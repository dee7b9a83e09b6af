"""Per-stage float64 references of the encoder's kernels and their per-element error bounds (device-agnostic torch).

Every function takes the 16-bit / fp32 values a kernel READ (exactly as the previous kernel stored them), computes the
op in float64 and returns (ref, bound): the stored output of a correct kernel satisfies |got - ref| <= bound element by
element.  The bounds come from the formats involved, never from observed errors; all constants live at the top.
check() reduces one comparison to the worst |got - ref| / bound, where it sits and how many outputs are not finite.

Symbols: u16 = 2^-8 (bf16) or 2^-11 (fp16), the unit roundoff of the stored format - where the other terms are small,
output rounding alone reaches ratios close to 1; u32 = 2^-24; gamma_K = K 2^-22, four times the IEEE worst case of a
K-term fp32 sum (margin for the tensor core's truncating alignment inside product groups)."""
import math
from dataclasses import dataclass

import torch

U_BF = 2.0 ** -8
U_F16 = 2.0 ** -11
U32 = 2.0 ** -24
F16_FLOOR = 2.0 ** -25      # absolute floor of fp16 outputs: spacing of the subnormals is 2^-24
GELU_POLY = 4e-6            # |gelu_erf - gelu| of the logistic-polynomial GELU in fp32 arithmetic (3.4e-6, common.cuh)
GELU_TANH_POLY = 7e-6       # same for the tanh-form gelu / gelu' polynomials of the fc2-dgrad epilogue (6.9e-6)
TANH_ABS = 2.0 ** -10.987   # tanh.approx.f32: maximum absolute error over the whole range (PTX ISA)
EXP2_REL = 2.0 ** -22       # ex2.approx.f32 relative error (PTX ISA: 2 ulp)
P_FLOOR = 2.0 ** -126       # ex2.approx.ftz flushes probabilities below the smallest normal fp32 value to 0
GELU_MAX_SLOPE = 1.13       # max |gelu'(x)| = 1.1289
LN_C = 2                    # c in the c C u32 of a LayerNorm row statistic: mean, then sum of squares


def gamma(K):
    return K * 2.0 ** -22


def unit(dtype):
    return {torch.bfloat16: U_BF, torch.float16: U_F16, torch.float32: U32, torch.float64: 0.0}[dtype]


def floor(dtype):
    return F16_FLOOR if dtype == torch.float16 else 0.0


def f64(t):
    return t.to(torch.float64)


@dataclass
class Result:
    name: str
    worst: float        # max |got - ref| / bound (inf where got is not finite or the bound is 0 and got != ref)
    where: tuple        # index of the worst element
    nonfinite: int      # count of NaN / inf outputs

    @property
    def ok(self):
        return self.nonfinite == 0 and self.worst <= 1.0

    def line(self):
        return "%-28s worst %.3e at %-22s nonfinite %d" % (self.name, self.worst, self.where, self.nonfinite)


def check(name, got, ref, bound):
    """Worst |got - ref| / bound over all elements (bound 0: exact equality required), its index, NaN / inf count."""
    g = f64(got)
    ref = f64(ref).expand_as(g)
    bound = f64(bound).expand_as(g)
    err = (g - ref).abs()
    fin = torch.isfinite(g)
    ratio = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err == 0, 0.0, math.inf))
    ratio = torch.where(fin, ratio, torch.full_like(ratio, math.inf))
    if ratio.numel() == 0:
        return Result(name, 0.0, (), 0)
    flat = int(torch.argmax(ratio.flatten()))
    where = tuple(int(i) for i in torch.unravel_index(torch.tensor(flat), ratio.shape))
    return Result(name, float(ratio.flatten()[flat]), where, int((~fin).sum()))


def _absmm(a, b):
    """|a| @ |b|^T in fp32 (a bound: relative accuracy 1e-6 is plenty, and it halves the float64 work)."""
    return (a.abs().float() @ b.abs().float().transpose(-1, -2)).double()


# ------------------------------------------------------------------------------------------------------------ GEMMs
def gemm(A, B, bias=None, res=None, out_dtype=torch.bfloat16):
    """y = A B^T (+ bias) (+ res), A [..., M, K], B [..., N, K] as the kernel read them.  fp32 accumulation over K, then
    the bias and the residual added in fp32, then one rounding to out_dtype.  Returns (ref, bound, acc_bound) with
    acc_bound the accumulation term alone (the GELU stage propagates it)."""
    A, B = f64(A), f64(B)
    K = A.shape[-1]
    r = A @ B.transpose(-1, -2)
    acc_bound = gamma(K) * _absmm(A, B)
    extra = 0.0
    if bias is not None:
        bias = f64(bias).unsqueeze(-2)
        r = r + bias
        extra = extra + bias.abs()
    if res is not None:
        res = f64(res)
        r = r + res
        extra = extra + res.abs()
    bound = unit(out_dtype) * r.abs() + acc_bound + U32 * extra + floor(out_dtype)
    if bias is not None:
        acc_bound = acc_bound + U32 * bias.abs()
    return r, bound, acc_bound


def gelu(x):
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def gelu_grad(x):
    return 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2.0 * math.pi)


def gelu_stage(r_u, acc_bound_u, out_dtype):
    """gelu of the fp32 accumulator of u (not of the rounded u): the accumulation error passes through a slope <= 1.13."""
    g = gelu(r_u)
    return g, unit(out_dtype) * g.abs() + GELU_MAX_SLOPE * acc_bound_u + GELU_POLY + floor(out_dtype)


def _tanh_form(u):
    """t = tanh(a(u)) and dd = a'(u) / 2 of the tanh-form GELU the fc2-dgrad epilogue evaluates (common.cuh)."""
    k = math.sqrt(2.0 / math.pi)
    t = torch.tanh(k * (u + 0.044715 * u ** 3))
    dd = 0.5 * k * (1.0 + 3 * 0.044715 * u * u)
    return t, dd


def gelu_grad_err(u):
    """|error| of the epilogue's gelu'(u) = sig + u (1 - t^2) dd with t from tanh.approx: sig = (1 + t) / 2 carries
    |dt| / 2, 1 - t^2 carries 2 |t| |dt| + dt^2; plus the polynomial fit."""
    t, dd = _tanh_form(u)
    return GELU_TANH_POLY + 0.5 * TANH_ABS + (u * dd).abs() * (2 * t.abs() * TANH_ABS + TANH_ABS ** 2)


def gelu_recompute_err(u):
    """|error| of the epilogue's gelu(u) = u (1 + t) / 2 (MFVIT_GELU_TWIN=0: the bf16 gelu of the fc2 weight gradient)."""
    return (GELU_TANH_POLY + 0.5 * TANH_ABS) * u.abs()


def dgelu_stage(dY, W, u):
    """dhid = bf16((dY W) * gelu'(u)), u = the stored bf16 pre-activation.  dY [..., M, N], W [..., N, K]."""
    dY, W, u = f64(dY), f64(W), f64(u)
    acc = dY @ W
    acc_b = gamma(dY.shape[-1]) * (dY.abs().float() @ W.abs().float()).double()
    dg = gelu_grad(u)
    r = acc * dg
    return r, U_BF * r.abs() + dg.abs() * acc_b + gelu_grad_err(u) * acc.abs()


# ------------------------------------------------------------------------------------------------------- LayerNorm
def ln_stats(x, eps=1e-6):
    x = f64(x)
    C = x.shape[-1]
    mean = x.mean(-1)
    var = ((x - mean.unsqueeze(-1)) ** 2).mean(-1)
    rstd = 1.0 / torch.sqrt(var + eps)
    tol = LN_C * C * U32
    return (mean, tol * x.abs().mean(-1) + U32 * mean.abs()), (rstd, tol * rstd)


def ln_fwd(x, w, b, out_dtype, eps=1e-6):
    """y = (x - mean) rstd w + b over the last dim.  Returns (y, bound)."""
    (mean, _), (rstd, _) = ln_stats(x, eps)
    x, w, b = f64(x), f64(w), f64(b)
    xh = (x - mean.unsqueeze(-1)) * rstd.unsqueeze(-1)
    y = xh * w + b
    C = x.shape[-1]
    return y, unit(out_dtype) * y.abs() + LN_C * C * U32 * (w.abs() * (xh.abs() + 1) + b.abs()) + floor(out_dtype)


def ln_bwd(dy, x, mean, rstd, w, dres=None, out_dtype=torch.bfloat16):
    """dx = rstd (g - mean(g) - xh mean(g xh)) + dres, g = w dy, with the kernel's stored mean / rstd.
    Returns (dx, bound, xh) - xh for the dgamma check."""
    dy, x, w = f64(dy), f64(x), f64(w)
    mean, rstd = f64(mean).unsqueeze(-1), f64(rstd).unsqueeze(-1)
    C = x.shape[-1]
    xh = (x - mean) * rstd
    g = w * dy
    c1 = g.mean(-1, keepdim=True)
    c2 = (g * xh).mean(-1, keepdim=True)
    dx = rstd * (g - c1 - xh * c2)
    bnd = LN_C * C * U32 * rstd * (g.abs() + g.abs().mean(-1, keepdim=True) + xh.abs() * (g * xh).abs().mean(-1, keepdim=True))
    if dres is not None:
        dres = f64(dres)
        dx = dx + dres
        bnd = bnd + U32 * dres.abs()
    return dx, unit(out_dtype) * dx.abs() + bnd + floor(out_dtype), xh


# ------------------------------------------------------------------------------------------------------ reductions
def colsum(Y, extra_rel=0.0):
    """sum over rows (dim -2) of Y [..., M, N]: bias gradients, dgamma / dbeta.  extra_rel: a rounding of every term the
    checked value did not see (u_bf: the bias sum of an fp32 dx checked against its stored bf16 copy)."""
    Y = f64(Y)
    M = Y.shape[-2]
    a = Y.abs().sum(-2)
    return Y.sum(-2), gamma(M) * a + extra_rel * a


def wgrad(dY, X):
    """dW = dY^T X over the M token rows: dY [..., M, N], X [..., M, K] -> [..., N, K]."""
    dY, X = f64(dY), f64(X)
    M = dY.shape[-2]
    r = dY.transpose(-1, -2) @ X
    return r, gamma(M) * (dY.abs().float().transpose(-1, -2) @ X.abs().float()).double()


# ------------------------------------------------------------------------------------------------------- attention
def _eps_s(q, k, scale):
    """Absolute error of a score in the exponent (natural-log units) per query row: fp32 q.k over D, the fp32 scaling into
    the log2 domain, ex2.approx."""
    D = q.shape[-1]
    qm = q.abs().amax(-1, keepdim=True)                      # [..., S, 1]
    km = k.abs().amax((-1, -2), keepdim=True)                # [..., 1, 1]
    return D * 2.0 ** -22 * scale * qm * km + EXP2_REL


def attn_fwd(q, k, v, scale, out_dtype, p_dtype, key_mask=None):
    """o = softmax(scale q k^T) v, lse.  q, k, v [..., S, D] as stored (the kernel reads them unconverted).  P is rounded
    to p_dtype for the P.V MMA; the row sum l and P.V accumulate in fp32 over S keys.  key_mask [S] (optional, bool):
    keys a correct kernel must ignore (tests only).  Returns (o, o_bound, lse, lse_bound)."""
    q, k, v = f64(q), f64(k), f64(v)
    S = k.shape[-2]
    s = scale * (q @ k.transpose(-1, -2))
    if key_mask is not None:
        s = s.masked_fill(~key_mask, -math.inf)
    lse = torch.logsumexp(s, -1)
    P = torch.exp(s - lse.unsqueeze(-1))
    o = P @ v
    eps = _eps_s(q, k, scale)
    pv = P @ v.abs()
    o_b = unit(out_dtype) * o.abs() + (unit(p_dtype) + eps + 2 * gamma(S)) * pv + floor(out_dtype)
    lse_b = eps.squeeze(-1) + gamma(S) + 2 * U32 * lse.abs()
    return o, o_b, lse, lse_b


def attn_bwd(q, k, v, o, do, lse, scale):
    """dq, dk, dv of o = softmax(scale q k^T) v from bf16 q / k / v / o / dO and the forward's lse, with P = exp(s - lse),
    delta = rowsum(dO o), dS = P (dP - delta); P and dS are rounded to bf16 for the MMAs.  Returns
    ((dq, dk, dv), (dq_b, dk_b, dv_b), (delta, delta_b))."""
    q, k, v, o, do, lse = (f64(t) for t in (q, k, v, o, do, lse))
    S, D = q.shape[-2], q.shape[-1]
    s = scale * (q @ k.transpose(-1, -2))
    P = torch.exp(s - lse.unsqueeze(-1))
    eps = _eps_s(q, k, scale)
    dv = P.transpose(-1, -2) @ do
    Pa = P.abs().float()
    dv_b = (U_BF * dv.abs() + (U_BF + eps.amax((-1, -2), keepdim=True) + gamma(S)) * (Pa.transpose(-1, -2) @ do.abs().float()).double()
            + P_FLOOR * do.abs().sum(-2, keepdim=True))
    dP = do @ v.transpose(-1, -2)
    delta = (do * o).sum(-1)
    delta_b = gamma(D) * (do * o).abs().sum(-1)
    dS = P * (dP - delta.unsqueeze(-1))
    e_dP = gamma(D) * _absmm(do, v) + delta_b.unsqueeze(-1)
    e_dS = U_BF * dS.abs() + (P * eps + P_FLOOR) * (dP.abs() + delta.abs().unsqueeze(-1)) + P * e_dP
    dSa = dS.abs().float()
    e_dS_f = e_dS.float()
    dq = scale * (dS @ k)
    dk = scale * (dS.transpose(-1, -2) @ q)
    dq_b = U_BF * dq.abs() + scale * ((e_dS_f @ k.abs().float()).double() + gamma(S) * (dSa @ k.abs().float()).double())
    dk_b = U_BF * dk.abs() + scale * ((e_dS_f.transpose(-1, -2) @ q.abs().float()).double()
                                      + gamma(S) * (dSa.transpose(-1, -2) @ q.abs().float()).double())
    return (dq, dk, dv), (dq_b, dk_b, dv_b), (delta, delta_b)


# ----------------------------------------------------------------------------------------------------- embedding
def im2col(images):
    """images f32 [B, 3, H, W] -> [B, np, 768] with k = c 256 + i 16 + j (the conv weight's own flattening)."""
    B, Cc, H, W = images.shape
    p = images.reshape(B, Cc, H // 16, 16, W // 16, 16).permute(0, 2, 4, 1, 3, 5)
    return p.reshape(B, (H // 16) * (W // 16), Cc * 256)
