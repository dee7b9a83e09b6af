"""Per-stage float64 references of the cross-attention fusion (csrc/fusion.cu) and their per-element error bounds.

Same conventions as tests/stage_ref.py: every function takes the fp32 values a kernel READ and returns (ref, bound) in
float64; a correct kernel's stored output satisfies |got - ref| <= bound element by element, and check() reduces a
comparison to its worst ratio.  The semantics are those of the comment at the head of fusion.cu: for instance
r = b 2 + d the query row is f0 = tok[d][b][0] and the keys are f0 itself plus tok[1-d][b][1..S-1], all LN1'd (eps
1e-5); q = Wq xh0, t_h = Wk_h^T q_h, u_h = sum_j softmax_j(scale t_h . xh_j) xh_j, o = Wv u, y = Wp o + bp,
c = f0 + y, e = f0 + LN2_{eps 1e-6}(c), fused_d = Wh e + bh, x_d = Wvh f0 + bvh.

Bounds.  A value the kernel computes as a tree of fp32 roundings of depth n is within gam(n) sum|terms| of the exact
value (Higham, Accuracy and Stability, 3.1), so each bound below is gam(depth) times the same expression evaluated on
absolute values, plus the error of any input the stage recomputes instead of reading (LN1 of the key rows, the
scores, P), plus the errors of the approximate intrinsics the kernels call:
    __expf(x) = ex2.approx.ftz(x log2 e): EXP2_REL relative, plus u32 |x| from rounding the product x log2 e;
    rsqrtf    = rsqrt.approx.f32: RSQRT_REL relative;
    __logf(x) = lg2.approx.f32(x) ln 2: LG2_ABS absolute (natural-log units, after the ln 2 factor), plus u32 |result|.
Stages whose inputs all come from `saved` have no input term (teacher forcing); the single-kernel path keeps fewer
intermediates, and there the caller passes the bound of the recomputed input (t_err, lse_err, du_err, y_err, ...)."""
import math

import torch

from stage_ref import EXP2_REL, LN_C, P_FLOOR, U32, Result, check, f64  # noqa: F401  (re-exported for the tests)

C = 384
CPL = C // 32           # columns per lane of a warp-held row
WARPS = 12              # FUS_THREADS / 32: warps of the streaming kernels
RSQRT_REL = 2.0 ** -22.9  # rsqrt.approx.f32 maximum relative error (PTX ISA)
LG2_ABS = 2.0 ** -22      # lg2.approx.f32 absolute error 2^-22.6 (PTX ISA), rounded up, times ln 2 < 1
# Depths of the fp32 reductions (counted from the loops in fusion.cu):
D_ROW = 20              # dot_row / warp_sum over C: 3 float4 groups of 4 fused products + 1 add each (<= 15 roundings
                        # per lane), then 5 butterfly levels
D_STAT = D_ROW + 2      # an LN row statistic: the warp sum, then * invC (invC = 1/384 is itself rounded)
EPS1, EPS2 = 1e-5, 1e-6  # LN1 (PreNorm) and LN2 (post LayerNorm)
assert LN_C * C >= D_STAT  # stage_ref's LayerNorm statistics tolerance is the looser of the two


def gam(n):
    return n * U32 / (1.0 - n * U32)


def expf_rel(arg_abs):
    """Relative error of __expf at |argument| <= arg_abs."""
    return EXP2_REL + U32 * arg_abs


def n_iter(S):
    """Rows one warp visits in a streaming pass (rows j = warp, warp + 12, ...)."""
    return (S + WARPS - 1) // WARPS


# ------------------------------------------------------------------------------------------------------ layout
def rec_offsets(heads):
    """Fus2Rec / fus_rec_floats (fusion.cu:29-31, 680-687): one record per instance, read by fusion_wgrad_kernel."""
    o, off = {}, 0
    for name, n in (("dq", 1), ("xh0", 1), ("q", 1), ("dt", heads), ("do", 1), ("u", heads), ("dy", 1), ("o", 1),
                    ("dz", 1), ("chat", 1), ("e", 1), ("f0", 1), ("dg1", 1), ("db1", 1)):
        o[name] = (off, n * C)
        off += n * C
    return o, off


def fwd_offsets(heads):
    """Fus2Off / fus2_fwd_floats (fusion.cu:671, 673-679): misc[0] rstd0, misc[1] rstd2, misc[4..4+heads) lse."""
    o, off = {}, 0
    for name, n in (("f0", 1), ("n0", 1), ("xh0", 1), ("q", 1), ("t", heads), ("u", heads), ("o", 1), ("y", 1),
                    ("chat", 1), ("e", 1)):
        o[name] = (off, n * C)
        off += n * C
    o["misc"] = (off, 16)
    return o, off + 16


def bwt_offsets(heads):
    """Fus2Bwt / fus2_bwt_floats (fusion.cu:672, 688-691)."""
    o = {"du": (0, heads * C), "dxh0": (heads * C, C), "df0": ((heads + 1) * C, C), "misc": ((heads + 2) * C, 16)}
    return o, (heads + 2) * C + 16


def saved_floats(B, heads):
    """mfv_fusion_saved_floats: [records 2B][forward state 2B][backward temporaries 2B] (fusion.cu:669, 1191-1195)."""
    return 2 * B * (rec_offsets(heads)[1] + fwd_offsets(heads)[1] + bwt_offsets(heads)[1])


def split_saved(saved, B, heads):
    """Views of `saved` [n] as dicts name -> [2B, ...] of the records, the forward state and the backward temporaries
    (instance r = b 2 + d along dim 0)."""
    ro, rf = rec_offsets(heads)
    fo, ff = fwd_offsets(heads)
    bo, bf = bwt_offsets(heads)
    R = 2 * B
    rec = saved[:R * rf].view(R, rf)
    fwd = saved[R * rf:R * (rf + ff)].view(R, ff)
    bwt = saved[R * (rf + ff):R * (rf + ff + bf)].view(R, bf)

    def cut(t, offs):
        return {k: t[:, a:a + n].reshape(R, n // C, C) if n % C == 0 and n >= C else t[:, a:a + n]
                for k, (a, n) in offs.items()}
    return cut(rec, ro), cut(fwd, fo), cut(bwt, bo)


# ------------------------------------------------------------------------------------------------------ LayerNorm
def ln(v, g, b, eps, v_err=None):
    """n = (v - mean) rstd, y = n g + b over the last dim, as ln_stats (fusion.cu:61-74) then one fma.  v_err: bound of
    an error already in v.  Returns dict of refs n, y, rstd and bounds n_b, y_b, rstd_b (rstd_b relative)."""
    v, g, b = f64(v), f64(g), f64(b)
    mean = v.mean(-1, keepdim=True)
    cen = v - mean
    var = (cen * cen).mean(-1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + eps)
    n = cen * rstd
    dv = torch.zeros_like(v) if v_err is None else f64(v_err).expand_as(v)
    dmean = gam(D_STAT) * v.abs().mean(-1, keepdim=True) + dv.mean(-1, keepdim=True)
    # var: squares of the rounded centred values (2u each) summed at depth D_STAT; a mean off by dm adds dm^2 exactly
    # (sum of the centred values is 0); an input error dv moves it by <= 2 mean(|cen| (|dv| + dm))
    dvar = (gam(D_STAT + 2) * var + dmean ** 2 + 2 * (cen.abs() * dv).mean(-1, keepdim=True)
            + 2 * cen.abs().mean(-1, keepdim=True) * dmean)
    rstd_rel = 0.5 * (dvar + U32 * (var + eps)) / (var + eps) + RSQRT_REL + U32
    n_b = rstd * (dv + dmean) + n.abs() * (rstd_rel + 2 * U32)
    y = n * g + b
    return dict(n=n, y=y, rstd=rstd.squeeze(-1), n_b=n_b, y_b=g.abs() * n_b + U32 * y.abs(), rstd_b=rstd_rel.squeeze(-1))


def ln_bwd(dxh, n, rstd, g, dres=None, dxh_err=None, n_err=None, rstd_rel=None, extra=0):
    """dx = rstd (G - mean G - n mean(G n)) (+ dres), G = dxh g, with the n / rstd the kernel uses (fusion.cu:478-492,
    538-558, 982-996, 1157-1171).  Errors already in dxh, n, rstd can be passed; extra: roundings that produced dxh
    (its abs replay is |dxh| only when dxh_err is given)."""
    dxh, n, g = f64(dxh), f64(n), f64(g)
    rstd = f64(rstd).unsqueeze(-1)
    G = dxh * g
    c1 = G.mean(-1, keepdim=True)
    c2 = (G * n).mean(-1, keepdim=True)
    dx = rstd * (G - c1 - n * c2)
    Ga = G.abs()
    absr = rstd * (Ga + Ga.mean(-1, keepdim=True) + n.abs() * (Ga * n.abs()).mean(-1, keepdim=True))
    bnd = gam(D_STAT + 3 + extra) * absr
    if dxh_err is not None:
        dG = g.abs() * f64(dxh_err)
        bnd = bnd + rstd * (dG + dG.mean(-1, keepdim=True) + n.abs() * (dG * n.abs()).mean(-1, keepdim=True))
    if n_err is not None:
        dn = f64(n_err)
        bnd = bnd + rstd * (dn * c2.abs() + n.abs() * (Ga * dn).mean(-1, keepdim=True))
    if rstd_rel is not None:
        bnd = bnd + f64(rstd_rel).unsqueeze(-1) * absr
    if dres is not None:
        dres = f64(dres)
        dx = dx + dres
        bnd = bnd + U32 * (dx.abs() + dres.abs())
    return dx, bnd


# ---------------------------------------------------------------------------------------------------- mat-vecs
def rowdot(W, vec, bias=None, vec_err=None, heads=None):
    """out[i] = W[i] . v (+ bias[i]): fus2_rowdot_kernel / matvec_rows / the single kernel's o and dq loops (dot_row,
    depth D_ROW, then the bias).  W [N, C]; vec [C], or [heads, C] with heads given: row i reads head i // (N / heads)."""
    W, vec = f64(W), f64(vec)
    if heads is not None:
        Wh = W.view(heads, W.shape[0] // heads, C)
        out = torch.einsum("hic,hc->hi", Wh, vec).reshape(-1)
        absr = torch.einsum("hic,hc->hi", Wh.abs(), vec.abs()).reshape(-1)
        err = 0.0 if vec_err is None else torch.einsum("hic,hc->hi", Wh.abs(), f64(vec_err)).reshape(-1)
    else:
        out = W @ vec
        absr = W.abs() @ vec.abs()
        err = 0.0 if vec_err is None else W.abs() @ f64(vec_err)
    depth = D_ROW
    if bias is not None:
        bias = f64(bias)
        out = out + bias
        absr = absr + bias.abs()
        depth += 1
    return out, gam(depth) * absr + err


def coldot(W, vec, heads=1, acc=None, vec_err=None):
    """out[..., s, c] = sum_{i in segment s} W[i][c] vec[..., i] (+ acc): W^T products, one sequential fma chain per
    column (fus2_coldot_kernel; the single kernel's t, do, du and Wq^T dq loops).  W [C, C], vec [..., C]."""
    W, vec = f64(W), f64(vec)
    hd = C // heads
    Ws = W.view(heads, hd, C)
    v = vec.view(*vec.shape[:-1], heads, hd)
    out = torch.einsum("sic,...si->...sc", Ws, v)
    absr = torch.einsum("sic,...si->...sc", Ws.abs(), v.abs())
    depth = hd
    err = 0.0 if vec_err is None else torch.einsum("sic,...si->...sc", Ws.abs(), f64(vec_err).view(v.shape))
    if acc is not None:
        acc = f64(acc).view(out.shape)
        out = out + acc
        absr = absr + acc.abs()
        depth += 1
    return out, gam(depth) * absr + err


# ---------------------------------------------------------------------------------------------- streaming passes
def key_rows(tok, b, d, f0=None):
    """The S rows instance (b, d) attends over: its own CLS row (f0 as stored, or tok[d][b][0]) and rows 1.. of the
    other branch.  tok [2, B, S, C]."""
    rows = tok[1 - d, b].clone()
    rows[0] = tok[d, b, 0] if f0 is None else f0
    return rows


def _scores(xh, xh_b, t, t_err, scale):
    """s [heads, S] and its bound from the row dot (depth D_ROW), the key rows' LN error, the error of t, and the
    rounding of the product by scale."""
    s = scale * (t @ xh.T)
    s_b = scale * (gam(D_ROW) * (t.abs() @ xh.abs().T) + t.abs() @ xh_b.T) + 2 * U32 * s.abs()  # scale: rounded, times
    if t_err is not None:
        s_b = s_b + scale * (f64(t_err) @ xh.abs().T)
    return s, s_b


def stream_fwd(rows, g1, b1, t, scale, t_err=None):
    """u_h = sum_j softmax_j(s_h) xh_j and lse_h for one instance (fus2_stream_fwd_kernel, fusion.cu:181-246, 845-910).
    rows [S, C] fp32 as read, t [heads, C].  Per-warp online softmax over n_iter(S) rows, then a 12-way merge: each
    weight picks up one __expf per rescale plus its own and the merge factor, and 2 roundings per row update."""
    S = rows.shape[0]
    L = ln(rows, g1, b1, EPS1)
    xh, xh_b = L["y"], L["y_b"]
    t = f64(t)
    s, s_b = _scores(xh, xh_b, t, t_err, scale)
    lse = torch.logsumexp(s, -1)
    P = torch.exp(s - lse.unsqueeze(-1))
    spread = (s.amax(-1) - s.amin(-1)).unsqueeze(-1) + s_b.amax(-1, keepdim=True) + math.log(S)  # |__expf arguments|
    it = n_iter(S)
    e_exp = (it + 3) * expf_rel(spread)
    ds_max = s_b.amax(-1, keepdim=True)
    lse_b = ds_max + e_exp + gam(it + WARPS + 2) + LG2_ABS + U32 * lse.abs().unsqueeze(-1)
    eps_p = s_b + lse_b + e_exp + gam(2 * it + WARPS + 2)
    u = P @ xh
    u_b = (P * eps_p + P_FLOOR) @ xh.abs() + P @ xh_b
    return dict(u=u, u_b=u_b, lse=lse, lse_b=lse_b.squeeze(-1), xh=xh, xh_b=xh_b, n=L["n"], n_b=L["n_b"],
                rstd=L["rstd"], rstd_b=L["rstd_b"], s=s, s_b=s_b)


def stream_bwd(rows, g1, b1, t, lse, u, du, scale, t_err=None, lse_err=None, du_err=None):
    """Second streaming pass for one instance (fus2_stream_bwd_kernel, fusion.cu:1038-1129; fusion_bwd_kernel 424-506):
    P = __expf(s - lse) with the lse READ, D_h = du_h . u_h, dS = P (xh . du_h - D_h) scale, dxh_j = sum_h P du_h + dS t_h,
    dtok_j = LN1'(dxh_j) for j >= 1; dt_h = sum_j dS xh_j; dg1 / db1 partials over j >= 1.  Returns dict."""
    S = rows.shape[0]
    it = n_iter(S)
    L = ln(rows, g1, b1, EPS1)
    xh, xh_b, n, n_b = L["y"], L["y_b"], L["n"], L["n_b"]
    t, lse, u, du = f64(t), f64(lse), f64(u), f64(du)
    heads = t.shape[0]
    s, s_b = _scores(xh, xh_b, t, t_err, scale)
    arg = (s - lse.unsqueeze(-1))
    P = torch.exp(arg)
    eps_p = s_b + expf_rel(arg.abs() + s_b) + U32 * arg.abs()
    if lse_err is not None:
        eps_p = eps_p + f64(lse_err).unsqueeze(-1)
    dP_b = P * eps_p + P_FLOOR
    D = (du * u).sum(-1)
    D_b = gam(D_ROW) * (du.abs() * u.abs()).sum(-1)
    dp = du @ xh.T                                                    # [heads, S]
    dp_b = gam(D_ROW) * (du.abs() @ xh.abs().T) + du.abs() @ xh_b.T
    if du_err is not None:
        du_err = f64(du_err)
        D_b = D_b + (du_err * u.abs()).sum(-1)
        dp_b = dp_b + du_err @ xh.abs().T
    diff = dp - D.unsqueeze(-1)
    dS = P * diff * scale
    dS_b = scale * (dP_b * diff.abs() + P * (dp_b + D_b.unsqueeze(-1)) + gam(3) * P * (dp.abs() + D.abs().unsqueeze(-1)))
    # dxh_j = sum_h P du_h + dS t_h: 2 heads fused terms per column
    dxh = P.T @ du + dS.T @ t
    dxh_absr = P.T @ du.abs() + dS.abs().T @ t.abs()
    dxh_b = gam(2 * heads) * dxh_absr + dP_b.T @ du.abs() + dS_b.T @ t.abs()
    if du_err is not None:
        dxh_b = dxh_b + P.T @ du_err
    if t_err is not None:
        dxh_b = dxh_b + dS.abs().T @ f64(t_err)
    dt = dS @ xh
    dt_b = gam(it + WARPS) * (dS.abs() @ xh.abs()) + dS_b @ xh.abs() + dS.abs() @ xh_b
    drows, drows_b = ln_bwd(dxh[1:], n[1:], L["rstd"][1:], g1, dxh_err=dxh_b[1:], n_err=n_b[1:],
                            rstd_rel=L["rstd_b"][1:])
    return dict(drows=drows, drows_b=drows_b, dt=dt, dt_b=dt_b, dxh=dxh, dxh_b=dxh_b, dxh_absr=dxh_absr, n=n, n_b=n_b,
                P=P, D=D)


def lnw_grads(st, dxh0, dxh0_b, n0):
    """dg1 = sum_{j>=1} dxh_j n_j + dxh0 n0, db1 = sum_j dxh_j (per-warp sums over n_iter(S) rows, a 12-way merge, then
    the CLS row's share added last: fus2_stream_bwd + fus2_bwd_row0, or the single kernel's record loop)."""
    S = st["dxh"].shape[0]
    depth = n_iter(S) + WARPS + 2
    dx, n = st["dxh"][1:], st["n"][1:]
    dxh0, n0 = f64(dxh0), f64(n0)
    dg = (dx * n).sum(0) + dxh0 * n0
    db = dx.sum(0) + dxh0
    dg_b = (gam(depth) * ((dx * n).abs().sum(0) + (dxh0 * n0).abs()) + (st["dxh_b"][1:] * n.abs()).sum(0)
            + (dx.abs() * st["n_b"][1:]).sum(0) + dxh0_b * n0.abs())
    db_b = gam(depth) * (dx.abs().sum(0) + dxh0.abs()) + st["dxh_b"][1:].sum(0) + dxh0_b
    return (dg, dg_b), (db, db_b)


# ------------------------------------------------------------------------------------------- LN2 and the heads
def ln2(f0, y, w2, b2, y_err=None):
    """c = f0 + y (one rounding), chat = LN2(c), e = f0 + chat w2 + b2 (two roundings).  Returns dict of chat, e, rstd2
    with bounds."""
    f0, y = f64(f0), f64(y)
    c = f0 + y
    c_err = U32 * c.abs() + (0.0 if y_err is None else f64(y_err))
    L = ln(c, w2, b2, EPS2, v_err=c_err)
    w2, b2 = f64(w2), f64(b2)
    e = f0 + L["n"] * w2 + b2
    e_b = w2.abs() * L["n_b"] + gam(2) * (f0.abs() + (L["n"] * w2).abs() + b2.abs())
    return dict(chat=L["n"], chat_b=L["n_b"], e=e, e_b=e_b, rstd2=L["rstd"], rstd2_b=L["rstd_b"])


def heads_bwd(chat, rstd2, d_fused, d_x, head_w, vhead_w, w2, chat_err=None, rstd2_rel=None):
    """dz = Wh^T dfused, df0 = dz + Wvh^T dx + dy, dy = LN2'(dz) with the chat / rstd2 read (fus2_bwd_heads_kernel,
    fusion.cu:371-403, 971-999).  d_fused [R, NC], d_x [R, NC] or None."""
    d_fused, head_w = f64(d_fused), f64(head_w)
    NC = head_w.shape[0]
    dz = d_fused @ head_w
    dz_b = gam(NC) * (d_fused.abs() @ head_w.abs())
    dv = torch.zeros_like(dz)
    dv_b = torch.zeros_like(dz)
    if d_x is not None and vhead_w is not None:
        dv = f64(d_x) @ f64(vhead_w)
        dv_b = gam(NC + 1) * (f64(d_x).abs() @ f64(vhead_w).abs())
    dy, dy_b = ln_bwd(dz, chat, rstd2, w2, dxh_err=dz_b, n_err=chat_err, rstd_rel=rstd2_rel)
    df0 = dz + dv + dy
    df0_b = dz_b + dv_b + dy_b + gam(2) * (dz.abs() + dv.abs() + dy.abs())
    return dict(dz=dz, dz_b=dz_b, dy=dy, dy_b=dy_b, df0=df0, df0_b=df0_b)


# ---------------------------------------------------------------------------------------------- weight gradients
def contract(L, Rv, G0=None):
    """sum_b L[b, i] R[b, c] (+ G0): fusion_wgrad_kernel's sequential fma over the batch, then one += .  L [Bd, N],
    Rv [Bd, N, C] (per-row right vector: the head slice) or [Bd, C]."""
    L, Rv = f64(L), f64(Rv)
    Bd = L.shape[0]
    if Rv.dim() == 3:
        r = torch.einsum("bi,bic->ic", L, Rv)
        a = torch.einsum("bi,bic->ic", L.abs(), Rv.abs())
    else:
        r = L.T @ Rv
        a = L.abs().T @ Rv.abs()
    return _acc(r, a, Bd, G0)


def vsum(V, G0=None):
    """sum over the batch of V [Bd, ...] (+ G0)."""
    V = f64(V)
    return _acc(V.sum(0), V.abs().sum(0), V.shape[0], G0)


def _acc(r, a, Bd, G0):
    b = gam(Bd) * a
    if G0 is not None:
        G0 = f64(G0)
        r = r + G0
        b = b + U32 * (r.abs() + G0.abs()) * (1 + gam(1))
    return r, b


def head_slices(v, heads, N=C):
    """[Bd, heads, C] -> [Bd, N, C]: the head vector each of the N output rows pairs with (row i -> head i // hd)."""
    hd = N // heads
    return v.repeat_interleave(hd, dim=1)


FIELDS = ("ln1_w", "ln1_b", "wq", "wk", "wv", "proj_w", "proj_b", "ln2_w", "ln2_b", "head_w", "head_b", "vhead_w",
          "vhead_b")


def run_stages(tok, P, heads, d_fused, d_x, got=None, G0=None, report=None, fill=None):
    """Replays the fusion stage by stage in float64.  tok [2, B, S, C]; P: name -> (t_d0, t_d1) (vhead_* may be None);
    d_fused [B, NC]; d_x [2, B, NC] or None.  got: stored kernel values, name -> [2B, ...] per instance r = b 2 + d
    (f0 n0 xh0 rstd0 q t u lse o y chat e rstd2 dz dy df0 do du dt dq dxh0 dg1 db1); each stage READS the stored value
    of its inputs where there is one, else the reference and its bound (so got=None is a plain chained replay).
    report(stage, b, d, got, ref, bound) is called for every stored value; G0: name -> (g_d0, g_d1) gradients the
    kernel accumulated onto.  Returns (out, grads): out has fused [B, NC], x [2, B, NC] | None, dtok [2, B, S, C] with
    bounds fused_b, x_b, dtok_b; grads: name -> ((ref, bound) for d in 0, 1) from the records the batch contraction
    reads.  fill (a dict): every stage reads the fp32 rounding of its own reference instead, stored into fill[name][r]
    (correctly rounded outputs of a kernel that matches the reference)."""
    got = got or {}
    dev = tok.device
    B, S = tok.shape[1], tok.shape[2]
    hd = C // heads
    scale = hd ** -0.5
    has_vh = P["vhead_w"][0] is not None
    NC = P["head_w"][0].shape[0]
    Z = lambda *sh: torch.zeros(*sh, dtype=torch.float64, device=dev)  # noqa: E731
    fused, fused_b = Z(B, NC), Z(B, NC)
    x, x_b = Z(2, B, NC), Z(2, B, NC)
    dtok, dtok_b = Z(2, B, S, C), Z(2, B, S, C)
    recs = {k: [[None] * B for _ in range(2)] for k in ("dq", "xh0", "q", "dt", "do", "u", "dy", "o", "dz", "chat",
                                                          "e", "f0", "dg1", "db1")}

    def use(name, r, ref, bound, b, d, shape=None):
        """The value the next stage reads: the stored one (checked here) or the reference, and its error bound."""
        if fill is not None:
            v = ref.float()
            fill.setdefault(name, {})[r] = v
            return f64(v), None
        if name in got:
            g = got[name][r]
            g = g.reshape(ref.shape) if shape is None else g.reshape(shape)
            if report is not None:
                report(name, b, d, g, ref, bound)
            return f64(g), None
        return ref, bound

    for b in range(B):
        for d in range(2):
            r = b * 2 + d
            p = {k: (v[d] if v[d] is not None else None) for k, v in P.items()}
            # ---- forward
            f0, _ = use("f0", r, f64(tok[d, b, 0]), torch.zeros(C, dtype=torch.float64, device=dev), b, d)
            L0 = ln(f0, p["ln1_w"], p["ln1_b"], EPS1)
            n0, n0_e = use("n0", r, L0["n"], L0["n_b"], b, d)
            rstd0, r0_e = use("rstd0", r, L0["rstd"].reshape(1), (L0["rstd_b"] * L0["rstd"]).reshape(1), b, d)
            r0_rel = None if r0_e is None else r0_e / rstd0
            xh0, xh0_e = use("xh0", r, L0["y"], L0["y_b"], b, d)
            q, q_e = use("q", r, *rowdot(p["wq"], xh0, vec_err=xh0_e), b, d)
            t_ref, t_b = coldot(p["wk"], q, heads, vec_err=q_e)
            t, t_e = use("t", r, t_ref, t_b, b, d)
            rows = key_rows(tok, b, d, f0=f0)
            F = stream_fwd(rows, p["ln1_w"], p["ln1_b"], t, scale, t_err=t_e)
            u, u_e = use("u", r, F["u"], F["u_b"], b, d)
            lse, lse_e = use("lse", r, F["lse"], F["lse_b"], b, d)
            o, o_e = use("o", r, *rowdot(p["wv"], u, vec_err=u_e, heads=heads), b, d)
            y, y_e = use("y", r, *rowdot(p["proj_w"], o, p["proj_b"], vec_err=o_e), b, d)
            L2 = ln2(f0, y, p["ln2_w"], p["ln2_b"], y_err=y_e)
            chat, chat_e = use("chat", r, L2["chat"], L2["chat_b"], b, d)
            e, e_e = use("e", r, L2["e"], L2["e_b"], b, d)
            rstd2, r2_e = use("rstd2", r, L2["rstd2"].reshape(1), (L2["rstd2_b"] * L2["rstd2"]).reshape(1), b, d)
            r2_rel = None if r2_e is None else r2_e / rstd2
            part, part_b = rowdot(p["head_w"], e, p["head_b"], vec_err=e_e)
            fused[b] += part
            fused_b[b] += part_b + U32 * part.abs()
            if has_vh:
                x[d, b], x_b[d, b] = rowdot(p["vhead_w"], f0, p["vhead_b"])
            # ---- backward
            dxd = d_x[d, b:b + 1] if (d_x is not None and has_vh) else None
            H = heads_bwd(chat.unsqueeze(0), rstd2, d_fused[b:b + 1], dxd, p["head_w"], p["vhead_w"], p["ln2_w"],
                          chat_err=None if chat_e is None else chat_e.unsqueeze(0), rstd2_rel=r2_rel)
            dz, dz_e = use("dz", r, H["dz"][0], H["dz_b"][0], b, d)
            dy, dy_e = use("dy", r, H["dy"][0], H["dy_b"][0], b, d)
            df0, df0_e = use("df0", r, H["df0"][0], H["df0_b"][0], b, d)
            do, do_e = use("do", r, *[v.reshape(C) for v in coldot(p["proj_w"], dy, 1, vec_err=dy_e)], b, d)
            du, du_e = use("du", r, *coldot(p["wv"], do, heads, vec_err=do_e), b, d)
            Bk = stream_bwd(rows, p["ln1_w"], p["ln1_b"], t, lse, u, du, scale, t_err=t_e, lse_err=lse_e,
                            du_err=du_e)
            dt, dt_e = use("dt", r, Bk["dt"], Bk["dt_b"], b, d)
            dq, dq_e = use("dq", r, *rowdot(p["wk"], dt, vec_err=dt_e, heads=heads), b, d)
            dx0_ref, dx0_b = coldot(p["wq"], dq, 1, acc=Bk["dxh"][0], vec_err=dq_e)
            dxh0, dxh0_e = use("dxh0", r, dx0_ref.reshape(C), dx0_b.reshape(C) + Bk["dxh_b"][0], b, d)
            row0, row0_b = ln_bwd(dxh0.unsqueeze(0), n0.unsqueeze(0), rstd0, p["ln1_w"], dres=df0.unsqueeze(0),
                                  dxh_err=None if dxh0_e is None else dxh0_e.unsqueeze(0),
                                  n_err=None if n0_e is None else n0_e.unsqueeze(0), rstd_rel=r0_rel)
            if df0_e is not None:
                row0_b = row0_b + df0_e
            dtok[d, b, 0], dtok_b[d, b, 0] = row0[0], row0_b[0]
            dtok[1 - d, b, 1:], dtok_b[1 - d, b, 1:] = Bk["drows"], Bk["drows_b"]
            (dg, dg_b), (db, db_b) = lnw_grads(Bk, dxh0, 0.0 if dxh0_e is None else dxh0_e, n0)
            dg, _ = use("dg1", r, dg, dg_b, b, d)
            db, _ = use("db1", r, db, db_b, b, d)
            for k, v in (("dq", dq), ("xh0", xh0), ("q", q), ("dt", dt), ("do", do), ("u", u), ("dy", dy), ("o", o),
                         ("dz", dz), ("chat", chat), ("e", e), ("f0", f0), ("dg1", dg), ("db1", db)):
                recs[k][d][b] = v.reshape(-1, C) if k in ("dt", "u") else v.reshape(C)
    # ---- weight gradients: the batch contraction of the records
    grads = {}
    for d in range(2):
        R_ = {k: torch.stack(v[d]) for k, v in recs.items()}
        g0 = (lambda k: None if G0 is None or G0[k][d] is None else G0[k][d])  # noqa: E731
        dfd = f64(d_fused)
        dxx = f64(d_x[d]) if (d_x is not None and has_vh) else torch.zeros_like(dfd)
        gd = {
            "wq": contract(R_["dq"], R_["xh0"], g0("wq")),
            "wk": contract(R_["q"], head_slices(R_["dt"], heads), g0("wk")),
            "wv": contract(R_["do"], head_slices(R_["u"], heads), g0("wv")),
            "proj_w": contract(R_["dy"], R_["o"], g0("proj_w")),
            "ln1_w": vsum(R_["dg1"], g0("ln1_w")), "ln1_b": vsum(R_["db1"], g0("ln1_b")),
            "ln2_w": vsum(R_["dz"] * R_["chat"], g0("ln2_w")), "ln2_b": vsum(R_["dz"], g0("ln2_b")),
            "proj_b": vsum(R_["dy"], g0("proj_b")),
            "head_w": contract(dfd, R_["e"], g0("head_w")), "head_b": vsum(dfd, g0("head_b")),
            "vhead_w": contract(dxx, R_["f0"], g0("vhead_w")), "vhead_b": vsum(dxx, g0("vhead_b")),
        }
        for k, v in gd.items():
            grads.setdefault(k, [None, None])[d] = v
    fused_b = fused_b + U32 * fused.abs()
    out = dict(fused=fused, fused_b=fused_b, x=x if has_vh else None, x_b=x_b, dtok=dtok, dtok_b=dtok_b)
    return out, grads


def _check_layout():
    for heads in (1, 2, 3, 4):
        assert rec_offsets(heads)[1] == C * (12 + 2 * heads)           # fus_rec_floats
        assert fwd_offsets(heads)[1] == C * (8 + 2 * heads) + 16       # fus2_fwd_floats
        assert bwt_offsets(heads)[1] == C * (2 + heads) + 16           # fus2_bwt_floats


_check_layout()
__all__ = ["Result", "check", "U32", "gam", "ln", "ln_bwd", "rowdot", "coldot", "stream_fwd", "stream_bwd", "ln2",
           "heads_bwd", "logits", "contract", "vsum", "lnw_grads", "key_rows", "split_saved", "saved_floats", "math"]
