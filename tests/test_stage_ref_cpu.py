"""The per-stage checker of tests/stage_ref.py is not vacuous: synthetic "kernel outputs" (fp32 arithmetic, explicit
16-bit rounding of what a kernel stores) pass with ratio < 1, and each of the defects the GPU stage test exists to catch
fails: an element 2 ulps off in the last row of a ragged tile, a dropped bias, the neighbouring group's output, LayerNorm
statistics of the wrong row, an unmasked padded key, a non-zero gradient gap, a NaN."""
import math
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import stage_ref as R  # noqa: E402

BF, F16, F32 = torch.bfloat16, torch.float16, torch.float32


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _rnd(shape, g, scale=1.0, dtype=BF):
    return (torch.randn(shape, generator=g) * scale).to(dtype)


def _ok(res):
    assert res.ok, res.line()
    return res


def _fails(res):
    assert not res.ok, res.line()
    return res


def _gemm_case(M=197, K=384, N=128, G=2, in_dtype=BF, seed=0):
    g = _gen(seed)
    A = _rnd((G, M, K), g, 1.0, in_dtype)
    W = _rnd((G, N, K), g, 0.05, in_dtype)
    b = torch.randn(G, N, generator=g) * 0.02
    acc = A.float() @ W.float().transpose(-1, -2)
    return A, W, b, acc


@pytest.mark.parametrize("out_dtype", [BF, F16])
def test_gemm_output_passes_and_two_ulps_in_the_ragged_last_row_fail(out_dtype):
    A, W, b, acc = _gemm_case(in_dtype=F16 if out_dtype == F16 else BF)
    got = (acc + b.unsqueeze(1)).to(out_dtype)
    ref, bound, _ = R.gemm(A, W, b, out_dtype=out_dtype)
    res = _ok(R.check("gemm", got, ref, bound))
    assert 0.05 < res.worst < 1.0  # output rounding dominates: the bound is not slack
    # 2 ulps away from the reference, in the last row (M = 197: row 196 is alone in its 256-row tile)
    row = got.shape[1] - 1
    room = (bound[:, row] / (ref[:, row].abs() * R.unit(out_dtype)))  # bound in units of u16 |r| (1 ulp >= u16 |r| / 2)
    gi, n = divmod(int(torch.argmin(room.flatten() + (ref[:, row].abs() < 1e-2).flatten().double() * 1e9)), room.shape[1])
    bad = got.clone()
    v = bad[gi, row, n]
    step = 1 if float(v) >= float(ref[gi, row, n]) else -1
    bits = v.view(torch.int16) + (2 if (float(v) >= 0) == (step > 0) else -2)
    bad[gi, row, n] = bits.view(out_dtype)
    res = _fails(R.check("gemm", bad, ref, bound))
    assert res.where == (gi, row, n)


def test_gemm_with_a_bias_left_out_fails():
    A, W, b, acc = _gemm_case()
    ref, bound, _ = R.gemm(A, W, b, out_dtype=BF)
    _ok(R.check("gemm", (acc + b.unsqueeze(1)).to(BF), ref, bound))
    _fails(R.check("gemm", acc.to(BF), ref, bound))


def test_gemm_output_of_the_neighbouring_group_fails():
    A, W, b, acc = _gemm_case()
    got = (acc + b.unsqueeze(1)).to(BF)
    ref, bound, _ = R.gemm(A, W, b, out_dtype=BF)
    swapped = got.clone()
    swapped[1] = got[0]  # group 1 stored the group-0 result (wrong weight / output group stride)
    res = _fails(R.check("gemm", swapped, ref, bound))
    assert res.where[0] == 1


def test_gemm_with_fp32_residual_passes():
    A, W, b, acc = _gemm_case(N=384)
    res = torch.randn(2, 197, 384, generator=_gen(3))
    got = (acc + b.unsqueeze(1)) + res
    ref, bound, _ = R.gemm(A, W, b, res, out_dtype=F32)
    _ok(R.check("resid", got, ref, bound))
    bad = got.clone()
    bad[0, 196] -= res[0, 196]  # residual of the ragged last row not added
    res_ = _fails(R.check("resid", bad, ref, bound))
    assert res_.where[:2] == (0, 196)


def test_gelu_from_the_fp32_accumulator_passes():
    A, W, b, acc = _gemm_case(N=256, in_dtype=F16)
    u32 = acc + b.unsqueeze(1)
    g32 = 0.5 * u32 * (1 + torch.erf(u32 / math.sqrt(2)))
    r_u, _, accb = R.gemm(A, W, b, out_dtype=BF)
    for dt in (F16, BF):
        ref, bound = R.gelu_stage(r_u, accb, dt)
        _ok(R.check("gelu", g32.to(dt), ref, bound))
    # gelu of the ROUNDED u (a kernel that re-read its own bf16 u) is a different function
    ref, bound = R.gelu_stage(r_u, accb, F16)
    ub = u32.to(BF).float()
    _fails(R.check("gelu", (0.5 * ub * (1 + torch.erf(ub / math.sqrt(2)))).to(F16), ref, bound))


def test_gelu_grad_epilogue_tanh_form_passes():
    g = _gen(5)
    dY = _rnd((1, 197, 384), g, 0.01)
    W = _rnd((1, 384, 512), g, 0.05)
    u = _rnd((1, 197, 512), g, 2.0)
    acc = dY.float() @ W.float()
    uf = u.float()
    k = math.sqrt(2 / math.pi)
    t = torch.tanh(k * (uf + 0.044715 * uf ** 3))
    dg = 0.5 * (1 + t) + uf * (1 - t * t) * 0.5 * k * (1 + 3 * 0.044715 * uf * uf)  # the epilogue's tanh form
    ref, bound = R.dgelu_stage(dY, W, u)
    _ok(R.check("dgelu", (acc * dg).to(BF), ref, bound))
    _fails(R.check("dgelu", acc.to(BF), ref, bound))  # gelu' left out


def test_layernorm_forward_passes_and_shifted_row_statistics_fail():
    g = _gen(7)
    x = torch.randn(2, 197, 384, generator=g) * 3 + 1.5
    w = 1 + torch.randn(384, generator=g) * 0.1
    b = torch.randn(384, generator=g) * 0.1
    mean = x.mean(-1)
    rstd = torch.rsqrt(((x - mean.unsqueeze(-1)) ** 2).mean(-1) + 1e-6)
    y = (x - mean.unsqueeze(-1)) * rstd.unsqueeze(-1) * w + b
    (rm, mb), (rr, rb) = R.ln_stats(x)
    _ok(R.check("ln.mean", mean, rm, mb))
    _ok(R.check("ln.rstd", rstd, rr, rb))
    for dt in (F16, BF, F32):
        ref, bound = R.ln_fwd(x, w, b, dt)
        _ok(R.check("ln.y", y.to(dt), ref, bound))
    # statistics of the next row (off-by-one row index in the reduction)
    sh_m, sh_r = torch.roll(mean, -1, 1), torch.roll(rstd, -1, 1)
    _fails(R.check("ln.mean", sh_m, rm, mb))
    _fails(R.check("ln.rstd", sh_r, rr, rb))
    ref, bound = R.ln_fwd(x, w, b, F16)
    _fails(R.check("ln.y", ((x - sh_m.unsqueeze(-1)) * sh_r.unsqueeze(-1) * w + b).to(F16), ref, bound))


@pytest.mark.parametrize("dres_dtype", [None, BF, F32])
def test_layernorm_backward_passes_and_dropped_residual_fails(dres_dtype):
    g = _gen(9)
    x = torch.randn(2, 197, 384, generator=g) * 2
    w = 1 + torch.randn(384, generator=g) * 0.1
    dy = _rnd((2, 197, 384), g, 1e-3)
    mean = x.mean(-1)
    rstd = torch.rsqrt(((x - mean.unsqueeze(-1)) ** 2).mean(-1) + 1e-6)
    xh = (x - mean.unsqueeze(-1)) * rstd.unsqueeze(-1)
    gg = w * dy.float()
    dx = rstd.unsqueeze(-1) * (gg - gg.mean(-1, keepdim=True) - xh * (gg * xh).mean(-1, keepdim=True))
    dres = None if dres_dtype is None else _rnd((2, 197, 384), g, 1e-3, dres_dtype)
    if dres is not None:
        dx = dx + dres.float()
    ref, bound, _ = R.ln_bwd(dy, x, mean, rstd, w, dres, BF)
    _ok(R.check("ln_bwd", dx.to(BF), ref, bound))
    ref32, bound32, _ = R.ln_bwd(dy, x, mean, rstd, w, dres, F32)
    _ok(R.check("ln_bwd32", dx, ref32, bound32))
    if dres is not None:
        _fails(R.check("ln_bwd", (dx - dres.float()).to(BF), ref, bound))
    # column sums: dgamma, dbeta and the bias gradient of the Linear in front (fp32 dx against its bf16 copy)
    dgw, dgw_b = R.colsum(dy.double() * R.ln_bwd(dy, x, mean, rstd, w)[2])
    _ok(R.check("dgamma", (dy.float() * xh).sum(1), dgw, dgw_b))
    cs, cs_b = R.colsum(dx.to(BF), extra_rel=R.U_BF)
    _ok(R.check("bias_from_dx", dx.sum(1), cs, cs_b))


def _attn_case(seed=11, S=197, D=64, nb=3):
    g = _gen(seed)
    q = _rnd((nb, S, D), g, 1.0, F16)
    k = _rnd((nb, S, D), g, 1.0, F16)
    v = _rnd((nb, S, D), g, 1.0, F16)
    return q, k, v, D ** -0.5


def _attn_kernel_fp32(q, k, v, scale, p_dtype, pad_keys=0):
    """fp32 attention with P rounded to p_dtype; pad_keys zero keys / values appended (a tile's padding) and NOT masked."""
    kk, vv = k.float(), v.float()
    if pad_keys:
        z = torch.zeros(kk.shape[0], pad_keys, kk.shape[2])
        kk, vv = torch.cat([kk, z], 1), torch.cat([vv, z], 1)
    s = (q.float() @ kk.transpose(-1, -2)) * scale
    m = s.amax(-1, keepdim=True)
    p = torch.exp(s - m)
    l = p.sum(-1, keepdim=True)
    o = (p.to(p_dtype).float() @ vv) / l
    return o, (m + torch.log(l)).squeeze(-1)


def test_attention_forward_passes_and_an_unmasked_padded_key_fails():
    q, k, v, scale = _attn_case()
    o, lse = _attn_kernel_fp32(q, k, v, scale, F16)
    ro, ob, rl, lb = R.attn_fwd(q, k, v, scale, F16, F16)
    _ok(R.check("attn.o", o.to(F16), ro, ob))
    _ok(R.check("attn.lse", lse, rl, lb))
    o2, lse2 = _attn_kernel_fp32(q, k, v, scale, F16, pad_keys=1)
    _fails(R.check("attn.o", o2.to(F16), ro, ob))
    _fails(R.check("attn.lse", lse2, rl, lb))
    # the same defect seen through an explicit key mask of the reference (mask of the 198-key problem)
    kp = torch.cat([k, torch.zeros(3, 1, 64, dtype=F16)], 1)
    vp = torch.cat([v, torch.zeros(3, 1, 64, dtype=F16)], 1)
    mask = torch.arange(198) < 197
    ro, ob, _, _ = R.attn_fwd(q, kp, vp, scale, F16, F16, key_mask=mask)
    _ok(R.check("attn.o", o.to(F16), ro, ob))
    _fails(R.check("attn.o", o2.to(F16), ro, ob))


def test_attention_backward_passes_and_a_wrong_delta_fails():
    q, k, v, scale = _attn_case(seed=13)
    qb, kb, vb = q.to(BF), k.to(BF), v.to(BF)
    o, lse = _attn_kernel_fp32(qb, kb, vb, scale, BF)
    ob = o.to(BF)
    do = _rnd(o.shape, _gen(14), 1e-2)
    s = (qb.float() @ kb.float().transpose(-1, -2)) * scale
    P = torch.exp(s - lse.unsqueeze(-1))
    delta = (do.float() * ob.float()).sum(-1)
    dP = do.float() @ vb.float().transpose(-1, -2)
    dS = (P * (dP - delta.unsqueeze(-1))).to(BF).float()
    dv = P.to(BF).float().transpose(-1, -2) @ do.float()
    dq = scale * dS @ kb.float()
    dk = scale * dS.transpose(-1, -2) @ qb.float()
    (rq, rk, rv), (bq, bk, bv), (rd, bd) = R.attn_bwd(qb, kb, vb, ob, do, lse, scale)
    _ok(R.check("attn.dq", dq.to(BF), rq, bq))
    _ok(R.check("attn.dk", dk.to(BF), rk, bk))
    _ok(R.check("attn.dv", dv.to(BF), rv, bv))
    _ok(R.check("attn.delta", delta, rd, bd))
    dS_bad = (P * dP).to(BF).float()  # delta dropped
    _fails(R.check("attn.dq", (scale * dS_bad @ kb.float()).to(BF), rq, bq))


def test_weight_gradient_split_k_passes_and_a_missing_split_fails():
    g = _gen(17)
    dY = _rnd((2, 1379, 384), g, 1e-2)
    X = _rnd((2, 1379, 256), g, 1.0)
    parts = [dY[:, i:i + 512].float().transpose(-1, -2) @ X[:, i:i + 512].float() for i in range(0, 1379, 512)]
    got = parts[0] + parts[1] + parts[2]
    ref, bound = R.wgrad(dY, X)
    _ok(R.check("wgrad", got, ref, bound))
    _fails(R.check("wgrad", parts[0] + parts[1], ref, bound))
    db, db_b = R.colsum(dY)
    _ok(R.check("bias", dY.float().sum(1), db, db_b))
    _fails(R.check("bias", dY[:, :-1].float().sum(1), db, db_b))  # last (ragged) row left out


def test_nonzero_gradient_gap_and_nan_fail():
    gap = torch.zeros(2, 40)
    _ok(R.check("gap", gap, torch.zeros(()), torch.zeros(())))
    gap[1, 17] = 1e-30
    res = _fails(R.check("gap", gap, torch.zeros(()), torch.zeros(())))
    assert res.where == (1, 17) and res.worst == math.inf
    A, W, b, acc = _gemm_case()
    got = (acc + b.unsqueeze(1)).to(BF)
    ref, bound, _ = R.gemm(A, W, b, out_dtype=BF)
    got[1, 100, 3] = float("nan")
    res = _fails(R.check("gemm", got, ref, bound))
    assert res.nonfinite == 1 and res.where == (1, 100, 3)


def test_im2col_order_matches_the_conv_weight():
    img = torch.randn(2, 3, 32, 48, generator=_gen(19))
    w = torch.randn(5, 3, 16, 16, generator=_gen(20))
    conv = torch.nn.functional.conv2d(img, w, stride=16)                     # [2, 5, 2, 3]
    mm = R.im2col(img) @ w.reshape(5, -1).t()                                # [2, 6, 5]
    assert torch.allclose(conv.flatten(2).transpose(1, 2), mm, atol=1e-4)
