"""The explain pass on the GPU: mfv_attn_probs, mfv_attn_rollout and mfv_fusion_attn checked per element against float64
replays of what they read (teacher forcing, derived bounds), the public calls against the fp32 oracle, and the absence
of side effects on the training path.

Bounds (stage_ref / fusion_stage_ref constants; never fitted):
  * probabilities: a score s_j = scale q.k is an fp32 FMA chain over exact 16-bit products, so it is off by at most
    e_j = scale gamma(D) sum|q_d k_d| + 2 u32 |s_j| (the product by the rounded scale).  The softmax is shift-invariant,
    so the error reaches P_j through its own score and the row maximum: |log(P~_j / P_j)| <= e_j + max_k e_k.  Then
    __expf (ex2.approx.ftz of x log2 e: EXP2_REL plus u32 |x| for the product, plus u32 |x| for the subtraction),
    the row sum (gamma(S) and the exp error of every term), and the correctly rounded division (u32).  Flushed
    exponentials add P_FLOOR absolute.  bound = P expm1(total) + P_FLOOR.
  * row sums of the kernel's own P: |sum_j P~_j - 1| <= gamma(S) + 2 u32, whatever the score errors.
  * head_mean against the float64 mean of the kernel's own probs: (gamma(H) + u32) mean|P~| + P_FLOOR.
  * rollout against a float64 chain over the kernel's own head means: per step v' = (v A + v) / 2 adds
    gamma(S + 1) (|v| A + |v|) / 2 and carries the previous error through (A + I) / 2.
  * cross maps: LN1 -> q -> t -> s composed from fusion_stage_ref (ln, rowdot, coldot, _scores), each stage's bound an
    absolute-value replay of its inputs' bounds, then the softmax bound above with e_j = the score bound."""
import math
import os
import sys

import pytest
import torch
import torch.nn.functional as Fn

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import e2e_common as E  # noqa: E402
import fusion_stage_ref as FS  # noqa: E402
import stage_ref as R  # noqa: E402

pytestmark = pytest.mark.gpu

BF, F16, F32 = torch.bfloat16, torch.float16, torch.float32
WORST = {}  # check name -> worst ratio seen (printed at the end of the module)


@pytest.fixture(scope="module", autouse=True)
def _exact_reference_math():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    for k, v in sorted(WORST.items()):
        print("[attn maps] %-34s worst %.4g" % (k, v))


def _note(name, res):
    WORST[name] = max(WORST.get(name, 0.0), res.worst)
    assert res.ok, res.line()


def _bits_equal(a, b):
    if a is None or b is None:
        return a is b
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    it = {2: torch.int16, 4: torch.int32, 8: torch.int64}[a.element_size()]
    return torch.equal(a.contiguous().view(it), b.contiguous().view(it))


def _scalar(v, like):
    return torch.full((), v, dtype=torch.float64, device=like.device)


# --------------------------------------------------------------------------------------------------- references
def softmax_ref(s, e):
    """float64 softmax of scores s [..., S] and the bound of a kernel whose scores are off by at most e [..., S]."""
    S = s.shape[-1]
    e_row = e.amax(-1, keepdim=True)
    arg = s - s.amax(-1, keepdim=True)
    P = torch.softmax(s, -1)
    e_exp = R.EXP2_REL + 2 * R.U32 * (arg.abs() + 2 * e_row)
    e_sum = R.EXP2_REL + 2 * R.U32 * (arg.abs().amax(-1, keepdim=True) + 2 * e_row) + R.gamma(S)
    rel = e + e_row + e_exp + e_sum + R.U32
    return P, P * torch.expm1(rel) + R.P_FLOOR


def probs_ref(qkv):
    """qkv 16-bit [NB, S, 3, H, D] as stored -> (P [NB, H, S, S], bound) in float64."""
    D = qkv.shape[-1]
    scale = D ** -0.5
    q = qkv[:, :, 0].permute(0, 2, 1, 3).double()
    k = qkv[:, :, 1].permute(0, 2, 1, 3).double()
    s = scale * (q @ k.transpose(-1, -2))
    e = scale * R.gamma(D) * (q.abs() @ k.abs().transpose(-1, -2)) + 2 * R.U32 * s.abs()
    return softmax_ref(s, e)


def check_probs(tag, qkv, probs, mean):
    NB, S, _, H, _ = qkv.shape
    P, bnd = probs_ref(qkv)
    _note("probs " + tag, R.check("probs", probs, P, bnd))
    _note("row sums " + tag, R.check("row sums", probs.double().sum(-1), _scalar(1.0, probs),
                                     _scalar(R.gamma(S) + 2 * R.U32, probs)))
    p64 = probs.double()
    _note("head_mean " + tag, R.check("head_mean", mean, p64.mean(1),
                                      (R.gamma(H) + R.U32) * p64.abs().mean(1) + R.P_FLOOR))


def rollout_ref(means):
    """float64 chain over the kernel's own head means [L, NB, S, S] -> (v [NB, S], bound)."""
    L, NB, S, _ = means.shape
    v = torch.zeros(NB, S, dtype=torch.float64, device=means.device)
    v[:, 0] = 1
    err = torch.zeros_like(v)
    for l in reversed(range(L)):
        A = means[l].double()
        va = (v.unsqueeze(1) @ A).squeeze(1)
        ea = (err.unsqueeze(1) @ A).squeeze(1)
        step = 0.5 * R.gamma(S + 1) * (((v.abs() + err).unsqueeze(1) @ A).squeeze(1) + v.abs() + err)
        v, err = 0.5 * (va + v), 0.5 * (ea + err) + step
    return v, err


# ---------------------------------------------------------------------------------------------- encoder runs
def _pair(B, img=224, seed=0, heads=6):
    if heads == 6:
        _, (o_f, o_c, o_e) = E.build_mfvit_pair(img_size=img, seed=seed)
        return (o_c, o_e), E.synthetic_pair(B, img, rank=seed, device="cuda")[:2]
    _, o = E.build_vit_pair(img_size=img, num_heads=heads, seed=seed)
    return (o,), E.synthetic_pair(B, img, rank=seed, device="cuda")[:1]


def _saving_forward(mods, images, bf16=False, wide=False):
    from mfvit.engine import engine_for
    if wide:  # q / k weights x8 in blocks 3 and 7: scores spread over hundreds, near one-hot rows
        with torch.no_grad():
            for m in mods:
                for i in (3, 7):
                    m.blocks[i].attn.qkv.weight[:2 * m.embed_dim].mul_(8.0)
    eng = engine_for(*mods)
    eng.adopt(images[0].device)
    if bf16:
        eng.fwd_f16 = False
        eng.invalidate_shadow()
    tokens, lease = eng.forward(list(images), save=True)
    lay = eng.layout
    D = lay.C // lay.H
    qkv = lease.ws.qkv.view(F16 if eng.fwd_f16 else BF).view(lay.depth, eng.G * images[0].shape[0], lay.S, 3, lay.H, D)
    return eng, tokens, lease, qkv


CONFIGS = [  # (G, B, heads, img, bf16, wide)
    (2, 1, 6, 224, False, False),
    (2, 7, 6, 224, False, False),
    (2, 32, 6, 224, False, False),
    (1, 7, 12, 224, False, False),
    (2, 2, 6, 384, False, False),
    (2, 7, 6, 224, True, False),
    (2, 7, 6, 224, False, True),
    (1, 3, 12, 384, True, True),
]


@pytest.mark.parametrize("G,B,heads,img,bf16,wide", CONFIGS,
                         ids=["G%d-B%d-H%d-%dpx%s%s" % (c[0], c[1], c[2], c[3], "-bf16" if c[4] else "",
                                                       "-wide" if c[5] else "") for c in CONFIGS])
def test_teacher_forced_probs_and_rollout(G, B, heads, img, bf16, wide):
    from mfvit import ops
    mods, images = _pair(B, img, seed=B + heads, heads=heads)
    assert len(mods) == G
    eng, _, lease, qkv = _saving_forward(mods, images, bf16=bf16, wide=wide)
    try:
        L, NB, S, _, H, D = qkv.shape
        assert qkv.dtype == BF or not bf16   # the fp16 forward switches itself to bf16 for out-of-range weights
        tag = "%s D%d S%d" % ("bf16" if qkv.dtype == BF else "fp16", D, S)
        means = torch.full((L, NB, S, S), math.nan, device="cuda")
        for l in range(L):
            probs = torch.full((NB, H, S, S), math.nan, device="cuda")
            ops.attn_probs(qkv[l], probs, means[l])
            torch.cuda.synchronize()
            check_probs(tag + (" wide" if wide else ""), qkv[l], probs, means[l])
            # the mean alone (the rollout path) writes the same bits
            alone = torch.full((NB, S, S), math.nan, device="cuda")
            ops.attn_probs(qkv[l], None, alone)
            assert _bits_equal(alone, means[l])
            del probs
        out = torch.full((NB, S), math.nan, device="cuda")
        ops.attn_rollout(means, out)
        v, err = rollout_ref(means)
        _note("rollout " + tag, R.check("rollout", out, v, err))
    finally:
        lease.release()


# ------------------------------------------------------------------------------------------------- cross maps
def _fusion_params(heads, seed, wide):
    """Random PreNorm / wq / wk of both directions (the only tensors mfv_fusion_attn reads), plus stand-ins."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    std = 0.2 if wide else 0.02
    C = 384

    def r(*shape, s=1.0, mean=0.0):
        return (torch.randn(*shape, generator=g, device="cuda") * s + mean).contiguous()
    ps = {"ln1_w": [r(C, s=0.1, mean=1.0) for _ in range(2)], "ln1_b": [r(C, s=0.1) for _ in range(2)],
          "wq": [r(C, C, s=std) for _ in range(2)], "wk": [r(C, C, s=std) for _ in range(2)]}
    return ps


def cross_ref(tok, ps, heads):
    """float64 probs [B, 2, heads, S] and bound from fp32 tok [2, B, S, C] (fusion_stage_ref stage bounds)."""
    _, B, S, C = tok.shape
    scale = (C // heads) ** -0.5
    P = torch.empty(B, 2, heads, S, dtype=torch.float64, device=tok.device)
    bnd = torch.empty_like(P)
    for d in range(2):
        g1, b1, wq, wk = ps["ln1_w"][d], ps["ln1_b"][d], ps["wq"][d], ps["wk"][d]
        L = FS.ln(torch.cat((tok[d, :, 0:1], tok[1 - d, :, 1:]), 1), g1, b1, FS.EPS1)   # [B, S, C] key rows
        xh, xh_b = L["y"], L["y_b"]
        for b in range(B):
            q, q_b = FS.rowdot(wq, xh[b, 0], vec_err=xh_b[b, 0])
            t, t_b = FS.coldot(wk, q, heads=heads, vec_err=q_b)
            s, s_b = FS._scores(xh[b], xh_b[b], t, t_b, scale)
            P[b, d], bnd[b, d] = softmax_ref(s, s_b)
    return P, bnd


@pytest.mark.parametrize("heads", [1, 2, 3, 4])
@pytest.mark.parametrize("S,B", [(197, 1), (197, 17), (197, 64), (577, 5)])
@pytest.mark.parametrize("wide", [False, True], ids=["init", "wide"])
def test_teacher_forced_cross_maps(heads, S, B, wide):
    from mfvit import ops
    from mfvit.functions import FUSION_FIELDS
    ps = _fusion_params(heads, seed=heads * 100 + S + B, wide=wide)
    g = torch.Generator(device="cuda").manual_seed(S + B)
    tok = torch.randn(2, B, S, 384, generator=g, device="cuda")
    tok = Fn.layer_norm(tok, (384,)) * 1.3 + 0.1   # final-normed-like rows
    full = {n: ps.get(n, [None, None]) for n in FUSION_FIELDS}
    out = torch.full((B, 2, heads, S), math.nan, device="cuda")
    ops.fusion_attn(tok, ops.fusion_param_struct({n: tuple(v) for n, v in full.items()}), heads, out)
    P, bnd = cross_ref(tok, ps, heads)
    _note("cross heads %d S %d%s" % (heads, S, " wide" if wide else ""), R.check("cross", out, P, bnd))
    _note("cross row sums", R.check("cross row sums", out.double().sum(-1), _scalar(1.0, out),
                                    _scalar(R.gamma(S) + 2 * R.U32, out)))


# ------------------------------------------------------------------------------------------- end to end: oracle
def _cos_rows(a, b):
    """Cosine similarity over the last dimension."""
    return Fn.cosine_similarity(a.double(), b.double(), dim=-1)


@pytest.mark.parametrize("img,B", [(224, 4), (384, 2)])
def test_end_to_end_against_the_fp32_oracle(img, B):
    from oracle import attention_ref as A
    (r_f, r_c, r_e), (o_f, o_c, o_e) = E.build_mfvit_pair(img_size=img, seed=3)
    img_c, img_e, _ = E.synthetic_pair(B, img, rank=3, device="cuda")
    ex = o_f.explain(o_c, o_e, img_c, img_e, blocks=range(12))
    with torch.no_grad():
        tc, mc = A.vit_attention(r_c, img_c)
        te, me = A.vit_attention(r_e, img_e)
        cross = A.cross_attention(r_f, tc, te)
    ref_maps = torch.stack((mc, me))                            # [2, B, L, H, S, S]
    ref_roll = torch.stack((A.rollout(mc.mean(2)), A.rollout(me.mean(2))))
    c_maps = _cos_rows(ex.maps.flatten(-2), ref_maps.flatten(-2))   # one cosine per (branch, image, block, head)
    c_roll = _cos_rows(ex.rollout, ref_roll)
    c_cross = _cos_rows(ex.cross, cross)
    for name, c in (("maps", c_maps), ("rollout", c_roll), ("cross", c_cross)):
        worst = float(c.min())
        WORST["e2e %dpx min cosine %s (1 - cos)" % (img, name)] = max(
            WORST.get("e2e %dpx min cosine %s (1 - cos)" % (img, name), 0.0), 1.0 - worst)
        assert worst >= 0.999, (name, worst)


def test_vit_public_calls_match_the_oracle_and_the_ops():
    """VisionTransformerMoCo.attention_maps / attention_rollout (single-branch engine, 12 heads of 32) equal the ops on
    the same stored qkv bit for bit and follow the oracle."""
    from mfvit import ops
    from mfvit.engine import engine_for
    from oracle import attention_ref as A
    ref, ours = E.build_vit_pair(num_heads=12, seed=4)
    x, _, _ = E.synthetic_pair(3, 224, rank=4, device="cuda")
    maps = ours.attention_maps(x, blocks=[0, 5, 11, 5])
    roll = ours.attention_rollout(x)
    assert maps.shape == (3, 4, 12, 197, 197) and roll.shape == (3, 197)
    assert not maps.requires_grad and not roll.requires_grad
    eng, _, lease, qkv = _saving_forward((ours,), [x])
    try:
        means = torch.empty(12, 3, 197, 197, device="cuda")
        for l in range(12):
            p = torch.empty(3, 12, 197, 197, device="cuda")
            ops.attn_probs(qkv[l], p, means[l])
            for k, b in enumerate([0, 5, 11, 5]):
                if b == l:
                    assert _bits_equal(maps[:, k], p), (k, b)
        assert _bits_equal(roll, ops.attn_rollout(means))
    finally:
        lease.release()
    assert _bits_equal(ours.attention_maps(x)[:, 5], maps[:, 1])   # blocks=None is all of them
    with torch.no_grad():
        _, rm = A.vit_attention(ref, x)
    assert float(_cos_rows(maps.flatten(-2), rm[:, [0, 5, 11, 5]].flatten(-2)).min()) >= 0.999
    assert float(_cos_rows(roll, A.rollout(rm.mean(2))).min()) >= 0.999
    assert eng is engine_for(ours)


# ---------------------------------------------------------------------------------------------- no side effects
def _engine_state(eng):
    return {"ptrs": [p.data_ptr() for p in eng.params_flat()], "master": eng.master.clone(),
            "shadow": eng.shadow.clone(), "shadow16": eng.shadow16.clone(),
            "grads": [None if g is None else g.clone() for g in eng.grads]}


def _same_state(a, b):
    return (a["ptrs"] == b["ptrs"] and all(_bits_equal(a[k], b[k]) for k in ("master", "shadow", "shadow16"))
            and all(_bits_equal(x, y) for x, y in zip(a["grads"], b["grads"])))


def test_explain_has_no_side_effects():
    from mfvit.engine import engine_for
    _, (o_f, o_c, o_e) = E.build_mfvit_pair(seed=6)
    img_c, img_e, tgt = E.synthetic_pair(8, 224, rank=6, device="cuda")
    o_f.train()
    E.mfvit_step(o_f, o_c, o_e, img_c, img_e, tgt)   # a training step: gradients exist, the engine is adopted
    eng = engine_for(o_c, o_e)
    with torch.no_grad():
        want = o_f(o_c, o_e, img_c, img_e)
    before = _engine_state(eng)
    grads_before = [p.grad.clone() for p in o_c.parameters() if p.grad is not None]
    ex = o_f.explain(o_c, o_e, img_c, img_e, blocks=(2, 9))
    ex2 = o_f.explain(o_c, o_e, img_c, img_e, blocks=(2, 9))
    torch.cuda.synchronize()
    for a, b in zip(want, (ex.fused, ex.x_cxr, ex.x_enh)):
        assert _bits_equal(a, b)
    for f in ("fused", "x_cxr", "x_enh", "rollout", "cross", "maps"):
        assert _bits_equal(getattr(ex, f), getattr(ex2, f)), f
        assert not getattr(ex, f).requires_grad, f
    assert ex.maps.shape == (2, 8, 2, 6, 197, 197) and ex.rollout.shape == (2, 8, 197)
    assert ex.cross.shape == (8, 2, 3, 197)
    assert _same_state(before, _engine_state(eng))
    assert all(_bits_equal(g, p.grad) for g, p in zip(grads_before, [p for p in o_c.parameters() if p.grad is not None]))
    assert o_f.explain(o_c, o_e, img_c, img_e).maps is None


def test_explain_between_a_training_forward_and_its_backward():
    """The saving forward of explain takes a workspace of its own: the training forward's saved activations stay
    bit-identical, and so do the gradients of its backward (when the backward itself is run-to-run reproducible; the
    split-K weight gradients add with red.global.add, so that is measured first)."""
    from mfvit.engine import engine_for
    _, (o_f, o_c, o_e) = E.build_mfvit_pair(seed=8)
    img_c, img_e, _ = E.synthetic_pair(7, 224, rank=8, device="cuda")
    eng = engine_for(o_c, o_e)
    eng.adopt(img_c.device)
    g = torch.Generator(device="cuda").manual_seed(8)
    dtok = torch.randn(2, 7, 197, 384, device="cuda", generator=g) * 1e-3

    def train_step(between=None):
        tokens, lease = eng.forward([img_c, img_e], save=True)
        snap = None
        if between is not None:
            snap = {f: getattr(lease.ws, f).clone() for f in ("x", "xn", "qkv", "attn_o", "lse", "u", "gact")}
            between()
            torch.cuda.synchronize()
            for f, t in snap.items():
                assert _bits_equal(t, getattr(lease.ws, f)), f
        return tokens, eng.backward(lease, dtok).clone()

    t0, g0 = train_step()
    t1, g1 = train_step()
    t2, g2 = train_step(lambda: o_f.explain(o_c, o_e, img_c, img_e, blocks=(0, 11)))
    assert _bits_equal(t0, t2)
    if _bits_equal(g0, g1):
        assert _bits_equal(g0, g2)
    else:
        spread = float((g0 - g1).abs().max())
        assert float((g0 - g2).abs().max()) <= 4 * spread, spread


# ---------------------------------------------------------------------------------------------------- contract
def test_errors():
    from mfvit import MfvError, ops
    _, ours = E.build_vit_pair(seed=9)
    x, _, _ = E.synthetic_pair(2, 224, rank=9, device="cuda")
    with pytest.raises(MfvError):
        ours.attention_maps(x.cpu())
    with pytest.raises(MfvError):
        ours.attention_rollout(x.cpu())
    for bad in (-1, 12, 1.5):
        with pytest.raises(MfvError):
            ours.attention_maps(x, blocks=[0, bad])
    with pytest.raises(MfvError):
        ops.attn_probs(torch.zeros(2, 5, 3, 4, 48, dtype=BF, device="cuda"), torch.empty(2, 4, 5, 5, device="cuda"))
    with pytest.raises(MfvError):   # S > 577
        ops.attn_probs(torch.zeros(1, 578, 3, 6, 64, dtype=BF, device="cuda"), None,
                       torch.empty(1, 578, 578, device="cuda"))
    with pytest.raises(MfvError):
        ops.attn_probs(torch.zeros(2, 5, 3, 6, 64, dtype=BF), torch.empty(2, 6, 5, 5))
    with pytest.raises(MfvError):   # fp32 qkv
        ops.attn_probs(torch.zeros(2, 5, 3, 6, 64, device="cuda"), torch.empty(2, 6, 5, 5, device="cuda"))
    with pytest.raises(MfvError):   # wrong output shape
        ops.attn_probs(torch.zeros(2, 5, 3, 6, 64, dtype=BF, device="cuda"), torch.empty(2, 6, 5, 4, device="cuda"))
    with pytest.raises(MfvError):   # non-contiguous output
        ops.attn_probs(torch.zeros(2, 5, 3, 6, 64, dtype=BF, device="cuda"),
                       torch.empty(2, 6, 5, 5, device="cuda").transpose(-1, -2))
    with pytest.raises(MfvError):
        ops.attn_rollout(torch.zeros(2, 1, 5, 5))
    with pytest.raises(MfvError):
        ops.fusion_attn(torch.zeros(2, 1, 197, 384), ops.fusion_param_struct({}), 3)
    (_, _, _), (o_f, o_c, o_e) = E.build_mfvit_pair(seed=9)
    with pytest.raises(MfvError):
        o_f.explain(o_e, o_c, x, x)   # backbones swapped
    with pytest.raises(MfvError):
        o_f.explain(o_c, o_e, x, x, blocks=[12])
    with pytest.raises(MfvError):
        o_f.explain(o_c, o_e, x.cpu(), x.cpu())


def test_fusion_explain_cross_equals_the_op():
    from mfvit import ops
    from mfvit.engine import engine_for
    _, (o_f, o_c, o_e) = E.build_mfvit_pair(seed=10)
    img_c, img_e, _ = E.synthetic_pair(5, 224, rank=10, device="cuda")
    with torch.enable_grad():
        ex = o_f.explain(o_c, o_e, img_c, img_e)
    eng = engine_for(o_c, o_e)
    with torch.no_grad():
        tok, lease = eng.forward([img_c, img_e], save=True)
        lease.release()
        params, _ = o_f._fusion_params(o_c, o_e)
        from mfvit.functions import FUSION_FIELDS
        ps = [None if p is None else p.detach().contiguous() for p in params]
        st = ops.fusion_param_struct({n: (ps[2 * i], ps[2 * i + 1]) for i, n in enumerate(FUSION_FIELDS)})
        assert _bits_equal(ex.cross, ops.fusion_attn(tok, st, o_f.heads))
