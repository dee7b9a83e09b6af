"""The fusion's stage checker (tests/fusion_stage_ref.py) is right and not vacuous, without a GPU.

The per-stage replays chained in float64 equal the oracle (oracle.fusion_ref.Fus_CrossViT, forward and autograd
backward in float64); correctly rounded fp32 outputs of every stage pass every bound; and each defect the GPU test
exists to catch fails at the stage and instance where it is planted: swapped LN eps, the wrong softmax scale, the other
branch's CLS row as key 0, a head reading its neighbour's slice, a dropped proj_b, another instance's or direction's
vector, an unwritten dtok row, a record missing from the batch contraction, a NaN."""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import fusion_stage_ref as F  # noqa: E402

C = F.C
ORDER = ("f0", "n0", "rstd0", "xh0", "q", "t", "u", "lse", "o", "y", "chat", "e", "rstd2", "dz", "dy", "df0", "do",
         "du", "dt", "dq", "dxh0", "dg1", "db1")


class _Stub:
    def features3D(self, x):
        return x


def _model(heads, NC, seed, dtype=torch.float64, perturb=0.05):
    from oracle.fusion_ref import Fus_CrossViT
    torch.manual_seed(seed)
    fus = Fus_CrossViT(_Stub(), _Stub(), num_classes=NC, heads=heads).to(dtype)
    vh = [torch.nn.Linear(C, NC).to(dtype) for _ in range(2)]
    with torch.no_grad():
        for p in list(fus.parameters()) + [p for m in vh for p in m.parameters()]:
            p.add_(torch.randn_like(p) * perturb)
    L = fus.multi_scale_transformers[0].cross_attn_layers[0]
    pre, post, hm = (L[0], L[2]), (L[3], L[1]), (fus.mlp_head_cxr[0], fus.mlp_head_enh[0])
    names = {
        "ln1_w": [m.norm.weight for m in pre], "ln1_b": [m.norm.bias for m in pre],
        "wq": [m.fn.wq.weight for m in pre], "wk": [m.fn.wk.weight for m in pre], "wv": [m.fn.wv.weight for m in pre],
        "proj_w": [m.fn.proj.weight for m in pre], "proj_b": [m.fn.proj.bias for m in pre],
        "ln2_w": [m.weight for m in post], "ln2_b": [m.bias for m in post],
        "head_w": [m.weight for m in hm], "head_b": [m.bias for m in hm],
        "vhead_w": [m.weight for m in vh], "vhead_b": [m.bias for m in vh],
    }
    return fus, vh, names


def _inputs(B, S, NC, seed, dtype=torch.float64):
    g = torch.Generator().manual_seed(seed)
    tok = torch.randn(2, B, S, C, generator=g, dtype=dtype) * 1.5
    tok[:, :, 0] *= 2e-3  # CLS rows with a variance near the LN eps: an eps mix-up is visible
    d_fused = torch.randn(B, NC, generator=g, dtype=dtype)
    d_x = torch.randn(2, B, NC, generator=g, dtype=dtype)
    return tok, d_fused, d_x


def _plain(names):
    return {k: tuple(t.detach() for t in v) for k, v in names.items()}


@pytest.mark.parametrize("NC", [1, 3])
@pytest.mark.parametrize("heads", [1, 2, 3, 4])
def test_chained_replay_equals_the_oracle_in_float64(heads, NC):
    B, S = 2, 9
    fus, vh, names = _model(heads, NC, seed=heads * 10 + NC)
    tok, d_fused, d_x = _inputs(B, S, NC, seed=1)
    tok.requires_grad_(True)
    fused = fus.fuse(tok[0], tok[1])
    x = torch.stack([vh[0](tok[0][:, 0]), vh[1](tok[1][:, 0])])
    ((fused.reshape(B, NC) * d_fused).sum() + (x * d_x).sum()).backward()  # NC = 1: fuse() squeezes the class dim
    out, grads = F.run_stages(tok.detach(), _plain(names), heads, d_fused, d_x)

    def close(a, ref, what):
        err = float((a - ref.reshape(a.shape)).abs().max())
        assert err <= 1e-12 * max(1.0, float(ref.abs().max())), (what, err)
    close(out["fused"], fused.detach(), "fused")
    close(out["x"], x.detach(), "x")
    close(out["dtok"], tok.grad, "dtok")
    for k, v in names.items():
        for d in range(2):
            close(grads[k][d][0], v[d].grad, "d%s[%d]" % (k, d))


# --------------------------------------------------------------------------------------- synthetic kernel outputs
HEADS, NC, B, S = 3, 3, 3, 13


@pytest.fixture(scope="module")
def case():
    _, _, names = _model(HEADS, NC, seed=7, dtype=torch.float32)
    P = _plain(names)
    tok, d_fused, d_x = _inputs(B, S, NC, seed=2, dtype=torch.float32)
    fill = {}
    out, grads = F.run_stages(tok, P, HEADS, d_fused, d_x, fill=fill)
    got = {k: torch.stack([v[r] for r in range(2 * B)]) for k, v in fill.items()}
    return dict(P=P, tok=tok, d_fused=d_fused, d_x=d_x, got=got, out=out, grads=grads)


def _run(case, got=None, outs=None, grads_got=None):
    """All stage results of `got` (+ optional outputs / gradients), in pipeline order."""
    rows = []
    out, grads = F.run_stages(case["tok"], case["P"], HEADS, case["d_fused"], case["d_x"], got=got or case["got"],
                              report=lambda n, b, d, g, r, bd: rows.append((n, b, d, F.check(n, g, r, bd))))
    o = outs or {k: case["out"][k].float() for k in ("fused", "x", "dtok")}
    for k in ("fused", "x", "dtok"):
        rows.append((k, -1, -1, F.check(k, o[k], out[k], out[k + "_b"])))
    gg = grads_got or {k: [v[d][0].float() for d in range(2)] for k, v in case["grads"].items()}
    for k, v in grads.items():
        for d in range(2):
            rows.append(("g_" + k, -1, d, F.check(k, gg[k][d], v[d][0], v[d][1])))
    return rows


def _failed(rows):
    return [(n, b, d) for n, b, d, res in rows if not res.ok]


def test_correctly_rounded_outputs_pass_every_bound(case):
    rows = _run(case)
    assert not _failed(rows), [res.line() for *_, res in rows if not res.ok]
    worst = max(res.worst for *_, res in rows)
    assert worst > 1e-3  # the bounds are not so loose that nothing could fail


def _mutated(case, **repl):
    got = {k: v.clone() for k, v in case["got"].items()}
    for k, fn in repl.items():
        for r in range(2 * B):
            v = fn(r)
            if v is not None:
                got[k][r] = v.reshape(got[k][r].shape).float()
    return got


def _first(rows):
    bad = _failed(rows)
    assert bad, "the mutation went unnoticed"
    return min(bad, key=lambda t: ORDER.index(t[0]) if t[0] in ORDER else len(ORDER))


def _p(case, d):
    return {k: v[d] for k, v in case["P"].items()}


def _rows(case, r, cls=None):
    b, d = divmod(r, 2)
    return F.key_rows(case["tok"], b, d, f0=cls)


def test_swapped_ln_eps_fail_at_ln1_and_ln2(case):
    g = case["got"]

    def ln1(key):
        return lambda r: F.ln(g["f0"][r], _p(case, r % 2)["ln1_w"], _p(case, r % 2)["ln1_b"], F.EPS2)[key]
    got = _mutated(case, n0=ln1("n"), xh0=ln1("y"))
    assert _first(_run(case, got))[0] == "n0"

    def ln2(key):
        return lambda r: F.ln2(g["f0"][r], g["y"][r], _p(case, r % 2)["ln2_w"], _p(case, r % 2)["ln2_b"])[key]
    F_EPS2 = F.EPS2
    try:
        F.EPS2 = F.EPS1
        got = _mutated(case, chat=ln2("chat"), e=ln2("e"))
    finally:
        F.EPS2 = F_EPS2
    assert _first(_run(case, got))[0] == "chat"


def _u_with(case, r, scale=None, cls=None, t=None):
    g = case["got"]
    p = _p(case, r % 2)
    sc = scale if scale is not None else (C // HEADS) ** -0.5
    return F.stream_fwd(_rows(case, r, cls if cls is not None else g["f0"][r]), p["ln1_w"], p["ln1_b"],
                        g["t"][r] if t is None else t, sc)


def test_scale_of_the_full_width_fails_at_the_streaming_pass(case):
    got = _mutated(case, u=lambda r: _u_with(case, r, scale=C ** -0.5)["u"],
                   lse=lambda r: _u_with(case, r, scale=C ** -0.5)["lse"])
    assert _first(_run(case, got))[0] == "u"


def test_other_branch_cls_row_as_key_zero_fails_at_the_streaming_pass(case):
    tok = case["tok"]
    got = _mutated(case, u=lambda r: _u_with(case, r, cls=tok[1 - r % 2, r // 2, 0])["u"])
    assert _first(_run(case, got))[0] == "u"


def test_a_head_reading_its_neighbours_slice_fails_at_that_stage(case):
    g = case["got"]

    def o_shift(r):  # row block of head 0 reads u_1 (a wrong `sel`)
        u = g["u"][r].clone()
        u[0] = u[1]
        return F.rowdot(_p(case, r % 2)["wv"], u, heads=HEADS)[0]
    assert _first(_run(case, _mutated(case, o=o_shift)))[0] == "o"

    def u_shift(r):  # head 2's scores taken against t_1
        t = g["t"][r].clone()
        t[2] = t[1]
        return _u_with(case, r, t=t)["u"]
    assert _first(_run(case, _mutated(case, u=u_shift)))[0] == "u"


def test_dropped_proj_bias_fails_at_y(case):
    got = _mutated(case, y=lambda r: F.rowdot(_p(case, r % 2)["proj_w"], case["got"]["o"][r])[0])
    assert _first(_run(case, got))[0] == "y"


def test_another_instance_or_direction_fails_at_that_instance(case):
    g = case["got"]
    target = 2 * 1 + 1  # instance (b=1, d=1) reads (b=2, d=1)'s xh0

    def q_inst(r):
        return F.rowdot(_p(case, 1)["wq"], g["xh0"][r + 2])[0] if r == target else None
    assert _first(_run(case, _mutated(case, q=q_inst))) == ("q", 1, 1)

    def q_dir(r):  # (b=0, d=0) reads direction 1's vector
        return F.rowdot(_p(case, 0)["wq"], g["xh0"][1])[0] if r == 0 else None
    assert _first(_run(case, _mutated(case, q=q_dir))) == ("q", 0, 0)


def test_unwritten_dtok_row_and_missing_record_and_nan_fail(case):
    outs = {k: case["out"][k].float().clone() for k in ("fused", "x", "dtok")}
    outs["dtok"][1, B - 1, S - 1] = float("nan")  # poisoned and never written
    assert ("dtok", -1, -1) in _failed(_run(case, outs=outs))
    outs["dtok"][1, B - 1, S - 1] = 0.0
    assert ("dtok", -1, -1) in _failed(_run(case, outs=outs))
    # the contraction misses the record of the last instance
    g = case["got"]
    gg = {k: [v[d][0].float() for d in range(2)] for k, v in case["grads"].items()}
    last = 2 * (B - 1) + 1
    gg["wq"][1] = gg["wq"][1] - (F.f64(g["dq"][last]).outer(F.f64(g["xh0"][last]))).float()
    assert _failed(_run(case, grads_got=gg)) == [("g_wq", -1, 1)]
    # a NaN in one stored value
    got = {k: v.clone() for k, v in g.items()}
    got["dt"][3, 1, 5] = float("nan")
    assert _first(_run(case, got)) == ("dt", 1, 1)
