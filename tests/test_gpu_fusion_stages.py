"""Stage checks of the cross-attention fusion (csrc/fusion.cu) on both of its paths, per element, against the float64
replays of tests/fusion_stage_ref.py.

Every buffer is NaN-poisoned before each call: `saved`, dtok, the outputs.  The batched path is teacher-forced: every
stage is recomputed from the fp32 values the previous kernel stored in `saved` and compared with what it stored
itself, so a wrong instance, head slice or ragged block shows up at a named stage and instance.  The single-kernel path
(MFVIT_FUSION_BATCHED=0, read once per process, so it runs in a child interpreter) keeps only the per-instance records
of its backward: each record, fused, x and every dtok row are checked from the records they depend on, with the bound
of the intermediates it does not keep carried forward.  The evaluation forward (fusion_fwd without `saved`) runs that
same kernel and must reproduce the child's checked outputs bit for bit.  Parameter gradients are accumulated onto known
values; the state reuse of the batched path and the deferred contraction must give bit-identical results."""
import ctypes
import json
import os
import subprocess
import sys
import tempfile

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (HERE, ROOT, os.path.join(ROOT, "multi-feature-vit_b200"), os.path.join(ROOT, "multi-feature-vit_b200", "dropin")):
    if _p not in sys.path:
        sys.path.insert(0, _p)
import fusion_stage_ref as F  # noqa: E402

pytestmark = pytest.mark.gpu

C = F.C
MFV_ERR_SHAPE = -1  # common.cuh
NAN = float("nan")
FIELDS = F.FIELDS


# ----------------------------------------------------------------------------------------------------- inputs
def make_params(heads, NC, regime, seed, vhead=True, dev=None):
    from oracle.fusion_ref import Fus_CrossViT
    dev = dev or ("cuda" if torch.cuda.is_available() else "cpu")

    class Stub:
        def features3D(self, x):
            return x
    torch.manual_seed(seed)
    fus = Fus_CrossViT(Stub(), Stub(), num_classes=NC, heads=heads)  # the model's init: trunc-normal 0.02, LN 1 / 0
    vh = [torch.nn.Linear(C, NC) for _ in range(2)]
    for m in vh:
        Fus_CrossViT._init_weights(m)
    if regime != "init":  # the op check's perturbed weights
        with torch.no_grad():
            for p in list(fus.parameters()) + [p for m in vh for p in m.parameters()]:
                p.add_(torch.randn_like(p) * 0.05)
    L = fus.multi_scale_transformers[0].cross_attn_layers[0]
    pre, post, hm = (L[0], L[2]), (L[3], L[1]), (fus.mlp_head_cxr[0], fus.mlp_head_enh[0])
    P = {
        "ln1_w": [m.norm.weight for m in pre], "ln1_b": [m.norm.bias for m in pre],
        "wq": [m.fn.wq.weight for m in pre], "wk": [m.fn.wk.weight for m in pre], "wv": [m.fn.wv.weight for m in pre],
        "proj_w": [m.fn.proj.weight for m in pre], "proj_b": [m.fn.proj.bias for m in pre],
        "ln2_w": [m.weight for m in post], "ln2_b": [m.bias for m in post],
        "head_w": [m.weight for m in hm], "head_b": [m.bias for m in hm],
        "vhead_w": [m.weight for m in vh] if vhead else [None, None],
        "vhead_b": [m.bias for m in vh] if vhead else [None, None],
    }
    return {k: tuple(None if t is None else t.detach().float().contiguous().to(dev) for t in v) for k, v in P.items()}


def make_inputs(B, S, NC, seed, dev=None):
    dev = dev or ("cuda" if torch.cuda.is_available() else "cpu")
    g = torch.Generator().manual_seed(seed)
    tok = torch.randn(2, B, S, C, generator=g) * 1.5
    return tok.to(dev), torch.randn(B, NC, generator=g).to(dev), torch.randn(2, B, NC, generator=g).to(dev)


def widen_scores(P, tok, heads, target=80.0):
    """Scale Wq until the score spread of instance (0, 0) reaches `target` in every head: each softmax is then nearly
    one-hot, and the online softmax rescales on almost every new maximum."""
    p = {k: v[0] for k, v in P.items()}
    L = F.ln(tok[0, 0, 0], p["ln1_w"], p["ln1_b"], F.EPS1)
    q = F.f64(p["wq"]) @ L["y"]
    t = F.coldot(p["wk"], q, heads)[0]
    xh = F.ln(F.key_rows(tok, 0, 0), p["ln1_w"], p["ln1_b"], F.EPS1)["y"]
    s = (C // heads) ** -0.5 * (t @ xh.T)
    k = target / float((s.amax(-1) - s.amin(-1)).min())
    return dict(P, wq=tuple((w * k).contiguous() for w in P["wq"]))


def make_case(B, heads=3, NC=3, S=197, regime="perturbed", seed=0, vhead=True, dx=True):
    P = make_params(heads, NC, regime, seed, vhead=vhead)
    tok, d_fused, d_x = make_inputs(B, S, NC, seed + 1)
    if regime == "wide":
        P = widen_scores(P, tok, heads)
    if regime == "zero_var":  # a key row and a CLS row whose LayerNorm variance is 0: rstd = 1/sqrt(eps)
        tok[1, 0, 3] = 0.3
        tok[0, B - 1, 0] = -1.7
    g = torch.Generator().manual_seed(seed + 2)
    G0 = {k: tuple(None if t is None else (torch.randn(t.shape, generator=g) * 0.1).to(t.device) for t in v)
          for k, v in P.items()}
    return dict(B=B, S=S, heads=heads, NC=NC, P=P, tok=tok, d_fused=d_fused, d_x=d_x if dx else None, G0=G0)


# --------------------------------------------------------------------------------------------------- the calls
def struct(P, grads=False):
    from mfvit import ops
    from mfvit._lib import FusionGrads, FusionParams
    return ops.fusion_param_struct(P, cls=FusionGrads if grads else FusionParams)


def fwd(cs, saved):
    """mfv_fusion_fwd into NaN-poisoned outputs."""
    from mfvit import ops
    B, NC = cs["B"], cs["NC"]
    fused = torch.full((B, NC), NAN, device="cuda")
    x = torch.full((2, B, NC), NAN, device="cuda")
    prm = struct(cs["P"])
    rc = ops._lib_for(cs["tok"]).mfv_fusion_fwd(ops._p(cs["tok"]), ctypes.byref(prm), ops._p(fused), ops._p(x),
                                                 ops._p(saved), B, cs["S"], C, cs["heads"], NC, ops._stream())
    ops.check(rc, "mfv_fusion_fwd")
    return fused, x


def new_saved(cs):
    from mfvit import ops
    n = ops.fusion_scratch(cs["tok"], cs["B"], cs["S"], C, cs["heads"]).numel()
    assert n == F.saved_floats(cs["B"], cs["heads"])
    return torch.full((n,), NAN, device="cuda")


def new_grads(cs):
    return {k: tuple(None if t is None else t.clone() for t in v) for k, v in cs["G0"].items()}


def bwd(cs, saved, grads, defer=False):
    from mfvit import ops
    dtok = torch.full_like(cs["tok"], NAN)
    ops.fusion_bwd(cs["tok"], struct(cs["P"]), struct(grads, True), cs["d_fused"], cs["d_x"], cs["B"], cs["S"], C,
                   cs["heads"], cs["NC"], dtok=dtok, scratch=saved, defer=defer)
    return dtok


def run_plain(cs):
    saved = new_saved(cs)
    fused, x = fwd(cs, saved)
    grads = new_grads(cs)
    dtok = bwd(cs, saved, grads)
    torch.cuda.synchronize()
    return dict(fused=fused, x=x, dtok=dtok, saved=saved, grads=grads)


# -------------------------------------------------------------------------------------------------- the checks
def stored_batched(saved, B, heads):
    rec, fw, bt = F.split_saved(saved, B, heads)
    got = {k: fw[k] for k in ("f0", "n0", "xh0", "q", "t", "u", "o", "y", "chat", "e")}
    got.update(rstd0=fw["misc"][:, 0:1], rstd2=fw["misc"][:, 1:2], lse=fw["misc"][:, 4:4 + heads])
    got.update({k: rec[k] for k in ("dz", "dy", "do", "dt", "dq", "dg1", "db1")})
    got.update(du=bt["du"], dxh0=bt["dxh0"], df0=bt["df0"])
    return got, rec, fw


def stored_single(saved, B, heads):
    rec, _, _ = F.split_saved(saved, B, heads)
    return {k: rec[k] for k in ("f0", "xh0", "q", "u", "o", "chat", "e", "dz", "dy", "do", "dt", "dq", "dg1", "db1")}


def check_run(cs, res, got):
    """Every stored stage value, the outputs and the 26 gradients.  Returns the list of (stage, b, d, Result)."""
    rows = []

    def rep(name, b, d, g, r, bd):
        rows.append((name, b, d, F.check(name, g, r, bd)))
    out, grads = F.run_stages(cs["tok"], cs["P"], cs["heads"], cs["d_fused"], cs["d_x"], got=got, G0=cs["G0"],
                              report=rep)
    rows.append(("fused", -1, -1, F.check("fused", res["fused"], out["fused"], out["fused_b"])))
    if out["x"] is not None:
        rows.append(("x", -1, -1, F.check("x", res["x"], out["x"], out["x_b"])))
    rows.append(("dtok", -1, -1, F.check("dtok", res["dtok"], out["dtok"], out["dtok_b"])))
    for k, v in grads.items():
        for d in range(2):
            if k in res["grads"] and res["grads"][k][d] is not None:
                rows.append(("g_" + k, -1, d, F.check(k, res["grads"][k][d], v[d][0], v[d][1])))
    return rows


def summary(rows):
    worst = {}
    for n, _, _, r in rows:
        worst[n] = max(worst.get(n, 0.0), r.worst)
    return worst


def assert_ok(rows, label):
    w = summary(rows)
    print("\n[%s] worst |got - ref| / bound per stage: %s" % (label, json.dumps({k: float("%.3g" % v)
                                                                                  for k, v in w.items()})))
    bad = [(n, b, d, r.line()) for n, b, d, r in rows if not r.ok]
    assert not bad, bad[:10]


def bits_equal(a, b):
    if a is None or b is None:
        return a is b
    return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))


@pytest.fixture(scope="module", autouse=True)
def _exact_reference_math():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield


# ------------------------------------------------------------------------------------------ a. batched path
CASES = ([dict(B=B) for B in (1, 2, 15, 16, 17, 32, 33, 64)]
         + [dict(B=17, heads=h) for h in (1, 2, 4)]
         + [dict(B=17, S=577), dict(B=17, NC=1), dict(B=17, NC=8)]
         + [dict(B=17, regime=r) for r in ("init", "wide", "zero_var")]
         + [dict(B=1, regime="init"), dict(B=32, regime="init")])


def _id(kw):
    return "-".join("%s%s" % (k, v) for k, v in kw.items())


@pytest.mark.parametrize("kw", CASES, ids=[_id(k) for k in CASES])
def test_batched_path_every_stage(kw):
    cs = make_case(**kw)
    res = run_plain(cs)
    got, rec, fw = stored_batched(res["saved"], cs["B"], cs["heads"])
    for k in ("xh0", "q", "o", "chat", "e", "f0", "u"):  # the records copy the forward state bit for bit
        assert bits_equal(rec[k], fw[k]), k
    assert_ok(check_run(cs, res, got), "batched " + _id(kw))


def test_corrupted_u_is_reported_at_its_stage_and_instance_only():
    cs = make_case(B=17)
    res = run_plain(cs)
    got, _, fw = stored_batched(res["saved"], cs["B"], cs["heads"])
    r = 16 * 2 + 1
    fw["u"][r, 1, 77] += 0.05 * float(fw["u"][r].abs().max())  # between the run and its checks
    rows = check_run(cs, res, got)
    bad = {(n, b, d) for n, b, d, x in rows if not x.ok}
    assert ("u", 16, 1) in bad
    order = ("f0", "n0", "rstd0", "xh0", "q", "t", "u")
    assert all(b == 16 and d == 1 and n not in order[:-1] for n, b, d in bad if b >= 0), bad
    assert all(n in ("dtok", "fused", "x") or n.startswith("g_") for n, b, _ in bad if b < 0), bad  # downstream only
    print("\ncorruption of u at (b=16, d=1) flagged at:", sorted(bad))


# --------------------------------------------------------------------------------------- e. contract
def test_without_backbone_heads_x_stays_poisoned_and_their_gradients_untouched():
    cs = make_case(B=17, vhead=False)
    cs["G0"]["vhead_w"] = tuple(torch.randn(3, C, device="cuda") for _ in range(2))
    cs["G0"]["vhead_b"] = tuple(torch.randn(3, device="cuda") for _ in range(2))
    res = run_plain(cs)
    assert torch.isnan(res["x"]).all()
    for k in ("vhead_w", "vhead_b"):
        for d in range(2):
            assert bits_equal(res["grads"][k][d], cs["G0"][k][d]), k
    res["grads"] = {k: v for k, v in res["grads"].items() if k not in ("vhead_w", "vhead_b")}
    got, _, _ = stored_batched(res["saved"], cs["B"], cs["heads"])
    assert_ok([r for r in check_run(cs, res, got) if not r[0].startswith("g_vhead")], "no vhead")


def test_without_d_x():
    cs = make_case(B=17, dx=False)
    res = run_plain(cs)
    got, _, _ = stored_batched(res["saved"], cs["B"], cs["heads"])
    assert_ok(check_run(cs, res, got), "d_x None")
    for k in ("vhead_w", "vhead_b"):
        for d in range(2):
            assert bits_equal(res["grads"][k][d], cs["G0"][k][d]), k


@pytest.mark.parametrize("heads,NC,Cd", [(5, 3, 384), (3, 9, 384), (3, 3, 768), (0, 3, 384)])
def test_unsupported_shapes_are_refused(heads, NC, Cd):
    from mfvit import ops
    cs = make_case(B=2, S=5)
    saved = torch.full((F.saved_floats(2, 4) * 2,), NAN, device="cuda")
    out = torch.full((64,), NAN, device="cuda")
    lib = ops._lib_for(cs["tok"])
    prm, gs = struct(cs["P"]), struct(new_grads(cs), True)
    rc = lib.mfv_fusion_fwd(ops._p(cs["tok"]), ctypes.byref(prm), ops._p(out), ops._p(out), ops._p(saved), 2, 5, Cd,
                            heads, NC, ops._stream())
    assert rc == MFV_ERR_SHAPE
    rc = lib.mfv_fusion_bwd(ops._p(cs["tok"]), ctypes.byref(prm), ops._p(saved), ops._p(out), ops._p(out),
                            ops._p(out), ctypes.byref(gs), 2, 5, Cd, heads, NC, ops._stream())
    assert rc == MFV_ERR_SHAPE
    torch.cuda.synchronize()
    assert torch.isnan(out).all()


# ---------------------------------------------------------------------------------- f. state reuse, ordering
def _same(a, b, what):
    assert bits_equal(a["dtok"], b["dtok"]), what + ": dtok"
    for k in FIELDS:
        for d in range(2):
            assert bits_equal(a["grads"][k][d], b["grads"][k][d]), "%s: %s[%d]" % (what, k, d)


def test_state_reuse_and_ordering_are_bit_identical():
    from mfvit import ops
    A, Bc = make_case(B=17, seed=0), make_case(B=33, seed=5)
    ref_a, ref_b = run_plain(A), run_plain(Bc)
    # the recompute branch: a backward on a buffer no forward filled
    s_other = new_saved(A)
    fwd(A, s_other)
    g = new_grads(A)
    r = dict(dtok=bwd(A, new_saved(A), g), grads=g)
    torch.cuda.synchronize()
    _same(r, ref_a, "recompute")
    # forward A, forward B into another buffer, backward A, backward B
    sa, sb = new_saved(A), new_saved(Bc)
    fwd(A, sa)
    fwd(Bc, sb)
    ga, gb = new_grads(A), new_grads(Bc)
    ra = dict(dtok=bwd(A, sa, ga), grads=ga)
    rb = dict(dtok=bwd(Bc, sb, gb), grads=gb)
    torch.cuda.synchronize()
    _same(ra, ref_a, "A B A B")
    _same(rb, ref_b, "A B A B (B)")
    # two backwards from one forward
    s = new_saved(A)
    fwd(A, s)
    g1, g2 = new_grads(A), new_grads(A)
    r1 = dict(dtok=bwd(A, s, g1), grads=g1)
    r2 = dict(dtok=bwd(A, s, g2), grads=g2)
    torch.cuda.synchronize()
    _same(r1, ref_a, "first of two backwards")
    _same(r2, ref_a, "second of two backwards")
    # deferred + join
    s = new_saved(A)
    fwd(A, s)
    g = new_grads(A)
    r = dict(dtok=bwd(A, s, g, defer=True), grads=g)
    ops.fusion_bwd_join()
    torch.cuda.synchronize()
    _same(r, ref_a, "deferred")
    # two deferred backwards on one buffer back to back, then one join
    s = new_saved(A)
    fwd(A, s)
    g1, g2 = new_grads(A), new_grads(A)
    r1 = dict(dtok=bwd(A, s, g1, defer=True), grads=g1)
    r2 = dict(dtok=bwd(A, s, g2, defer=True), grads=g2)
    ops.fusion_bwd_join()
    torch.cuda.synchronize()
    _same(r1, ref_a, "first of two deferred")
    _same(r2, ref_a, "second of two deferred")
    # a plain backward while a deferred one is pending, onto the same gradients: G0 + 2 x the contraction
    s = new_saved(A)
    fwd(A, s)
    g = new_grads(A)
    bwd(A, s, g, defer=True)
    fwd(A, s)
    bwd(A, s, g)
    ops.fusion_bwd_join()
    gg = new_grads(A)
    for _ in range(2):
        fwd(A, s)
        bwd(A, s, gg)
    torch.cuda.synchronize()
    _same(dict(dtok=ref_a["dtok"], grads=g), dict(dtok=ref_a["dtok"], grads=gg), "deferred then plain")


# -------------------------------------------------------------------------------------- b. single-kernel path
SINGLE = [dict(B=17, heads=1), dict(B=1), dict(B=17), dict(B=32), dict(B=17, heads=2), dict(B=17, heads=4),
          dict(B=2, S=577), dict(B=17, NC=8), dict(B=17, regime="wide"), dict(B=17, regime="zero_var")]


def _child(path_in, path_out):
    """Runs in an interpreter started with MFVIT_FUSION_BATCHED=0: the single-kernel forward and backward."""
    cases = torch.load(path_in)
    outs = []
    for kw in cases:
        cs = make_case(**kw)
        outs.append({k: (v.cpu() if torch.is_tensor(v) else {kk: tuple(None if t is None else t.cpu() for t in vv)
                                                              for kk, vv in v.items()})
                     for k, v in run_plain(cs).items()})
    torch.save(outs, path_out)


@pytest.fixture(scope="module")
def single_results():
    with tempfile.TemporaryDirectory() as tmp:
        pin, pout = os.path.join(tmp, "in.pt"), os.path.join(tmp, "out.pt")
        torch.save(SINGLE, pin)
        env = dict(os.environ, MFVIT_FUSION_BATCHED="0")
        subprocess.run([sys.executable, os.path.abspath(__file__), pin, pout], env=env, cwd=ROOT, check=True,
                       timeout=1800)
        return torch.load(pout)


@pytest.mark.parametrize("i", range(len(SINGLE)), ids=[_id(k) for k in SINGLE])
def test_single_kernel_path_every_record(single_results, i):
    cs = make_case(**SINGLE[i])
    res = {k: (v.cuda() if torch.is_tensor(v) else {kk: tuple(None if t is None else t.cuda() for t in vv)
                                                     for kk, vv in v.items()})
           for k, v in single_results[i].items()}
    got = stored_single(res["saved"], cs["B"], cs["heads"])
    assert_ok(check_run(cs, res, got), "single " + _id(SINGLE[i]))
    # the evaluation forward (no saved buffer) in this process: the same kernel, bit for bit
    fused, x = fwd(cs, None)
    torch.cuda.synchronize()
    assert bits_equal(fused, res["fused"]) and bits_equal(x, res["x"])


if __name__ == "__main__":
    _child(sys.argv[1], sys.argv[2])
