"""GPU: the fused LARS step (mfv_lars_step_dev, moco/optimizer.py:10-43) against a float64 replay, its determinism and
CUDA-graph capture, and MoCoPretrainer(optimizer='lars' | 'adam') against the reference loop body (MAIN_PRE:510-548).

Per-element bound of one step (derived from the formats; every step is replayed in float64 from the fp32 state the
kernel read, with the fp32 values of lr, weight decay, momentum and eta the kernel used):
  q      : |q - q64| <= q64 * Q_REL(n).  A norm^2 is a fp32 sum of non-negative terms in a fixed tree of depth
           D(n) = 32 (serial FMAs per lane) + 10 (lanes, warp, CTA) + ceil(chunks / 256) + 8 (chunk partials): relative
           error <= D u.  dp^2 adds 2u (dp = fma(wd, p, g) is rounded), each square root halves and adds u, eta * ||p||
           and the division add u each: (D + 5) u to first order, Q_REL = (D + 8) u with room for the products.
  mu     : x = q dp, mu64 = momentum mu + x;  |mu - mu64| <= |x| (Q_REL + 3u) + u |mu64|  (x = fl(fl(dp) q) is off by
           Q_REL + 2u relative, then one fma rounding).  Vectors: Q_REL = 0 (q = 1 and dp = g are exact).
  p      : p64 = p - lr mu64;  |p - p64| <= lr B_mu (1 + u) + u |p64|  (one fma rounding).
u = 2^-24.  Shadows: bit-identical to the round-to-nearest casts of the new fp32 master."""
import importlib
import math
import os
import sys
from functools import partial
from types import SimpleNamespace

import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import e2e_common as E  # noqa: E402
import stage_ref as R  # noqa: E402

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
LANE_TERMS = 32768 // (4 * 256)     # MFV_LARS_CHUNK / (float4 x 256 threads)
MOM, ETA, WD = 0.9, 0.001, 0.1
LRS = (0.6, 2.4, 0.15)               # one learning rate per step, read from lr_dev


def f32(x):
    return float(torch.tensor(x, dtype=torch.float32))


def depth(n):
    chunks = -(-n // 32768)
    return LANE_TERMS + 10 + -(-chunks // 256) + 8


def q_rel(n):
    return (depth(n) + 8) * U


# --------------------------------------------------------------------------------------------------- the test table
SMALL = [  # projector (base_encoder.head) and predictor of MoCo_ViT(dim 256, mlp_dim 4096), then the edge cases
    ("proj.0.weight", (4096, 384)), ("proj.1.weight", (4096,)), ("proj.1.bias", (4096,)),
    ("proj.3.weight", (4096, 4096)), ("proj.4.weight", (4096,)), ("proj.4.bias", (4096,)),
    ("proj.6.weight", (256, 4096)),
    ("pred.0.weight", (4096, 256)), ("pred.1.weight", (4096,)), ("pred.1.bias", (4096,)), ("pred.3.weight", (256, 4096)),
    ("odd_matrix", (7, 143)), ("odd_vector", (13,)), ("zero_weight", (3, 5)), ("zero_update", (2, 6)),
    ("cls_like", (1, 1, 5)), ("vector6", (6,)),
]
FROZEN = ("pos_embed", "patch_embed.proj.weight", "patch_embed.proj.bias")  # fixed table; stop_grad_conv1


class Case:
    """An encoder layout's flat buffers (gaps and frozen tensors included) plus a packed buffer of SMALL, 4-aligned."""

    def __init__(self, seed=0, device="cuda"):
        from mfvit.engine import ViTLayout
        gen = torch.Generator().manual_seed(seed)
        lay = ViTLayout(224, 16, 384, 12, 6, 1536)
        self.tensors = []   # (name, shape, which, off)
        for name, shape, off in lay.entries:
            if name not in FROZEN:
                self.tensors.append((name, shape, "enc", off))
        off = 0
        for name, shape in SMALL:
            self.tensors.append((name, shape, "sm", off))
            off += (math.prod(shape) + 3) // 4 * 4
        n = {"enc": lay.P, "sm": off}
        self.buf = {}
        for w in ("enc", "sm"):
            p = torch.randn(n[w], generator=gen) * 0.02
            g = torch.randn(n[w], generator=gen) * 1e-3
            self.buf[w] = dict(p=p.to(device), g=g.to(device), mu=torch.zeros(n[w], device=device),
                               sb=torch.full((n[w],), -7.0, device=device, dtype=torch.bfloat16),
                               sh=torch.full((n[w],), -7.0, device=device, dtype=torch.float16))
        wd = f32(WD)
        for name, shape, w, o in self.tensors:
            k = math.prod(shape)
            b = self.buf[w]
            if name == "zero_weight":
                b["p"][o:o + k] = 0.0
            if name == "zero_update":  # powers of two: wd * p is exact in fp32, so g + wd * p == 0 exactly
                pv = torch.tensor([0.5, -1.0, 2.0, -0.25, 1.0, 4.0] * 2, device=device)
                b["p"][o:o + k] = pv
                b["g"][o:o + k] = -(pv * wd)
        self.mask = {w: torch.zeros(n[w], dtype=torch.bool, device=device) for w in ("enc", "sm")}
        for name, shape, w, o in self.tensors:
            self.mask[w][o:o + math.prod(shape)] = True

    def records(self):
        out = []
        for name, shape, w, o in self.tensors:
            sl = slice(o, o + math.prod(shape))
            b = self.buf[w]
            out.append((b["p"][sl], b["g"][sl], b["mu"][sl], b["sb"][sl], b["sh"][sl], len(shape) > 1))
        return out

    def state(self):
        return {w: {k: v.clone() for k, v in b.items()} for w, b in self.buf.items()}

    def load(self, st):
        for w, b in self.buf.items():
            for k, v in b.items():
                v.copy_(st[w][k])


def replay_check(name, p0, g, mu0, p_got, mu_got, q_got, lr, wd, mom, eta):
    """One LARS step replayed in float64 from the fp32 state (p0, g, mu0) the kernel read, against what it wrote
    (p_got, mu_got, trust ratio q_got), with the bounds of the module docstring.  Returns [(key, stage_ref.Result)]."""
    from oracle import lars_ref
    p64, mu64 = p0.double().clone(), mu0.double().clone()
    q64 = float(lars_ref.lars_update_(p64, g.double(), mu64, lr, wd, mom, eta))
    qr = q_rel(p0.numel()) if p0.dim() > 1 and q64 != 1.0 else 0.0
    x = (mu64 - mom * mu0.double()).abs()
    b_mu = x * (qr + 3 * U) + U * mu64.abs()
    b_p = lr * b_mu * (1 + U) + U * p64.abs()
    rq = abs(q_got - q64) / (q64 * qr) if qr > 0 else (0.0 if q_got == q64 else math.inf)
    return [("mu", R.check(name, mu_got, mu64, b_mu)), ("p", R.check(name, p_got, p64, b_p)),
            ("q", R.Result(name, rq, (), 0))]


def _lars(case, table, ws, lr_dev, q):
    from mfvit import ops
    tab, nt, nc = table
    ops.lars_step_dev_(tab, nt, nc, ws, lr_dev, MOM, WD, ETA, q_out=q)


def _prepare(case):
    from mfvit import ops
    table = ops.make_lars_table(case.records(), torch.device("cuda"))
    ws = ops.lars_workspace(table[2], torch.device("cuda"))
    q = torch.full((table[1],), float("nan"), device="cuda")
    return table, ws, q


def test_lars_op_matches_the_fp64_replay_per_element():
    case = Case(seed=1)
    table, ws, q = _prepare(case)
    lr_dev = torch.zeros(1, device="cuda")
    wd, mom, eta = f32(WD), f32(MOM), f32(ETA)
    worst = {"p": (0.0, ""), "mu": (0.0, ""), "q": (0.0, "")}
    before0 = case.state()
    for step, lr in enumerate(LRS):
        lr_dev.fill_(lr)
        lr32 = float(lr_dev)
        before = case.state()
        _lars(case, table, ws, lr_dev, q)
        torch.cuda.synchronize()
        for i, (name, shape, w, o) in enumerate(case.tensors):
            k = math.prod(shape)
            sl = slice(o, o + k)
            got_q = float(q[i])
            trust = len(shape) > 1
            for key, res in replay_check(name, before[w]["p"][sl].view(shape), before[w]["g"][sl].view(shape),
                                         before[w]["mu"][sl].view(shape), case.buf[w]["p"][sl].view(shape),
                                         case.buf[w]["mu"][sl].view(shape), got_q, lr32, wd, mom, eta):
                if not res.ok:
                    pytest.fail("step %d %s %s: %s" % (step, key, name, res.line()))
                if res.worst > worst[key][0]:
                    worst[key] = (res.worst, "%s (step %d)" % (name, step))
            if (name == "zero_weight" and step == 0) or name == "zero_update" or not trust:
                assert got_q == 1.0, (name, step, got_q)
        for w, b in case.buf.items():
            m = case.mask[w]
            assert torch.equal(b["sb"][m], b["p"][m].to(torch.bfloat16)), "bf16 shadow (%s, step %d)" % (w, step)
            assert torch.equal(b["sh"][m], b["p"][m].to(torch.float16)), "fp16 shadow (%s, step %d)" % (w, step)
            for key in ("p", "mu", "sb", "sh", "g"):  # gaps, pos_embed, the frozen conv: not one bit changed
                assert torch.equal(b[key][~m], before0[w][key][~m]), "%s outside the table (%s, step %d)" % (key, w, step)
    print("LARS op vs fp64 replay, worst |err| / bound over 3 steps:",
          {k: "%.3f at %s" % v for k, v in worst.items()})
    assert int(case.mask["enc"].sum()) + int(case.mask["sm"].sum()) > 42_800_000  # the whole ViT-S MoCo trainable set


def test_lars_op_is_deterministic_and_capturable():
    case = Case(seed=2)
    table, ws, q = _prepare(case)
    lr_dev = torch.zeros(1, device="cuda")
    s0 = case.state()

    def run_eager():
        case.load(s0)
        qs = []
        for lr in LRS:
            lr_dev.fill_(lr)
            _lars(case, table, ws, lr_dev, q)
            qs.append(q.clone())
        torch.cuda.synchronize()
        return case.state(), qs

    a, qa = run_eager()
    b, qb = run_eager()
    for w in a:
        for k in a[w]:
            assert torch.equal(a[w][k], b[w][k]), (w, k)
    assert all(torch.equal(x, y) for x, y in zip(qa, qb))
    # capture once, replay with the learning rate changed between replays
    case.load(s0)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        _lars(case, table, ws, lr_dev, q)
    torch.cuda.synchronize()
    for w in s0:  # capturing executes nothing
        assert torch.equal(case.buf[w]["p"], s0[w]["p"]) and torch.equal(case.buf[w]["mu"], s0[w]["mu"])
    qg = []
    for lr in LRS:
        lr_dev.fill_(lr)
        graph.replay()
        qg.append(q.clone())
    torch.cuda.synchronize()
    for w in a:
        for k in a[w]:
            assert torch.equal(case.buf[w][k], a[w][k]), ("graph", w, k)
    assert all(torch.equal(x, y) for x, y in zip(qa, qg))


def test_lars_table_rejects_misaligned_and_mismatched_tensors():
    from mfvit import MfvError, ops
    x = torch.zeros(64, device="cuda")
    with pytest.raises(MfvError, match="16-byte"):
        ops.make_lars_table([(x[1:9], x[16:24], x[32:40], None, None, True)], torch.device("cuda"))
    s = torch.zeros(64, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(MfvError, match="8-byte"):
        ops.make_lars_table([(x[0:8], x[16:24], x[32:40], s[2:10], None, True)], torch.device("cuda"))
    with pytest.raises(MfvError, match="contiguous"):
        ops.make_lars_table([(x[0:8], x[16:20], x[32:40], None, None, True)], torch.device("cuda"))


# --------------------------------------------------------------------------------------------------- the pretrainer
def _moco_pair(T=0.2):
    import vits
    from oracle import moco_ref, vit_ref
    bm = importlib.import_module("moco.builder_vit_mocov3structure_mocov2loss")
    torch.manual_seed(0)
    ours = bm.MoCo_ViT(partial(vits.vit_small, stop_grad_conv1=True), SimpleNamespace(arch="vit_small"), 256, 4096, T)
    with torch.no_grad():
        for p in ours.base_encoder.parameters():
            p.add_(torch.randn_like(p) * 0.01)
    ref = moco_ref.MoCoViT(partial(vit_ref.vit_small, stop_grad_conv1=True), 256, 4096, T)
    ref.load_state_dict(ours.state_dict(), strict=True)
    return ref.cuda().train(), ours.cuda().train()


@pytest.mark.parametrize("optimizer", ["lars", "adam"])
def test_pretrain_step_with_lars_or_adam_follows_the_reference_loop_body(optimizer):
    """MAIN_PRE:510-548 over the oracle model (fp16 autocast + GradScaler, oracle LARS or torch.optim.Adam, cosine lr
    with warm-up, cosine momentum) against MoCoPretrainer(optimizer=...) over the drop-in.  LARS runs with MoCo-v3's
    weight decay of 1e-6, so every matrix moves along its gradient rather than along -p.

    The two paths compute their gradients differently (the oracle under fp16 autocast, the kernels with fp16 forward /
    bf16 backward operands), so their per-tensor gradients agree to a cosine of about 0.98-0.999 at this batch, not
    exactly.  The LARS checks therefore separate the optimizer from the gradients: (1) the last step of the pretrainer is
    replayed in float64 from its own state (parameters, gradients, momentum, learning rate) and must match per element
    within the op's bound - the table covers the right tensors, nothing else moves; (2) the movement of every matrix
    follows the reference loop as closely as the gradients that drive it do: its cosine is at least the worst per-step
    gradient cosine of that matrix minus 0.005 (the trust ratios weight the steps slightly differently)."""
    import moco_dp_common as M
    from mfvit import _lib
    from mfvit import schedules as S
    from mfvit.pretrain import MoCoPretrainer
    from oracle import lars_ref
    ref, ours = _moco_pair()
    B, epochs, warm, iters = 32, 100, 10, 4
    if optimizer == "lars":
        lr0, wd = S.base_lr(0.6, 16), 1e-6                                # lr 0.6 at batch 16 -> 2.4
        opt = lars_ref.LARS(ref.parameters(), lr0, weight_decay=wd)        # MAIN_PRE:340-342
    else:
        lr0, wd = S.base_lr(1.5e-4, 16), 0.1
        opt = torch.optim.Adam(ref.parameters(), lr0, weight_decay=wd)     # MAIN_PRE:343-345
    scaler = torch.amp.GradScaler("cuda")
    pre = MoCoPretrainer(ours, lr=lr0, weight_decay=wd, epochs=epochs, warmup_epochs=warm, moco_m=0.99,
                         optimizer=optimizer)
    names = {id(p): n for n, p in ours.named_parameters()}
    ref_params = dict(ref.named_parameters())
    mats = [n for n, p in ours.named_parameters() if p.requires_grad and p.dim() > 1]
    start = {n: p.detach().clone() for n, p in ours.named_parameters() if p.requires_grad}
    gcos = {n: 1.0 for n in mats}
    losses = []
    lib = _lib.load()
    for i in range(3):
        im_q, im_k = M.structured_views(B, 224, i, "cuda")
        ep = 2 + i / iters
        for g in opt.param_groups:
            g["lr"] = S.pretrain_lr(ep, lr0, epochs, warm)
        with torch.autocast("cuda", dtype=torch.float16):
            out, tgt = ref(im_q, im_k, S.moco_momentum(ep, epochs, 0.99))
            loss_r = F.cross_entropy(out, tgt)
        opt.zero_grad()
        scaler.scale(loss_r).backward()
        scaler.step(opt)                                                   # unscales the .grad tensors in place
        scaler.update()
        if i == 2 and optimizer == "lars":  # the state the last LARS step reads
            before = {id(p): p.detach().clone() for p in ours.parameters()}
            mu_before = (pre._mu_e.clone(), pre._mu_s.clone())
        n0 = lib.mfv_launch_count()
        loss_o = pre.step(im_q, im_k, ep)
        launches = lib.mfv_launch_count() - n0
        losses.append((float(loss_r), float(loss_o)))
        for n in mats:
            gcos[n] = min(gcos[n], E.cos(ours.get_parameter(n).grad, ref_params[n].grad))
    print("%s: pretrain losses (reference loop over oracle, MoCoPretrainer over drop-in): %s; GradScaler scale %.0f; "
          "%d libmfvit launches in the last step" % (optimizer, losses, scaler.get_scale(), launches))
    assert scaler.get_scale() == 65536.0, "the reference skipped a step (fp16 overflow): the comparison is void"
    for a, b in losses:
        assert abs(a - b) <= 2e-2 * max(1.0, abs(a)), losses
    moved = {n: p.detach() - start[n] for n, p in ours.named_parameters() if p.requires_grad}
    moved_r = {n: p.detach() - start[n] for n, p in ref.named_parameters() if p.requires_grad}
    if optimizer == "adam":
        assert int(pre._step_dev) == 3
        big = [n for n in moved if moved_r[n].numel() >= 384 * 384]
        cs = [E.cos(moved[n], moved_r[n]) for n in big]
        print("adam: parameter movement cosine after 3 steps: min %.4f" % min(cs))
        assert min(cs) >= 0.9, sorted(zip(cs, big))[:3]
        return
    # (1) the last step, replayed in float64 from the pretrainer's own state, tensor by tensor in table order
    eng, sm = pre.engine, pre._small
    lr32, wd32, mom32, eta32 = float(pre._lr_dev), f32(wd), f32(0.9), f32(ETA)
    worst = {"p": (0.0, ""), "mu": (0.0, ""), "q": (0.0, "")}
    for p, qo in zip(pre.lars_params, pre.lars_q.tolist()):
        n = names[id(p)]
        base, mu_all = ((eng.master, mu_before[0]) if id(p) in {id(t) for _, t in eng._params[0]}
                        else (sm.master, mu_before[1]))
        off = (p.data_ptr() - base.data_ptr()) // 4
        mu_now = (pre._mu_e if base is eng.master else pre._mu_s).view(-1)[off:off + p.numel()].view(p.shape)
        mu0 = mu_all.view(-1)[off:off + p.numel()].view(p.shape)
        for key, res in replay_check(n, before[id(p)], p.grad.detach(), mu0, p.detach(), mu_now, qo, lr32, wd32, mom32,
                                     eta32):
            assert res.ok, "last step, %s: %s" % (key, res.line())
            if res.worst > worst[key][0]:
                worst[key] = (res.worst, n)
        if p.dim() <= 1:
            assert qo == 1.0, n
    assert len(pre.lars_params) == sum(1 for p in ours.parameters() if p.requires_grad)
    for n, p in ours.base_encoder.named_parameters():  # pos_embed and the stop_grad_conv1 conv did not move
        if not p.requires_grad:
            assert torch.equal(p.detach(), before[id(p)]), n
    # (2) against the reference loop
    rel = []
    for p, qo in zip(pre.lars_params, pre.lars_q.tolist()):
        if p.dim() > 1:
            qr = float(opt.state[ref_params[names[id(p)]]]["q"])
            rel.append((abs(qo - qr) / qr, names[id(p)]))
    rel.sort()
    cs = sorted((E.cos(moved[n], moved_r[n]) - gcos[n], E.cos(moved[n], moved_r[n]), gcos[n], n) for n in mats)
    print("lars: last step vs its fp64 replay, worst |err| / bound: %s" % {k: "%.3f at %s" % v for k, v in worst.items()})
    print("lars: trust ratios vs the reference loop, median relative difference %.2e, worst %s"
          % (rel[len(rel) // 2][0], [("%.2e" % r, n) for r, n in rel[-3:]]))
    print("lars: movement cosine after 3 steps minus the worst gradient cosine of the same matrix, lowest three:",
          [("%+.4f" % d, "%.4f" % c, "%.4f" % g, n) for d, c, g, n in cs[:3]])
    assert cs[0][0] >= -0.005, cs[:3]
