"""Teacher-forced stage checks of the native encoder (mfv_vit_forward / mfv_vit_backward_range), in place.

The real engine runs on NaN-poisoned workspaces: a saving forward, then a backward of one segment per block whose
single-slot buffers are cloned after every segment (vit.cu keeps cur == 0 at a block boundary, so dx16[0] then holds the
gradient of the block's input and dx16[1] that of its mid residual).  Every stage is then recomputed in float64 from the
16-bit / fp32 values its kernel READ - exactly as the previous kernel stored them - and every stored output is compared
element by element against the bound of tests/stage_ref.py.  Rounding never compounds, so the bound is as tight at block
11 as at block 0, and a wrong slot, group, tile or row shows up as a violation at a named stage.

The two intermediates a segment overwrites (the head LayerNorm-backward output, the fc1-dgrad output) are rebuilt by
re-issuing the same calls through mfvit.ops; that the LayerNorm backward and the dgrad GEMM are deterministic is asserted
first.  Besides the per-element bounds: the rebuilt patch matrix, dacc and every gap of the gradient buffer are checked
bit for bit, every slice the backward reports final is bit-identical to the end result, and two forwards on the same
inputs store bit-identical buffers."""
import math
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import e2e_common as E  # noqa: E402
import stage_ref as R  # noqa: E402

pytestmark = pytest.mark.gpu

BF, F16, F32 = torch.bfloat16, torch.float16, torch.float32
# mfv_set_option keys this file switches, with the runtime defaults they are restored to (include/mfvit.h)
DEFAULTS = {"fuse_ln": 1, "patch_tma": 1, "dx32": 0, "rows96": 0, "legacy_attention": 0, "pdl": 1, "side_stream": 1}
FWD_FIELDS = ("patches", "x", "xn", "stats", "qkv", "attn_o", "lse", "u", "gact", "patches_bf", "xn_bf", "attn_o_bf",
              "gact_bf")
SNAP_FIELDS = ("dx0", "dx1", "dx16_0", "dx16_1", "dhid", "dxn", "d_o", "dqkv", "delta")


def _set_option(key, value):
    from mfvit import _lib
    assert _lib.load().mfv_set_option(key.encode(), int(value)) == 0, key


@pytest.fixture(scope="module", autouse=True)
def _exact_reference_math():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield


# ------------------------------------------------------------------------------------------------------- the run
class Run:
    """One saving forward + segmented backward of the real engine, with everything the checks read."""

    def __init__(self, mods, images, seed=0, corrupt=None, backward=True):
        from mfvit import ops
        from mfvit.engine import engine_for
        self.eng = eng = engine_for(*mods)
        dev = images[0].device
        eng.adopt(dev)
        lay = self.lay = eng.layout
        self.G, self.B = eng.G, images[0].shape[0]
        self.images = images
        ws = eng._workspace(self.B, True)
        bwd = ws.ensure_bwd(lay, dev)
        for t in [getattr(ws, f) for f in FWD_FIELDS] + list(bwd.values()):
            if t is not None:
                t.fill_(float("nan"))
        self.f16 = eng.fwd_f16
        tokens, lease = eng.forward(images, save=True)
        assert lease.ws is ws
        first = {f: getattr(ws, f).clone() for f in FWD_FIELDS if getattr(ws, f) is not None}
        tok0 = tokens.clone()
        lease.release()
        tokens, lease = eng.forward(images, save=True)  # same inputs, same workspace: bit-identical buffers
        assert lease.ws is ws
        torch.cuda.synchronize()
        self.nondeterministic = [f for f, t in first.items() if not _bits_equal(t, getattr(ws, f))]
        if not _bits_equal(tok0, tokens):
            self.nondeterministic.append("tokens")
        self.ws, self.tokens = ws, tokens
        if corrupt is not None:
            corrupt(self)
        self.snap, self.final_slices = {}, []
        self.lease = lease
        if not backward:
            lease.release()
            return
        g = torch.Generator(device=dev).manual_seed(seed)
        self.dtokens = torch.randn(tokens.shape, device=dev, generator=g) * 1e-3
        depth = lay.depth

        def on_segment(grad, lo, hi):
            blk = depth - 1 - len(self.snap)
            self.snap[blk] = {k: (bwd[k].clone() if bwd[k] is not None else None) for k in SNAP_FIELDS}
            if ws.gact_bf is not None and not ws.gact_twin:
                self.snap[blk]["gact_bf1"] = ws.gact_bf.clone()  # one slot, recomputed by the fc2-dgrad epilogue
            self.final_slices.append((lo, hi, grad[:, lo:hi].clone()))

        self.grad = eng.backward(lease, self.dtokens, segments=[(b, b) for b in range(depth - 1, -1, -1)],
                                 on_segment=on_segment)
        self.dacc = bwd["dacc"].clone()
        self.ops = ops
        torch.cuda.synchronize()


def _bits_equal(a, b):
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    it = {2: torch.int16, 4: torch.int32, 8: torch.int64}[a.element_size()]
    return torch.equal(a.view(it), b.view(it))


# ---------------------------------------------------------------------------------------------------- the checks
class Report:
    def __init__(self):
        self.rows = []  # (stage, block, group, Result)

    def add(self, stage, block, got, ref, bound):
        """got / ref / bound with the group as their leading dimension."""
        for g in range(got.shape[0]):
            self.rows.append((stage, block, g, R.check(stage, got[g], ref[g] if ref.dim() else ref,
                                                        bound[g] if bound.dim() else bound)))

    def exact(self, stage, block, got, want):
        for g in range(got.shape[0]):
            same = _bits_equal(got[g].contiguous(), want[g].contiguous())
            self.rows.append((stage, block, g, R.Result(stage, 0.0 if same else math.inf, (), 0)))

    def failures(self):
        return [(s, b, g, r) for s, b, g, r in self.rows if not r.ok]

    def summary(self, tag):
        worst = {}
        for s, b, g, r in self.rows:
            if s not in worst or not (r.worst <= worst[s][0]):
                worst[s] = (r.worst, b, g, r.where, r.nonfinite)
        lines = ["[%s] %d checks" % (tag, len(self.rows))]
        for s, (w, b, g, where, nf) in worst.items():
            lines.append("  %-16s worst %.3e  block %-4s group %d at %s%s" % (s, w, b, g, where,
                                                                           "  nonfinite %d" % nf if nf else ""))
        for s, b, g, r in self.failures():
            lines.append("  FAIL %s block %s group %d: %s" % (s, b, g, r.line()))
        print("\n".join(lines), flush=True)


def _param(run, name, src):
    lay, G = run.lay, run.G
    off, shape = lay.offset[name], lay.shape[name]
    n = math.prod(shape)
    return src[:, off:off + n].reshape((G,) + tuple(shape))


def check_forward(run, rep):
    eng, lay, ws, G, B = run.eng, run.lay, run.ws, run.G, run.B
    S, C, H, Hd, depth, npch = lay.S, lay.C, lay.H, lay.hidden, lay.depth, lay.np
    D, M = C // H, B * S
    fdt = F16 if run.f16 else BF
    wsrc = eng.shadow16 if run.f16 else eng.shadow

    def p32(name):
        return _param(run, name, eng.master)

    def w16(name):  # forward GEMM operand: the fp16 (or, all-bf16 forward, bf16) shadow
        return _param(run, name, wsrc)

    x = ws.x.view(-1, G, M, C)
    xn = ws.xn.view(-1, G, M, C).view(fdt)
    xn_bf = ws.xn_bf.view(-1, G, M, C) if run.f16 else None
    stats = ws.stats.view(-1, 2, G, M)
    qkv = ws.qkv.view(depth, G, M, 3 * C).view(fdt)
    ao = ws.attn_o.view(depth, G, M, C).view(fdt)
    ao_bf = ws.attn_o_bf.view(depth, G, M, C) if run.f16 else None
    lse = ws.lse.view(depth, G, B, H, S)
    u = ws.u.view(depth, G, M, Hd)
    gact = ws.gact.view(depth, G, M, Hd).view(fdt)
    gact_bf = ws.gact_bf.view(-1, G, M, Hd) if (run.f16 and ws.gact_twin) else None

    # ---- embedding: x(0) = [cls + pos0 ; im2col(img) W^T + b + pos[1:]]
    cols = torch.stack([R.im2col(im) for im in run.images])                # [G, B, np, 768] fp32
    pe_w = w16("patch_embed.proj.weight").reshape(G, C, 768)
    pos = p32("pos_embed").reshape(G, 1, S, C)
    ref, bnd, _ = R.gemm(cols.to(fdt).reshape(G, B * npch, 768), pe_w, p32("patch_embed.proj.bias"),
                         pos[:, :, 1:].expand(G, B, npch, C).reshape(G, B * npch, C), out_dtype=F32)
    x0 = x[0].view(G, B, S, C)
    rep.add("embed", "-", x0[:, :, 1:].reshape(G, B * npch, C), ref, bnd)
    cls = (p32("cls_token").reshape(G, 1, C) + pos[:, :, 0]).double()                # [G, 1, C]
    rep.add("embed.cls", "-", x0[:, :, 0], cls.expand(G, B, C), 2 * R.U32 * cls.abs().expand(G, B, C))
    if ws.patches is not None and not torch.isnan(ws.patches[:1]).all():  # written by the forward only with patch_tma=0
        rep.exact("patches", "-", ws.patches.view(G, B, npch, 768).view(fdt), cols.to(fdt))
        if run.f16:
            rep.exact("patches_bf", "-", ws.patches_bf.view(G, B, npch, 768), cols.to(BF))

    def ln(stage, blk, i, xin, w, b):
        (rm, mb), (rr, rb) = R.ln_stats(xin)
        rep.add(stage + ".mean", blk, stats[i, 0], rm, mb)
        rep.add(stage + ".rstd", blk, stats[i, 1], rr, rb)
        y, yb = R.ln_fwd(xin, w.unsqueeze(1), b.unsqueeze(1), fdt)
        rep.add(stage + ".y", blk, xn[i], y, yb)
        if xn_bf is not None:
            y, yb = R.ln_fwd(xin, w.unsqueeze(1), b.unsqueeze(1), BF)
            rep.add(stage + ".y_bf", blk, xn_bf[i], y, yb)

    for l in range(depth):
        pre = "blocks.%d." % l
        ln("ln1", l, 2 * l, x[2 * l], p32(pre + "norm1.weight"), p32(pre + "norm1.bias"))
        ref, bnd, _ = R.gemm(xn[2 * l], w16(pre + "attn.qkv.weight"), p32(pre + "attn.qkv.bias"), out_dtype=fdt)
        rep.add("qkv", l, qkv[l], ref, bnd)
        del ref, bnd
        t = qkv[l].view(G, B, S, 3, H, D).permute(3, 0, 1, 4, 2, 5)        # [3, G, B, H, S, D]
        o, ob, ls, lb = R.attn_fwd(t[0], t[1], t[2], D ** -0.5, fdt, fdt)
        rep.add("attn_fwd.o", l, ao[l].view(G, B, S, H, D).transpose(2, 3), o, ob)
        if ao_bf is not None:
            o, ob, _, _ = R.attn_fwd(t[0], t[1], t[2], D ** -0.5, BF, fdt)
            rep.add("attn_fwd.o_bf", l, ao_bf[l].view(G, B, S, H, D).transpose(2, 3), o, ob)
        rep.add("attn_fwd.lse", l, lse[l], ls, lb)
        del o, ob, ls, lb
        ref, bnd, _ = R.gemm(ao[l], w16(pre + "attn.proj.weight"), p32(pre + "attn.proj.bias"), x[2 * l], out_dtype=F32)
        rep.add("proj+res", l, x[2 * l + 1], ref, bnd)
        ln("ln2", l, 2 * l + 1, x[2 * l + 1], p32(pre + "norm2.weight"), p32(pre + "norm2.bias"))
        r_u, bnd, accb = R.gemm(xn[2 * l + 1], w16(pre + "mlp.fc1.weight"), p32(pre + "mlp.fc1.bias"), out_dtype=BF)
        rep.add("fc1.u", l, u[l], r_u, bnd)
        g_ref, g_b = R.gelu_stage(r_u, accb, fdt)
        rep.add("fc1.gelu", l, gact[l], g_ref, g_b)
        if gact_bf is not None:
            g_ref, g_b = R.gelu_stage(r_u, accb, BF)
            rep.add("fc1.gelu_bf", l, gact_bf[l], g_ref, g_b)
        del r_u, bnd, accb, g_ref, g_b
        ref, bnd, _ = R.gemm(gact[l], w16(pre + "mlp.fc2.weight"), p32(pre + "mlp.fc2.bias"), x[2 * l + 1],
                             out_dtype=F32)
        rep.add("fc2+res", l, x[2 * l + 2], ref, bnd)
        del ref, bnd
    last = 2 * depth
    (rm, mb), (rr, rb) = R.ln_stats(x[last])
    rep.add("norm.mean", "-", stats[last, 0], rm, mb)
    rep.add("norm.rstd", "-", stats[last, 1], rr, rb)
    y, yb = R.ln_fwd(x[last], p32("norm.weight").unsqueeze(1), p32("norm.bias").unsqueeze(1), F32)
    rep.add("tokens", "-", run.tokens.view(G, M, C), y, yb)


def check_backward(run, rep, dx32):
    eng, lay, ws, G, B = run.eng, run.lay, run.ws, run.G, run.B
    ops = run.ops
    S, C, H, Hd, depth, npch, P = lay.S, lay.C, lay.H, lay.hidden, lay.depth, lay.np, lay.P
    D, M = C // H, B * S
    fdt = F16 if run.f16 else BF
    grad, snap = run.grad, run.snap
    x = ws.x.view(-1, G, M, C)
    stats = ws.stats.view(-1, 2, G, M)
    xn_b = (ws.xn_bf if run.f16 else ws.xn).view(-1, G, M, C)
    qkv = ws.qkv.view(depth, G, M, 3 * C).view(fdt)
    ao_b = (ws.attn_o_bf if run.f16 else ws.attn_o).view(depth, G, M, C)
    lse = ws.lse.view(depth, G * B, H, S)
    u = ws.u.view(depth, G, M, Hd)

    def p32(name):
        return _param(run, name, eng.master)

    def w16(name):  # backward GEMM operand: the bf16 shadow
        return _param(run, name, eng.shadow)

    def gr(name):
        return _param(run, name, grad)

    def v(t, *shape):
        return t.view(*shape)

    def ln_bwd_issue(dy, xi, st, w, dres, want_f32):
        """The LayerNorm backward exactly as vit.cu issues it, into fresh buffers (no gradient accumulation)."""
        return ops.layernorm_bwd(dy, xi, st[0], st[1], w, dres=dres, want_f32=want_f32)

    # ---- head: final-norm backward, rebuilt (its output is overwritten by block depth-1)
    last = 2 * depth
    dtok = run.dtokens.view(G, M, C)
    head32, head16 = ln_bwd_issue(dtok, x[last], stats[last], p32("norm.weight"), None, True)
    ref, bnd, xh = R.ln_bwd(dtok, x[last], stats[last, 0], stats[last, 1], p32("norm.weight").unsqueeze(1), None, BF)
    rep.add("head_ln_bwd", "-", head16, ref, bnd)
    rep.add("head_ln_bwd32", "-", head32, *R.ln_bwd(dtok, x[last], stats[last, 0], stats[last, 1],
                                                    p32("norm.weight").unsqueeze(1), None, F32)[:2])
    rep.add("dgamma", "norm", gr("norm.weight"), *R.colsum(dtok.double() * xh))
    rep.add("dbeta", "norm", gr("norm.bias"), *R.colsum(dtok))
    del ref, bnd, xh

    for l in range(depth - 1, -1, -1):
        pre = "blocks.%d." % l
        sn = snap[l]
        if l == depth - 1:
            d_in16, d_in32 = head16, head32
        else:
            d_in16, d_in32 = snap[l + 1]["dx16_0"].view(G, M, C), snap[l + 1]["dx0"].view(G, M, C)
        dres_mlp = d_in32 if dx32 else d_in16
        # fc2 bias: column sums of the fp32 dx of the LayerNorm backward that produced this block's output gradient
        src = d_in32 if dx32 else d_in16
        rep.add("bias.fc2", l, gr(pre + "mlp.fc2.bias"), *R.colsum(src, extra_rel=0.0 if dx32 else R.U_BF))
        # ---- MLP half
        dhid = v(sn["dhid"], G, M, Hd)
        ref, bnd = R.dgelu_stage(d_in16, w16(pre + "mlp.fc2.weight"), u[l])
        rep.add("fc2_dgrad.dgelu", l, dhid, ref, bnd)
        del ref, bnd
        if ws.gact_bf is not None and not ws.gact_twin:
            gb = v(sn["gact_bf1"], G, M, Hd)
            ug = R.f64(u[l])
            rep.add("fc2_dgrad.gelu_bf", l, gb, R.gelu(ug), R.U_BF * R.gelu(ug).abs() + R.gelu_recompute_err(ug))
            del ug
        else:
            gb = (ws.gact_bf.view(-1, G, M, Hd)[l] if run.f16 else ws.gact.view(depth, G, M, Hd)[l])
        # fc1 dgrad: dxn of the LayerNorm-2 backward, overwritten later in the segment -> re-issued
        wfc1 = w16(pre + "mlp.fc1.weight")                                   # [G, Hd, C]
        dxn2 = torch.empty(G, M, C, device=dhid.device, dtype=BF)
        off = lay.offset[pre + "mlp.fc1.weight"]
        ops.gemm(dhid, eng.shadow.view(-1)[off:], dxn2, M=M, N=C, K=Hd, G=G, lda=Hd, ldb=C, ldc=C, a_gstride=M * Hd,
                 b_gstride=P, c_gstride=M * C, b_mn=True, epilogue=ops.EPI_BF16)
        ref, bnd, _ = R.gemm(dhid, wfc1.transpose(-1, -2), out_dtype=BF)
        rep.add("fc1_dgrad", l, dxn2, ref, bnd)
        del ref, bnd
        # LayerNorm-2 backward -> gradient of the mid residual
        ref, bnd, xh = R.ln_bwd(dxn2, x[2 * l + 1], stats[2 * l + 1, 0], stats[2 * l + 1, 1],
                                p32(pre + "norm2.weight").unsqueeze(1), dres_mlp, BF)
        rep.add("ln2_bwd", l, v(sn["dx16_1"], G, M, C), ref, bnd)
        if dx32:
            rep.add("ln2_bwd32", l, v(sn["dx1"], G, M, C), *R.ln_bwd(
                dxn2, x[2 * l + 1], stats[2 * l + 1, 0], stats[2 * l + 1, 1], p32(pre + "norm2.weight").unsqueeze(1),
                dres_mlp, F32)[:2])
        rep.add("dgamma", l, gr(pre + "norm2.weight"), *R.colsum(R.f64(dxn2) * xh))
        rep.add("dbeta", l, gr(pre + "norm2.bias"), *R.colsum(dxn2))
        del ref, bnd, xh
        mid16 = v(sn["dx16_1"], G, M, C)
        mid = v(sn["dx1"], G, M, C) if dx32 else mid16
        rep.add("bias.proj", l, gr(pre + "attn.proj.bias"), *R.colsum(mid, extra_rel=0.0 if dx32 else R.U_BF))
        # MLP weight gradients
        rep.add("wgrad.fc2", l, gr(pre + "mlp.fc2.weight"), *R.wgrad(d_in16, gb))
        rep.add("wgrad.fc1", l, gr(pre + "mlp.fc1.weight"), *R.wgrad(dhid, xn_b[2 * l + 1]))
        rep.add("bias.fc1", l, gr(pre + "mlp.fc1.bias"), *R.colsum(dhid))
        # ---- attention half
        d_o = v(sn["d_o"], G, M, C)
        ref, bnd, _ = R.gemm(mid16, w16(pre + "attn.proj.weight").transpose(-1, -2), out_dtype=BF)
        rep.add("proj_dgrad", l, d_o, ref, bnd)
        del ref, bnd
        t = qkv[l].view(G * B, S, 3, H, D).permute(2, 0, 3, 1, 4).to(BF)   # [3, NB, H, S, D] (bf16, as the kernel)
        oo = ao_b[l].view(G * B, S, H, D).transpose(1, 2)
        dd = d_o.view(G * B, S, H, D).transpose(1, 2)
        refs, bnds, (dl, dlb) = R.attn_bwd(t[0], t[1], t[2], oo, dd, lse[l], D ** -0.5)
        dqkv = v(sn["dqkv"], G * B, S, 3, H, D).permute(2, 0, 3, 1, 4)
        for i, nm in enumerate(("dq", "dk", "dv")):
            rep.add("attn_bwd." + nm, l, dqkv[i].reshape(G, B, H, S, D), refs[i].reshape(G, B, H, S, D),
                    bnds[i].reshape(G, B, H, S, D))
        if not torch.isnan(sn["delta"]).all():  # stored only by the kernels that take delta from a separate pass
            rep.add("attn_bwd.delta", l, v(sn["delta"], G, B, H, S), dl.reshape(G, B, H, S), dlb.reshape(G, B, H, S))
        del refs, bnds, dl, dlb, t
        dqkv = v(sn["dqkv"], G, M, 3 * C)
        dxn1 = v(sn["dxn"], G, M, C)
        ref, bnd, _ = R.gemm(dqkv, w16(pre + "attn.qkv.weight").transpose(-1, -2), out_dtype=BF)
        rep.add("qkv_dgrad", l, dxn1, ref, bnd)
        del ref, bnd
        # determinism of the re-issued kernels: the qkv dgrad and this block's LayerNorm-1 backward
        again = torch.empty_like(dxn1)
        off = lay.offset[pre + "attn.qkv.weight"]
        ops.gemm(dqkv, eng.shadow.view(-1)[off:], again, M=M, N=C, K=3 * C, G=G, lda=3 * C, ldb=C, ldc=C,
                 a_gstride=M * 3 * C, b_gstride=P, c_gstride=M * C, b_mn=True, epilogue=ops.EPI_BF16)
        rep.exact("reissue.qkv_dgrad", l, again, dxn1)
        a32, a16 = ln_bwd_issue(dxn1, x[2 * l], stats[2 * l], p32(pre + "norm1.weight"), mid, True)
        rep.exact("reissue.ln1_bwd", l, a16, v(sn["dx16_0"], G, M, C))
        if l == depth - 1:
            b32, b16 = ln_bwd_issue(dtok, x[last], stats[last], p32("norm.weight"), None, True)
            rep.exact("reissue.head_ln_bwd", "-", b16, head16)
        ref, bnd, xh = R.ln_bwd(dxn1, x[2 * l], stats[2 * l, 0], stats[2 * l, 1], p32(pre + "norm1.weight").unsqueeze(1),
                                mid, BF)
        rep.add("ln1_bwd", l, v(sn["dx16_0"], G, M, C), ref, bnd)
        if dx32 or l == 0:
            rep.add("ln1_bwd32", l, v(sn["dx0"], G, M, C), *R.ln_bwd(
                dxn1, x[2 * l], stats[2 * l, 0], stats[2 * l, 1], p32(pre + "norm1.weight").unsqueeze(1), mid, F32)[:2])
        rep.add("dgamma", l, gr(pre + "norm1.weight"), *R.colsum(R.f64(dxn1) * xh))
        rep.add("dbeta", l, gr(pre + "norm1.bias"), *R.colsum(dxn1))
        del ref, bnd, xh
        rep.add("wgrad.proj", l, gr(pre + "attn.proj.weight"), *R.wgrad(mid16, ao_b[l]))
        rep.add("wgrad.qkv", l, gr(pre + "attn.qkv.weight"), *R.wgrad(dqkv, xn_b[2 * l]))
        rep.add("bias.qkv", l, gr(pre + "attn.qkv.bias"), *R.colsum(dqkv))

    # ---- tail: embedding backward
    dx0 = v(snap[0]["dx0"], G, B, S, C)
    dacc = run.dacc.view(G, B, npch, C)
    rep.exact("dacc", "-", dacc, dx0[:, :, 1:].to(BF))
    rep.add("grad.cls", "-", gr("cls_token").reshape(G, C), *R.colsum(dx0[:, :, 0]))
    frozen_conv = not run.eng._params[0][2][1].requires_grad
    if not frozen_conv:
        rep.add("grad.pe_bias", "-", gr("patch_embed.proj.bias"), *R.colsum(dacc.reshape(G, B * npch, C)))
        cols = torch.stack([R.im2col(im) for im in run.images]).to(BF)       # [G, B, np, 768]
        pb = (ws.patches_bf if run.f16 else ws.patches).view(G, B, npch, 768)
        rep.exact("patches_bf(bwd)", "-", pb, cols)
        rep.add("wgrad.pe", "-", gr("patch_embed.proj.weight").reshape(G, C, 768),
                *R.wgrad(dacc.reshape(G, B * npch, C), pb.reshape(G, B * npch, 768)))
    # ---- the gradient buffer: gaps, the frozen pos_embed (and conv) ranges exactly 0
    live = torch.zeros(P, dtype=torch.bool, device=grad.device)
    for name, shape, off in lay.entries:
        if name == "pos_embed" or (frozen_conv and name.startswith("patch_embed.")):
            continue
        live[off:off + math.prod(shape)] = True
    rep.exact("grad.gaps+frozen", "-", torch.where(live, torch.zeros((), device=grad.device), grad),
              torch.zeros_like(grad))
    # ---- every slice reported final is final
    for lo, hi, sl in run.final_slices:
        rep.exact("grad.final_slice", "%d:%d" % (lo, hi), sl, grad[:, lo:hi])


def _run_and_check(tag, mods, images, dx32=False, seed=0):
    run = Run(mods, images, seed=seed)
    rep = Report()
    for f in run.nondeterministic:
        rep.rows.append(("fwd_repeat." + f, "-", 0, R.Result(f, math.inf, (), 0)))
    with torch.no_grad():
        check_forward(run, rep)
        check_backward(run, rep, dx32)
    rep.summary(tag)
    bad = rep.failures()
    assert not bad, ["%s block %s group %d: %s" % (s, b, g, r.line()) for s, b, g, r in bad[:20]]
    return rep


def _pair(B, img=224, seed=0):
    _, (o_f, o_c, o_e) = E.build_mfvit_pair(img_size=img, seed=seed)
    img_c, img_e, _ = E.synthetic_pair(B, img, rank=seed, device="cuda")
    return (o_c, o_e), [img_c, img_e]


# ------------------------------------------------------------------------------------------------------ the tests
@pytest.mark.parametrize("B", [1, 7, 32])
def test_stages_default_path(B):
    """G = 2 (the two MF-ViT backbones, distinct weights), M = 197 (one partial pair tile), 1 379 (ragged), 6 304 (bench)."""
    mods, images = _pair(B, seed=B)
    _run_and_check("default B=%d" % B, mods, images, seed=B)


def test_stages_384px():
    """S = 577: the flash forward across key blocks, the key-block attention backward with its fp32 dQ workspace."""
    mods, images = _pair(2, img=384, seed=3)
    _run_and_check("384px B=2", mods, images)


def test_stages_12_heads_single_group():
    """D = 32 (the mma.sync attention kernels), G = 1."""
    _, ours = E.build_vit_pair(num_heads=12, seed=5)
    img, _, _ = E.synthetic_pair(7, 224, device="cuda")
    _run_and_check("12 heads G=1 B=7", (ours,), [img])


def test_stages_wide_scores():
    """q / k rows of blocks 3 and 7 scaled x8: scores spread far beyond 2^8 between key blocks, so the forward's lazy
    reference maximum moves (O rescaled) inside a row."""
    mods, images = _pair(7, seed=9)
    with torch.no_grad():
        for m in mods:
            for i in (3, 7):
                m.blocks[i].attn.qkv.weight[:2 * m.embed_dim].mul_(8.0)
    _run_and_check("wide scores B=7", mods, images)


def test_stages_bf16_forward():
    mods, images = _pair(7, seed=11)
    from mfvit.engine import engine_for
    eng = engine_for(*mods)
    eng.fwd_f16 = False
    eng.invalidate_shadow()
    _run_and_check("bf16 forward B=7", mods, images)


@pytest.mark.parametrize("opts", [{"fuse_ln": 0}, {"patch_tma": 0}, {"dx32": 1}, {"rows96": 1},
                                  {"legacy_attention": 1}, {"pdl": 0, "side_stream": 0}],
                         ids=lambda o: "+".join("%s=%d" % kv for kv in o.items()))
def test_stages_runtime_options(opts):
    mods, images = _pair(7, seed=13)
    try:
        for k, val in opts.items():
            _set_option(k, val)
        _run_and_check("options %s B=7" % opts, mods, images, dx32=bool(opts.get("dx32", 0)))
    finally:
        for k in opts:
            _set_option(k, DEFAULTS[k])


def test_stages_gelu_recomputed_in_the_fc2_dgrad(monkeypatch):
    """MFVIT_GELU_TWIN=0: one bf16 gelu(u) slot that the fc2-dgrad epilogue rewrites per block (read when the workspace
    is created)."""
    monkeypatch.setenv("MFVIT_GELU_TWIN", "0")
    mods, images = _pair(7, seed=15)
    _run_and_check("gelu twin=0 B=7", mods, images)


def test_stages_stop_grad_conv1():
    mods, images = _pair(7, seed=17)
    for m in mods:
        m.patch_embed.proj.weight.requires_grad = False
        m.patch_embed.proj.bias.requires_grad = False
    _run_and_check("stop_grad_conv1 B=7", mods, images)


def test_a_corrupted_qkv_element_is_reported_at_its_stage_only():
    """One element of block 5's stored qkv (group 1) changed after the forward: the qkv GEMM check of block 5 sees its
    output changed and the attention-forward check of block 5 sees an input its outputs do not match; nothing upstream
    and nothing in group 0 may move."""
    mods, images = _pair(1, seed=19)
    lay_C, H = mods[0].embed_dim, mods[0].num_heads

    def corrupt(run):
        M = run.B * run.lay.S
        q = run.ws.qkv.view(run.lay.depth, run.G, M, 3 * lay_C)
        fdt = F16 if run.f16 else BF
        e = q[5, 1].view(fdt)
        e[40, lay_C + 2 * (lay_C // H) + 7] += 4.0  # a key element of token 40, head 2

    run = Run(mods, images, corrupt=corrupt, backward=False)
    rep = Report()
    with torch.no_grad():
        check_forward(run, rep)
    rep.summary("corrupted qkv[5] group 1")
    bad = {(s.split(".")[0], b, g) for s, b, g, r in rep.failures()}
    assert ("attn_fwd", 5, 1) in bad, bad
    assert bad <= {("attn_fwd", 5, 1), ("qkv", 5, 1)}, bad
