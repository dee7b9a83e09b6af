"""Fused LARS step (mfv_lars_step_dev) over the whole MoCo ViT-S trainable set, against a device-to-device copy of the
same byte count, the fused AdamW step on the same set and the eager LARS the reference runs (oracle/lars_ref.py, one
ATen launch sequence per tensor); then whole MoCoPretrainer steps at 128 images x 2 views, K = 65 536, with 'lars'
and 'adamw' alternated.  Prints one JSON line.   usage: python tests/gpu_lars_bench.py [--reps 50] [--steps 10]

Algorithmic bytes of one LARS step: the norm pass reads p and g of every matrix (8 B), the update pass reads p, g, mu
and writes p, mu (20 B) of every tensor, and rewrites the encoder's two 16-bit shadows (4 B).  The 0.7 GB working set
is several times the 126 MB L2, so every pass streams from HBM."""
import argparse
import json
import os
import subprocess
import sys
from functools import partial
from types import SimpleNamespace

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "multi-feature-vit_b200"), os.path.join(ROOT, "multi-feature-vit_b200", "dropin"),
          os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return name, out or "unknown"


def device_ms(fn, reps):
    """Device time per call: `reps` calls captured in one CUDA graph (no Python time between kernels), best of 3."""
    fn()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(3):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        g.replay()
        b.record()
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b) / reps)
    return best


def wall_ms(fn, reps):
    """Eager calls, events around the whole run (host launch time included, as the reference pays it)."""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--steps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gpu_lars_bench.py measures on a CUDA device; none is present")
    import importlib

    import moco_dp_common as M
    import vits
    from mfvit import ops
    from mfvit.pretrain import MoCoPretrainer
    from oracle import lars_ref
    torch.backends.cuda.matmul.allow_tf32 = False
    bm = importlib.import_module("moco.builder_vit_mocov3structure_mocov2loss")
    dev = torch.device("cuda", 0)

    def model(seed):
        torch.manual_seed(seed)
        return bm.MoCo_ViT(partial(vits.vit_small, stop_grad_conv1=True), SimpleNamespace(arch="vit_small"), 256, 4096,
                           0.2).to(dev).train()

    B = 128
    im_q, im_k = M.structured_views(B, 224, 0, dev)
    pres = {"lars": MoCoPretrainer(model(0), lr=2.4, weight_decay=1e-6, epochs=100, warmup_epochs=10,
                                   optimizer="lars"),
            "adamw": MoCoPretrainer(model(0), lr=6e-4, weight_decay=0.1, epochs=100, warmup_epochs=10)}
    for pre in pres.values():
        pre.step(im_q, im_k, 2.0)
    torch.cuda.synchronize()

    # ---- the optimizer steps alone, over the set the pretrainer steps
    pl = pres["lars"]
    eng = pl.engine
    grad = eng.grads[eng.grad_idx]
    table = pl._lars_table(grad)
    enc_ids = {id(p) for _, p in eng._params[0]}
    n_all = sum(p.numel() for p in pl.lars_params)
    n_mat = sum(p.numel() for p in pl.lars_params if p.dim() > 1)
    n_enc = sum(p.numel() for p in pl.lars_params if id(p) in enc_ids)
    shadow_b = 4 if eng.fwd_f16 else 2
    nbytes = 8 * n_mat + 20 * n_all + shadow_b * n_enc
    lars_ms = device_ms(lambda: ops.lars_step_dev_(table[0], table[1], table[2], pl._lars_ws, pl._lr_dev, 0.9, 1e-6,
                                                   0.001, q_out=pl.lars_q), args.reps)
    src = torch.empty(nbytes // 2, device=dev, dtype=torch.uint8)
    dst = torch.empty_like(src)
    copy_ms = wall_ms(lambda: dst.copy_(src), args.reps)  # eager: a graph's memcpy node may go to a copy engine
    del src, dst

    pa = pres["adamw"]
    ea = pa.engine
    ga = ea.grads[ea.grad_idx]

    def adamw():
        pa._step_dev.add_(1)
        for lo, hi in pa._runs:
            sl = slice(lo, hi)
            ops.adam_step_dev_(ea.master[0, sl], ga[0, sl], pa._m1_e[0, sl], pa._m2_e[0, sl], ea.shadow[0, sl],
                               pa._lr_dev, pa.betas, pa.eps, pa.wd, True, pa._step_dev,
                               shadow16=ea.shadow16[0, sl] if ea.fwd_f16 else None)
        sm = pa._small
        ops.adam_step_dev_(sm.master, sm.grad, pa._m1_s, pa._m2_s, None, pa._lr_dev, pa.betas, pa.eps, pa.wd, True,
                           pa._step_dev)
    adamw_ms = device_ms(adamw, args.reps)

    # ---- the eager LARS as the reference runs it, on tensors of the same shapes
    eager = [torch.nn.Parameter(p.detach().clone()) for p in pl.lars_params]
    for p in eager:
        p.grad = torch.randn_like(p) * 1e-3
    opt = lars_ref.LARS(eager, lr=0.5, weight_decay=1e-6)
    eager_ms = wall_ms(opt.step, max(args.reps // 5, 5))
    del eager, opt

    # ---- whole pretraining steps, 'lars' and 'adamw' alternated
    times = {"lars": [], "adamw": []}
    for i in range(args.steps + 2):
        for name, pre in pres.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            pre.step(im_q, im_k, 2.0 + i / 100)
            b.record()
            times[name].append((a, b))
    torch.cuda.synchronize()
    step_ms = {k: sorted(a.elapsed_time(b) for a, b in v[2:]) for k, v in times.items()}

    name, power = card()
    print(json.dumps({
        "card": name, "power_limit": power,
        "params": n_all, "params_matrix": n_mat, "params_encoder": n_enc, "tensors": table[1], "chunks": table[2],
        "lars_fused_ms": round(lars_ms, 4), "lars_bytes": nbytes, "lars_gbs": round(nbytes / lars_ms / 1e6, 1),
        "copy_same_bytes_ms": round(copy_ms, 4), "copy_gbs": round(nbytes / copy_ms / 1e6, 1),
        "lars_vs_copy": round(copy_ms / lars_ms, 3),
        "adamw_fused_ms": round(adamw_ms, 4), "lars_eager_reference_ms": round(eager_ms, 3),
        "step_batch": B, "step_K": 65536,
        "step_lars_ms_median": round(step_ms["lars"][len(step_ms["lars"]) // 2], 3),
        "step_adamw_ms_median": round(step_ms["adamw"][len(step_ms["adamw"]) // 2], 3),
        "step_lars_ms_min": round(step_ms["lars"][0], 3), "step_adamw_ms_min": round(step_ms["adamw"][0], 3),
        "reps": args.reps, "steps": args.steps,
    }), flush=True)


if __name__ == "__main__":
    main()
