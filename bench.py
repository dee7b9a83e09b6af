#!/usr/bin/env python
"""bench.py - MF-ViT CA training throughput (image-pairs/s, fwd+bwd+optimizer step) on N B200 GPUs of one node.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --gpus 1 --steps K --warmup W      # the reference path on the host CPU cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR    # + what the last timed step computed, DIR/*.npy

Workload (BASELINE.json): MF-ViT CA = two ViT-S/16 branches (CXR + enhanced CXR) + CLS cross-attention fusion + two summed
aux heads, 224x224 synthetic CXR tensors, random-init weights.  N=1: configs[1] (32 pairs); N>1: configs[2] (64 pairs per
GPU, data parallel, gradient all-reduce over NCCL/NVLink).  One "step" = H-resident batch -> forward -> CE(fused+x_cxr+
x_enh) -> backward through both backbones and the fusion -> [all-reduce] -> SGD-momentum step on every parameter.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "multi-feature-vit_b200"), os.path.join(ROOT, "multi-feature-vit_b200", "dropin"),
          os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "MF-ViT CA train image-pairs/s"
UNIT = "pairs/s"


# ------------------------------------------------------------------------------------------------ work accounting
def vit_fwd_flops(img, C=384, depth=12, hidden=1536):
    """2*MAC FLOPs of one ViT-S/16 forward for one image (SURVEY 8(d): 9.197 GF @224)."""
    np_ = (img // 16) ** 2
    S = np_ + 1
    patch = 2 * np_ * 768 * C
    blk = 2 * S * C * 3 * C + 4 * S * S * C + 2 * S * C * C + 4 * S * C * hidden
    return patch + depth * blk


def pair_flops(img):
    """fwd+bwd FLOPs of one MF-ViT CA pair on the de-duplicated graph (BASELINE.md section 3: 55.65 GF @224)."""
    C, S = 384, (img // 16) ** 2 + 1
    vit = vit_fwd_flops(img)
    fusion = 2 * (2 * 2 * S * C * C)  # both directions, wk/wv GEMMs as written
    fwd = 2 * vit + fusion
    patch = 2 * (img // 16) ** 2 * 768 * C
    return fwd + 2 * fwd - 2 * patch  # no dgrad for the pixels


def gemm_class_flops(img, B, G=2, C=384, depth=12, hidden=1536):
    """FLOPs per step of the three GEMM kernel classes (forward, dgrad, wgrad) for G branches of B images."""
    np_ = (img // 16) ** 2
    S = np_ + 1
    lin = 2 * S * C * (3 * C + C + 2 * hidden) * depth  # per image, all Linear layers
    patch = 2 * np_ * 768 * C
    return {"gemm_fwd": G * B * (lin + patch), "gemm_dgrad": G * B * lin, "gemm_wgrad": G * B * (lin + patch)}


def ln_class_bytes(img, B, G=2, C=384, depth=12):
    """Algorithmic HBM bytes per step of the LayerNorm classes (DESIGN.md 3.3): forward = x f32 in, fp16 + bf16 copies
    out, mean / rstd; backward = x f32, dy bf16, residual gradient f32 in, dx f32 + bf16 out, mean / rstd."""
    rows = G * B * ((img // 16) ** 2 + 1)
    return {"ln_fwd": 2 * depth * rows * (C * (4 + 2 + 2) + 8) + rows * (C * (4 + 4) + 8),
            "ln_bwd": 2 * depth * rows * (C * (4 + 2 + 4 + 4 + 2) + 8) + rows * (C * (4 + 4 + 4 + 2) + 8)}


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t_begin = self.t_end = None

    def start(self):
        """Started BEFORE the warm-up steps: the first nvidia-smi answer on a fresh box can take longer than the whole
        timed region (20 steps are ~90 ms), which left the record without a single sample."""
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def wait_ready(self, timeout=15.0):
        """Block until the sampler has delivered its first row (or the timeout passes)."""
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.01)

    def begin(self):
        self.t_begin = time.time()

    def end(self):
        self.t_end = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if self.t_end is None:
            self.t_end = time.time()
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def digest(rows):
            sm, smax, reasons = [], None, set()
            for _, r in rows:
                f = [x.strip() for x in r.split(",")]
                if len(f) < 7:
                    continue
                try:
                    sm.append(float(f[0]))
                    smax = float(f[1])
                except ValueError:
                    continue
                for n, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            return sm, smax, reasons

        lo = self.t_begin if self.t_begin is not None else 0.0
        inside = [r for r in self.rows if lo <= r[0] <= self.t_end + 0.02]
        sm, smax, reasons = digest(inside)
        out = {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
               "samples": len(sm), "window": "the device-resident and end-to-end timed regions"}
        if not sm:  # nothing landed inside the window: say so and give what the whole run saw
            sm, smax, reasons = digest(self.rows)
            out.update({"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                        "samples": 0, "samples_whole_run": len(sm)})
        return out


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"bf16_burst": d.get("bf16_tflops", 1590.0), "bf16_sustained": d.get("bf16_tflops_sustained", 1400.0),
                "hbm": d.get("hbm_gbs", 6650.0), "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "source": "fallback (B200_PROFILING.md)"}


# ------------------------------------------------------------------------------------------------ CPU reference arm
def build_oracle(img):
    """The reference path on CPU: oracle restatement of timm ViT-S/16 x2 + Fus_CrossViT (as written, FUS:126-157)."""
    from oracle import fusion_ref, vit_ref
    import e2e_common as E
    torch.manual_seed(0)
    cxr, enh = vit_ref.vit_small(img_size=img), vit_ref.vit_small(img_size=img)
    for v in (cxr, enh):
        E.reference_head_init_(v)
    fus = fusion_ref.Fus_CrossViT(cxr, enh)
    params = [p for m in (fus, cxr, enh) for p in m.parameters() if p.requires_grad]
    opt = torch.optim.SGD(params, lr=1e-3, momentum=0.9)
    return fus, cxr, enh, opt


def cpu_reference_rate(img, sample_pairs, steps, warmup):
    """pairs/s of the reference's own CPU path (fp32, all host threads), as written: 4 backbone passes per step."""
    import e2e_common as E
    torch.set_num_threads(os.cpu_count() or 1)
    fus, cxr, enh, opt = build_oracle(img)
    img_c, img_e, tgt = E.synthetic_pair(sample_pairs, img)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        fused, x_c, x_e = fus(cxr, enh, img_c, img_e)  # MAIN_CA:862
        loss = torch.nn.functional.cross_entropy(fused + x_c + x_e, tgt)  # MAIN_CA:868-873
        loss.backward()
        opt.step()
        float(loss.detach())
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    return sample_pairs / dt, dt, torch.get_num_threads()


def cublas_same_shapes(img, B, device, reps=20):
    """Measuring stick, not product path: the bare contractions of one encoder block at THIS step's shapes (two branches
    batched, bf16, no bias / activation / residual / LayerNorm) on cuBLAS through torch.bmm, graph-timed with warm
    inputs.  A [2 x 6304 x 384] problem is a handful of waves of tiles: cuBLAS itself reaches a fraction of its 8192^3
    rate here, and that - not the large-matrix peak - is what a fused GEMM at these shapes can be held against."""
    S = (img // 16) ** 2 + 1
    M, C, Hd = B * S, 384, 1536
    shapes = [("qkv", M, 3 * C, C), ("proj", M, C, C), ("fc1", M, Hd, C), ("fc2", M, C, Hd)]
    out = {"what": "torch.bmm (cuBLAS) bf16 [2 x M x K] @ [2 x K x N], CUDA-graph timed, bare contraction", "M": M, "shapes": {}}
    tot_us, tot_fl = 0.0, 0.0
    for name, m, n, k in shapes:
        a = torch.randn(2, m, k, device=device, dtype=torch.bfloat16)
        w = torch.randn(2, k, n, device=device, dtype=torch.bfloat16)
        c = torch.empty(2, m, n, device=device, dtype=torch.bfloat16)
        for _ in range(3):
            torch.bmm(a, w, out=c)
        torch.cuda.synchronize()
        side = torch.cuda.Stream(device=device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for _ in range(reps):
                torch.bmm(a, w, out=c)
        g.replay()
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) / reps)
        fl = 2.0 * 2 * m * n * k
        out["shapes"][name] = {"N": n, "K": k, "us": best * 1e3, "tflops": fl / (best * 1e-3) / 1e12}
        tot_us += best * 1e3
        tot_fl += fl
        del a, w, c, g
    out["block_forward_us"] = tot_us
    out["block_forward_tflops"] = tot_fl / (tot_us * 1e-6) / 1e12
    torch.cuda.empty_cache()
    return out


def gpu_eager_reference(img, B, device, steps=8, warmup=3):
    """The "kernel to beat" on the same B200 (SURVEY 8(d) last row, BASELINE.md section 5): the reference graph in stock
    PyTorch - cuBLASLt / ATen library kernels - (i) fp32 as written (4 backbone passes, FUS:128-135), (ii) fp32
    de-duplicated, (iii) bf16 autocast de-duplicated, (iv) the same with F.scaled_dot_product_attention (flash / cuDNN
    kernels) in place of the explicit softmax.  fwd + bwd + SGD step on every parameter, like the measured step.  A
    baseline leg like cpu_baseline: it runs the oracle port, after and outside every timed region of this repo's path."""
    import torch.nn.functional as F

    import e2e_common as E
    from oracle import vit_ref
    out = {"unit": UNIT, "pairs_per_step": B, "steps": steps,
           "what": "oracle port of the reference modules under stock PyTorch %s on the same GPU, fwd+bwd+SGD, "
                   "CUDA-event timed" % torch.__version__}
    fus, cxr, enh, opt = build_oracle(img)
    for m in (fus, cxr, enh):
        m.to(device)
    opt = torch.optim.SGD([p for m in (fus, cxr, enh) for p in m.parameters() if p.requires_grad], lr=1e-3, momentum=0.9)
    img_c, img_e, tgt = (t.to(device) for t in E.synthetic_pair(B, img))
    plain_attention = vit_ref.Attention.forward

    def sdpa_attention(self, x):
        Bq, N, C = x.shape
        qkv = self.qkv(x).reshape(Bq, N, 3, self.num_heads, C // self.num_heads).permute(2, 0, 3, 1, 4)
        o = F.scaled_dot_product_attention(qkv[0], qkv[1], qkv[2], scale=self.scale)
        return self.proj(o.transpose(1, 2).reshape(Bq, N, C))

    def timed(dedup, autocast, sdpa):
        vit_ref.Attention.forward = sdpa_attention if sdpa else plain_attention
        try:
            def one():
                opt.zero_grad(set_to_none=True)
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                    fused, x_c, x_e = fus(cxr, enh, img_c, img_e, dedup=dedup)
                    loss = F.cross_entropy((fused + x_c + x_e).float(), tgt)
                loss.backward()
                opt.step()
            for _ in range(warmup):
                one()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps):
                one()
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b) / steps
            return {"pairs_per_s": B / ms * 1e3, "ms_per_step": ms}
        finally:
            vit_ref.Attention.forward = plain_attention

    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        out["fp32_as_written"] = timed(False, False, False)
        out["fp32_dedup"] = timed(True, False, False)
        out["bf16_autocast_dedup"] = timed(True, True, False)
        out["bf16_autocast_dedup_sdpa"] = timed(True, True, True)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32
    del fus, cxr, enh, opt
    torch.cuda.empty_cache()
    return out


def dp_gradient_check(trainer, device, rank, world, img, pairs=8):
    """Data-parallel correctness on the hardware the scaling numbers come from: the all-reduced gradient of `pairs`
    pairs per rank equals the gradient ONE rank computes on the concatenated batch (same replica, all-reduce off).
    Runs through MFViTCATrainer.forward_backward + all_reduce, i.e. the same NCCL path as the timed step."""
    import torch.distributed as dist

    import e2e_common as E
    c, e, t = (x.to(device) for x in E.synthetic_pair(pairs, img, rank=900 + rank))
    graph, trainer._graph = trainer._graph, None
    local0, ovl0 = trainer.local_only, trainer.overlap_optimizer
    try:
        trainer.local_only = False
        trainer.overlap_optimizer = False  # gradients only: nothing may be stepped between the two passes
        _, g = trainer.forward_backward(c, e, t, reduce_async=True)
        trainer.all_reduce(g)
        g_dp, s_dp = g.clone(), trainer._small.grad.clone()
        gc = [torch.empty_like(c) for _ in range(world)]
        ge = [torch.empty_like(e) for _ in range(world)]
        gt = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(gc, c), dist.all_gather(ge, e), dist.all_gather(gt, t)
        trainer.local_only = True
        _, g1 = trainer.forward_backward(torch.cat(gc), torch.cat(ge), torch.cat(gt))
        s1 = trainer._small.grad
        cos = lambda a, b: float(torch.nn.functional.cosine_similarity(a.flatten().double(), b.flatten().double(), dim=0))
        res = {"pairs_per_rank": pairs, "encoder_grad_cos": cos(g_dp, g1), "fusion_grad_cos": cos(s_dp, s1),
               "encoder_grad_max_rel": float((g_dp - g1).abs().max() / g1.abs().max().clamp_min(1e-30)),
               "what": "all-reduced gradient of %d pairs/rank vs one rank on the concatenated %d pairs"
                       % (pairs, pairs * world)}
        res["ok"] = res["encoder_grad_cos"] >= 0.9999 and res["fusion_grad_cos"] >= 0.9999
        return res
    finally:
        trainer.local_only, trainer.overlap_optimizer = local0, ovl0
        trainer._graph = graph


def run_reference(args, rank):
    if rank != 0:
        return
    sample = args.cpu_sample_pairs
    rate, dt, cores = cpu_reference_rate(args.img_size, sample, args.steps, max(args.warmup, 1))
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(args, per_gpu=args.pairs_per_gpu),
                       reference_arm_ran="ONE process on the host cores, %d pairs per step, no GPU and no data "
                                         "parallelism (the reference's MAIN_CA is single-device, MAIN_CA:59-60); the "
                                         "value is that process's pairs/s whatever --gpus says" % sample),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d pairs per step, as-written graph (4 backbone passes, FUS:128-135), oracle port of "
                                   "the reference (timm ViT is absent from the reference tree), fp32, %d threads"
                                   % (sample, cores)},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


DUMP_SAMPLE = 1 << 22  # parameters kept per encoder by --dump-outputs: 16 MB of its 87 MB


def dump_step_outputs(out_dir, trainer, loss, fus, cxr, enh):
    """--dump-outputs: what one training step hands its caller, as float32 .npy files - the loss, the three logit sets
    (fused, CXR head, enhanced head) and the parameters after the optimizer step: every one of the fusion's, and a fixed
    seeded sample of DUMP_SAMPLE of each encoder's (module.parameters() order, flattened), so that the files of two builds
    run with the same arguments compare element for element."""
    import numpy as np
    fused, x_c, x_e = trainer.logits()
    out = {"loss": loss, "logits_fused": fused, "logits_cxr": x_c, "logits_enh": x_e,
           "params_fusion": torch.cat([p.detach().reshape(-1) for p in fus.parameters()])}
    for name, m in (("cxr", cxr), ("enh", enh)):
        flat = torch.cat([p.detach().reshape(-1) for p in m.parameters()])
        idx = np.sort(np.random.default_rng(0).choice(flat.numel(), DUMP_SAMPLE, replace=False))
        out["params_%s_sample" % name] = flat[torch.from_numpy(idx).to(flat.device)]
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def workload_config(args, per_gpu):
    return {
        "workload": "MF-ViT CA: 2x ViT-S/16 (CXR + enhanced) + CLS cross-attention fusion + 2 summed aux heads, "
                    "fwd+bwd+SGD step, %dx%d, %d pairs/GPU" % (args.img_size, args.img_size, per_gpu),
        "pairs_per_gpu": per_gpu, "global_batch": per_gpu * args.gpus, "img_size": args.img_size,
        "tokens_per_branch": (args.img_size // 16) ** 2 + 1, "parallelism": "dp%d" % args.gpus,
        "baseline_config": "configs[1]" if args.gpus == 1 and per_gpu == 32 else "configs[2]",
        "l2_policy": "per-step working set (activations of 24 blocks, >2 GB) and 4 rotating input batches exceed the "
                     "126 MB L2; no explicit flush",
    }


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="mfvit", choices=["mfvit", "reference"])
    ap.add_argument("--pairs-per-gpu", type=int, default=0, help="default: 32 at N=1 (configs[1]), 64 at N>1 (configs[2])")
    ap.add_argument("--img-size", type=int, default=224)
    ap.add_argument("--cpu-sample-pairs", type=int, default=32, help="pairs per CPU step (32 = the batch of configs[1])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-moco", action="store_true", help="skip the MoCo pretraining-step leg (key moco_dp)")
    ap.add_argument("--moco-batch", type=int, default=128, help="images per GPU and view of the MoCo leg (configs[3])")
    ap.add_argument("--no-gpu-reference", action="store_true", help="skip the stock-PyTorch GPU baseline leg (N = 1)")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying the "
                                                            "CUDA graph of the step (single-GPU runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed (loss, "
                                                          "logits, parameters after the step) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "mfvit":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl mfvit)")
    if args.warmup < 3 and args.impl == "mfvit":
        args.warmup = 3
    if args.pairs_per_gpu <= 0:
        args.pairs_per_gpu = 32 if args.gpus == 1 else 64

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return 0

    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "WARN").upper() in ("VERSION", "WARN"):
            # at these two levels NCCL prints its version banner to stdout, in front of the one JSON line (the level
            # may come from the box's nccl.conf, so it is overridden rather than unset); INFO / TRACE from the caller
            # are left alone
            os.environ["NCCL_DEBUG"] = "NONE"
        dist.init_process_group("nccl", device_id=device)

    import importlib

    import e2e_common as E
    import vits_returnftrs as vits
    from mfvit import _lib
    from mfvit.trainer import MFViTCATrainer
    lib = _lib.init(local_rank)

    B, img = args.pairs_per_gpu, args.img_size
    torch.manual_seed(0)  # identical replicas on every rank
    fm = importlib.import_module(E.FUS_MOD)
    cxr, enh = vits.vit_small(img_size=img), vits.vit_small(img_size=img)
    for v in (cxr, enh):
        E.reference_head_init_(v)
    fus = fm.Fus_CrossViT(cxr, enh)
    cxr.to(device), enh.to(device), fus.to(device)
    from mfvit.data import EpochMetrics
    metrics = EpochMetrics(capacity=B * max(args.steps, 1), num_classes=3, device=device)
    trainer = MFViTCATrainer(fus, cxr, enh, lr=1e-3, momentum=0.9, weight_decay=0.0, metrics=metrics, train_backbones=True)

    # synthetic data: 4 rotating batches per rank, pinned host copies for the end-to-end leg
    nb = 4
    host = []
    for i in range(nb):
        c, e, t = E.synthetic_pair(B, img, rank=rank * 16 + i)
        host.append((c.pin_memory(), e.pin_memory(), t.pin_memory()))
    dev_batches = [(c.to(device), e.to(device), t.to(device)) for c, e, t in host]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)  # nvidia-smi loop: up and answering before the timed regions begin
    if rank == 0:
        sampler.start()
    # ---- warm-up (allocations, cudaFuncSetAttribute, NCCL channels)
    for i in range(args.warmup):
        trainer.step(*dev_batches[i % nb])
    barrier()
    use_graph = not args.no_graph and (world == 1 or os.environ.get("MFVIT_GRAPH_DDP", "1") == "1")
    if use_graph:  # the whole step (fwd, loss, bwd, optimizer) as one CUDA graph; data-parallel runs stay eager
        trainer.capture_graph(*dev_batches[0])
        for i in range(2):
            trainer.step(*dev_batches[i % nb])
        barrier()

    # ---- timed: device-resident inputs
    if rank == 0:
        sampler.wait_ready()
        sampler.begin()
    launches0 = lib.mfv_launch_count() + trainer.graph_replays * trainer.graph_launches
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    start.record()
    for i in range(args.steps):
        loss = trainer.step(*dev_batches[i % nb])
    end.record()
    barrier()
    elapsed_ms = start.elapsed_time(end)
    if args.dump_outputs and rank == 0:
        dump_step_outputs(args.dump_outputs, trainer, loss, fus, cxr, enh)
    # kernels of libmfvit.so per step: eager launches are counted by the library, graph replays re-issue the launches
    # counted while the step was captured
    launches = (lib.mfv_launch_count() + trainer.graph_replays * trainer.graph_launches - launches0) / args.steps
    loss_val = float(loss)

    # ---- timed: end to end (pinned host -> device copies in, loss read back, every step)
    copy_stream = torch.cuda.Stream(device=device)
    slots = [[torch.empty_like(t, device=device) for t in dev_batches[0]] for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def prefetch(step):
        s = step % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[s])
            for dst, src in zip(slots[s], host[step % nb]):
                dst.copy_(src, non_blocking=True)
            ready[s].record(copy_stream)

    for s in range(2):
        consumed[s].record()
    barrier()
    e_start, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_steps = args.steps
    e_start.record()
    prefetch(0)
    for i in range(e_steps):
        s = i % 2
        torch.cuda.current_stream().wait_event(ready[s])
        loss_e = trainer.step(*slots[s])
        consumed[s].record()
        if i + 1 < e_steps:  # enqueued AFTER this step's launch: the host work of the copies runs under the step
            prefetch(i + 1)
        loss_host = float(loss_e)  # device -> host read of the step's result (synchronises, as MAIN_CA:884 does)
    e_end.record()
    barrier()
    e2e_ms = e_start.elapsed_time(e_end)
    if rank == 0:
        sampler.end()
    clocks = sampler.stop() if rank == 0 else None

    # ---- timed: the same loop fed by the paired uint8 input pipeline (mfvit.data, SURVEY 8(f) row 3): pinned uint8
    # store -> host gather -> H2D of uint8 -> flip / rotate / crop / normalise kernel -> step -> loss read back
    from mfvit.data import PairedDeviceLoader, PairedU8Store
    gu = torch.Generator().manual_seed(4096 + rank)
    # one pass covers the timed steps when that fits ~0.6 GB of pinned memory per image type (a pass restart costs one
    # un-prefetched batch; real epochs are hundreds of batches long)
    n_store = max(3, min(args.steps + 2, int(6e8 // (B * img * img * 3)))) * B
    store = PairedU8Store(torch.randint(0, 256, (n_store, img, img, 3), dtype=torch.uint8, generator=gu),
                          torch.randint(0, 256, (n_store, img, img, 3), dtype=torch.uint8, generator=gu),
                          torch.randint(0, 3, (n_store,), generator=gu))
    loader = PairedDeviceLoader(store, B, crop=img, degrees=True, training=True, device=device, seed=rank, drop_last=True)

    def loader_batches(n):
        done, epoch = 0, 0
        while done < n:
            loader.set_epoch(epoch)
            for batch in loader:
                yield batch
                done += 1
                if done == n:
                    return
            epoch += 1

    for xc, xe, y in loader_batches(2):
        trainer.step(xc, xe, y)
    barrier()
    u_start, u_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    u_start.record()
    for xc, xe, y in loader_batches(e_steps):
        loss_u = trainer.step(xc, xe, y)
        loss_host = float(loss_u)
    u_end.record()
    barrier()
    u8_ms = u_start.elapsed_time(u_end)
    # the same loop the way the pipeline is meant to be driven: loss / hits / scores accumulate on the device
    # (mfv_epoch_metrics inside the captured step), one device -> host read at the end of the pass
    metrics.reset()
    barrier()
    u_start.record()
    for xc, xe, y in loader_batches(e_steps):
        trainer.step(xc, xe, y)
    ep_loss, ep_auc, ep_acc = metrics.result()
    u_end.record()
    barrier()
    u8_nosync_ms = u_start.elapsed_time(u_end)

    # ---- data-parallel correctness on this hardware (N > 1): all-reduced gradient == one rank on the concatenated batch.
    # Runs while the replicas are still identical (the same-work leg below steps every rank on its own, unsynchronised).
    dp_check = None
    if world > 1:
        try:
            dp_check = dp_gradient_check(trainer, device, rank, world, img)
        except Exception as exc:  # noqa: BLE001 - a failed self-check must not lose the measured line
            dp_check = {"ok": False, "error": "%s: %s" % (type(exc).__name__, exc)}

    # ---- data-parallel runs only: the same per-GPU work with the gradient all-reduce switched off (every rank steps its
    # own replica), i.e. the single-GPU rate at THIS batch size - the denominator a weak-scaling efficiency needs
    # (N = 1 of this benchmark runs configs[1], 32 pairs, not the 64 pairs per GPU of configs[2])
    local_ms = None
    if world > 1:
        trainer._graph = None
        trainer.local_only = True
        if use_graph:
            trainer.capture_graph(*dev_batches[0])
        for i in range(3):
            trainer.step(*dev_batches[i % nb])
        barrier()
        l_start, l_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l_start.record()
        for i in range(args.steps):
            trainer.step(*dev_batches[i % nb])
        l_end.record()
        barrier()
        local_ms = l_start.elapsed_time(l_end)

    # ---- per-kernel-class device time (CUDA events on the launching stream), 3 extra steps; the library serialises the
    # weight-gradient side stream while profiling so that every class time is that class alone
    breakdown, dominant = {}, None
    if rank == 0:
        import ctypes as C
        nl = lib.mfv_prof_num_labels()
        ms = (C.c_float * nl)()
        cnt = (C.c_int * nl)()
        lib.mfv_prof_enable(1)
        psteps = 3
        for i in range(psteps):
            trainer.forward_backward(*dev_batches[i % nb])
        lib.mfv_prof_read(ms, cnt, nl)
        lib.mfv_prof_enable(0)
        for i in range(nl):
            if cnt[i]:
                breakdown[lib.mfv_prof_label_name(i).decode()] = {"ms_per_step": ms[i] / psteps,
                                                                  "launches_per_step": cnt[i] / psteps}
        dominant = max(breakdown, key=lambda k: breakdown[k]["ms_per_step"]) if breakdown else None
    if world > 1:
        t = torch.tensor([elapsed_ms, e2e_ms, u8_ms, u8_nosync_ms, local_ms], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms, e2e_ms, u8_ms, u8_nosync_ms, local_ms = (float(v) for v in t)

    graph_launches = trainer.graph_launches

    # ---- BASELINE configs[3]: the MoCo-v3-structure / v2-loss pretraining step under SyncBatchNorm + DDP over NCCL
    # (MAIN_PRE:297,312), 128 images per GPU, K = 65 536, with its self-checks (tests/moco_dp_common.py).  N = 1 runs it
    # over a 1-rank NCCL group.
    moco_dp = None
    if not args.no_moco:
        trainer._graph = None
        torch.cuda.empty_cache()
        try:
            import moco_dp_common
            if world == 1 and not dist.is_initialized():
                import socket
                sk = socket.socket()
                sk.bind(("127.0.0.1", 0))
                port = sk.getsockname()[1]
                sk.close()
                dist.init_process_group("nccl", init_method="tcp://127.0.0.1:%d" % port, rank=0, world_size=1,
                                        device_id=device)
            moco_dp = moco_dp_common.run(device, rank, world, batch=args.moco_batch, steps=min(args.steps, 10), warmup=3)
        except Exception as exc:  # noqa: BLE001
            moco_dp = {"ok": False, "error": "%s: %s" % (type(exc).__name__, exc)}
        if world == 1 and dist.is_initialized():
            try:
                dist.destroy_process_group()
            except Exception:  # noqa: BLE001
                pass

    # ---- the kernel to beat: the reference graph under stock PyTorch on this GPU (rank 0, N = 1 only)
    eager_ref = None
    if world == 1 and not args.no_gpu_reference:
        try:
            eager_ref = gpu_eager_reference(img, B, device)
        except Exception as exc:  # noqa: BLE001
            eager_ref = {"error": "%s: %s" % (type(exc).__name__, exc)}
    cublas_ref = None
    if world == 1 and not args.no_gpu_reference:
        try:
            cublas_ref = cublas_same_shapes(img, B, device)
        except Exception as exc:  # noqa: BLE001
            cublas_ref = {"error": "%s: %s" % (type(exc).__name__, exc)}

    if rank == 0:
        peaks = measured_peaks()
        pairs = B * world
        value = pairs * args.steps / (elapsed_ms * 1e-3)
        e2e_value = pairs * e_steps / (e2e_ms * 1e-3)
        gf = gemm_class_flops(img, B)
        roof = None
        # DRAM bytes per launch of each kernel class from the committed ncu capture of the same step (cold-cache,
        # serialised launches; profiles/r02_kernel_traffic.json) - only meaningful for the configuration it was taken on
        traffic = {}
        tpath = os.path.join(ROOT, "profiles", "r02_kernel_traffic.json")
        if os.path.exists(tpath) and B == 32 and img == 224:
            with open(tpath) as f:
                traffic = {k: v.get("dram_bytes_per_launch") for k, v in json.load(f).get("classes", {}).items()}
        if dominant in gf:
            # The dominant kernel is gemm_bf16_kernel: every Linear of the step, forward, dgrad and weight gradient, runs on
            # it (145 launches, ~65 % of the serialised step in the ncu launch list).  achieved = the algorithmic FLOPs
            # of all of those launches / their summed in-step time; by_class splits the same numbers.  Since round 2 the
            # forward launches also carry the residual add + LayerNorm (proj, fc2), GELU (fc1) and the patch-embedding
            # epilogue work that used to be separate kernels - their time counts here, their FLOPs do not.
            cls = [k for k in ("gemm_fwd", "gemm_dgrad", "gemm_wgrad") if k in breakdown]
            ms = sum(breakdown[k]["ms_per_step"] for k in cls)
            n_l = sum(breakdown[k]["launches_per_step"] for k in cls)
            ach = sum(gf[k] for k in cls) / (ms * 1e-3) / 1e12
            tr_b = [traffic.get(k) for k in cls]
            roof = {"kernel": "gemm_bf16_kernel (all %d launches of the step: forward, dgrad, weight gradient)" % round(n_l),
                    "bound": "tensor", "achieved": ach, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                    "frac": ach / peaks["bf16_sustained"],
                    "traffic": (sum(t * breakdown[k]["launches_per_step"] for t, k in zip(tr_b, cls)) / n_l
                                if all(tr_b) else None),
                    "traffic_source": "ncu dram__bytes_read.sum + dram__bytes_write.sum per launch (mean over the three "
                                      "classes), profiles/r02_kernel_traffic.json" if all(tr_b) else None,
                    "peak_source": peaks["source"] + ", sustained figure (kernel timed inside a long step)",
                    "launches_per_step": n_l, "ms_per_step": ms,
                    "by_class": {k: {"achieved": gf[k] / (breakdown[k]["ms_per_step"] * 1e-3) / 1e12,
                                     "frac": gf[k] / (breakdown[k]["ms_per_step"] * 1e-3) / 1e12 / peaks["bf16_sustained"],
                                     "ms_per_step": breakdown[k]["ms_per_step"],
                                     "launches_per_step": breakdown[k]["launches_per_step"]} for k in cls}}
        elif dominant is not None:
            d = breakdown[dominant]
            roof = {"kernel": dominant, "bound": "hbm", "achieved": None, "peak": peaks["hbm"], "unit": "GB/s",
                    "frac": None, "traffic": traffic.get(dominant), "ms_per_step": d["ms_per_step"]}
        # the largest HBM-bound class of the same profiled pass, against the measured copy bandwidth
        roof_hbm = None
        lb = ln_class_bytes(img, B)
        hb = [k for k in lb if k in breakdown]
        if hb:
            k = max(hb, key=lambda n: breakdown[n]["ms_per_step"])
            gbs = lb[k] / (breakdown[k]["ms_per_step"] * 1e-3) / 1e9
            roof_hbm = {"kernel": k + "_kernel (%d launches of the step)" % round(breakdown[k]["launches_per_step"]),
                        "bound": "hbm", "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs / peaks["hbm"],
                        "traffic": traffic.get(k), "ms_per_step": breakdown[k]["ms_per_step"],
                        "peak_source": peaks["source"],
                        "note": "in-step class time from CUDA events around every launch (cold inputs, ~2 us of event "
                                "bracketing per launch); the kernel alone, graph-timed over a ring larger than L2: "
                                "profiles/r01_hbm_bench.log"}
        if roof is not None and cublas_ref and "block_forward_tflops" in cublas_ref:
            # what the library reaches on the bare forward contractions of a block at these shapes (no epilogues): the
            # practical ceiling of a GEMM at this problem size, beside the large-matrix peak the fraction is quoted on
            roof["cublas_same_shapes"] = cublas_ref
            fwd = roof.get("by_class", {}).get("gemm_fwd")
            if fwd:
                roof["gemm_fwd_vs_cublas_bare"] = fwd["achieved"] / cublas_ref["block_forward_tflops"]
        step_tf = value * pair_flops(img) / 1e12
        h2d = sum(t.numel() * t.element_size() for t in host[0])
        same_work = None if local_ms is None else {
            "value_per_gpu": B * args.steps / (local_ms * 1e-3), "unit": UNIT + " per GPU",
            "ms_per_step": local_ms / args.steps,
            "exposed_allreduce_ms": elapsed_ms / args.steps - local_ms / args.steps,
            "what": "every rank stepping its own replica on the same %d pairs with the all-reduce switched off (max "
                    "over ranks): the single-GPU rate at THIS per-GPU batch, i.e. the weak-scaling denominator (N = 1 "
                    "of this benchmark runs configs[1], 32 pairs)" % B}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "fp16 operands fwd / bf16 operands bwd, fp32 accumulate + fp32 residual stream and master weights",
            "data": "synthetic",
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": e2e_ms / e_steps},
            "gpu_launches": launches,
            # data-parallel runs: the honest weak-scaling denominator and the correctness of the reduction, up front
            "same_work_no_allreduce": same_work,
            "dp_gradient_check": dp_check,
            "moco_dp": moco_dp,
            "roofline": roof,
            "config": dict(workload_config(args, per_gpu=B),
                           trained_parameters="all: both ViT-S/16 encoders, their heads and the fusion (full fine-tuning, "
                                              "MFViTCATrainer(train_backbones=True)); the reference as written steps "
                                              "only the fusion's 22 tensors (MAIN_CA:435-449)"),
            "clocks": clocks,
            "gpu_eager_reference": eager_ref,
            "e2e_u8_loader": {"value": pairs * e_steps / (u8_ms * 1e-3), "unit": UNIT,
                              "h2d_bytes_per_step": loader.h2d_bytes_per_batch, "d2h_bytes_per_step": 4,
                              "ms_per_step": u8_ms / e_steps,
                              "value_epoch_metrics_on_device": pairs * e_steps / (u8_nosync_ms * 1e-3),
                              "epoch_metrics": {"loss": ep_loss, "auc": ep_auc, "acc": ep_acc,
                                                "d2h": "once per pass (loss sum, hit count, scores for the AUC)"},
                              "path": "pinned uint8 store -> gather -> H2D -> mfv_augment_u8 (flip, +-1 deg rotation, "
                                      "crop, normalise) x 2 on the copy stream -> step; not the headline e2e (that one copies the float32 "
                                      "tensors the reference's loaders produce)"},
            "launch_mode": "CUDA graph of the whole step (%d kernels per replay)" % graph_launches
                           if use_graph else "eager stream launches",
            "roofline_hbm": roof_hbm,
            "step_tflops": step_tf,
            "step_frac_of_bf16_peak": {"measured_sustained": step_tf / peaks["bf16_sustained"] / world,
                                       "measured_burst": step_tf / peaks["bf16_burst"] / world,
                                       "spec_2250": step_tf / 2250.0 / world},
            "kernel_breakdown_ms": {k: round(v["ms_per_step"], 4) for k, v in breakdown.items()},
            "final_loss": loss_val,
        }
        if world == 1 and not args.no_cpu_baseline:
            rate, dt, cores = cpu_reference_rate(img, args.cpu_sample_pairs, 3, 1)
            line["cpu_baseline"] = {
                "value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": "%d pairs per step x (1 warm-up + 3 timed) steps of the as-written reference graph (4 backbone "
                          "passes), oracle port, fp32" % args.cpu_sample_pairs}
        print(json.dumps(line), flush=True)
    if world > 1:
        # Tear-down: drop the captured graph (it references NCCL kernels) before the communicator goes away, and leave
        # through os._exit so that a slow NCCL destructor can never hold the launcher after the result line is out.
        trainer._graph = None
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    return 0


if __name__ == "__main__":
    sys.exit(main())
