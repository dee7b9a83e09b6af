"""Times the explain pass on the GPU (a script, not a test):

    python tests/gpu_attn_maps_bench.py [--pairs 32] [--img 224] [--iters 10] [--out results.json]

  * Fus_CrossViT.explain at `pairs` image pairs, without maps (rollout + cross maps) and with the maps of all 12 blocks,
    next to the plain no-grad forward it extends;
  * the three kernels alone (mfv_attn_probs with probs + head mean for one block, mfv_attn_rollout over 12 blocks,
    mfv_fusion_attn), CUDA events over `iters` launches after a warm-up;
  * the eager fp32 oracle (oracle/attention_ref.py: both encoders replayed block by block, rollout, cross maps) on the
    same GPU.
Prints the card name and its power limit with the numbers."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import e2e_common as E  # noqa: E402


def card():
    name = torch.cuda.get_device_name()
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power.strip() or "unknown"


def timed(fn, iters, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=32)
    ap.add_argument("--img", type=int, default=224)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device (B200)")
    torch.backends.cuda.matmul.allow_tf32 = False
    from mfvit import ops
    from mfvit.engine import engine_for
    from mfvit.functions import FUSION_FIELDS
    from oracle import attention_ref as A
    (r_f, r_c, r_e), (o_f, o_c, o_e) = E.build_mfvit_pair(img_size=a.img, seed=0)
    img_c, img_e, _ = E.synthetic_pair(a.pairs, a.img, device="cuda")
    res = {"card": None, "pairs": a.pairs, "img": a.img}
    res["card"], res["power_limit"] = card()
    with torch.no_grad():
        res["forward_nograd_ms"] = timed(lambda: o_f(o_c, o_e, img_c, img_e), a.iters)
    res["explain_no_maps_ms"] = timed(lambda: o_f.explain(o_c, o_e, img_c, img_e), a.iters)
    res["explain_all_maps_ms"] = timed(lambda: o_f.explain(o_c, o_e, img_c, img_e, blocks=range(12)), a.iters)

    eng = engine_for(o_c, o_e)
    with torch.no_grad():
        tok, lease = eng.forward([img_c, img_e], save=True)
    lay = eng.layout
    NB, S, H, L = 2 * a.pairs, lay.S, lay.H, lay.depth
    qkv = lease.ws.qkv.view(torch.float16 if eng.fwd_f16 else torch.bfloat16).view(L, NB, S, 3, H, lay.C // H)
    probs = torch.empty(NB, H, S, S, device="cuda")
    means = torch.empty(L, NB, S, S, device="cuda")
    res["kernel_attn_probs_block_ms"] = timed(lambda: ops.attn_probs(qkv[5], probs, means[5]), 5 * a.iters)
    res["kernel_attn_probs_mean_only_block_ms"] = timed(lambda: ops.attn_probs(qkv[5], None, means[5]), 5 * a.iters)
    for l in range(L):
        ops.attn_probs(qkv[l], None, means[l])
    res["kernel_attn_rollout_ms"] = timed(lambda: ops.attn_rollout(means), 5 * a.iters)
    params, _ = o_f._fusion_params(o_c, o_e)
    ps = [None if p is None else p.detach().contiguous() for p in params]
    st = ops.fusion_param_struct({n: (ps[2 * i], ps[2 * i + 1]) for i, n in enumerate(FUSION_FIELDS)})
    res["kernel_fusion_attn_ms"] = timed(lambda: ops.fusion_attn(tok, st, o_f.heads), 5 * a.iters)
    lease.release()
    # bytes the probs kernel must write for one block (probs + mean), and its rate
    wbytes = 4 * NB * S * S * (H + 1)
    res["attn_probs_write_GBps"] = wbytes / res["kernel_attn_probs_block_ms"] / 1e6
    del probs, means

    def oracle():
        with torch.no_grad():
            tc, mc = A.vit_attention(r_c, img_c)
            te, me = A.vit_attention(r_e, img_e)
            A.rollout(mc.mean(2)), A.rollout(me.mean(2)), A.cross_attention(r_f, tc, te)
    res["eager_oracle_fp32_ms"] = timed(oracle, max(2, a.iters // 2), warmup=1)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
