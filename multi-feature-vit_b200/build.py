"""Builds libmfvit.so (all hand-written sm_100a kernels + the C ABI) in-tree with nvcc.

    python multi-feature-vit_b200/build.py [--force]

nvcc cross-compiles without a GPU; the resulting .so is git-ignored but travels with the repo snapshot to the GPU box.
"""
import concurrent.futures as cf
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "mfvit")
LIB = os.path.join(OUT_DIR, "libmfvit.so")
OBJ_DIR = os.path.join(HERE, "build")
SOURCES = ["runtime.cu", "gemm.cu", "ln.cu", "attn.cu", "attn_tc.cu", "attn_maps.cu", "elementwise.cu", "lars.cu", "augment.cu", "fusion.cu", "infonce.cu", "patch_embed.cu", "vit.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
              "--expt-relaxed-constexpr", "-diag-suppress", "550"]


def _digest():
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for name in sorted(os.listdir(root)):
            if name.endswith((".cu", ".cuh", ".h")):
                with open(os.path.join(root, name), "rb") as f:
                    h.update(name.encode())
                    h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    os.makedirs(OBJ_DIR, exist_ok=True)
    stamp = os.path.join(OBJ_DIR, "stamp")
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig:
        return LIB
    nvcc = os.environ.get("NVCC", "nvcc")

    def compile_one(src):
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with cf.ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    r = subprocess.run([nvcc, "-shared", "-o", LIB, *objs, "-cudart", "static"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    with open(stamp, "w") as f:
        f.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
