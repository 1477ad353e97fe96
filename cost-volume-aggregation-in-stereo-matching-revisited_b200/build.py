"""Build recipe for libdca_b200.so (hand-written sm_100a kernels + C ABI).  In-tree, nvcc only.

    python build.py            # incremental
    python build.py --force
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libdca_b200.so")
SOURCES = ["volume.cu", "conv_direct.cu", "conv_tc.cu", "dca_ops.cu", "halo_p2p.cu", "abi_composites.cu", "metrics.cu",
           "confidence.cu", "lr_check.cu", "reproject.cu", "rectify.cu", "wls.cu", "tsdf.cu", "track.cu",
           "guide.cu", "stixel.cu", "motion.cu", "occupancy.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "--use_fast_math=false"]
FLAGS = [f for f in FLAGS if f != "--use_fast_math=false"]
# 16-bit plane format: fp16 by default (DESIGN.md section 3); DCA_PLANE_FORMAT=bf16 python build.py --force builds the
# bf16 variant (8 more exponent bits for un-normalised checkpoints, 60x the representation error)
if os.environ.get("DCA_PLANE_FORMAT", "fp16").lower() == "bf16":
    FLAGS.append("-DDCA_F16_PLANES=0")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(os.path.dirname(HERE), "include", "dca_b200.h"))     # metrics.cu includes the C ABI header
    objs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(CSRC, s[:-3] + ".o")
        objs.append(obj)
        if force or _stale(obj, [src] + hdrs):
            cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            print(" ".join(cmd), flush=True)
            subprocess.check_call(cmd)
    if force or _stale(OUT, objs):
        cmd = [NVCC, "-shared", "-o", OUT] + objs + ["-lcuda"]
        print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
