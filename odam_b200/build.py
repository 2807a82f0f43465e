"""Build odam_b200/lib/libodam_sq.so (hand-written sm_100a CUDA + the C ABI of include/odam_sq.h).

    python -m odam_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  -fmad=false: the sampler restates the reference's fp32 rounding
sequence, so every fused multiply-add in the kernels is written explicitly (__fmaf_rn).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = [os.path.join(HERE, "csrc", "sq_kernels.cu")]
DEPS = SRC + [os.path.join(HERE, "csrc", "sq_device.cuh"), os.path.join(HERE, "csrc", "sq_math.cuh"), os.path.join(HERE, "csrc", "sq_glibc_data.h"), os.path.join(HERE, "csrc", "sq_postproc.cuh"), os.path.join(HERE, "csrc", "sq_stage.h"), os.path.join(HERE, "csrc", "sq_autograd.cuh"), os.path.join(HERE, "..", "include", "odam_sq.h")]
OUT = os.path.join(HERE, "lib", "libodam_sq.so")
# -regUsageLevel=10: ptxas trades registers for better code more aggressively (default 5); inside the same launch
# bounds it is worth +0.4..1.6 % on the dense configs (profiles/r02_ptxas_regusage.txt), nothing changes numerically
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false",
              "-Xptxas", "-regUsageLevel=10", "-Xcompiler", "-fPIC", "-shared"]


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(d) > t for d in DEPS)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", OUT] + SRC
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode:
        raise RuntimeError("nvcc failed building libodam_sq.so")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
