"""Build odam_b200/lib/libodam_sq.so (hand-written sm_100a CUDA + the C ABI of include/odam_sq.h).

    python -m odam_b200.build [--force] [--verbose] [--out PATH]

--out writes the library elsewhere with the same flags, e.g. one build per source tree for A/B timing
(odam_b200/lib/ab/libodam_sq_<name>.so, run by tools/ab_run.sh <name>).
nvcc cross-compiles without a GPU.  -fmad=false: the sampler restates the reference's fp32 rounding
sequence, so every fused multiply-add in the kernels is written explicitly (__fmaf_rn).
"""
import argparse
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


def needs_build(out=OUT):
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(d) > t for d in DEPS)


def build(force=False, verbose=False, out=OUT):
    if not force and not needs_build(out):
        return out
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", out] + SRC
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode:
        raise RuntimeError(f"nvcc failed building {out}")
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser(prog="python -m odam_b200.build")
    ap.add_argument("--force", action="store_true", help="rebuild even when the library is newer than its sources")
    ap.add_argument("--verbose", action="store_true", help="print nvcc's output, with ptxas resource usage")
    ap.add_argument("--out", default=OUT, help="library to write (default: %(default)s)")
    a = ap.parse_args()
    print(build(force=a.force, verbose=a.verbose, out=a.out))
