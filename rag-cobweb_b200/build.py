"""Builds libcobweb_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

Strict-arithmetic translation units (ifit, categorize, index) are compiled with -fmad=false so
every fp32 operation is a single IEEE operation (DESIGN.md "Arithmetic contract"); the dense
scoring unit keeps FMA contraction.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libcobweb_b200.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--use_fast_math=false"]
UNITS = [
    ("cw_api.cu", []),
    ("cw_ifit.cu", ["-fmad=false"]),
    ("cw_categorize.cu", ["-fmad=false"]),
    ("cw_index.cu", ["-fmad=false"]),
    ("cw_dense.cu", []),
    ("cw_half.cu", []),
    ("cw_whiten.cu", []),
    ("cw_grad.cu", []),
    ("cw_pairs.cu", []),
]


def nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def sources():
    out = [os.path.join(CSRC, u) for u, _ in UNITS]
    out += [os.path.join(CSRC, "cw_common.cuh"), os.path.join(CSRC, "cw_nvtx.h"), os.path.join(os.path.dirname(HERE), "include", "cobweb_b200.h")]
    return out


def needs_build():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    return any(os.path.getmtime(s) > t for s in sources())


def build(force=False, verbose=False):
    if not force and not needs_build():
        return SO
    objs = []
    common = [f for f in COMMON if not f.startswith("--use_fast_math")]
    for unit, extra in UNITS:
        obj = os.path.join(CSRC, unit.replace(".cu", ".o"))
        if unit == "cw_ifit.cu" and os.environ.get("CW_IFIT_FINE_TIMERS"):
            extra = extra + ["-DCW_IFIT_FINE_TIMERS"]  # per-step timers of the lead thread (tools/ifit_phases.py)
        cmd = [nvcc()] + ARCH + common + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, unit), "-o", obj]
        subprocess.check_call(cmd)
        objs.append(obj)
    subprocess.check_call([nvcc()] + ARCH + ["-shared", "-o", SO] + objs)
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
