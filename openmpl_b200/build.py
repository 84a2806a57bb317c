"""Build libmpl_b200.so (hand-written CUDA for sm_100a) in-tree with nvcc.

    python -m openmpl_b200.build [--force]

The library has no torch dependency: it links the CUDA runtime only and resolves the one driver entry point it needs
(cuTensorMapEncodeTiled) at run time, so it builds on a machine without a GPU or driver.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.environ.get("MPL_B200_BUILD_LIB") or os.path.join(HERE, "libmpl_b200.so")
SOURCES = ["model.cu", "kernels_generic.cu", "gemm_tcgen05.cu", "metric_inputs.cu", "spt_fused.cu", "io_kernels.cu",
           "calibrate_rig.cu", "associate.cu", "track.cu"]
HEADERS = ["common.cuh", "kernels.cuh", "ptx.cuh", "so3.cuh", "shared.cuh", os.path.join("..", "..", "include", "mpl_b200.h")]
# per-file extra nvcc flags; MPL_GEMM_DEFS="-DMPL_LN_STAGES=6 ..." builds an experiment variant of the GEMM kernel
EXTRA_FLAGS = {"gemm_tcgen05.cu": os.environ.get("MPL_GEMM_DEFS", "").split(),
               "spt_fused.cu": os.environ.get("MPL_SPT_DEFS", "").split()}
# second compilation of spt_fused.cu: the 16-set / 9-warp shape, exporting launch_fpt_kp_fused_alt only (see the file's header)
VARIANTS = [("spt_fused.cu", "spt_fused_alt.o", ["-DMPL_SPT_ALT"])]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
              "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found; libmpl_b200.so cannot be built")


def _stale(target: str, deps: list) -> bool:
    if not os.path.isfile(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.isfile(d))


def build(force: bool = False, verbose: bool = False) -> str:
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.isfile(os.path.join(CSRC, s))]
    hdrs = [os.path.normpath(os.path.join(CSRC, h)) for h in HEADERS]
    objdir = os.path.join(CSRC, "build")
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()
    objs, procs = [], []
    # (source, object name, extra flags): every source once, plus the second shape of the single-kernel transformer
    units = [(s, os.path.basename(s)[:-3] + ".o", EXTRA_FLAGS.get(os.path.basename(s), [])) for s in srcs]
    units += [(os.path.join(CSRC, s), o, f) for s, o, f in VARIANTS if os.path.isfile(os.path.join(CSRC, s))]
    for s, oname, flags in units:
        o = os.path.join(objdir, oname)
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            log = open(o + ".log", "w")
            procs.append((s, log, subprocess.Popen([nvcc, *NVCC_FLAGS, *flags, "-c", s, "-o", o], stdout=log, stderr=subprocess.STDOUT)))
    failed = []
    for s, log, p in procs:
        rc = p.wait()
        log.close()
        text = open(log.name).read()
        if verbose or rc != 0:
            print(text)
        if rc != 0:
            failed.append(s)
    if failed:
        raise RuntimeError("nvcc failed for: " + ", ".join(failed))
    if force or procs or _stale(LIB, objs):
        subprocess.check_call([nvcc, "-shared", "-o", LIB, *objs, "-lcudart"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
