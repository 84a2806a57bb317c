"""Kernel time of mpl_triangulate (linear multi-view triangulation) at a batch well over the L2.

    python scripts/triangulate_bench.py [--poses 1048576] [--iters 20] [--out FILE]

For V in {2, 4, 5, 8} on the h36m and cmu rigs, plus the evaluation's 65 536-pose micro-batch (hm0, V = 4): device
synthetic pixels (`inputs.synth_project`), warm-up launches, then CUDA events around `--iters` back-to-back launches.
B = 1 048 576 poses makes pix 816 MB at V = 4, so every launch streams its input from HBM (L2 is 126 MB).
One JSON line per configuration: ms per launch, poses/s, and bytes/s over the algorithmic bytes (V J 12 in, J 16 out per
pose) with that rate's share of the 7.7 TB/s HBM3e data-sheet figure, next to the GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from openmpl_b200 import inputs, synth  # noqa: E402

HBM_BYTES_PER_S = 7.7e12        # HGX B200 data sheet, one GPU


def gpu_identity() -> dict:
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        power, clock = [x.strip() for x in q.stdout.strip().split(",")]
    except (OSError, ValueError, subprocess.SubprocessError):
        power, clock = "unknown", "unknown"
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def measure(kind: str, V: int, B: int, iters: int, warmup: int) -> dict:
    rig = synth.make_rig(V, kind)
    pix, _, calib = inputs.synth_project(B, rig, seed=1)
    J = pix.shape[2]
    for _ in range(warmup):
        points, used = inputs.triangulate(pix, calib)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        inputs.triangulate(pix, calib)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    nbytes = B * (V * J * 12 + J * 16)
    return {"kernel": "triangulate_kernel", "rig": kind, "V": V, "J": J, "poses": B, "iters": iters, "ms": ms,
            "poses_per_s": B / (ms / 1e3), "algorithmic_bytes": nbytes, "bytes_per_s": nbytes / (ms / 1e3),
            "hbm_share": nbytes / (ms / 1e3) / HBM_BYTES_PER_S,
            "under_determined_share": float((used < 2).float().mean())}


def main(argv=None):
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--poses", type=int, default=1 << 20)
    p.add_argument("--iters", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = p.parse_args(argv)
    if a.iters < 20:
        p.error("--iters must be at least 20")
    if not torch.cuda.is_available():
        sys.exit("triangulate_bench.py needs a CUDA device")
    ident = gpu_identity()
    configs = [(k, V, a.poses) for k in ("h36m", "cmu") for V in (2, 4, 5, 8)] + [("h36m", 4, 65536)]
    out = open(a.out, "a") if a.out else None
    for kind, V, B in configs:
        line = json.dumps({**measure(kind, V, B, a.iters, a.warmup), **ident})
        print(line, flush=True)
        if out:
            out.write(line + "\n")
        torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
