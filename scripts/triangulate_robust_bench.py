"""Kernel time of mpl_triangulate_robust next to mpl_triangulate on the same noisy detections, at a batch well over the L2.

    python scripts/triangulate_robust_bench.py [--poses 1048576] [--iters 20] [--out FILE]

For V in {2, 4, 5, 8, 16} on the h36m and cmu rigs, plus the evaluation's 65 536-pose micro-batch (hm0, V = 4): device
synthetic pixels (`inputs.synth_project`) corrupted on the device (`inputs.add_detector_noise`: sigma = 2 px / conf, 10 %
confident false detections, no misses), warm-up launches, then CUDA events around `--iters` back-to-back launches of each
kernel.  One JSON line per configuration: ms per launch and poses/s of both kernels, the robust / linear time ratio, the
number of two-view hypotheses per item (V (V - 1) / 2), the detector-noise kernel's time for the same pixels, and the
GPU name and power limit read in the same run.
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

SIGMA_PX, P_OUTLIER = 2.0, 0.10


def gpu_identity() -> dict:
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        power, clock = [x.strip() for x in q.stdout.strip().split(",")]
    except (OSError, ValueError, subprocess.SubprocessError):
        power, clock = "unknown", "unknown"
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def _time(fn, iters: int, warmup: int) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def measure(kind: str, V: int, B: int, iters: int, warmup: int) -> dict:
    rig = synth.make_rig(V, kind)
    clean, target, calib = inputs.synth_project(B, rig, seed=1)
    pix = clean.clone()
    inputs.add_detector_noise(pix, calib, 1, 0, SIGMA_PX, P_OUTLIER, 0.0)
    J = pix.shape[2]
    scratch = clean.clone()
    ms_noise = _time(lambda: inputs.add_detector_noise(scratch, calib, 1, 0, SIGMA_PX, P_OUTLIER, 0.0), iters, warmup)
    del scratch
    ms_lin = _time(lambda: inputs.triangulate(pix, calib), iters, warmup)
    ms_rob = _time(lambda: inputs.triangulate_robust(pix, calib), iters, warmup)
    lin, used = inputs.triangulate(pix, calib)
    rob, inl = inputs.triangulate_robust(pix, calib)
    err_l = (lin - target).norm(dim=-1)[used >= 2]
    err_r = (rob - target).norm(dim=-1)[inl != 0]
    return {"kernel": "triangulate_robust_kernel", "rig": kind, "V": V, "J": J, "poses": B, "iters": iters,
            "pixel_noise_px": SIGMA_PX, "outlier_rate": P_OUTLIER, "pairs_per_item": V * (V - 1) // 2,
            "ms": ms_rob, "poses_per_s": B / (ms_rob / 1e3),
            "linear_ms": ms_lin, "linear_poses_per_s": B / (ms_lin / 1e3), "robust_over_linear": ms_rob / ms_lin,
            "noise_ms": ms_noise,
            "median_err_cm": {"robust": float(err_r.median()) * 100, "linear": float(err_l.median()) * 100},
            "rejected_share": float(((inl == 0) & (used >= 2)).float().mean())}


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
        sys.exit("triangulate_robust_bench.py needs a CUDA device")
    ident = gpu_identity()
    configs = [(k, V, a.poses) for k in ("h36m", "cmu") for V in (2, 4, 5, 8, 16)] + [("h36m", 4, 65536)]
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
