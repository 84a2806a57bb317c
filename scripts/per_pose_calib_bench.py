"""Kernel time of every calibration-taking entry point with one shared calibration and with a calibration per pose, on
the same pixels, at a batch well over the L2; plus the random camera generator alone.

    python scripts/per_pose_calib_bench.py [--poses 1048576] [--iters 20] [--out FILE]

For V in {2, 4, 5, 8, 16} on the h36m rig: device synthetic pixels (`inputs.synth_project`) corrupted on the device
(`inputs.add_detector_noise`: sigma = 2 px / conf, 10 % confident false detections, no misses).  The per-pose calibration
is the rig repeated in every row of a [B, V, 18] tensor, so both paths do the same arithmetic on the same data (their
results are bitwise equal) and the difference is what reading and staging a calibration per pose costs.  Warm-up
launches, then CUDA events around `--iters` back-to-back launches of each consumer: mpl_build_inputs, mpl_synth_project,
mpl_synth_detector_noise (in place on a scratch copy), mpl_triangulate and mpl_triangulate_robust, and mpl_synth_cameras.
One JSON line per (V, consumer): ms per launch for both paths, their ratio, the extra calibration bytes per pose (144 V)
and the GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from openmpl_b200 import inputs, synth  # noqa: E402
from triangulate_robust_bench import gpu_identity, _time  # noqa: E402

SIGMA_PX, P_OUTLIER = 2.0, 0.10


def measure(V: int, B: int, iters: int, warmup: int) -> list:
    rig = synth.make_rig(V, "h36m")
    clean, _, calib = inputs.synth_project(B, rig, seed=1)
    tiled = calib.expand(B, V, 18).contiguous()
    pix = inputs.add_detector_noise(clean.clone(), calib, 1, 0, SIGMA_PX, P_OUTLIER, 0.0)
    J = pix.shape[2]
    scratch = clean.clone()
    consumers = {
        "build_inputs": lambda c: inputs.build_inputs(pix, c),
        "synth_project": lambda c: inputs.synth_project(B, rig, seed=1, cameras=c if c.dim() == 3 else None),
        "detector_noise": lambda c: inputs.add_detector_noise(scratch, c, 1, 0, SIGMA_PX, P_OUTLIER, 0.0),
        "triangulate": lambda c: inputs.triangulate(pix, c),
        "triangulate_robust": lambda c: inputs.triangulate_robust(pix, c),
    }
    lines = []
    for name, fn in consumers.items():
        ms_shared = _time(lambda: fn(calib), iters, warmup)
        ms_pose = _time(lambda: fn(tiled), iters, warmup)
        lines.append({"consumer": name, "V": V, "J": J, "poses": B, "iters": iters, "ms_shared": ms_shared,
                      "ms_per_pose": ms_pose, "per_pose_over_shared": ms_pose / ms_shared,
                      "calib_bytes_per_pose": 144 * V})
        torch.cuda.empty_cache()
    del scratch, tiled
    ms_cam = _time(lambda: inputs.synth_cameras(B, V, "h36m", seed=1), iters, warmup)
    lines.append({"consumer": "synth_cameras", "V": V, "poses": B, "iters": iters, "ms": ms_cam,
                  "bytes_written_per_pose": 144 * V, "write_GBps": B * 144 * V / (ms_cam / 1e3) / 1e9})
    return lines


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
        sys.exit("per_pose_calib_bench.py needs a CUDA device")
    ident = gpu_identity()
    out = open(a.out, "a") if a.out else None
    for V in (2, 4, 5, 8, 16):
        for rec in measure(V, a.poses, a.iters, a.warmup):
            line = json.dumps({**rec, **ident})
            print(line, flush=True)
            if out:
                out.write(line + "\n")
        torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
