"""Kernel time of mpl_triangulate_refine next to mpl_triangulate on the same noisy detections, at a batch well over the L2.

    python scripts/triangulate_refine_bench.py [--poses 1048576] [--iters 20] [--out FILE]

For V in {2, 4, 5, 8, 16} on the h36m rig: device synthetic pixels (`inputs.synth_project`) corrupted on the device
(`inputs.add_detector_noise`: sigma = 2 px / conf, 10 % confident false detections, no misses), triangulated by both
kernels.  Warm-up launches, then CUDA events around `--iters` back-to-back launches of: the linear kernel; the refinement
of the linear points over every candidate view; the refinement of the robust points over their inliers; both
refinements again with the rig repeated in a [B, V, 18] calibration per pose.  The refinements run with the default cap
of 20 iterations.  One JSON line per V: ms per launch, the refine / linear ratios, the algorithmic bytes per pose and the
rate they move at, the mean joint error before and after each refinement, and the GPU name and power limit read in the
same run.
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


def _mean_cm(points, target, mask):
    return float((points - target).norm(dim=-1)[mask].mean()) * 100


def measure(V: int, B: int, iters: int, warmup: int) -> dict:
    rig = synth.make_rig(V, "h36m")
    pix, target, calib = inputs.synth_project(B, rig, seed=1)
    inputs.add_detector_noise(pix, calib, 1, 0, SIGMA_PX, P_OUTLIER, 0.0)
    J = pix.shape[2]
    tiled = calib.expand(B, V, 18).contiguous()
    lin, used = inputs.triangulate(pix, calib)
    rob, inl = inputs.triangulate_robust(pix, calib)
    ms = {"linear_ms": _time(lambda: inputs.triangulate(pix, calib), iters, warmup)}
    for name, c in (("", calib), ("_per_pose", tiled)):
        ms[f"refine_linear{name}_ms"] = _time(lambda: inputs.refine_triangulation(pix, c, lin), iters, warmup)
        ms[f"refine_robust{name}_ms"] = _time(lambda: inputs.refine_triangulation(pix, c, rob, view_mask=inl), iters, warmup)
    ref_lin, rp_lin = inputs.refine_triangulation(pix, calib, lin)
    ref_rob, rp_rob = inputs.refine_triangulation(pix, calib, rob, view_mask=inl)
    # pixels, init, mask in; points, reproj_px out (the linear refinement reads no mask)
    bytes_per_pose = V * J * 12 + J * (12 + 4 + 12 + 4)
    return {"kernel": "triangulate_refine_kernel", "rig": "h36m", "V": V, "J": J, "poses": B, "iters": iters,
            "pixel_noise_px": SIGMA_PX, "outlier_rate": P_OUTLIER, "max_iters": 20, **ms,
            "refine_linear_over_linear": ms["refine_linear_ms"] / ms["linear_ms"],
            "refine_robust_over_linear": ms["refine_robust_ms"] / ms["linear_ms"],
            "bytes_per_pose": bytes_per_pose,
            "refine_robust_TBps": B * bytes_per_pose / (ms["refine_robust_ms"] / 1e3) / 1e12,
            "mean_err_cm": {"linear": _mean_cm(lin, target, used >= 2), "linear_refined": _mean_cm(ref_lin, target, used >= 2),
                            "robust": _mean_cm(rob, target, inl != 0), "robust_refined": _mean_cm(ref_rob, target, inl != 0)},
            "refined_share": {"linear": float((~torch.isnan(rp_lin))[used >= 2].float().mean()),
                              "robust": float((~torch.isnan(rp_rob))[inl != 0].float().mean())}}


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
        sys.exit("triangulate_refine_bench.py needs a CUDA device")
    ident = gpu_identity()
    out = open(a.out, "a") if a.out else None
    for V in (2, 4, 5, 8, 16):
        line = json.dumps({**measure(V, a.poses, a.iters, a.warmup), **ident})
        print(line, flush=True)
        if out:
            out.write(line + "\n")
        torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
