"""Cost and effect of lens distortion: kernel times of mpl_distort_pixels / mpl_undistort_pixels next to mpl_triangulate,
the triangulation error on distorted detections with and without undistortion, and the evaluation with and without
--lens-distortion.

    python scripts/lens_distortion_bench.py [--poses 1048576] [--iters 20] [--out-prefix profiles/r10]

kernels (PREFIX_lens_kernels.jsonl): for both rigs (each with its lens of LENSES) and V in {2, 4, 5, 8, 16}, device synthetic
pixels of `--poses` poses, distorted; CUDA events around `--iters` back-to-back launches (after warm-up) of the distortion
and the undistortion (out of place, margin half the image), with one calibration for the batch and with the rig repeated
in a [B, V, 18] calibration per pose, and of mpl_triangulate on the same pixels.  Bytes are the algorithmic traffic
(12 B read + 12 B written per entry, plus 144 B of calibration per pose and view when it is per pose); the rate is set
against the B200's 7.7 TB/s HBM.
errors (PREFIX_lens_triangulation.jsonl): V = 4 on both rigs, exact and noisy (sigma = 2 px / conf, 10 % outliers)
distorted detections: mean joint error of the linear, robust and refined (linear over the candidates, robust over its
inliers) triangulations of (a) the raw pixels with the pinhole calibration and (b) the undistorted pixels with the
shifted calibration.
evaluation (PREFIX_lens_eval.jsonl): `evaluate.run` of hm0, V = 4, `--poses` poses, detector noise, every triangulation
flag, without and with --lens-distortion (the h36m lens).
Every line carries the GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from openmpl_b200 import _lib, evaluate, inputs, synth  # noqa: E402
from triangulate_robust_bench import gpu_identity, _time  # noqa: E402

# illustrative coefficient sets (k1, k2, p1, p2, k3): H36M's magnitude on the h36m rig, a stronger one on the cmu rig
LENSES = {"h36m": (-0.207, 0.248, -0.0009, -0.0016, -0.0031), "cmu": (-0.30, 0.10, 0.001, -0.001, 0.0)}
HBM_TBPS = 7.7


def _lens_call(undistort, pin, pout, calib, cstride, dist, dstride, mx, my):
    B, V, J, _ = pin.shape
    s = torch.cuda.current_stream().cuda_stream
    L = _lib.lib()
    if undistort:
        st = L.mpl_undistort_pixels_strided(pin.data_ptr(), pout.data_ptr(), calib.data_ptr(), cstride, dist.data_ptr(),
                                            dstride, mx, my, B, V, J, s)
    else:
        st = L.mpl_distort_pixels_strided(pin.data_ptr(), pout.data_ptr(), calib.data_ptr(), cstride, dist.data_ptr(),
                                          dstride, B, V, J, s)
    _lib.check(st)


def kernels(kind: str, V: int, B: int, iters: int, warmup: int) -> dict:
    rig = synth.make_rig(V, kind)
    w, h = rig.image_size
    ideal, _, calib = inputs.synth_project(B, rig, seed=1)
    dist = torch.tensor([LENSES[kind]] * V, dtype=torch.float64, device="cuda")
    pix = inputs.distort_pixels(ideal.clone(), calib, dist)
    out = torch.empty_like(pix)
    tiled = calib.expand(B, V, 18).contiguous()
    J = pix.shape[2]
    res = {}
    for name, c, cs in (("shared", calib, 0), ("per_pose", tiled, 18 * V)):
        res[f"distort_{name}_ms"] = _time(lambda: _lens_call(False, ideal, out, c, cs, dist, 0, 0.0, 0.0), iters, warmup)
        res[f"undistort_{name}_ms"] = _time(lambda: _lens_call(True, pix, out, c, cs, dist, 0, w / 2, h / 2), iters, warmup)
    res["triangulate_ms"] = _time(lambda: inputs.triangulate(pix, calib), iters, warmup)
    entries = B * V * J
    rates = {}
    for name in ("shared", "per_pose"):
        nbytes = entries * 24 + (B * V * 144 if name == "per_pose" else 0)
        for op in ("distort", "undistort"):
            rates[f"{op}_{name}_TBps"] = nbytes / (res[f"{op}_{name}_ms"] / 1e3) / 1e12
    und, _ = inputs.undistort_pixels(pix, calib, dist, margin=(w / 2, h / 2))
    live = pix[..., 2] != 0
    return {"kernel": "distort_pixels_kernel / undistort_pixels_kernel", "rig": kind, "lens": LENSES[kind], "V": V, "J": J,
            "poses": B, "iters": iters, **res, **rates, "hbm_TBps": HBM_TBPS,
            "undistort_over_triangulate": res["undistort_shared_ms"] / res["triangulate_ms"],
            "bytes_per_entry": 24, "entries": entries,
            "undistorted_share": float((und[..., 2] != 0)[live].float().mean())}


def _mean_cm(points, target, mask):
    return float((points - target).norm(dim=-1)[mask].mean()) * 100


def _errors(pix, calib, target) -> dict:
    lin, used = inputs.triangulate(pix, calib)
    rob, inl = inputs.triangulate_robust(pix, calib)
    return {"linear": _mean_cm(lin, target, used >= 2), "robust": _mean_cm(rob, target, inl != 0),
            "linear_refined": _mean_cm(inputs.refine_triangulation(pix, calib, lin)[0], target, used >= 2),
            "robust_refined": _mean_cm(inputs.refine_triangulation(pix, calib, rob, view_mask=inl)[0], target, inl != 0),
            "triangulated_share": float((used >= 2).float().mean())}


def triangulation_errors(kind: str, V: int, B: int) -> list:
    rig = synth.make_rig(V, kind)
    w, h = rig.image_size
    dist = torch.tensor([LENSES[kind]] * V, dtype=torch.float64, device="cuda")
    lines = []
    for noise in ((0.0, 0.0), (2.0, 0.1)):
        pix, target, calib = inputs.synth_project(B, rig, seed=1)
        inputs.distort_pixels(pix, calib, dist)
        if noise[0]:
            inputs.add_detector_noise(pix, calib, 1, 0, noise[0], noise[1], 0.0)
        und, calib_u = inputs.undistort_pixels(pix, calib, dist, margin=(w / 2, h / 2))
        lines.append({"rig": kind, "lens": LENSES[kind], "V": V, "poses": B, "pixel_noise_px": noise[0], "outlier_rate": noise[1],
                      "mean_err_cm": {"raw_pixels": _errors(pix, calib, target),
                                      "undistorted_pixels": _errors(und, calib_u, target)}})
    return lines


def evaluation(B: int) -> list:
    kw = dict(arch="hm0", views=4, poses=B, pixel_noise=2.0, outlier_rate=0.1, triangulate=True, triangulate_robust=True,
              refine_triangulations=True, triangulation_pmpjpe=True)
    return [evaluate.run(**kw), evaluate.run(**kw, lens_distortion=LENSES["h36m"])]


def main(argv=None):
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--poses", type=int, default=1 << 20)
    p.add_argument("--iters", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--out-prefix", default=None, help="append the JSON lines to PREFIX_lens_{kernels,triangulation,eval}.jsonl")
    a = p.parse_args(argv)
    if not torch.cuda.is_available():
        sys.exit("lens_distortion_bench.py needs a CUDA device")
    ident = gpu_identity()

    def emit(section, d):
        line = json.dumps({**d, **ident})
        print(line, flush=True)
        if a.out_prefix:
            with open(f"{a.out_prefix}_lens_{section}.jsonl", "a") as f:
                f.write(line + "\n")

    for kind in ("h36m", "cmu"):
        for V in (2, 4, 5, 8, 16):
            emit("kernels", kernels(kind, V, a.poses, a.iters, a.warmup))
            torch.cuda.empty_cache()
    for kind in ("h36m", "cmu"):
        for line in triangulation_errors(kind, 4, a.poses):
            emit("triangulation", line)
    for line in evaluation(a.poses):
        emit("eval", line)


if __name__ == "__main__":
    main()
