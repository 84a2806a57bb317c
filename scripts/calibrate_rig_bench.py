"""Cost and effect of rig calibration: the time of mpl_calibrate_rig and the evaluation under calibration errors with and
without recalibration.

    python scripts/calibrate_rig_bench.py [--poses 262144] [--repeats 3] [--out-prefix profiles/r11]

timing (PREFIX_calibrate_rig_bench.jsonl): for N in {1024, 4096, 16384, 65536} poses and V in {2, 4, 8, 16} views of the h36m
ring, device synthetic pixels (1 px detector noise), the rig perturbed by 0.5 deg / 20 mm and init = the linear
triangulation under it; CUDA events around whole `inputs.calibrate_rig` calls (after one warm-up call of the same shape),
the median of `--repeats`.  ms_total is the call with max_iters = CALIBRATE_MAX_ITERS, as the evaluation makes it; it stops
after k iterations, and the launches after the stop return at once.  The call is deterministic, so max_iters = k runs the
same k iterations with no idle launch: ms_per_iteration = (t(k) - t(1)) / (k - 1), and ms_fixed = t(1) - ms_per_iteration
is the rest (item selection, mu0, outputs, workspace allocation).
evaluation (PREFIX_calibrate_rig_eval.jsonl): `evaluate.run` of hm0, V = 4, depth 2, `--poses` poses, 1 px detector noise,
--triangulate --triangulation-pmpjpe, at calibration noise 0; 0.25 deg, 10 mm; 1 deg, 50 mm, each with the perturbed rig
and recalibrated on 16384 poses.  The lifter has random-init weights: its MPJPE measures how its inputs move, not a
trained accuracy.
Every line carries the GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from openmpl_b200 import evaluate, inputs, synth  # noqa: E402
from triangulate_robust_bench import gpu_identity  # noqa: E402


def timing(V: int, N: int, repeats: int) -> dict:
    rig = synth.make_rig(V, "h36m")
    pix, _, calib = inputs.synth_project(N, rig, seed=1)
    inputs.add_detector_noise(pix, calib, 1, 0, 1.0, 0.0, 0.0)
    noisy = inputs.calibration_noise(calib, 7, 0, math.radians(0.5), 0.02)
    init = inputs.triangulate(pix, noisy)[0]

    def median_ms(max_iters):
        run = lambda: inputs.calibrate_rig(pix, noisy, init, sigma_rot=math.radians(0.5), sigma_pos=0.02,
                                           max_iters=max_iters)
        run()
        times = []
        for _ in range(repeats):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _, _, rep = run()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        return float(np.median(times)), rep.cpu().numpy()

    total, rep = median_ms(evaluate.CALIBRATE_MAX_ITERS)
    k = int(rep[6])
    t1, _ = median_ms(1)
    tk, rep_k = median_ms(k) if k > 1 else (t1, rep)
    assert int(rep_k[6]) == k
    per_it = (tk - t1) / (k - 1) if k > 1 else float("nan")
    return {"V": V, "poses": N, "items": int(rep[0]), "observations": int(rep[1]), "iterations": k, "accepted": int(rep[7]),
            "rms_px": [float(rep[4]), float(rep[5])], "ms_total": total, "ms_per_iteration": per_it,
            "ms_fixed": t1 - per_it, "ms_max_iters_k": tk, "ms_max_iters_1": t1}


def main():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--poses", type=int, default=262144)
    p.add_argument("--repeats", type=int, default=3)
    p.add_argument("--out-prefix", default="profiles/r11")
    a = p.parse_args()
    ident = gpu_identity()
    with open(f"{a.out_prefix}_calibrate_rig_bench.jsonl", "w") as f:
        for V in (2, 4, 8, 16):
            for N in (1024, 4096, 16384, 65536):
                line = {**timing(V, N, a.repeats), **ident}
                print(json.dumps(line), flush=True)
                f.write(json.dumps(line) + "\n")
    kw = dict(arch="hm0", views=4, depth=2, poses=a.poses, micro_batch=65536, precision="bf16", triangulate=True,
              triangulation_pmpjpe=True, pixel_noise=1.0)
    with open(f"{a.out_prefix}_calibrate_rig_eval.jsonl", "w") as f:
        for noise in ((0.0, 0.0), (0.25, 10.0), (1.0, 50.0)):
            for cal in ((0,) if noise[0] == 0 else (0, 16384)):
                line = evaluate.run(**kw, calib_noise=noise, calibrate_rig=cal)
                t = line["triangulation"]
                out = {"calib_noise": {"deg": noise[0], "mm": noise[1]}, "calibrate_rig_poses": cal,
                       "lifter_mpjpe_cm": line["mpjpe_cm"]["absolute"],
                       "lifter_p_mpjpe_cm": line["mpjpe_cm"]["procrustes_aligned"],
                       "triangulation_mpjpe_cm": t["mpjpe_cm"]["absolute"],
                       "triangulation_p_mpjpe_cm": t["procrustes_aligned"]["p_mpjpe_cm"],
                       "rig_calibration": line.get("rig_calibration"), "ms_total": line["ms_total"], **ident}
                print(json.dumps(out), flush=True)
                f.write(json.dumps(out) + "\n")


if __name__ == "__main__":
    main()
