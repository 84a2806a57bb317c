"""Time of the motion synthesis (mpl_synth_motion) and the tracking (mpl_track_people) next to the cross-view association of
the same person-frames.

    python scripts/track_bench.py [--person-frames 65536] [--frames 64] [--iters 20] [--out profiles/r13_track_bench.jsonl]

For (V, P) in the association bench's shapes {(4, 4), (5, 8), (8, 16), (16, 8)}: S = person_frames / (T P) sequences of
T = 64 frames on the h36m ring (cmu for V = 5) with noisy detections (2 px / conf Gaussian noise, 10 % confident false
detections, 5 % misses), put into random slots, associated, gathered and robustly triangulated.  CUDA events around `--iters`
back-to-back launches after 3 warm-up launches of: mpl_synth_motion (pixels and targets of all rows), mpl_associate_people,
and mpl_track_people of the K = P rows from a zeroed state (max_tracks = 2 P; the zeroing of the state is timed with it) and
mpl_tracking_score.  The inputs fit in L2 after the first launch, which is how the evaluation calls them right after
generating them.  Every line carries the GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from openmpl_b200 import inputs, synth  # noqa: E402
from associate_bench import SHAPES, events_ms  # noqa: E402
from triangulate_robust_bench import gpu_identity  # noqa: E402


def bench(V: int, P: int, total: int, T: int, iters: int) -> dict:
    kind = "cmu" if V == 5 else "h36m"
    S = total // (T * P)
    rig = synth.make_rig(V, kind)
    out = {}
    sms = events_ms(lambda: out.update(r=inputs.synth_motion(S, T, P, rig, seed=1)), iters)
    pix, _, calib = out["r"]
    inputs.add_detector_noise(pix, calib, 1, 0, 2.0, 0.1, 0.05)
    scene, perm = inputs.synth_people(pix, P, 1, 0)
    ams = events_ms(lambda: out.update(a=inputs.associate_people(scene, calib)), iters)
    members, labels, _ = out["a"]
    owner, _ = inputs.association_score(members, labels, perm)
    points, _ = inputs.triangulate_robust(inputs.gather_people(scene, members).view(S * T * P, V, 17, 3), calib)
    points = points.view(S, T, P, 17, 3)
    owner = owner.view(S, T, P)
    tms = events_ms(lambda: out.update(t=inputs.track_people(points, max_tracks=2 * P)), iters)
    ids = out["t"][0]
    scms = events_ms(lambda: inputs.tracking_score(ids, owner, P), iters)
    a = inputs.tracking_score(ids, owner, P).cpu().numpy()
    return {"V": V, "P": P, "sequences": S, "frames_per_sequence": T, "person_frames": S * T * P, "rig": kind,
            "noise": "2 px / conf, 10 % outliers, 5 % misses", "synth_motion_ms": sms, "associate_ms": ams,
            "track_ms": tms, "tracking_score_ms": scms, "track_person_frames_per_s": S * T * P / (tms / 1e3),
            "mota": float(1 - (a[4] + a[5] + a[6]) / a[2]), "id_switches": int(a[6]), "tracks_per_person": float(a[10] / (S * P)),
            "track_params": {"max_dist_m": 0.2, "max_age": 5, "min_joints": 3, "max_tracks": 2 * P}}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--person-frames", type=int, default=65536)
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args(argv)
    ident = gpu_identity()
    lines = []
    for V, P in SHAPES:
        line = {**bench(V, P, a.person_frames, a.frames, a.iters), **ident}
        print(json.dumps(line), flush=True)
        lines.append(line)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
