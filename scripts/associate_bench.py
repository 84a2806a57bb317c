"""Time of the cross-view association (mpl_associate_people) next to the lifter forward of the same people.

    python scripts/associate_bench.py [--people-total 65536] [--iters 20] [--out profiles/r12_associate_bench.jsonl]

For (V, P) in {(4, 4), (5, 8), (8, 16), (16, 8)}: F = people_total / P frames of the h36m ring (cmu for V = 5) with noisy
detections (2 px / conf Gaussian noise, 10 % confident false detections, 5 % misses), put into random slots by
mpl_synth_people.  CUDA events around `--iters` back-to-back launches of mpl_associate_people after 3 warm-up launches; the
inputs (F P V 17 x 12 bytes of pixels) fit in L2 after the first launch, which is how the evaluation calls it right after
generating them.  Next to it, the same way: mpl_gather_people of the K = P rows and the bf16 forward of the cmu0 lifter
(depth 2, V views) on the F P gathered rows.  Every line carries the GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from openmpl_b200 import evaluate, inputs, spec, synth  # noqa: E402
from openmpl_b200.models.multiview_mpl_b200 import MultiView_MPL  # noqa: E402
from triangulate_robust_bench import gpu_identity  # noqa: E402

SHAPES = [(4, 4), (5, 8), (8, 16), (16, 8)]


def events_ms(fn, iters: int, warmup: int = 3) -> float:
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


def bench(V: int, P: int, total: int, iters: int) -> dict:
    kind = "cmu" if V == 5 else "h36m"
    F = total // P
    rig = synth.make_rig(V, kind)
    pix, _, calib = inputs.synth_project(F * P, rig, seed=1)
    inputs.add_detector_noise(pix, calib, 1, 0, 2.0, 0.1, 0.05)
    scene, perm = inputs.synth_people(pix, P, 1, 0)
    out = {}
    ms = events_ms(lambda: out.update(r=inputs.associate_people(scene, calib)), iters)
    members, labels, people = out["r"]
    _, acc = inputs.association_score(members, labels, perm)
    a = acc.cpu().numpy()
    gms = events_ms(lambda: inputs.gather_people(scene, members), iters)
    rows = inputs.gather_people(scene, members).view(F * P, V, 17, 3)
    line = {"V": V, "P": P, "frames": F, "people": F * P, "rig": kind, "noise": "2 px / conf, 10 % outliers, 5 % misses",
            "associate_ms": ms, "frames_per_s": F / (ms / 1e3), "people_per_s": F * P / (ms / 1e3), "gather_ms": gms,
            "pair_precision": float(a[6] / a[5]), "pair_recall": float(a[6] / a[7]),
            "complete_fraction": float(a[4] / a[1]), "mean_people_per_frame": float(people.float().mean())}
    kw = dict(num_joints=17, embed_dim_ratio=32, num_heads=8, depth=2, num_views=V, drop_path_rate=0.1,
              **evaluate.ARCHS["cmu0"])
    try:
        model = MultiView_MPL(**kw, precision="bf16")
        model.load_state_dict({k: torch.from_numpy(v) for k, v in
                               synth.named_weights(spec.param_spec(spec.make_config(**kw)), seed=0).items()})
        model = model.cuda().eval()
        p, r, c = inputs.build_inputs(rows, calib)
        with torch.no_grad():
            fms = events_ms(lambda: model(p, rays=r, centers=c), iters)
        line.update(lifter="cmu0 depth 2 bf16", lifter_forward_ms=fms, lifter_people_per_s=F * P / (fms / 1e3))
    except Exception as e:                             # a view count the lifter does not serve: say so in the line
        line.update(lifter="cmu0 depth 2 bf16", lifter_forward_ms=None, lifter_error=f"{type(e).__name__}: {e}")
    return line


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--people-total", type=int, default=65536)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args(argv)
    ident = gpu_identity()
    lines = []
    for V, P in SHAPES:
        line = {**bench(V, P, a.people_total, a.iters), **ident}
        print(json.dumps(line), flush=True)
        lines.append(line)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
