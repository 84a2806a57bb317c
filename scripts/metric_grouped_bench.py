"""Kernel time of the grouped MPJPE and the masked / grouped P-MPJPE accumulators next to their ungrouped kernels.

    python scripts/metric_grouped_bench.py [--poses 1048576] [--iters 20] [--out FILE]

B = 1 048 576 poses of J = 17 joints (random fp32 poses on the device, 428 MB of pred + gt, well over the L2), each
accumulating into a zeroed fp64 buffer.  Warm-up launches, then CUDA events around `--iters` back-to-back launches of:
`mpl_mpjpe_accumulate`; `mpl_mpjpe_accumulate_grouped` with G = 1, G = 15 sorted (a DataLoader over one action at a time),
G = 15 shuffled (shared block sums) and G = 4 096 shuffled (global atomics); `mpl_pmpjpe_accumulate`;
`mpl_pmpjpe_accumulate_masked` with every joint used, with 20 % of the joints masked off, and with G = 15 shuffled.  One
JSON line per case: ms per launch, the algorithmic bytes per pose (pred, gt, and the group and mask entries it reads) and
the rate they move at, the ratio to the case's base kernel, and the GPU's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from openmpl_b200 import _lib  # noqa: E402
from triangulate_robust_bench import gpu_identity, _time  # noqa: E402

J = 17


def cases(B: int):
    gen = torch.Generator(device="cuda").manual_seed(0)
    gt = torch.randn(B, J, 3, device="cuda", generator=gen) * 0.3
    pred = gt + 0.05 * torch.randn(B, J, 3, device="cuda", generator=gen)
    g15 = torch.randint(0, 15, (B,), device="cuda", generator=gen, dtype=torch.int32)
    g4k = torch.randint(0, 4096, (B,), device="cuda", generator=gen, dtype=torch.int32)
    sorted15 = torch.sort(g15).values.contiguous()
    ones = torch.ones(B, J, device="cuda")
    off20 = (torch.rand(B, J, device="cuda", generator=gen) >= 0.2).float()
    L = _lib.lib()
    s = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
    p, g = pred.data_ptr(), gt.data_ptr()
    pose = 2 * J * 3 * 4

    def mpjpe(G, grp):
        acc = torch.zeros(max(G, 1), 11 * J + 1, dtype=torch.float64, device="cuda")
        if G == 0:
            return acc, lambda: _lib.check(L.mpl_mpjpe_accumulate(p, g, None, B, J, 100.0, None, acc.data_ptr(), s()))
        gp = None if grp is None else grp.data_ptr()
        return acc, lambda: _lib.check(L.mpl_mpjpe_accumulate_grouped(p, g, None, gp, G, B, J, 100.0, None, acc.data_ptr(), s()))

    def pmpjpe(G, mask, grp):
        if G == 0:
            acc = torch.zeros(J + 3, dtype=torch.float64, device="cuda")
            return acc, lambda: _lib.check(L.mpl_pmpjpe_accumulate(p, g, B, J, 100.0, 1, -1, acc.data_ptr(), s()))
        acc = torch.zeros(G, 2 * J + 4, dtype=torch.float64, device="cuda")
        mp, gp = None if mask is None else mask.data_ptr(), None if grp is None else grp.data_ptr()
        return acc, lambda: _lib.check(L.mpl_pmpjpe_accumulate_masked(p, g, mp, gp, G, B, J, 100.0, 1, -1, acc.data_ptr(), s()))

    keep = (pred, gt, g15, g4k, sorted15, ones, off20)
    yield "mpjpe", "ungrouped", None, pose, *mpjpe(0, None), keep
    yield "mpjpe_grouped", "G=1", "ungrouped", pose, *mpjpe(1, None), keep
    yield "mpjpe_grouped", "G=15 sorted", "ungrouped", pose + 4, *mpjpe(15, sorted15), keep
    yield "mpjpe_grouped", "G=15 shuffled", "ungrouped", pose + 4, *mpjpe(15, g15), keep
    yield "mpjpe_grouped", "G=4096 shuffled (global atomics)", "ungrouped", pose + 4, *mpjpe(4096, g4k), keep
    yield "pmpjpe", "unmasked", None, pose, *pmpjpe(0, None, None), keep
    yield "pmpjpe_masked", "every joint used", "unmasked", pose + 4 * J, *pmpjpe(1, ones, None), keep
    yield "pmpjpe_masked", "20% of joints off", "unmasked", pose + 4 * J, *pmpjpe(1, off20, None), keep
    yield "pmpjpe_masked", "G=15 shuffled, every joint used", "unmasked", pose + 4 * J + 4, *pmpjpe(15, ones, g15), keep


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--poses", type=int, default=1 << 20)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args(argv)
    if not torch.cuda.is_available():
        sys.exit("metric_grouped_bench.py needs a CUDA device")
    ident = gpu_identity()
    out = open(a.out, "a") if a.out else None
    base = {}
    for kernel, case, base_case, bytes_per_pose, acc, fn, _ in cases(a.poses):
        ms = _time(fn, a.iters, a.warmup)
        if base_case is None:
            base[kernel] = ms
        ref = base["mpjpe" if kernel.startswith("mpjpe") else "pmpjpe"]
        line = json.dumps({"kernel": kernel, "case": case, "poses": a.poses, "J": J, "iters": a.iters, "ms": ms,
                           "bytes_per_pose": bytes_per_pose, "TBps": a.poses * bytes_per_pose / (ms / 1e3) / 1e12,
                           "over_base": ms / ref, **ident})
        print(line, flush=True)
        if out:
            out.write(line + "\n")
    if out:
        out.close()


if __name__ == "__main__":
    main()
