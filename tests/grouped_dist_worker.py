"""Worker of tests/test_grouped_metrics_cpu.py: one process per rank (gloo, CPU).  Each rank fills grouped MPJPE and masked
P-MPJPE accumulators with its own oracle sums (no GPU here), all-reduces once, and rank 0 writes the reduced tensors."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import masked_pmpjpe_oracle as mpo  # noqa: E402
from openmpl_b200 import dist as mdist, metric  # noqa: E402
from test_grouped_metrics_cpu import rank_batch  # noqa: E402


def main():
    out_path, G = sys.argv[1], int(sys.argv[2])
    rank, world, _ = mdist.init_from_env("gloo")
    pred, gt, group, mask = rank_batch(rank)
    acc = metric.MpjpeAccumulator(17, device="cpu", num_groups=G)
    acc.acc += torch.from_numpy(mpo.grouped_metric_sums(pred, gt, group, G))
    acc.all_reduce()
    pacc = metric.PmpjpeAccumulator(17, device="cpu", num_groups=G)
    pacc.acc += torch.from_numpy(mpo.masked_pmpjpe_sums(pred, gt, mask, group, G))
    pacc.all_reduce()
    if rank == 0:
        json.dump({"world": world, "mpjpe": acc.acc.tolist(), "pmpjpe": pacc.acc.tolist()}, open(out_path, "w"))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
