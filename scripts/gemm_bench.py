"""Microbenchmark of the tcgen05 projection kernel on the four FPT shapes (CUDA events, L2-cold inputs by size).

    python scripts/gemm_bench.py [--dtype bf16|tf32] [--rows 131072] [--iters 10] [--shapes qkv,proj,fc1,fc2]
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from openmpl_b200 import _lib  # noqa: E402

p = argparse.ArgumentParser()
p.add_argument("--dtype", default="bf16")
p.add_argument("--rows", type=int, default=131072)
p.add_argument("--iters", type=int, default=10)
p.add_argument("--shapes", default="qkv,proj,fc1,fc2")
p.add_argument("--D", type=int, default=1088)
a = p.parse_args()
L = _lib.lib()
D, M = a.D, a.rows
shapes = {"qkv": (3 * D, D, 0, 0), "proj": (D, D, 2, 1), "fc1": (2 * D, D, 1, 0), "fc2": (D, 2 * D, 2, 1)}
split = a.dtype == "tf32"      # fp32-grade mode: two bf16 planes per matrix
mk = lambda x: torch.stack([x.to(torch.bfloat16), (x - x.to(torch.bfloat16).float()).to(torch.bfloat16)]).contiguous() if split else x.to(torch.bfloat16)
stream = torch.cuda.current_stream().cuda_stream
for name in a.shapes.split(","):
    N, K, epi, out_fp32 = shapes[name]
    A = mk(torch.randn(M, K, device="cuda"))
    W = mk(torch.randn(N, K, device="cuda") / K ** 0.5)
    bias = torch.randn(N, device="cuda")
    Y = torch.zeros(M, N, device="cuda", dtype=torch.float32) if out_fp32 else torch.zeros((2 if split else 1) * M, N, device="cuda", dtype=torch.bfloat16)
    run = lambda: _lib.check(L.mpl_test_gemm(A.data_ptr(), W.data_ptr(), bias.data_ptr(), Y.data_ptr(), M, N, K,
                                             _lib.PRECISIONS[a.dtype], epi, out_fp32, stream))
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.iters):
        run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / a.iters
    print(f"{a.dtype} {name:5s} M={M} N={N} K={K} epi={epi}: {ms:.3f} ms  {2.0 * M * N * K / ms / 1e9:.1f} TFLOP/s", flush=True)
