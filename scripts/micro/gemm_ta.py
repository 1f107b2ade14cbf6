"""E-sized dense layer (M = 252 798, K = N = 128, 3xTF32): the A-in-tensor-memory kernel, forward and dgrad.
Usage: python scripts/micro/gemm_ta.py"""
import os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from lcaonet_b200 import ops  # noqa: E402
from scripts.bench_kernels import timeit  # noqa: E402
M, K, N = 252798, 128, 128
x = torch.randn(M, K, device="cuda"); w = torch.randn(N, K, device="cuda") / K**0.5
y = torch.empty(M, N, device="cuda"); pre = torch.empty(M, N, device="cuda")
P, st = ops.ptr, ops.stream_ptr
m = ops.GEMM_MODES["tf32x3"]
t0 = timeit(lambda: ops._call("lcao_linear_fwd", P(x), K, P(w), None, P(y), N, None, N, M, K, N, 0, m, st()), reps=9)
t1 = timeit(lambda: ops._call("lcao_linear_fwd", P(x), K, P(w), None, P(y), N, P(pre), N, M, K, N, 1, m, st()), reps=9)
t2 = timeit(lambda: ops._call("lcao_linear_dgrad", P(y), N, None, 0, 0, P(w), P(x), K, M, K, N, 0, m, None, st()), reps=9)
print(f"fwd {t0*1e3:.1f} us | fwd+pre+silu {t1*1e3:.1f} us | dgrad {t2*1e3:.1f} us", flush=True)
