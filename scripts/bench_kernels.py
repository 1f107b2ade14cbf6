"""Micro-benchmarks of single C-ABI kernels on the BASELINE configs[1] shapes (CUDA events, L2 flushed
between repetitions by a 512 MB write).  Usage: python scripts/bench_kernels.py [gemm|edge|all]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lcaonet_b200 import _lib, ops  # noqa: E402
from lcaonet_b200.synth import qm9_like_batch  # noqa: E402

DEV = "cuda"
FLUSH = None


def timeit(fn, reps=5, warm=2):
    global FLUSH
    if os.environ.get("LCAO_BENCH_ONCE"):  # one launch per kernel: for ncu captures
        reps, warm = 1, 0
    if FLUSH is None:
        FLUSH = torch.empty(128 * 1024 * 1024, device=DEV)
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        FLUSH.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2]


def gemm_small():
    """latency of the dense-layer kernels at the node / table sized shapes of one step"""
    P, st = ops.ptr, ops.stream_ptr
    for M, K, N in ((128, 128, 128), (2048, 128, 128), (10952, 128, 128), (18470, 128, 128), (18470, 128, 256), (252798, 128, 128)):
        x = torch.randn(M, K, device=DEV)
        w = torch.randn(N, K, device=DEV) / K**0.5
        dy = torch.randn(M, N, device=DEV)
        y, dx = torch.empty(M, N, device=DEV), torch.empty(M, K, device=DEV)
        dw = torch.zeros(N, K, device=DEV)
        for mode in ("fp32", "tf32x3"):
            m = ops.GEMM_MODES[mode]
            n_scr = int(_lib.load().lcao_linear_bwd_scratch(P(dy), N, None, 0, 0, None, P(x), K, None, 0, M, K, N, m))
            scr = torch.empty(max(n_scr, 1), device=DEV)
            t_f = timeit(lambda: ops._call("lcao_linear_fwd", P(x), K, P(w), None, P(y), N, None, N, M, K, N, 0, m, st()), reps=9)
            t_d = timeit(lambda: ops._call("lcao_linear_dgrad", P(dy), N, None, 0, 0, P(w), P(dx), K, M, K, N, 0, m, None, st()), reps=9)
            t_w = timeit(lambda: ops._call("lcao_linear_wgrad", P(dy), N, None, 0, 0, P(x), K, P(dw), None, M, K, N, m, P(scr), st()), reps=9)
            print(f"gemm {mode:7s} M={M:7d} K={K} N={N}: fwd {t_f*1e3:7.1f} us | dgrad {t_d*1e3:7.1f} us | wgrad {t_w*1e3:7.1f} us", flush=True)


def gemm():
    M, K, N = 2_022_384, 128, 128
    x = torch.randn(M, K, device=DEV)
    w = torch.randn(N, K, device=DEV) / K**0.5
    dy = torch.randn(M, N, device=DEV)
    y, pre, dx = torch.empty(M, N, device=DEV), torch.empty(M, N, device=DEV), torch.empty(M, K, device=DEV)
    dw = torch.zeros(N, K, device=DEV)
    P, st = ops.ptr, ops.stream_ptr
    for mode in ("fp32", "tf32x3", "tf32"):
        m = ops.GEMM_MODES[mode]
        t_f = timeit(lambda: ops._call("lcao_linear_fwd", P(x), K, P(w), None, P(y), N, P(pre), N, M, K, N, 1, m, st()))
        t_f0 = timeit(lambda: ops._call("lcao_linear_fwd", P(x), K, P(w), None, P(y), N, None, N, M, K, N, 0, m, st()))
        t_d = timeit(lambda: ops._call("lcao_linear_dgrad", P(dy), N, None, 0, 0, P(w), P(dx), K, M, K, N, 0, m, None, st()))
        t_w = timeit(lambda: ops._call("lcao_linear_wgrad", P(dy), N, None, 0, 0, P(x), K, P(dw), None, M, K, N, m, None, st()))
        gb = lambda nbytes, ms: nbytes / ms / 1e6  # noqa: E731
        fl = 2.0 * M * K * N
        print(f"gemm {mode:7s} M={M} K={K} N={N}: fwd+silu+pre {t_f:.3f} ms ({gb(4*M*(K+2*N), t_f):.0f} GB/s, {fl/t_f/1e9:.0f} TF/s) | "
              f"fwd plain {t_f0:.3f} ms ({gb(4*M*(K+N), t_f0):.0f} GB/s) | dgrad {t_d:.3f} ms ({gb(4*M*(K+N), t_d):.0f} GB/s) | "
              f"wgrad {t_w:.3f} ms ({gb(4*M*(K+N), t_w):.0f} GB/s)", flush=True)


def edge():
    g = qm9_like_batch(1024, seed=1000).to(DEV)
    N, E, C, NL, O = g["z"].shape[0], g["edge_index"].shape[1], 128, 3, 8
    gi = ops.GraphIndex(g["edge_index"], N)
    P, st = ops.ptr, ops.stream_ptr
    # ---- pair-table contraction (f_coeffs evaluated on the (max_z+1)^2 species-pair table)
    Zd = 37
    z = g["z"]
    pair = (z[g["edge_index"][0]] * Zd + z[g["edge_index"][1]]).contiguous()
    tab = torch.randn(Zd * Zd, O, C, device=DEV)
    rb = torch.randn(E, O, device=DEV)
    lgrp = torch.tensor([0, 0, 1, 0, 1, 0, 2, 1], dtype=torch.int32, device=DEV)
    B = torch.empty(E, NL, C, device=DEV)
    gram = torch.empty(E, NL * (NL + 1) // 2, dtype=torch.float64, device=DEV)
    t_pf = timeit(lambda: ops._call("lcao_pair_contract_fwd", P(tab), P(pair), P(rb), None, P(lgrp), E, O, C, NL, 0, P(B), P(gram), None, st()))
    kptr, kperm = ops.bucket_sort(pair, Zd * Zd, stable=False)
    dBr = torch.randn(E, NL, C, device=DEV)
    d_tab = torch.empty_like(tab)
    nbytes = int(_lib.load().lcao_pair_contract_bwd_scratch(E, Zd * Zd, O, C, 0))
    scratch = torch.empty(nbytes // 4 + 4, dtype=torch.int32, device=DEV)
    t_pb = timeit(lambda: ops._call("lcao_pair_contract_bwd", P(tab), P(pair), P(kptr), P(kperm), P(rb), None, P(lgrp), P(dBr), E,
                                    Zd * Zd, O, C, NL, 0, P(d_tab), None, P(scratch), st()))
    bpf = E * (4 * NL * C + 4 * O + 8 + 8 * 6)
    bpb = E * (4 * NL * C + 4 * O + 4)
    print(f"pair_contract E={E}: fwd {t_pf:.3f} ms ({bpf/t_pf/1e6:.0f} GB/s) | bwd {t_pb:.3f} ms ({bpb/t_pb/1e6:.0f} GB/s)", flush=True)
    # ---- three-body
    unit = torch.nn.functional.normalize(torch.randn(E, 3, device=DEV), dim=1)
    xk = torch.sigmoid(torch.randn(N, C, device=DEV))  # gate rows
    tbw, dB, q = torch.empty(E, C, device=DEV), torch.empty(E, NL, C, device=DEV), torch.empty(E, C, device=DEV)
    du1, du2 = torch.empty(E, 3, device=DEV), torch.empty(E, 3, device=DEV)
    d_tbw = torch.randn(E, C, device=DEV)
    args = (P(B), NL, P(gram), P(unit), P(xk), xk.stride(0), P(gi.in_ptr), P(gi.in_edge), P(gi.in_src), P(gi.out_ptr),
            P(gi.out_edge), N, E, C, NL)
    t_f = timeit(lambda: ops._call("lcao_threebody_fwd", *args, P(tbw), st()))
    t_b = timeit(lambda: ops._call("lcao_threebody_bwd", *args, P(d_tbw), None, P(dB), P(q), None, None, st()))
    t_bf = timeit(lambda: ops._call("lcao_threebody_bwd", *args, P(d_tbw), None, P(dB), P(q), P(du1), P(du2), st()))
    T = gi.num_triplets()
    bf = E * (4 * NL * C + 48 + 12 + 8 + 4 * C) + N * (4 * C + 8)
    bb = E * (4 * NL * C + 48 + 4 * C + 12 + 8 + 4 * NL * C + 4 * C) + N * (4 * C + 8)
    print(f"threebody N={N} E={E} T={T}: "
          f"fwd {t_f:.3f} ms ({bf/t_f/1e6:.0f} GB/s, {T/t_f/1e6:.2f} Gtriplets/s) | "
          f"bwd {t_b:.3f} ms ({bb/t_b/1e6:.0f} GB/s, {T/t_b/1e6:.2f} Gtriplets/s) | bwd+forces {t_bf:.3f} ms", flush=True)
    t_i = timeit(lambda: ops.GraphIndex(g["edge_index"], N))
    print(f"graph index build: {t_i:.3f} ms", flush=True)


def tb():
    """three-body kernels alone, QM9-shape (config 2) and crystal (config 4, 64 cells) graphs; realistic B / Gram from
    the pair-table kernel so the coefficient chain sees sane norms"""
    from lcaonet_b200.synth import crystal_like_batch
    P, st = ops.ptr, ops.stream_ptr
    C, NL, O = 128, 3, 8
    for name, g in (("qm9 1024 mol", qm9_like_batch(1024, seed=1000)), ("crystal 64 cells", crystal_like_batch(64, seed=1000))):
        g = g.to(DEV)
        N, E = g["z"].shape[0], g["edge_index"].shape[1]
        gi = ops.GraphIndex(g["edge_index"], N)
        Zd = 37
        z = g["z"]
        pair = (z[g["edge_index"][0]] * Zd + z[g["edge_index"][1]]).contiguous()
        torch.manual_seed(0)
        tab = torch.randn(Zd * Zd, O, C, device=DEV)
        rb = torch.randn(E, O, device=DEV)
        lgrp = torch.tensor([0, 0, 1, 0, 1, 0, 2, 1], dtype=torch.int32, device=DEV)
        B = torch.empty(E, NL, C, device=DEV)
        gram = torch.empty(E, NL * (NL + 1) // 2, dtype=torch.float64, device=DEV)
        ops._call("lcao_pair_contract_fwd", P(tab), P(pair), P(rb), None, P(lgrp), E, O, C, NL, 0, P(B), P(gram), None, st())
        unit = torch.nn.functional.normalize(torch.randn(E, 3, device=DEV), dim=1)
        xk = torch.sigmoid(torch.randn(N, C, device=DEV))
        tbw, dB, q = torch.empty(E, C, device=DEV), torch.empty(E, NL, C, device=DEV), torch.empty(E, C, device=DEV)
        du1, du2 = torch.empty(E, 3, device=DEV), torch.empty(E, 3, device=DEV)
        d_tbw = torch.randn(E, C, device=DEV)
        args = (P(B), NL, P(gram), P(unit), P(xk), xk.stride(0), P(gi.in_ptr), P(gi.in_edge), P(gi.in_src), P(gi.out_ptr),
                P(gi.out_edge), N, E, C, NL)
        t_f = timeit(lambda: ops._call("lcao_threebody_fwd", *args, P(tbw), st()), reps=9)
        t_b = timeit(lambda: ops._call("lcao_threebody_bwd", *args, P(d_tbw), None, P(dB), P(q), None, None, st()), reps=9)
        t_bf = timeit(lambda: ops._call("lcao_threebody_bwd", *args, P(d_tbw), None, P(dB), P(q), P(du1), P(du2), st()), reps=9)
        T = gi.num_triplets()
        bf = E * (4 * NL * C + 48 + 12 + 8 + 4 * C) + N * (4 * C + 8)
        bb = E * (4 * NL * C + 48 + 4 * C + 12 + 8 + 4 * NL * C + 4 * C) + N * (4 * C + 8)
        peak = 6556.5
        print(f"threebody {name}: N={N} E={E} T={T}: fwd {t_f:.3f} ms ({bf/t_f/1e6:.0f} GB/s, "
              f"{bf/t_f/1e6/peak:.2f}) | bwd {t_b:.3f} ms ({bb/t_b/1e6:.0f} GB/s, {bb/t_b/1e6/peak:.2f}) | bwd+forces {t_bf:.3f} ms "
              f"({bb/t_bf/1e6/peak:.2f})", flush=True)
        print(f"  checksums: tbw {float(tbw.double().abs().sum()):.9e} dB {float(dB.double().abs().sum()):.9e} q "
              f"{float(q.double().abs().sum()):.9e} du {float((du1 + du2).double().abs().sum()):.9e}", flush=True)


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "all"
    if what in ("gemm", "all"):
        gemm()
    if what in ("gemm_small", "all"):
        gemm_small()
    if what in ("edge", "all"):
        edge()
    if what in ("tb", "all"):
        tb()
