"""Every dense-layer kernel path of the C ABI, called directly, against FP64 torch on the same FP32 inputs.

`linear.cu` dispatches each entry point to one of several kernels: the CUDA-core `k_tiny_rows` / `k_tiny_wgrad` /
`k_gemm` (vectorised or scalar loads) of gemm_simt.cu, and the tcgen05 `k_tc_rows<EPI8>`, `k_tc_rows<false>`,
`k_tc_rows_ta`, `k_tc_wgrad` and `k_wgrad_reduce_batch` of gemm_tc.cu.  The helpers below restate that dispatch from
the shapes, the alignment and the SM count, so every case id names the kernel it runs and the shapes follow the part.

Every operand and output is a view into a larger NaN-filled buffer (row offset, leading dimension wider than the view,
NaN rows after the last one): a kernel that reads outside its operand picks up NaN, and one that writes outside its
output changes the padding, which is checked bitwise.  The error bound is componentwise,
    |y - y64| <= c_mode * (|X| |W|^T)      (for the weight gradient (|dY|^T |X|), plus |initial value| for `+=` outputs)
so one wrong row, column, tail tile or contraction chunk fails even when the global relative error would not see it.
"""
from __future__ import annotations

import ctypes
import math

import pytest
import torch

from lcaonet_b200 import _lib, ops
from lcaonet_b200._lib import ACT

pytestmark = pytest.mark.gpu
DEV = "cuda"

NSM = torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148
MODES = {"fp32": _lib.GEMM_FP32, "tf32x3": _lib.GEMM_TF32X3, "tf32": _lib.GEMM_TF32}

# Componentwise error bound per arithmetic mode, in units of the abs-product: the largest |y - y64| / abs-product over
# every case of this file, measured on an NVIDIA B200 (1000 W power limit), times a margin of at most 4
C_MODE = {"fp32": 1.4e-6,     # observed 3.74e-7 (CUDA-core forward, pre-activation with bias)
          "tf32x3": 5.0e-6,   # observed 1.25e-6 (tcgen05 forward, pre-activation with bias)
          "tf32": 5.2e-3}     # observed 1.31e-3 (k_tc_rows<false> data gradient through tanh', contraction 32)
# Extra bound of an activation (or its derivative) evaluated in FP32 in an epilogue or an elementwise pass, per unit
# of the abs-product of the value it is applied to; observed 6.0e-7 (lcao_act_bwd, SiLU')
C_ACT = 2.3e-6
# Lipschitz constant of the activations used here: |SiLU'| <= 1.0999, |tanh'| <= 1
LIP = {"none": 1.0, "silu": 1.1, "tanh": 1.0}

# M by row-block count (128-row tiles) against the SM count: lcao_tc_rows takes k_tc_rows<EPI8> for at most one tile per
# SM, k_tc_rows<false> up to two, and k_tc_rows_ta in 3xTF32 mode from two tiles per SM on
M_EPI8 = NSM * 128 - 61          # the largest EPI8 grid, with a partial last tile
M_ROWS = NSM * 128 + 77          # one tile more than SMs
M_ROWS2 = 2 * NSM * 128 - 133    # the last row count below the tensor-memory kernel
M_TA = 2 * NSM * 128 + 77        # the smallest row count that selects k_tc_rows_ta

NAN_BITS = 0x7FC00000
TAIL = 5  # NaN rows after the last row of every matrix
# layout -> (row offset, column offset, ld - column offset - width).  "wide": 32-byte aligned rows (256-bit stores),
# "narrow": 16- but not 32-byte aligned (the 128-bit store epilogue), "odd": unaligned, odd ld (scalar loads and stores)
LAYOUT = {"wide": (1, 0, 8), "narrow": (1, 4, 12), "odd": (1, 1, 2)}


# ---------------------------------------------------------------------------------------------- dispatch restated
def _tc_rows_kernel(M, mode):
    """lcao_tc_rows: the tcgen05 row kernel for M rows (shared memory always fits for Kc, Nb <= 128)."""
    nblocks = -(-M // 128)
    if mode == "tf32x3" and nblocks >= 2 * NSM:
        return "ta"
    if nblocks <= NSM:
        return "epi8"
    return "rows_x3" if mode == "tf32x3" else "rows_tf32"


def fwd_path(M, K, Nout, mode, aligned):
    """lcao_linear_fwd.  `aligned`: X, W, bias, Y, pre 16-byte aligned and every ld a multiple of 4."""
    if mode != "fp32" and Nout % 16 == 0 and K % 32 == 0 and 32 <= K <= 128 and M >= 512 and aligned:
        return _tc_rows_kernel(M, mode)
    if M <= 512 and K <= 256:
        return "tiny"
    return "simt_vec" if aligned and K % 4 == 0 else "simt_scalar"


def dgrad_path(M, K, Nout, mode, aligned):
    """lcao_linear_dgrad (after the act' pass into scratch, which is always aligned)."""
    if mode != "fp32" and Nout % 32 == 0 and K % 16 == 0 and M >= 512 and aligned:
        return _tc_rows_kernel(M, mode)
    if M <= 512 and Nout <= 256:
        return "tiny"
    return "simt"


def dgrad_act_path(M, K, Nout, mode, aligned, g_aligned, act):
    """lcao_linear_dgrad_act: the SiLU' factor fused into the tcgen05 epilogue, a separate pass otherwise."""
    p = dgrad_path(M, K, Nout, mode, aligned)
    if p in ("tiny", "simt") or not g_aligned:
        return "fallback"
    return "fused_" + p if act == "silu" else "nonsilu"


def wgrad_path(M, K, Nout, mode, aligned):
    """lcao_linear_wgrad / lcao_linear_wgrad_deferred."""
    if mode != "fp32" and Nout % 128 == 0 and M >= 512 and K % 32 == 0 and 32 <= K <= 128 and aligned:
        return "tc_x3" if mode == "tf32x3" else "tc_tf32"
    return "tiny" if M <= 64 else "splitk"


def _is_tc(path):
    return path not in ("tiny", "simt", "simt_vec", "simt_scalar", "splitk", "fallback")


def _aligned(*ts_and_lds):
    ok = True
    for t in ts_and_lds:
        if t is None:
            continue
        if isinstance(t, int):
            ok &= t % 4 == 0
        else:
            ok &= t.data_ptr() % 16 == 0
    return ok


# ---------------------------------------------------------------------------------------------- padded operands
def _mat(M, N, layout, fill=None):
    """(buffer, view): an (M, N) view into a NaN buffer with the layout's offsets and ld; `fill` = values or None."""
    if layout.startswith("half"):  # one half of an (M, 2N) buffer, as the interaction layer passes its operands
        r0, c0, ld = 0, (N if layout == "half_right" else 0), 2 * N
    else:
        r0, c0, extra = LAYOUT[layout]
        ld = c0 + N + extra
    buf = torch.full((r0 + M + TAIL, ld), float("nan"), device=DEV)
    v = buf[r0:r0 + M, c0:c0 + N]
    if fill is not None:
        v.copy_(fill)
    return buf, v


def _flat(shape, fill, off):
    """a contiguous tensor of `shape` at element offset `off` inside a NaN buffer"""
    n = math.prod(shape)
    buf = torch.full((off + n + 16,), float("nan"), device=DEV)
    v = buf[off:off + n].view(*shape)
    v.copy_(fill)
    return buf, v


def _padding_untouched(buf, view, what):
    mask = torch.ones(buf.numel(), dtype=torch.bool, device=DEV)
    inner = torch.as_strided(torch.arange(buf.numel(), device=DEV), view.shape, view.stride(), view.storage_offset())
    mask[inner.reshape(-1)] = False
    bits = buf.reshape(-1).view(torch.int32)[mask]
    assert bool((bits == NAN_BITS).all()), f"{what}: {int((bits != NAN_BITS).sum())} padding elements written"


def _check(what, got, ref, absprod, tol):
    """componentwise: |got - ref| <= tol * absprod, no NaN"""
    assert not bool(torch.isnan(got).any()), f"{what}: NaN in the output (a read outside the operand?)"
    err = (got.double() - ref).abs()
    ratio = float((err / absprod.clamp_min(1e-300)).max())
    bad = err > tol * absprod
    if bool(bad.any()):
        first = torch.nonzero(bad)[0].tolist()
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements over the bound, first at {first} "
                             f"(got {float(got[tuple(first)]):.8g}, want {float(ref[tuple(first)]):.8g}); "
                             f"max ratio {ratio:.3g} > {tol:.3g}")


def _act64(act, z):
    return {"none": lambda v: v, "silu": torch.nn.functional.silu, "tanh": torch.tanh}[act](z)


def _dact64(act, z):
    if act == "silu":
        s = torch.sigmoid(z)
        return s * (1 + z * (1 - s))
    if act == "tanh":
        return 1 - torch.tanh(z) ** 2
    return torch.ones_like(z)


def _launches():
    return _lib.launch_count()


P, ST = ops.ptr, ops.stream_ptr


# ---------------------------------------------------------------------------------------------- lcao_linear_fwd
# (path, mode, M, K, Nout, act, pre, bias, layout)
FWD = [
    ("tiny", "tf32x3", 300, 20, 48, "silu", True, True, "wide"),
    ("tiny", "tf32x3", 37, 200, 144, "tanh", True, False, "narrow"),
    ("simt_vec", "fp32", 1000, 96, 144, "silu", True, True, "wide"),
    ("simt_vec", "tf32x3", 700, 200, 48, "none", False, True, "narrow"),
    ("simt_vec", "fp32", M_TA, 128, 256, "silu", True, True, "wide"),
    ("simt_scalar", "tf32x3", 900, 20, 48, "tanh", True, True, "odd"),
    ("simt_scalar", "fp32", 1300, 200, 16, "none", False, False, "odd"),
    ("epi8", "tf32x3", M_EPI8, 96, 144, "silu", True, True, "narrow"),
    ("epi8", "tf32x3", 1029, 32, 384, "none", False, True, "wide"),
    ("epi8", "tf32x3", 777, 128, 16, "tanh", True, False, "wide"),
    ("epi8", "tf32", 2049, 128, 16, "silu", False, True, "wide"),
    ("rows_x3", "tf32x3", M_ROWS, 128, 256, "silu", True, True, "narrow"),
    ("rows_x3", "tf32x3", M_ROWS2, 96, 48, "tanh", True, True, "wide"),
    ("rows_x3", "tf32x3", M_ROWS, 32, 144, "none", False, False, "wide"),
    ("rows_tf32", "tf32", M_TA, 128, 144, "silu", True, True, "narrow"),
    ("rows_tf32", "tf32", M_ROWS, 96, 256, "tanh", False, True, "wide"),
    ("ta", "tf32x3", M_TA, 128, 256, "silu", True, True, "narrow"),
    ("ta", "tf32x3", M_TA, 96, 48, "tanh", True, False, "wide"),
    ("ta", "tf32x3", M_TA, 32, 384, "none", False, True, "wide"),
    ("ta", "tf32x3", M_TA, 128, 144, "silu", False, False, "wide"),
]


def _fwd_id(c):
    path, mode, M, K, N, act, pre, bias, layout = c
    return f"{path}-{mode}-M{M}-K{K}-N{N}-{act}{'-pre' if pre else ''}{'-bias' if bias else ''}-{layout}"


@pytest.mark.parametrize("case", FWD, ids=[_fwd_id(c) for c in FWD])
def test_linear_fwd(case):
    path, mode, M, K, N, act, want_pre, want_bias, layout = case
    torch.manual_seed(M * 7 + K + N)
    woff = 1 if layout == "odd" else 4
    xb, x = _mat(M, K, layout, torch.randn(M, K, device=DEV))
    wb, w = _flat((N, K), torch.randn(N, K, device=DEV) / K**0.5, woff)
    bb, b = _flat((N,), torch.randn(N, device=DEV), woff) if want_bias else (None, None)
    yb, y = _mat(M, N, layout)
    pb, pre = _mat(M, N, layout) if want_pre else (None, None)
    aligned = _aligned(x, w, b, y, pre, x.stride(0), y.stride(0), pre.stride(0) if want_pre else 0)
    assert fwd_path(M, K, N, mode, aligned) == path
    n0 = _launches()
    ops._call("lcao_linear_fwd", P(x), x.stride(0), P(w), P(b), P(y), y.stride(0), P(pre), pre.stride(0) if want_pre else 0,
              M, K, N, ACT[act], MODES[mode], ST())
    n_launch = _launches() - n0
    if _is_tc(path):  # one launch per 128 output columns; a non-SiLU activation is one elementwise pass after them
        assert n_launch == -(-N // 128) + (act not in ("none", "silu")), n_launch
    else:
        assert n_launch == 1, n_launch
    torch.cuda.synchronize()
    x64, w64 = x.double(), w.double()
    z = x64 @ w64.T
    a = x64.abs() @ w64.abs().T
    if want_bias:
        z, a = z + b.double(), a + b.double().abs()
    tol = C_MODE[mode]
    if want_pre:
        _check(f"{mode} fwd pre", pre, z, a, tol)
        _padding_untouched(pb, pre, "pre")
    tol_y = tol * LIP[act] + (C_ACT if act != "none" else 0.0)
    _check(f"{mode} fwd{'' if act == 'none' else ' act'}", y, _act64(act, z), a, tol_y)
    _padding_untouched(yb, y, "Y")
    for buf, v, what in ((xb, x, "X"), (wb, w, "W")):
        _padding_untouched(buf, v, what)


# ---------------------------------------------------------------------------------------------- lcao_linear_dgrad
# (path, mode, M, K, Nout, accumulate, act (H), layout)
DGRAD = [
    ("tiny", "tf32x3", 300, 144, 32, 1, "none", "wide"),
    ("tiny", "fp32", 500, 16, 256, 0, "silu", "narrow"),
    ("simt", "fp32", 2000, 256, 160, 1, "tanh", "wide"),
    ("simt", "fp32", 4000, 144, 32, 0, "none", "narrow"),
    ("simt", "tf32x3", 1100, 144, 160, 1, "none", "odd"),
    ("epi8", "tf32x3", 3001, 256, 160, 1, "none", "wide"),
    ("epi8", "tf32x3", 1500, 16, 32, 0, "silu", "narrow"),
    ("epi8", "tf32", 2500, 144, 160, 1, "none", "wide"),
    ("rows_x3", "tf32x3", M_ROWS, 144, 256, 1, "none", "narrow"),
    ("rows_x3", "tf32x3", M_ROWS2, 16, 160, 0, "silu", "wide"),
    ("rows_tf32", "tf32", M_ROWS2, 256, 32, 0, "tanh", "wide"),
    ("ta", "tf32x3", M_TA, 144, 256, 1, "none", "wide"),
    ("ta", "tf32x3", M_TA, 16, 160, 0, "silu", "narrow"),
    ("ta", "tf32x3", M_TA, 256, 32, 1, "tanh", "wide"),
    ("ta", "tf32x3", M_TA, 144, 160, 0, "none", "narrow"),
]


def _dgrad_id(c):
    path, mode, M, K, N, acc, act, layout = c
    return f"{path}-{mode}-M{M}-K{K}-N{N}{'-acc' if acc else ''}-H{act}-{layout}"


def _scratch(n):
    """exactly n floats followed by a NaN guard"""
    buf = torch.full((n + 256,), float("nan"), device=DEV)
    return buf, buf[:n]


@pytest.mark.parametrize("case", DGRAD, ids=[_dgrad_id(c) for c in DGRAD])
def test_linear_dgrad(case):
    path, mode, M, K, N, accumulate, act, layout = case
    torch.manual_seed(M * 5 + K + N)
    dyb, dy = _mat(M, N, layout, torch.randn(M, N, device=DEV))
    hb, h = _mat(M, N, layout, 2 * torch.randn(M, N, device=DEV)) if act != "none" else (None, None)
    wb, w = _flat((N, K), torch.randn(N, K, device=DEV) / N**0.5, 1 if layout == "odd" else 4)
    dxb, dx = _mat(M, K, layout, torch.randn(M, K, device=DEV) if accumulate else None)
    dx0 = dx.double() if accumulate else None
    ldh = h.stride(0) if h is not None else 0
    n_scr = int(_lib.load().lcao_linear_bwd_scratch(P(dy), dy.stride(0), P(h), ldh, ACT[act], P(w), None, 0, P(dx),
                                                    dx.stride(0), M, K, N, MODES[mode]))
    assert n_scr == (M * N if act != "none" else 0)
    sb, scr = _scratch(n_scr)
    # with an activation the GEMM reads dY * act'(H) from the (packed, aligned) scratch
    aligned = _aligned(w, dx, dx.stride(0)) and (act != "none" or _aligned(dy, dy.stride(0)))
    assert dgrad_path(M, K, N, mode, aligned) == path
    n0 = _launches()
    ops._call("lcao_linear_dgrad", P(dy), dy.stride(0), P(h), ldh, ACT[act], P(w), P(dx), dx.stride(0), M, K, N, accumulate,
              MODES[mode], P(sb), ST())
    n_launch = _launches() - n0
    want = (-(-K // 128)) * (-(-N // 128)) if _is_tc(path) else 1
    assert n_launch == want + (act != "none"), n_launch
    torch.cuda.synchronize()
    g = dy.double() * _dact64(act, h.double()) if act != "none" else dy.double()
    ref, a = g @ w.double(), g.abs() @ w.double().abs()
    if accumulate:
        ref, a = ref + dx0, a + dx0.abs()
    _check(f"{mode} dgrad{'' if act == 'none' else ' act'}", dx, ref, a, C_MODE[mode] + (C_ACT if act != "none" else 0.0))
    _padding_untouched(dxb, dx, "dX")
    bits = sb[n_scr:].view(torch.int32)
    assert bool((bits == NAN_BITS).all()), "scratch written past the queried size"


# ---------------------------------------------------------------------------------------------- lcao_linear_dgrad_act
# (path, mode, M, K, Nout, act, layout, G layout)
DGRAD_ACT = [
    ("fused_epi8", "tf32x3", 2500, 144, 160, "silu", "wide", "narrow"),
    ("fused_epi8", "tf32x3", 1700, 16, 256, "silu", "narrow", "wide"),
    ("fused_rows_x3", "tf32x3", M_ROWS, 128, 256, "silu", "narrow", "wide"),
    ("fused_rows_tf32", "tf32", M_ROWS, 144, 256, "silu", "wide", "narrow"),
    ("fused_ta", "tf32x3", M_TA, 256, 160, "silu", "wide", "wide"),
    ("fused_ta", "tf32x3", M_TA, 16, 384, "silu", "narrow", "narrow"),
    ("nonsilu", "tf32x3", 3000, 144, 256, "tanh", "wide", "narrow"),
    ("nonsilu", "tf32x3", M_TA, 128, 160, "tanh", "narrow", "wide"),
    ("fallback", "tf32x3", 2000, 144, 160, "silu", "wide", "odd"),        # G unaligned, ldg odd
    ("fallback", "tf32x3", 2100, 128, 256, "silu", "wide", "misaligned"),  # G 4-byte aligned, ldg % 4 == 0
    ("fallback", "fp32", 1000, 144, 160, "silu", "narrow", "wide"),
    ("fallback", "tf32x3", 1200, 20, 160, "tanh", "odd", "odd"),
]


def _dgrad_act_id(c):
    path, mode, M, K, N, act, layout, glayout = c
    return f"{path}-{mode}-M{M}-K{K}-N{N}-{act}-{layout}-G{glayout}"


@pytest.mark.parametrize("case", DGRAD_ACT, ids=[_dgrad_act_id(c) for c in DGRAD_ACT])
def test_linear_dgrad_act(case):
    path, mode, M, K, N, act, layout, glayout = case
    torch.manual_seed(M * 3 + K + N)
    dyb, dy = _mat(M, N, layout, torch.randn(M, N, device=DEV))
    wb, w = _flat((N, K), torch.randn(N, K, device=DEV) / N**0.5, 1 if layout == "odd" else 4)
    gvals = 2 * torch.randn(M, K, device=DEV)
    if glayout == "misaligned":  # row stride a multiple of 4, rows 4 bytes off a 16-byte boundary
        gb = torch.full((M + TAIL + 1, K + 8), float("nan"), device=DEV)
        G = gb.view(-1)[1 + (K + 8):1 + (K + 8) * (M + 1)].view(M, K + 8)[:, :K]
        G.copy_(gvals)
    else:
        gb, G = _mat(M, K, glayout, gvals)
    dxb, dx = _mat(M, K, layout)
    aligned = _aligned(w, dy, dx, dy.stride(0), dx.stride(0))
    g_aligned = _aligned(G, G.stride(0))
    assert dgrad_act_path(M, K, N, mode, aligned, g_aligned, act) == path
    n0 = _launches()
    ops._call("lcao_linear_dgrad_act", P(dy), dy.stride(0), P(w), P(G), G.stride(0), ACT[act], P(dx), dx.stride(0), M, K, N,
              MODES[mode], ST())
    n_launch = _launches() - n0
    gemm = (-(-K // 128)) * (-(-N // 128)) if path != "fallback" else 1
    assert n_launch == gemm + (not path.startswith("fused")), n_launch
    torch.cuda.synchronize()
    z, a = dy.double() @ w.double(), dy.double().abs() @ w.double().abs()
    f = _dact64(act, G.double())
    _check(f"{mode} dgrad_act act", dx, z * f, a, C_MODE[mode] * LIP[act] + C_ACT)
    _padding_untouched(dxb, dx, "dX")
    _padding_untouched(gb, G, "G")


# ---------------------------------------------------------------------------------------------- lcao_linear_wgrad
# (path, mode, M, K, Nout, bias, act (H), layout); "halves": dY and X are halves of (M, 2 Nout) / (M, 2 K) buffers
WGRAD = [
    ("tc_x3", "tf32x3", 512, 32, 128, True, "none", "halves"),
    ("tc_x3", "tf32x3", 513, 96, 256, False, "silu", "wide"),
    ("tc_x3", "tf32x3", 1000, 128, 128, True, "tanh", "narrow"),
    ("tc_x3", "tf32x3", 4127, 96, 256, True, "none", "halves"),
    ("tc_x3", "tf32x3", 18945, 128, 128, True, "none", "halves"),
    ("tc_x3", "tf32x3", M_TA + 77, 32, 256, True, "silu", "halves"),
    ("tc_x3", "tf32x3", 3 * 128 * NSM // 4 + 1, 128, 256, False, "none", "halves"),
    ("tc_tf32", "tf32", 4127, 128, 256, True, "none", "halves"),
    ("tc_tf32", "tf32", M_TA + 77, 96, 128, False, "none", "wide"),
    ("splitk", "fp32", 18945, 128, 256, True, "none", "halves"),
    ("splitk", "fp32", 1000, 96, 128, False, "tanh", "wide"),
    ("splitk", "fp32", 4127, 32, 256, True, "silu", "halves"),
    ("splitk", "tf32x3", 513, 96, 128, True, "none", "odd"),
    ("tiny", "tf32x3", 64, 128, 128, True, "none", "halves"),
    ("tiny", "fp32", 37, 96, 256, False, "silu", "wide"),
]


def _wgrad_id(c):
    path, mode, M, K, N, bias, act, layout = c
    return f"{path}-{mode}-M{M}-K{K}-N{N}{'-bias' if bias else ''}-H{act}-{layout}"


def _wgrad_operands(M, K, N, layout, act):
    dy_l, x_l = ("half_right", "half_left") if layout == "halves" else (layout, layout)
    dyb, dy = _mat(M, N, dy_l, torch.randn(M, N, device=DEV))
    xb, x = _mat(M, K, x_l, torch.randn(M, K, device=DEV))
    hb, h = _mat(M, N, layout if layout != "halves" else "wide", 2 * torch.randn(M, N, device=DEV)) if act != "none" else (None, None)
    return dyb, dy, xb, x, hb, h


@pytest.mark.parametrize("case", WGRAD, ids=[_wgrad_id(c) for c in WGRAD])
def test_linear_wgrad(case):
    path, mode, M, K, N, want_bias, act, layout = case
    torch.manual_seed(M * 11 + K + N)
    dyb, dy, xb, x, hb, h = _wgrad_operands(M, K, N, layout, act)
    dw0 = torch.randn(N, K, device=DEV)  # dW += / db += : start from random values
    db0 = torch.randn(N, device=DEV) if want_bias else None
    ldh = h.stride(0) if h is not None else 0
    aligned = _aligned(x, x.stride(0)) and (act != "none" or _aligned(dy, dy.stride(0)))
    assert wgrad_path(M, K, N, mode, aligned) == path
    n_scr = int(_lib.load().lcao_linear_bwd_scratch(P(dy), dy.stride(0), P(h), ldh, ACT[act], None, P(x), x.stride(0), None,
                                                    0, M, K, N, MODES[mode]))

    def run():
        wb, dw = _flat((N, K), dw0, 4)
        bb, db = _flat((N,), db0, 4) if want_bias else (None, None)
        sb, _ = _scratch(n_scr)
        n0 = _launches()
        ops._call("lcao_linear_wgrad", P(dy), dy.stride(0), P(h), ldh, ACT[act], P(x), x.stride(0), P(dw), P(db), M, K, N,
                  MODES[mode], P(sb), ST())
        n_launch = _launches() - n0
        torch.cuda.synchronize()
        return wb, dw, bb, db, sb, n_launch

    wb, dw, bb, db, sb, n_launch = run()
    passes = N // 128
    want = {"tiny": 1, "splitk": 1 + want_bias}.get(path, 2 * passes)  # tcgen05: stage 1 + the reduction per pass
    assert n_launch == want + (act != "none"), n_launch
    g = dy.double() * _dact64(act, h.double()) if act != "none" else dy.double()
    tol = C_MODE[mode] + (C_ACT if act != "none" else 0.0)
    _check(f"{mode} wgrad{'' if act == 'none' else ' act'}", dw, dw0.double() + g.T @ x.double(),
           dw0.double().abs() + g.abs().T @ x.double().abs(), tol)
    _padding_untouched(wb, dw, "dW")
    if want_bias:
        _check(f"{mode} wgrad db", db, db0.double() + g.sum(0), db0.double().abs() + g.abs().sum(0), tol)
        _padding_untouched(bb, db, "db")
    bits = sb[n_scr:].view(torch.int32)
    assert bool((bits == NAN_BITS).all()), "scratch written past the queried size"
    if _is_tc(path):  # fixed-order two-stage reduction: a rerun is bitwise the same
        _, dw2, _, db2, _, _ = run()
        assert torch.equal(dw2.view(torch.int32), dw.view(torch.int32))
        if want_bias:
            assert torch.equal(db2.view(torch.int32), db.view(torch.int32))


# ---------------------------------------------------------------------------------------------- deferred weight gradients
def _deferred_specs():
    """21 weight gradients of mixed K, Nout (1-3 passes of 128 columns) and bias: 42 descriptors, two batch launches"""
    return [(600 + 131 * i, (32, 96, 128, 64)[i % 4], 128 * (i % 3 + 1), i % 2 == 0) for i in range(21)]


DEFERRED = [("tc_x3", "tf32x3"), ("tc_tf32", "tf32"), ("ndesc0", "fp32")]


@pytest.mark.parametrize("path,mode", DEFERRED, ids=[f"{p}-{m}" for p, m in DEFERRED])
def test_linear_wgrad_deferred_batch(path, mode):
    torch.manual_seed(17)
    items = []
    for M, K, N, want_bias in _deferred_specs():
        dyb, dy, xb, x, _, _ = _wgrad_operands(M, K, N, "halves", "none")
        p = wgrad_path(M, K, N, mode, _aligned(dy, x, dy.stride(0), x.stride(0)))
        assert p == path if _is_tc(p) else path == "ndesc0"
        dw0 = torch.randn(N, K, device=DEV)
        db0 = torch.randn(N, device=DEV) if want_bias else None
        items.append((M, K, N, dy, x, dw0, db0))
    descs, keep = [], []
    n0 = _launches()
    for M, K, N, dy, x, dw0, db0 in items:
        passes = N // 128
        n_scr = int(_lib.load().lcao_linear_bwd_scratch(P(dy), dy.stride(0), None, 0, 0, None, P(x), x.stride(0), None, 0, M,
                                                        K, N, MODES[mode]))
        sb, _ = _scratch(n_scr * passes)
        wb, dw = _flat((N, K), dw0, 4)
        bb, db = _flat((N,), db0, 4) if db0 is not None else (None, None)
        desc, nd = (ctypes.c_int64 * (6 * passes))(), ctypes.c_int32(-1)
        m0 = _launches()
        ops._call("lcao_linear_wgrad_deferred", P(dy), dy.stride(0), P(x), x.stride(0), P(dw), P(db), M, K, N, MODES[mode],
                  P(sb), desc, ctypes.byref(nd), ST())
        if mode == "fp32":
            assert nd.value == 0 and _launches() - m0 == 1 + (db0 is not None)
        else:  # stage 1 only: one launch per pass, nothing more until the batch reduction
            assert nd.value == passes and _launches() - m0 == passes
            assert (sb[n_scr * passes:].view(torch.int32) == NAN_BITS).all()
        descs.extend(desc[: 6 * nd.value])
        keep.append((wb, dw, bb, db, sb))
    torch.cuda.synchronize()
    if mode != "fp32":
        for (M, K, N, dy, x, dw0, db0), (wb, dw, bb, db, sb) in zip(items, keep):
            assert torch.equal(dw.view(torch.int32), dw0.view(torch.int32)), "stage 1 wrote dW"
            if db0 is not None:
                assert torch.equal(db.view(torch.int32), db0.view(torch.int32)), "stage 1 wrote db"
        n = len(descs) // 6
        assert n == sum(N // 128 for _, _, N, _ in _deferred_specs()) and n > 32
        arr = (ctypes.c_int64 * len(descs))(*descs)
        m0 = _launches()
        ops._call("lcao_wgrad_reduce_batch", arr, n, ST())
        assert _launches() - m0 == -(-n // 32)
        torch.cuda.synchronize()
    else:
        assert not descs and _launches() - n0 == sum(1 + b for _, _, _, b in _deferred_specs())
    for (M, K, N, dy, x, dw0, db0), (wb, dw, bb, db, sb) in zip(items, keep):
        what = f"{mode} deferred wgrad M{M} K{K} N{N}"
        x64, g = x.double(), dy.double()
        _check(what, dw, dw0.double() + g.T @ x64, dw0.double().abs() + g.abs().T @ x64.abs(), C_MODE[mode])
        _padding_untouched(wb, dw, "dW")
        if db0 is not None:
            _check(what + " db", db, db0.double() + g.sum(0), db0.double().abs() + g.abs().sum(0), C_MODE[mode])
            _padding_untouched(bb, db, "db")
        if mode != "fp32":  # the same kernels and summation order as the immediate weight gradient
            n_scr = int(_lib.load().lcao_linear_bwd_scratch(P(dy), dy.stride(0), None, 0, 0, None, P(x), x.stride(0), None, 0,
                                                            M, K, N, MODES[mode]))
            scr = torch.empty(n_scr, device=DEV)
            dw_i, db_i = dw0.clone(), (db0.clone() if db0 is not None else None)
            ops._call("lcao_linear_wgrad", P(dy), dy.stride(0), None, 0, 0, P(x), x.stride(0), P(dw_i), P(db_i), M, K, N,
                      MODES[mode], P(scr), ST())
            torch.cuda.synchronize()
            assert torch.equal(dw_i.view(torch.int32), dw.view(torch.int32)), what
            if db0 is not None:
                assert torch.equal(db_i.view(torch.int32), db.view(torch.int32)), what


# ---------------------------------------------------------------------------------------------- lcao_act_bwd
@pytest.mark.parametrize("act", ["silu", "tanh", "gelu"])
@pytest.mark.parametrize("M,C,layout", [(3001, 128, "wide"), (777, 48, "narrow"), (1029, 37, "odd")])
def test_act_bwd_in_place(act, M, C, layout):
    """dH = dY * act'(H) written over dY, with dY and H at different strides; "odd": unaligned rows, odd width and lds."""
    torch.manual_seed(M + C)
    dyb, dy = _mat(M, C, layout, torch.randn(M, C, device=DEV))
    hvals = 2 * torch.randn(M, C, device=DEV)
    if layout == "odd":  # H in a layout of its own, so that the two row strides differ
        hb = torch.full((M + TAIL, C + 6), float("nan"), device=DEV)
        h = hb[1:M + 1, 2:C + 2]
        h.copy_(hvals)
    else:
        hb, h = _mat(M, C, "narrow" if layout == "wide" else "wide", hvals)
    assert dy.stride(0) != h.stride(0)
    g64 = dy.double()
    hd = h.double().requires_grad_(True)
    fn = {"silu": torch.nn.functional.silu, "tanh": torch.tanh, "gelu": torch.nn.functional.gelu}[act]
    (d,) = torch.autograd.grad(fn(hd).sum(), hd)
    n0 = _launches()
    ops._call("lcao_act_bwd", P(dy), dy.stride(0), P(h), h.stride(0), P(dy), dy.stride(0), M, C, ACT[act], ST())
    assert _launches() - n0 == 1
    torch.cuda.synchronize()
    _check(f"act_bwd {act}", dy, g64 * d, g64.abs() * d.abs().clamp_min(1.0), C_ACT)
    _padding_untouched(dyb, dy, "dH")


# ---------------------------------------------------------------------------------------------- coverage of the table
REQUIRED = {
    "fwd": {"tiny", "simt_vec", "simt_scalar", "epi8", "rows_x3", "rows_tf32", "ta"},
    "dgrad": {"tiny", "simt", "epi8", "rows_x3", "ta"},
    "dgrad_act": {"fused_epi8", "fused_rows_x3", "fused_ta", "nonsilu", "fallback"},
    "wgrad": {"tc_x3", "tc_tf32", "splitk", "tiny"},
    "deferred": {"tc_x3", "ndesc0"},
}
_COVERED = {"fwd": {c[0] for c in FWD}, "dgrad": {c[0] for c in DGRAD}, "dgrad_act": {c[0] for c in DGRAD_ACT},
            "wgrad": {c[0] for c in WGRAD}, "deferred": {p for p, _ in DEFERRED}}
for _ep, _paths in REQUIRED.items():
    assert _paths <= _COVERED[_ep], f"{_ep}: no case for {_paths - _COVERED[_ep]}"
# the declared path of every case follows from its shape, mode and layout under the restated dispatch
for _c in FWD:
    assert fwd_path(_c[2], _c[3], _c[4], _c[1], _c[8] != "odd") == _c[0], _c
for _c in DGRAD:
    assert dgrad_path(_c[2], _c[3], _c[4], _c[1], _c[7] != "odd") == _c[0], _c
for _c in DGRAD_ACT:
    assert dgrad_act_path(_c[2], _c[3], _c[4], _c[1], _c[6] != "odd", _c[7] not in ("odd", "misaligned"), _c[5]) == _c[0], _c
for _c in WGRAD:
    assert wgrad_path(_c[2], _c[3], _c[4], _c[1], _c[7] != "odd") == _c[0], _c
