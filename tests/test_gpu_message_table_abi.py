"""Every message-passing and embedding-table kernel path of the C ABI, called directly, against exact and FP64 references.

The entry points (edge_ops.cu, table_norm.cu, graph_index.cu):
  - `lcao_edge_pair_fwd`  a1 = act(u_a[s] + u_b[t] + b) of every interaction block;
  - `lcao_segment_sum`    the message sum, the backward through act' and the node pooling (sorted segments, no atomics);
  - `lcao_msg_bwd`        the backward of the message sum, h given or recomputed from pre_h;
  - `lcao_gather_rows`    node-table and pair-table gathers and the backward of the segment reduce;
  - `lcao_reduce_by_key`  the backward of every table gather (32 sorted entries per CTA, atomic flushes);
  - `lcao_act_fwd`        the activations the GEMM epilogue does not fuse;
  - `lcao_table_norm_fwd` / `_bwd`, `lcao_pair_outer_fwd` / `_bwd`, `lcao_histogram`: the embedding tables.
The helpers below restate their dispatch (18 kernels), so every case id names the kernels it runs; one test checks that
the cases reach all of them, another (where cuobjdump is available) that the library holds no kernel that no test claims.

Every sum runs twice:
  - exact inputs: small integers, so every FP32 product and partial sum is an integer below 2^24 and each output must
    EQUAL the FP64 reference whatever the summation order (+0 and -0 compare equal);
  - random inputs: normal values.  Outputs formed with one rounding (gathers with `mul`, the edge-pair `pre`, d_bw from
    a given h, the pair-outer forward) must be bitwise torch FP32 on the same inputs; a segment sum without y must be
    bitwise the sequential FP32 sum in perm order; every other sum is bounded componentwise by gamma_n * (the same sum
    over absolute values), gamma_n = n u / (1 - n u), u = 2^-24, with n from the kernel's own summation order.
Activations are compared with FP64 torch of the same FP32 argument: |got - ref| <= K u mag + 2^-119, where mag is the
magnitude of the terms the kernel forms (for SSP softplus(x) + ln 2: the subtraction cancels near 0) and the 2^-119
allows for results that underflow.  K is 4x the largest ratio observed on a B200 (values next to the constants).
Special arguments (+-0, the softplus threshold 19.99 / 20 / 20.01, +-88 .. +-100 where expf overflows in the sigmoid,
+-1e30 and NaN) are part of every activation case.  NaN in gives NaN out; a derivative at a NaN argument is NaN or,
as torch's, the passed-through gradient.

Every operand is a view into a NaN-filled buffer with NaN rows before and after it (index operands: -1), row strides
wider than the view where the API takes one, and one-float row offsets to reach the scalar paths.  Inputs must stay
bitwise unchanged, output padding untouched, empty segments and keys no entry reaches exact, and two identical calls
must agree bitwise, except k_reduce_by_key and k_hist_f, which flush with atomics (DESIGN.md R8): their determinism is
checked with exact data only.
"""
from __future__ import annotations

import functools
import math
import os
import re
import shutil
import subprocess

import pytest
import torch

from lcaonet_b200 import _lib, ops
from lcaonet_b200.csrc.build import LIB

pytestmark = pytest.mark.gpu
DEV = "cuda"
P_, ST = ops.ptr, ops.stream_ptr
NAN_BITS = 0x7FC00000
PAD = 4               # NaN rows before and after every operand
U = 2.0 ** -24        # unit roundoff of FP32
TINY = 2.0 ** -119    # absolute allowance of an activation for results that underflow
WARP_PASS = 128       # warp-per-row kernels: floats one warp covers per pass (32 lanes x float4)
RBK_CHUNK = 32        # k_reduce_by_key: sorted entries per CTA
RBK_PASS = 1024       # k_reduce_by_key: floats one CTA covers per column pass (256 threads x float4)
OUTER_CAP = 148 * 8   # k_pair_outer_fwd: grid cap, CTAs of 256 threads with one float4 each per pass
ACT_NAMES = ["none", "silu", "ssp", "softplus", "relu", "tanh", "sigmoid", "gelu", "elu", "leaky_relu"]

# K of the activation bounds, forward and derivative, per LCAO_ACT_* kind: 4x the largest err / (u mag) observed over
# every case of this file on an NVIDIA B200 at its 1000 W power limit (observed values in the comments; 0 = exact).
#       none  silu  ssp  softplus relu tanh  sigmoid gelu  elu  leaky_relu
K_FWD = [0, 14.6, 7.1, 12.0, 0, 13.4, 11.6, 8.6, 6.7, 5.5]
#   observed 0     3.65  1.76  2.99     0    3.33  2.89    2.14  1.67  1.36
K_GRAD = [0, 14.8, 7.2, 7.5, 0, 4.8, 10.2, 5.1, 6.0, 0.005]
#   observed 0     3.68  1.80  1.86     0    1.18  2.53    1.27  1.48  0.00106 (0.01f for 0.01)
# Largest |got - ref| / bound per analytic bound (a ratio <= 1 passes), same GPU:
#   segment_sum y 0.64, act 0.44, grad 0.47; msg_bwd d_bw 1.0 (one product, rounded to nearest: the bound is its half
#   ulp), d_pre_h 0.50; edge_pair / act_fwd 0.13; reduce_by_key 0.11; pair_outer d_fe 0.39, d_za and d_zb 0.79;
#   table_norm save_mean 0.13, save_rstd 0.35, y 0.81, running statistics 0.42, dbeta 0.07, dgamma 0.08, dx 0.89
OBSERVED: dict = {}


def gamma(n):
    n = torch.as_tensor(n, dtype=torch.float64, device=DEV)
    return n * U / (1 - n * U)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for k in sorted(OBSERVED):
        print(f"observed {k}: {OBSERVED[k]:.3g}")


# ---------------------------------------------------------------------------------------------- dispatch restated
def _b(x):
    return "true" if x else "false"


def _aligned(t):
    return t is None or t.data_ptr() % 16 == 0


def edge_pair_kernels(E, act):
    """lcao_edge_pair_fwd: SiLU and no activation take the SiLU-only instantiation"""
    return [f"k_edge_pair_fwd<{_b(act not in (0, 1))}>"] if E > 0 else []


def segsum_vec(C, x, y, out):
    """the float4 path needs C, every row stride and every base 16-byte aligned"""
    return (C % 4 == 0 and x.stride(0) % 4 == 0 and out.stride(0) % 4 == 0 and (y is None or y.stride(0) % 4 == 0)
            and _aligned(x) and _aligned(y) and _aligned(out))


def segsum_kernels(R, C, vec, mode):
    """lcao_segment_sum: the generic-activation instantiation only when bit 1 or 2 asks for a kind other than SiLU
    (the activation field 0 means SiLU); the scalar path is always generic"""
    if R == 0 or C == 0:
        return []
    kind = (mode >> 4) & 15
    gen = bool(mode & 6) and kind > 1
    return [f"k_segment_sum<true,{_b(gen)}>" if vec else "k_segment_sum<false,true>"]


def msg_bwd_kernels(E, act):
    return [f"k_msg_bwd<{_b(act != 1)}>"] if E > 0 else []


def gather_vec(W, table, mul, out):
    return (W % 4 == 0 and table.stride(0) % 4 == 0 and out.stride(0) % 4 == 0 and _aligned(table) and _aligned(out)
            and (mul is None or (mul.stride(0) % 4 == 0 and _aligned(mul))))


def gather_kernels(n, W, is64, vec):
    return [f"k_gather_rows<{'int64_t' if is64 else 'int32_t'},{_b(vec)}>"] if n and W else []


def rbk_kernels(n):
    return ["k_reduce_by_key"] if n > 0 else []


def outer_grid_strides(Zd, O, K):
    """k_pair_outer_fwd takes more than one grid-stride pass when the float4 count exceeds the capped grid"""
    return math.ceil(Zd * Zd * O * (K // 4) / 256) > OUTER_CAP


ALL_KERNELS = ({f"k_edge_pair_fwd<{v}>" for v in ("false", "true")}
               | {"k_segment_sum<true,false>", "k_segment_sum<true,true>", "k_segment_sum<false,true>"}
               | {f"k_msg_bwd<{v}>" for v in ("false", "true")}
               | {f"k_gather_rows<{t},{v}>" for t in ("int64_t", "int32_t") for v in ("false", "true")}
               | {"k_reduce_by_key", "k_act_fwd", "k_wbn_fwd", "k_wbn_bwd", "k_pair_outer_fwd", "k_pair_outer_bwd",
                  "k_hist_f"})


def _kid(names):
    return "+".join(k.replace("<", ".").replace(">", "").replace(",", ".").replace("_t", "") for k in names) or "none"


# ---------------------------------------------------------------------------------------------- padded operands
def _mat(M, W, ld=None, off=0, fill=None, dtype=torch.float32):
    """(buffer, view): an (M, W) view with row stride ld, starting `off` elements into row PAD of a NaN buffer"""
    ld = W if ld is None else ld
    buf = torch.full(((M + 2 * PAD) * ld + off,), float("nan"), dtype=dtype, device=DEV)
    v = buf.as_strided((M, W), (ld, 1), PAD * ld + off)
    if fill is not None:
        v.copy_(fill.reshape(M, W))
    return buf, v


def _irows(n, fill, dtype):
    """(buffer, view): n index entries with PAD entries of the sentinel -1 before and after them"""
    buf = torch.full((n + 2 * PAD,), -1, dtype=dtype, device=DEV)
    v = buf[PAD:PAD + n]
    v.copy_(fill.reshape(-1))
    return buf, v


def _padding_untouched(buf, view, what):
    mask = torch.ones(buf.numel(), dtype=torch.bool, device=DEV)
    inner = torch.as_strided(torch.arange(buf.numel(), device=DEV), view.shape, view.stride(), view.storage_offset())
    mask[inner.reshape(-1)] = False
    if buf.dtype == torch.float32:
        bits = buf.view(torch.int32)[mask]
        assert bool((bits == NAN_BITS).all()), f"{what}: {int((bits != NAN_BITS).sum())} padding elements written"
    else:
        assert bool((buf[mask] == -1).all()), f"{what}: padding written"


def _same_bits(a, b):
    if a is None or b is None:
        return a is b
    if not a.is_floating_point():
        return torch.equal(a, b)
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _same_or_nan(a, b):
    """bitwise equal, NaN payloads aside"""
    nan = torch.isnan(a)
    return torch.equal(nan, torch.isnan(b)) and _same_bits(torch.where(nan, 0.0, a), torch.where(nan, 0.0, b))


def _check(name, what, got, ref, lim, nan_ok=None):
    """|got - ref| <= lim componentwise (FP64 ref and lim).  Where ref is NaN, got must be NaN; got may be NaN where ref
    is finite only where nan_ok is set."""
    g = got.double()
    ref_nan, got_nan = torch.isnan(ref), torch.isnan(g)
    miss = ref_nan & ~got_nan
    assert not bool(miss.any()), f"{what}: NaN swallowed at {torch.nonzero(miss)[0].tolist()} (got {float(g[miss][0])!r})"
    extra = got_nan & ~ref_nan
    if nan_ok is not None:
        extra &= ~nan_ok
    assert not bool(extra.any()), f"{what}: NaN at {torch.nonzero(extra)[0].tolist()} where the reference is finite"
    live = ~ref_nan & ~got_nan
    err = torch.where(live, (g - ref).abs(), 0.0)
    err = torch.where(live & (g == ref), 0.0, err)   # equal infinities
    lim = torch.where(live, torch.as_tensor(lim, dtype=torch.float64, device=DEV).expand_as(err), math.inf)
    ratio = float((err / lim.clamp_min(1e-300)).max()) if err.numel() else 0.0
    bad = err > lim
    if not bool(bad.any()):
        OBSERVED[name] = max(OBSERVED.get(name, 0.0), ratio)
    else:
        idx = tuple(torch.nonzero(bad)[0].tolist())
        raise AssertionError(f"{what}: over the bound at {list(idx)} (got {float(g[idx]):.9g}, want {float(ref[idx]):.9g}, "
                             f"bound {float(lim[idx]):.3g}); {int(bad.sum())} elements, max ratio {ratio:.3g}")


def _exact(what, got, ref):
    """got equals the FP64 reference exactly (finite; +0 == -0)"""
    g = got.double()
    ok = torch.isfinite(g) & (g == ref)
    if not bool(ok.all()):
        idx = tuple(torch.nonzero(~ok)[0].tolist())
        raise AssertionError(f"{what}: not exact at {list(idx)}: got {float(g[idx])!r}, want {float(ref[idx])!r} "
                             f"({int((~ok).sum())} elements differ)")


class Launch:
    """counts the kernels a block of calls launched"""

    def __enter__(self):
        self.n0 = _lib.launch_count()
        return self

    def __exit__(self, *exc):
        self.n = _lib.launch_count() - self.n0


def _call(kernels, name, *args):
    with Launch() as n:
        ops._call(name, *args)
    torch.cuda.synchronize()
    assert n.n == len(kernels), (name, n.n, kernels)


def _values(shape, exact, g, scale=1.0, lo=-4, hi=4):
    if exact:
        return torch.randint(lo, hi + 1, shape, generator=g, device=DEV).float()
    return torch.randn(shape, generator=g, device=DEV) * scale


# ---------------------------------------------------------------------------------------------- activations in FP64
F = torch.nn.functional
SPECIALS = [0.0, -0.0, 19.99, 20.0, 20.01, -19.99, -20.0, 88.0, 89.0, 90.0, 100.0, -88.0, -89.0, -90.0, -100.0,
            9.0, -9.0, 15.0, -15.0, 1e-30, -1e-30, 1e30, -1e30, float("nan")]
NS = len(SPECIALS)
NAN_COL = NS - 1
_ACT64 = [lambda v: v, F.silu, lambda v: F.softplus(v) - math.log(2.0), F.softplus, F.relu, torch.tanh, torch.sigmoid,
          F.gelu, F.elu, F.leaky_relu]


def act64(kind, x):
    return _ACT64[kind](x.double())


def dact64(kind, x):
    """torch's derivative (autograd in FP64) of the activation at the same argument"""
    x = x.double().detach().clone().requires_grad_(True)
    (g,) = torch.autograd.grad(_ACT64[kind](x).sum(), x)
    return g


def act_mag(kind, x):
    """magnitude of the terms the kernel forms for act(x)"""
    x = x.double()
    if kind == 1:
        return (x * torch.sigmoid(x)).abs()
    if kind == 2:
        return F.softplus(x) + math.log(2.0)
    if kind == 3:
        return F.softplus(x)
    if kind == 6:
        return torch.sigmoid(x)
    if kind == 7:
        return 0.5 * x.abs() * (1 + torch.erf(x / math.sqrt(2.0)).abs())
    return act64(kind, x).abs()


def dact_mag(kind, x):
    """magnitude of the terms the kernel forms for act'(x)"""
    x = x.double()
    s = torch.sigmoid(x)
    if kind == 1:
        return s * (1 + x.abs() * (1 + s))
    if kind in (2, 3):
        return torch.where(x > 20, 1.0, s)
    if kind == 5:
        return 1 + torch.tanh(x) ** 2
    if kind == 6:
        return s * (1 + s)
    if kind == 7:
        return 0.5 * (1 + torch.erf(x / math.sqrt(2.0)).abs()) + x.abs() * torch.exp(-0.5 * x * x) / math.sqrt(2 * math.pi)
    if kind == 8:
        return torch.where(x > 0, 1.0, torch.exp(x))
    return torch.ones_like(x)


def _act_units(name, got, ref, mag, slack=TINY):
    """records the activation error in units of u mag (the quantity K bounds), after `slack`: the underflow allowance
    and the roundings of the products the output also carries"""
    ok = torch.isfinite(ref) & torch.isfinite(got.double()) & torch.isfinite(mag)
    err = torch.where(ok, ((got.double() - ref).abs() - slack).clamp_min(0), 0.0)
    r = float((err / torch.where(ok, U * mag, 1.0).clamp_min(1e-300)).max()) if err.numel() else 0.0
    OBSERVED[name] = max(OBSERVED.get(name, 0.0), r)


def _act_lim(kind, x, grad):
    K = (K_GRAD if grad else K_FWD)[kind]
    return K * U * (dact_mag if grad else act_mag)(kind, x) + TINY


# ---------------------------------------------------------------------------------------------- graphs and segments
@functools.lru_cache(None)
def _graph(kind):
    """(edge_index (2, E) int64 on the host, N).  "bounds": out-degrees 0, 1, 31, 32, 33 and 300 (the hub), in-degrees
    300, 33, 32, 31 and 1, self-loops, nodes without in-edges and isolated nodes 600..639.  "big": 20 000 nodes."""
    g = torch.Generator().manual_seed(3 if kind == "bounds" else 4)
    if kind == "bounds":
        N = 640
        deg = torch.randint(0, 5, (N,), generator=g)
        deg[:6] = torch.tensor([0, 1, 31, 32, 33, 300])
        deg[600:] = 0
        src = torch.repeat_interleave(torch.arange(N), deg)
        E = src.numel()
        fixed = torch.cat([torch.full((n,), t) for t, n in ((10, 300), (11, 33), (12, 32), (13, 31), (14, 1))])
        rnd = torch.randint(15, 600, (E - fixed.numel(),), generator=g)
        dst = torch.cat([fixed, rnd])[torch.randperm(E, generator=g)]
        dst = torch.where((torch.arange(E) % 41 == 0) & (dst >= 15), src, dst)
    else:
        N, E = 20000, 100000
        src = torch.randint(0, N - 100, (E,), generator=g)
        dst = torch.randint(0, N - 100, (E,), generator=g)
    return torch.stack([src, dst]), N


@functools.lru_cache(None)
def _gi(kind):
    ei, N = _graph(kind)
    return ops.GraphIndex(ei.to(DEV), N)


@functools.lru_cache(None)
def _segments(kind, order):
    """(ptr, perm or None, R, E): the out-CSR, the in-CSR, the out-CSR with a hand-shuffled order inside every segment,
    or the out-CSR pointers with perm = NULL (items in storage order)"""
    gi = _gi(kind)
    if order == "in":
        return gi.in_ptr, gi.in_edge, gi.N, gi.E
    if order in ("out", "identity"):
        return gi.out_ptr, (None if order == "identity" else gi.out_edge), gi.N, gi.E
    cnt = (gi.out_ptr[1:] - gi.out_ptr[:-1]).long()
    seg = torch.repeat_interleave(torch.arange(gi.N, device=DEV), cnt)
    r = torch.randperm(gi.E, generator=torch.Generator(device=DEV).manual_seed(9), device=DEV)
    order_ = r[torch.sort(seg[r], stable=True).indices]
    return gi.out_ptr, gi.out_edge[order_].contiguous(), gi.N, gi.E


def _items(ptr, perm, E):
    """(row of every sorted position, segment of every sorted position, count per segment)"""
    cnt = (ptr[1:] - ptr[:-1]).long()
    rows = perm.long() if perm is not None else torch.arange(E, device=DEV)
    seg = torch.repeat_interleave(torch.arange(cnt.numel(), device=DEV), cnt)
    return rows, seg, cnt


def _layout(C, layout):
    """(ld, off): "vec" a row stride wider than C, "off1" one float past an aligned row start, "ldodd" an odd stride"""
    if layout == "off1":
        return C + 4 - C % 4, 1
    if layout == "ldodd":
        return C + 1, 0
    return C + 4 - C % 4, 0


# ---------------------------------------------------------------------------------------------- segment sum
# (graph, perm, C, layout, y mode, activation field, mean bit)
SEG_CASES = [
    ("bounds", "out", 128, "vec", "none", 0, 0),
    ("bounds", "in", 132, "vec", "y", 0, 1),
    ("bounds", "shuffled", 124, "vec", "act", 0, 0),       # field 0 = SiLU
    ("bounds", "identity", 260, "vec", "grad", 1, 0),
    ("bounds", "out", 128, "vec", "act", 7, 1),
    ("bounds", "in", 4, "vec", "grad", 2, 0),
    ("bounds", "out", 33, "vec", "none", 0, 1),           # odd C: scalar
    ("bounds", "shuffled", 128, "off1", "y", 0, 0),
    ("bounds", "out", 127, "ldodd", "act", 5, 0),
    ("bounds", "identity", 129, "vec", "grad", 4, 1),
    ("bounds", "in", 1, "vec", "grad", 8, 0),
    ("bounds", "out", 256, "off1", "none", 0, 0),
    ("bounds", "in", 128, "ldodd", "none", 0, 0),
    ("bounds", "out", 64, "vec", "act", 9, 0),
    ("big", "out", 128, "vec", "act", 1, 0),
    ("big", "in", 64, "off1", "none", 0, 1),
    ("big", "shuffled", 132, "vec", "grad", 9, 0),
    ("big", "identity", 128, "vec", "y", 0, 0),
]
YBITS = {"none": 0, "y": 0, "act": 2, "grad": 4}


def _seg_mode(ymode, kind, mean):
    return mean | YBITS[ymode] | (kind << 4)


def _seg_is_vec(C, layout, ymode):
    ld, off = _layout(C, layout)
    return C % 4 == 0 and ld % 4 == 0 and off == 0


def _seg_case_kernels(case):
    graph, order, C, layout, ymode, kind, mean = case
    R = _graph(graph)[1]
    return segsum_kernels(R, C, _seg_is_vec(C, layout, ymode), _seg_mode(ymode, kind, mean))


def _seg_id(c):
    return f"{_kid(_seg_case_kernels(c))}-{c[0]}-{c[1]}-C{c[2]}-{c[3]}-{c[4]}" + (f"-{ACT_NAMES[c[5]]}" if c[4] in ("act", "grad") else "") + ("-mean" if c[6] else "")


def _segsum(x, y, ptr, perm, R, C, mode, ld, off):
    """one call with padded index operands and a NaN-padded output of stride ld at offset off"""
    pb, p = _irows(R + 1, ptr, torch.int32)
    mb, m = _irows(perm.numel(), perm, torch.int32) if perm is not None else (None, None)
    ob, out = _mat(R, C, ld, off)
    before = [(b, b.clone()) for b in (pb, mb) if b is not None]
    ks = segsum_kernels(R, C, segsum_vec(C, x, y, out), mode)
    _call(ks, "lcao_segment_sum", P_(x), x.stride(0), P_(y), y.stride(0) if y is not None else 0, P_(p), P_(m), R, C,
          mode, P_(out), out.stride(0), ST())
    _padding_untouched(ob, out, "out")
    for b, b0 in before:
        assert _same_bits(b, b0), "an index operand was written"
    return out


def _seq_sum32(x, rows, ptr, R):
    """the sequential FP32 sum of every segment in perm order"""
    cnt = (ptr[1:] - ptr[:-1]).long()
    acc = torch.zeros(R, x.shape[1], device=DEV)
    start = ptr[:-1].long()
    for k in range(int(cnt.max()) if cnt.numel() else 0):
        live = cnt > k
        acc[live] = acc[live] + x[rows[start[live] + k]]
    return acc


def _seg_reference(x, y, ymode, kind, rows, seg, cnt, R):
    """(ref, mag, act allowance): FP64 sum of the terms, of their magnitudes, and sum |x| (K u mag_act(y) + tiny)"""
    xr = x[rows].double()
    C = x.shape[1]
    extra = None
    if ymode == "none":
        t = xr
    elif ymode == "y":
        t = xr * y[rows].double()
    else:
        k = kind if kind else 1
        yr = y[rows]
        f = act64(k, yr) if ymode == "act" else dact64(k, yr)
        t = xr * f
        extra = torch.zeros(R, C, dtype=torch.float64, device=DEV).index_add_(0, seg, xr.abs() * _act_lim(k, yr, ymode == "grad"))
    z = functools.partial(torch.zeros, R, C, dtype=torch.float64, device=DEV)
    ref = z().index_add_(0, seg, t)
    mag = z().index_add_(0, seg, t.abs())
    return ref, mag, (extra if extra is not None else z())


@pytest.mark.parametrize("case", SEG_CASES, ids=[_seg_id(c) for c in SEG_CASES])
def test_segment_sum(case):
    graph, order, C, layout, ymode, kind, mean = case
    ptr, perm, R, E = _segments(graph, order)
    rows, seg, cnt = _items(ptr, perm, E)
    ld, off = _layout(C, layout)
    mode = _seg_mode(ymode, kind, mean)
    for exact in ((True, False) if ymode in ("none", "y") else (False,)):
        g = torch.Generator(device=DEV).manual_seed(C + 17 * exact + 3 * len(order))
        xb, x = _mat(E, C, ld, off, _values((E, C), exact, g))
        yb, y = _mat(E, C, ld, off, _values((E, C), exact, g, scale=3.0)) if ymode != "none" else (None, None)
        inputs = [(b, b.clone()) for b in (xb, yb) if b is not None]
        out = _segsum(x, y, ptr, perm, R, C, mode, ld, off)
        again = _segsum(x, y, ptr, perm, R, C, mode, ld, off)
        assert _same_bits(out, again), "two identical calls differ"
        for b, b0 in inputs:
            assert _same_bits(b, b0), "an input buffer (operand or padding) was written"
        assert bool((out[cnt == 0] == 0).all()), "an empty segment is not exactly zero"
        kindname = "exact" if exact else "random"
        ref, mag, extra = _seg_reference(x, y, ymode, kind, rows, seg, cnt, R)
        scale = (1.0 / cnt.clamp_min(1).float()).unsqueeze(1) if mean else None
        if exact:
            want = ref.float()
            if mean:
                want = scale * want            # fp32(fp32(1 / count) * sum), the sum itself exact
            assert _same_bits(out, want), f"{kindname}: not the exact sum"
        elif ymode == "none":
            want = _seq_sum32(x, rows, ptr, R)
            if mean:
                want = scale * want
            assert _same_bits(out, want), "not bitwise the sequential FP32 sum in perm order"
            # the other path (vector <-> scalar) on the same values: bitwise the same
            ld2, off2 = _layout(C, "off1" if _seg_is_vec(C, layout, ymode) else "vec")
            xb2, x2 = _mat(E, C, ld2, off2, x)
            assert _same_bits(_segsum(x2, None, ptr, perm, R, C, mode, ld2, off2), out), "scalar and vector paths differ"
        else:
            n = (cnt + 2).double().unsqueeze(1)
            if mean:
                d = cnt.clamp_min(1).double().unsqueeze(1)
                ref, mag, extra = ref / d, mag / d, extra / d
            _check(f"segment_sum {ymode}", f"{kindname} out", out, ref, gamma(n) * mag + extra * (1 + gamma(n)))


def test_segment_sum_bounds_single_out_one_term():
    """removing one item of the 300-item hub segment from the reference makes the random-case bound fail"""
    ptr, perm, R, E = _segments("bounds", "out")
    rows, seg, cnt = _items(ptr, perm, E)
    C = 128
    g = torch.Generator(device=DEV).manual_seed(1)
    _, x = _mat(E, C, C + 4, 0, _values((E, C), False, g))
    _, y = _mat(E, C, C + 4, 0, _values((E, C), False, g, scale=3.0))
    out = _segsum(x, y, ptr, perm, R, C, 0, C + 4, 0)
    ref, mag, _ = _seg_reference(x, y, "y", 0, rows, seg, cnt, R)
    n = (cnt + 2).double().unsqueeze(1)
    _check("segment_sum y", "out", out, ref, gamma(n) * mag)
    hub = 5
    assert int(cnt[hub]) == 300
    j = int(ptr[hub]) + 150
    t = (x[rows[j]].double() * y[rows[j]].double())
    bad = (out[hub].double() - (ref[hub] - t)).abs() > gamma(302) * (mag[hub] - t.abs())
    assert bool(bad.any()), "the bound accepts the hub's sum without one of its 300 items"


@pytest.mark.parametrize("mode", [0, 1, 2 | (7 << 4), 4 | (1 << 4)])
def test_segment_sum_without_items(mode):
    """an edge-less batch passes x = y = NULL, also with bit 1 or 2: every segment is empty and out is zero-filled"""
    R, C = 50, 128
    ptr = torch.zeros(R + 1, dtype=torch.int32, device=DEV)
    ob, out = _mat(R, C, C + 4, 0)
    _call(segsum_kernels(R, C, True, mode), "lcao_segment_sum", None, C, None, C, P_(ptr), None, R, C, mode, P_(out),
          out.stride(0), ST())
    _padding_untouched(ob, out, "out")
    assert bool((out == 0).all())


# ---------------------------------------------------------------------------------------------- edge pair
# (graph, C, extra row stride of a and b, bias, pre, act)
EP_CASES = [
    ("bounds", 128, 4, True, True, 1), ("bounds", 4, 0, False, True, 0), ("bounds", 124, 8, True, False, 0),
    ("bounds", 132, 4, True, True, 7), ("bounds", 260, 0, False, True, 1), ("big", 128, 4, True, True, 1),
    ("big", 256, 0, True, False, 5), ("bounds", 128, 0, True, True, 4),
]


def _ep_id(c):
    E = _graph(c[0])[0].shape[1]
    return (f"{_kid(edge_pair_kernels(E, c[5]))}-{c[0]}-C{c[1]}-ld+{c[2]}{'-bias' if c[3] else ''}{'-pre' if c[4] else ''}"
            f"-{ACT_NAMES[c[5]]}")


def _edge_pair(a, b, bias, gi, C, act, want_pre):
    E = gi.E
    ob, out = _mat(E, C)
    pb, pre = _mat(E, C) if want_pre else (None, None)
    _call(edge_pair_kernels(E, act), "lcao_edge_pair_fwd", P_(a), a.stride(0), P_(b), b.stride(0), P_(bias),
          P_(gi.src32), P_(gi.dst32), E, C, act, P_(out), P_(pre), ST())
    _padding_untouched(ob, out, "out")
    if want_pre:
        _padding_untouched(pb, pre, "pre")
    return out, pre


@pytest.mark.parametrize("case", EP_CASES, ids=[_ep_id(c) for c in EP_CASES])
def test_edge_pair_fwd(case):
    graph, C, extra, with_bias, want_pre, act = case
    gi = _gi(graph)
    N, E = gi.N, gi.E
    s, t = gi.src32.long(), gi.dst32.long()
    for exact in (True, False):
        g = torch.Generator(device=DEV).manual_seed(C + exact)
        ab, a = _mat(N, C, C + extra, 0, _values((N, C), exact, g))
        bb, b = _mat(N, C, C + extra, 0, _values((N, C), exact, g))
        cb, bias = _mat(1, C, fill=_values((C,), exact, g)) if with_bias else (None, None)
        bias = bias.view(C) if with_bias else None
        inputs = [(q, q.clone()) for q in (ab, bb, cb) if q is not None]
        out, pre = _edge_pair(a, b, bias, gi, C, act, want_pre)
        out2, pre2 = _edge_pair(a, b, bias, gi, C, act, True)
        out3, _ = _edge_pair(a, b, bias, gi, C, act, want_pre)
        assert _same_bits(out, out3) and _same_bits(out, out2), "out differs between identical calls or with pre"
        for q, q0 in inputs:
            assert _same_bits(q, q0), "an input buffer (operand or padding) was written"
        want = a[s] + b[t]
        if with_bias:
            want = want + bias
        assert _same_bits(pre2, want), "pre is not fp32(fp32(a[s] + b[t]) + bias)"
        if want_pre:
            assert _same_bits(pre, pre2)
        if exact:
            ref = a[s].double() + b[t].double() + (bias.double() if with_bias else 0)
            _exact("exact pre", pre2, ref)
        if act == 0:
            assert _same_bits(out, pre2), "out is not pre without an activation"
        else:
            ref = act64(act, pre2)
            _act_units(f"act fwd {ACT_NAMES[act]}", out, ref, act_mag(act, pre2))
            _check(f"edge_pair act", "out", out, ref, _act_lim(act, pre2, False))


# ---------------------------------------------------------------------------------------------- message backward
# (graph, C, extra row stride of d_agg, act)
MB_CASES = [("bounds", 128, 4, 1), ("bounds", 4, 0, 3), ("bounds", 132, 8, 6), ("big", 128, 0, 1), ("bounds", 260, 4, 9),
            ("bounds", 124, 4, 4)]


def _mb_id(c):
    E = _graph(c[0])[0].shape[1]
    return f"{_kid(msg_bwd_kernels(E, c[3]))}-{c[0]}-C{c[1]}-ld+{c[2]}-{ACT_NAMES[c[3]]}"


def _msg_bwd(d_agg, src32, h, bw, pre_h, E, C, act, expect=None):
    db, d_bw = _mat(E, C)
    pb, d_pre = _mat(E, C)
    if expect is None:
        _call(msg_bwd_kernels(E, act), "lcao_msg_bwd", P_(d_agg), d_agg.stride(0), P_(src32), P_(h), P_(bw), P_(pre_h),
              E, C, act, P_(d_bw), P_(d_pre), ST())
    else:
        rc = _lib.load().lcao_msg_bwd(P_(d_agg), d_agg.stride(0), P_(src32), P_(h), P_(bw), P_(pre_h), E, C, act, P_(d_bw),
                                      P_(d_pre), ST())
        torch.cuda.synchronize()
        assert rc == expect
    _padding_untouched(db, d_bw, "d_bw")
    _padding_untouched(pb, d_pre, "d_pre_h")
    return d_bw, d_pre


def _msg_bwd_refs(g, b, p, act):
    """(d_bw from act(p): ref, lim), (d_pre_h: ref, lim) in FP64"""
    g64, b64 = g.double(), b.double()
    a = act64(act, p)
    ref_bw = g64 * a
    lim_bw = g64.abs() * _act_lim(act, p, False) * (1 + U) + U * ref_bw.abs()
    da = dact64(act, p)
    ref_d = g64 * b64 * da
    lim_d = (g64 * b64).abs() * _act_lim(act, p, True) * (1 + gamma(2)) + gamma(2) * ref_d.abs()
    return (ref_bw, lim_bw), (ref_d, lim_d)


def _msg_units(act, ga, bw, p, d_bw, rb, d_pre, rd):
    g1, g2 = ga.double().abs(), (ga.double() * bw.double()).abs()
    _act_units(f"act fwd {ACT_NAMES[act]}", d_bw, rb, g1 * act_mag(act, p), g1 * TINY + U * rb.abs())
    _act_units(f"act grad {ACT_NAMES[act]}", d_pre, rd, g2 * dact_mag(act, p), g2 * TINY + gamma(2) * rd.abs())


@pytest.mark.parametrize("case", MB_CASES, ids=[_mb_id(c) for c in MB_CASES])
def test_msg_bwd(case):
    graph, C, extra, act = case
    gi = _gi(graph)
    N, E = gi.N, gi.E
    s = gi.src32.long()
    for exact in (True, False):
        g = torch.Generator(device=DEV).manual_seed(C + act + exact)
        ab, d_agg = _mat(N, C, C + extra, 0, _values((N, C), exact, g))
        hb, h = _mat(E, C, fill=_values((E, C), exact, g))
        wb, bw = _mat(E, C, fill=_values((E, C), exact, g))
        pb, pre_h = _mat(E, C, fill=_values((E, C), False, g, scale=3.0))
        inputs = [(q, q.clone()) for q in (ab, hb, wb, pb)]
        d_bw_h, d_pre_h = _msg_bwd(d_agg, gi.src32, h, bw, pre_h, E, C, act)
        d_bw, d_pre = _msg_bwd(d_agg, gi.src32, None, bw, pre_h, E, C, act)
        d_bw2, d_pre2 = _msg_bwd(d_agg, gi.src32, None, bw, pre_h, E, C, act)
        assert _same_bits(d_bw, d_bw2) and _same_bits(d_pre, d_pre2), "two identical calls differ"
        assert _same_bits(d_pre, d_pre_h), "d_pre_h depends on whether h is given"
        for q, q0 in inputs:
            assert _same_bits(q, q0), "an input buffer (operand or padding) was written"
        ga = d_agg[s]
        assert _same_bits(d_bw_h, ga * h), "d_bw is not fp32(d_agg[src] * h)"
        if exact:
            _exact("exact d_bw", d_bw_h, ga.double() * h.double())
        (rb, lb), (rd, ld_) = _msg_bwd_refs(ga, bw, pre_h, act)
        _msg_units(act, ga, bw, pre_h, d_bw, rb, d_pre, rd)
        _check("msg_bwd d_bw", "d_bw (h recomputed)", d_bw, rb, lb)
        _check("msg_bwd d_pre_h", "d_pre_h", d_pre, rd, ld_)


# ---------------------------------------------------------------------------------------------- every activation
@pytest.mark.parametrize("kind", range(10), ids=[f"{ACT_NAMES[k]}" for k in range(10)])
def test_activation_in_every_entry_point(kind):
    """act_fwd, edge_pair, segment_sum bits 1 and 2 (vector and scalar path) and msg_bwd with and without h, each with
    the special arguments in columns 0..23 of every row (NaN in column 23)"""
    C = 128
    spec = torch.tensor(SPECIALS, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(40 + kind)
    name = ACT_NAMES[kind]
    nan_col = torch.zeros(C, dtype=torch.bool, device=DEV)
    nan_col[NAN_COL] = True

    # lcao_act_fwd, out of place and in place
    M = 300
    X = torch.randn(M, C, generator=g, device=DEV) * 4
    X[:, :NS] = spec
    xb, x = _mat(M, C, C + 8, 0, X)
    yb, y = _mat(M, C, C + 4, 0)
    x0 = xb.clone()
    _call(["k_act_fwd"], "lcao_act_fwd", P_(x), x.stride(0), P_(y), y.stride(0), M, C, kind, ST())
    _padding_untouched(yb, y, "Y")
    assert _same_bits(xb, x0), "X was written"
    ref = act64(kind, x)
    _act_units(f"act fwd {name}", y, ref, act_mag(kind, x))
    _check("act_fwd", f"act_fwd {name}", y, ref, _act_lim(kind, x, False))
    _call(["k_act_fwd"], "lcao_act_fwd", P_(x), x.stride(0), P_(x), x.stride(0), M, C, kind, ST())
    assert _same_or_nan(x, y), "act_fwd in place differs from out of place"
    _padding_untouched(xb, x, "X in place")

    # lcao_edge_pair_fwd: pre = a[s] in the special columns (b and bias are zero there)
    gi = _gi("bounds")
    N, E = gi.N, gi.E
    A = torch.randn(N, C, generator=g, device=DEV) * 2
    A[:, :NS] = spec
    Bt = torch.randn(N, C, generator=g, device=DEV) * 2
    Bt[:, :NS] = 0
    bias_v = torch.randn(C, generator=g, device=DEV)
    bias_v[:NS] = 0
    _, a = _mat(N, C, C + 4, 0, A)
    _, b = _mat(N, C, C + 4, 0, Bt)
    _, bias = _mat(1, C, fill=bias_v)
    out, pre = _edge_pair(a, b, bias.view(C), gi, C, kind, True)
    assert _same_or_nan(pre, (a[gi.src32.long()] + b[gi.dst32.long()]) + bias.view(C)), "pre is not the FP32 sum"
    ref = act64(kind, pre)
    _act_units(f"act fwd {name}", out, ref, act_mag(kind, pre))
    _check("edge_pair act", f"edge_pair {name}", out, ref, _act_lim(kind, pre, False))

    # lcao_segment_sum, bits 1 and 2, vector and scalar paths (the field's 0 is SiLU)
    k = kind if kind else 1
    ptr, perm, R, E = _segments("bounds", "out")
    rows, seg, cnt = _items(ptr, perm, E)
    Xs = torch.randn(E, C, generator=g, device=DEV)
    Ys = torch.randn(E, C, generator=g, device=DEV) * 4
    Ys[:, :NS] = spec
    results = {}
    for layout in ("vec", "off1"):
        ld, off = _layout(C, layout)
        _, xs = _mat(E, C, ld, off, Xs)
        _, ys = _mat(E, C, ld, off, Ys)
        for ymode in ("act", "grad"):
            mode = YBITS[ymode] | (kind << 4)
            o = _segsum(xs, ys, ptr, perm, R, C, mode, ld, off)
            results[(layout, ymode)] = o
            t_ref, t_mag, t_extra = _seg_reference(xs, ys, ymode, kind, rows, seg, cnt, R)
            n = (cnt + 2).double().unsqueeze(1)
            nan_ok = (nan_col.unsqueeze(0) & (cnt > 0).unsqueeze(1)) if ymode == "grad" else None
            _check(f"segment_sum {ymode}", f"segment_sum {ymode} {name} {layout}", o, t_ref,
                   gamma(n) * t_mag + t_extra * (1 + gamma(n)), nan_ok=nan_ok)
            if kind == 0:   # field 0 and field SiLU run the same kernel: bitwise the same
                o1 = _segsum(xs, ys, ptr, perm, R, C, YBITS[ymode] | (1 << 4), ld, off)
                assert _same_or_nan(o, o1)

    # lcao_msg_bwd: the activation's derivative is the point; NONE is rejected (the message has an activation)
    d_agg = torch.randn(N, C, generator=g, device=DEV)
    _, bw = _mat(E, C, fill=torch.randn(E, C, generator=g, device=DEV))
    _, h = _mat(E, C, fill=torch.randn(E, C, generator=g, device=DEV))
    Pp = torch.randn(E, C, generator=g, device=DEV) * 4
    Pp[:, :NS] = spec
    _, pre_h = _mat(E, C, fill=Pp)
    if kind == 0:
        _msg_bwd(d_agg, gi.src32, h, bw, pre_h, E, C, 0, expect=-1)
        return
    ga = d_agg[gi.src32.long()]
    d_bw_h, d_pre_h = _msg_bwd(d_agg, gi.src32, h, bw, pre_h, E, C, kind)
    d_bw, d_pre = _msg_bwd(d_agg, gi.src32, None, bw, pre_h, E, C, kind)
    assert _same_bits(d_bw_h, ga * h) and _same_or_nan(d_pre, d_pre_h)
    (rb, lb), (rd, ld_) = _msg_bwd_refs(ga, bw, pre_h, kind)
    _check("msg_bwd d_bw", f"msg_bwd d_bw {name}", d_bw, rb, lb)
    _check("msg_bwd d_pre_h", f"msg_bwd d_pre_h {name}", d_pre, rd, ld_, nan_ok=nan_col.expand(E, C))
    _msg_units(kind, ga, bw, pre_h, d_bw, rb, d_pre, rd)


def test_relu_propagates_nan_like_torch():
    """ReLU(NaN) is NaN and its derivative passes the gradient (torch.relu / threshold_backward)"""
    x = torch.tensor([float("nan"), -0.0, 0.0, -1.0, 2.0, float("-inf")] + [0.0] * 2, device=DEV).view(2, 4)
    _, y = _mat(2, 4)
    _call(["k_act_fwd"], "lcao_act_fwd", P_(x), 4, P_(y), 4, 2, 4, 4, ST())
    want = torch.relu(x)
    assert torch.equal(torch.isnan(y), torch.isnan(want)) and bool((y == want)[~torch.isnan(want)].all()), y
    ptr = torch.arange(9, dtype=torch.int32, device=DEV)
    ones = torch.ones(8, 4, device=DEV)
    xx = torch.tensor([float("nan"), -0.0, 0.0, -1.0, 2.0, float("-inf"), 3.0, -3.0], device=DEV).view(8, 1).expand(8, 4).contiguous()
    d = _segsum(ones, xx, ptr, None, 8, 4, 4 | (4 << 4), 4, 0)
    xr = xx.double().requires_grad_(True)
    (want,) = torch.autograd.grad(torch.relu(xr).sum(), xr)
    assert torch.equal(d.double(), want), (d, want)


# ---------------------------------------------------------------------------------------------- gather rows
# (n, W, extra table stride, row offset, int64 index, mul, extra out / mul stride)
GATHER_CASES = [
    (5000, 128, 4, 0, True, True, 0), (5000, 1792, 0, 0, False, False, 4), (3000, 33, 0, 0, True, False, 0),
    (3000, 128, 4, 1, False, True, 0), (100000, 4, 0, 0, False, False, 0), (777, 130, 2, 0, True, True, 2),
    (1, 1, 0, 0, False, True, 0), (4000, 256, 4, 0, True, False, 0), (4000, 128, 0, 1, True, False, 4),
]
T_ROWS = 37


def _gather_is_vec(c):
    n, W, te, off, is64, mul, oe = c
    return W % 4 == 0 and (W + te) % 4 == 0 and (W + oe) % 4 == 0 and off == 0


def _gather_id(c):
    n, W, te, off, is64, mul, oe = c
    return f"{_kid(gather_kernels(n, W, is64, _gather_is_vec(c)))}-n{n}-W{W}-ldt+{te}-off{off}{'-mul' if mul else ''}-ldo+{oe}"


@pytest.mark.parametrize("case", GATHER_CASES, ids=[_gather_id(c) for c in GATHER_CASES])
def test_gather_rows(case):
    n, W, te, off, is64, with_mul, oe = case
    for exact in (True, False):
        g = torch.Generator(device=DEV).manual_seed(n + W + exact)
        tb, table = _mat(T_ROWS, W, W + te, off, _values((T_ROWS, W), exact, g))
        idx = torch.randint(0, T_ROWS - 3, (n,), generator=g, device=DEV)   # the last three rows are never gathered
        ib, ix = _irows(n, idx, torch.int64 if is64 else torch.int32)
        mb, mul = _mat(n, W, W + oe, off, _values((n, W), exact, g)) if with_mul else (None, None)
        inputs = [(q, q.clone()) for q in (tb, ib, mb) if q is not None]
        outs = []
        for _ in range(2):
            ob, out = _mat(n, W, W + oe, off)
            ks = gather_kernels(n, W, is64, gather_vec(W, table, mul, out))
            assert ks == gather_kernels(n, W, is64, _gather_is_vec(case))
            _call(ks, "lcao_gather_rows", P_(table), table.stride(0), P_(ix), int(is64), P_(mul),
                  mul.stride(0) if with_mul else 0, n, W, P_(out), out.stride(0), ST())
            _padding_untouched(ob, out, "out")
            outs.append(out)
        assert _same_bits(outs[0], outs[1]), "two identical calls differ"
        for q, q0 in inputs:
            assert _same_bits(q, q0), "an input buffer (operand or padding) was written"
        want = table[idx]
        if with_mul:
            want = want * mul
        assert _same_bits(outs[0], want), "not bitwise table[idx] (* mul)"
        if exact:
            _exact("exact gather", outs[0], table[idx].double() * (mul.double() if with_mul else 1))


# ---------------------------------------------------------------------------------------------- reduce by key
RUN_SIZES = (1, 31, 32, 33, 64, 1000)


@functools.lru_cache(None)
def _key_layout(kind):
    """(counts per key (host int64), nkeys): "runs" puts a run of every RUN_SIZES length on, one before and one after a
    32-entry chunk boundary, separated by filler keys and empty keys, with two leading and three trailing empty keys;
    "one" is nkeys = 1; "big" 60 000 entries over 1369 keys"""
    if kind == "one":
        return torch.tensor([1000]), 1
    if kind == "big":
        g = torch.Generator().manual_seed(12)
        k = torch.randint(0, 1369, (60000,), generator=g)
        k = torch.where(k % 50 == 0, k + 1, k)        # every 50th key empty
        return torch.bincount(k, minlength=1369), 1369
    counts, pos = [0, 0], 0
    for size in RUN_SIZES:
        for target in (0, 31, 1):                      # on, one before, one after a boundary
            fill = (target - pos) % RBK_CHUNK
            counts += [fill, 0]
            counts.append(size)
            pos += fill + size
    counts += [0, 0, 0]
    return torch.tensor(counts), len(counts)


def _run_starts(counts):
    starts = torch.cumsum(counts, 0) - counts
    return {(int(c), int(s) % RBK_CHUNK) for c, s in zip(counts, starts) if c > 0}


def _flushes(kptr):
    """chunks each key's run touches: one atomic flush of every column per chunk"""
    lo, hi = kptr[:-1].long(), kptr[1:].long()
    return torch.where(hi > lo, (hi - 1) // RBK_CHUNK - lo // RBK_CHUNK + 1, 0)


# (key layout, W, extra row stride of x)
RBK_CASES = [("runs", 128, 4), ("runs", 4, 0), ("runs", 1024, 0), ("runs", 1028, 4), ("runs", 1792, 0), ("one", 260, 4),
             ("big", 1792, 0), ("big", 128, 4)]


class KeyOps:
    def __init__(self, kind, W, extra, exact, seed):
        counts, nkeys = _key_layout(kind)
        n = int(counts.sum())
        g = torch.Generator(device=DEV).manual_seed(seed)
        self.W, self.n, self.nkeys = W, n, nkeys
        kptr = torch.zeros(nkeys + 1, dtype=torch.int32)
        kptr[1:] = torch.cumsum(counts, 0)
        self.kpb, self.kptr = _irows(nkeys + 1, kptr.to(DEV), torch.int32)
        self.kmb, self.kperm = _irows(n, torch.randperm(n, generator=g, device=DEV).int(), torch.int32)
        self.xb, self.x = _mat(n, W, W + extra, 0, _values((n, W), exact, g))
        self.init = _values((nkeys, W), exact, g)
        self.keys = torch.repeat_interleave(torch.arange(nkeys, device=DEV), counts.to(DEV))
        self.inputs = [(q, q.clone()) for q in (self.kpb, self.kmb, self.xb)]

    def run(self, init=None):
        ab, acc = _mat(self.nkeys, self.W, fill=self.init if init is None else init)
        _call(rbk_kernels(self.n), "lcao_reduce_by_key", P_(self.x), self.x.stride(0), P_(self.kptr), P_(self.kperm),
              self.nkeys, self.n, self.W, P_(acc), ST())
        _padding_untouched(ab, acc, "acc")
        for q, q0 in self.inputs:
            assert _same_bits(q, q0), "an input buffer (operand or padding) was written"
        return acc

    def reference(self):
        xr = self.x[self.kperm.long()].double()
        ref = self.init.double().index_add(0, self.keys, xr)
        mag = self.init.double().abs().index_add(0, self.keys, xr.abs())
        return ref, mag


def _rbk_id(c):
    counts, nkeys = _key_layout(c[0])
    return f"k_reduce_by_key-{c[0]}-n{int(counts.sum())}-keys{nkeys}-W{c[1]}-ldx+{c[2]}"


@pytest.mark.parametrize("case", RBK_CASES, ids=[_rbk_id(c) for c in RBK_CASES])
def test_reduce_by_key(case):
    kind, W, extra = case
    for exact in (True, False):
        k = KeyOps(kind, W, extra, exact, seed=W + 5 * exact)
        acc = k.run()
        empty = (k.kptr[1:] == k.kptr[:-1])
        assert _same_bits(acc[empty], k.init[empty]), "a key without entries changed"
        ref, mag = k.reference()
        if exact:
            _exact("exact acc", acc, ref)      # also pins +=: init is non-zero
            assert _same_bits(acc, k.run()), "two identical calls differ on exact data"
        else:
            n = (RBK_CHUNK + _flushes(k.kptr) + 1).double().unsqueeze(1)
            _check("reduce_by_key", "random acc", acc, ref, gamma(n) * mag)


def test_reduce_by_key_bound_single_out_one_entry():
    """removing the entry at a 32-entry chunk boundary inside the 1000-entry run from the reference fails the bound"""
    k = KeyOps("runs", 128, 4, False, seed=3)
    acc = k.run()
    ref, mag = k.reference()
    n = (RBK_CHUNK + _flushes(k.kptr) + 1).double().unsqueeze(1)
    _check("reduce_by_key", "acc", acc, ref, gamma(n) * mag)
    cnt = (k.kptr[1:] - k.kptr[:-1]).long()
    key = int(torch.nonzero(cnt == 1000)[0])
    j = int(k.kptr[key])
    j += (-j) % RBK_CHUNK + RBK_CHUNK                  # a chunk start inside the run
    assert int(k.keys[j]) == key and j % RBK_CHUNK == 0
    t = k.x[int(k.kperm[j])].double()
    bad = (acc[key].double() - (ref[key] - t)).abs() > gamma(n[key]) * (mag[key] - t.abs())
    assert bool(bad.any()), "the bound accepts the key's sum without one of its 1000 entries"


# ---------------------------------------------------------------------------------------------- histogram
HIST_CASES = [(100000, 1369), (5000, 37), (3000, 1), (1, 5), (0, 9)]


@pytest.mark.parametrize("n,nb", HIST_CASES, ids=[f"{_kid(['k_hist_f'] if n else [])}-n{n}-nb{nb}" for n, nb in HIST_CASES])
def test_histogram(n, nb):
    g = torch.Generator(device=DEV).manual_seed(n + nb)
    keys = torch.randint(-3, nb + 3, (n,), generator=g, device=DEV)
    if n > 10:
        keys[:4] = torch.tensor([-(2 ** 62), 2 ** 62, nb, -1], device=DEV)
        keys[4:1000] = nb // 2                          # one hot key: whole warps agree
    kb, k = _irows(n, keys, torch.int64)
    k0 = kb.clone()
    res = []
    for _ in range(2):
        cb, counts = _mat(1, nb)
        _call(["k_hist_f"] if n else [], "lcao_histogram", P_(k) if n else None, n, nb, P_(counts), ST())
        _padding_untouched(cb, counts, "counts")
        res.append(counts.view(nb))
    assert _same_bits(kb, k0), "keys were written"
    inr = keys[(keys >= 0) & (keys < nb)]
    want = torch.bincount(inr, minlength=nb).double()
    _exact("counts (out-of-range keys dropped)", res[0], want)
    assert _same_bits(res[0], res[1])


# ---------------------------------------------------------------------------------------------- pair outer
PO_CASES = [(1, 1, 4), (9, 5, 12), (20, 3, 128), (37, 14, 128), (5, 64, 260)]


def _po_id(c):
    return f"k_pair_outer_fwd+k_pair_outer_bwd-Zd{c[0]}-O{c[1]}-K{c[2]}{'-grid-stride' if outer_grid_strides(*c) else ''}"


def _pair_outer(Zd, O, K, exact, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    fb, fe = _mat(Zd * O, K, fill=_values((Zd * O, K), exact, g))
    ab, za = _mat(Zd, K, fill=_values((Zd, K), exact, g, scale=0.5))
    bb, zb = _mat(Zd, K, fill=_values((Zd, K), exact, g, scale=0.5))
    db, dpre = _mat(Zd * Zd * O, K, fill=_values((Zd * Zd * O, K), exact, g))
    inputs = [(q, q.clone()) for q in (fb, ab, bb, db)]
    res = []
    for _ in range(2):
        pb, pre = _mat(Zd * Zd * O, K)
        _call(["k_pair_outer_fwd"], "lcao_pair_outer_fwd", P_(fe), P_(za), P_(zb), Zd, O, K, P_(pre), ST())
        _padding_untouched(pb, pre, "pre")
        outs = [_mat(Zd * O, K), _mat(Zd, K), _mat(Zd, K)]
        _call(["k_pair_outer_bwd"], "lcao_pair_outer_bwd", P_(dpre), P_(fe), P_(za), P_(zb), Zd, O, K,
              *[P_(v) for _, v in outs], ST())
        for (b_, v), nm in zip(outs, ("d_fe", "d_za", "d_zb")):
            _padding_untouched(b_, v, nm)
        res.append((pre, *[v for _, v in outs]))
    for a, b in zip(*res):
        assert _same_bits(a, b), "two identical calls differ"
    for q, q0 in inputs:
        assert _same_bits(q, q0), "an input buffer (operand or padding) was written"
    v = dict(fe=fe.view(Zd, O, K), za=za, zb=zb, dpre=dpre.view(Zd, Zd, O, K))
    return v, [r.view(s) for r, s in zip(res[0], ((Zd, Zd, O, K), (Zd, O, K), (Zd, K), (Zd, K)))]


def _po_reference(v):
    fe, za, zb, dp = (v[k].double() for k in ("fe", "za", "zb", "dpre"))
    fac = 1 + za[:, None, None, :] + zb[None, :, None, :]             # (s, t, 1, K)
    facm = 1 + za.abs()[:, None, None, :] + zb.abs()[None, :, None, :]
    d_fe = (dp * fac).sum(0), (dp.abs() * facm).sum(0)
    d_za = (dp * fe[None]).sum((1, 2)), (dp.abs() * fe.abs()[None]).sum((1, 2))
    d_zb = (dp * fe[None]).sum((0, 2)), (dp.abs() * fe.abs()[None]).sum((0, 2))
    return fe[None] * fac, d_fe, d_za, d_zb


@pytest.mark.parametrize("case", PO_CASES, ids=[_po_id(c) for c in PO_CASES])
def test_pair_outer(case):
    Zd, O, K = case
    for exact in (True, False):
        v, (pre, d_fe, d_za, d_zb) = _pair_outer(Zd, O, K, exact, seed=Zd + O + K + exact)
        pre_ref, (fr, fm), (ar, am), (br, bm) = _po_reference(v)
        want = v["fe"][None] * ((1 + v["za"][:, None, None, :]) + v["zb"][None, :, None, :])
        assert _same_bits(pre, want), "pre is not fp32(fe * fp32(fp32(1 + za) + zb))"
        if exact:
            _exact("exact pre", pre, pre_ref)
            _exact("exact d_fe", d_fe, fr)
            _exact("exact d_za", d_za, ar)
            _exact("exact d_zb", d_zb, br)
        else:
            # d_fe: Zd FMAs after the two roundings of the factor; d_za, d_zb: Zd O FMAs
            _check("pair_outer d_fe", "d_fe", d_fe, fr, gamma(Zd + 2) * fm)
            _check("pair_outer d_za", "d_za", d_za, ar, gamma(Zd * O) * am)
            _check("pair_outer d_zb", "d_zb", d_zb, br, gamma(Zd * O) * bm)


def test_pair_outer_bound_single_out_one_term():
    """removing the s = 17 term of one d_fe element from the reference fails the bound"""
    Zd, O, K = 37, 14, 128
    v, (pre, d_fe, _, _) = _pair_outer(Zd, O, K, False, seed=5)
    _, (fr, fm), _, _ = _po_reference(v)
    _check("pair_outer d_fe", "d_fe", d_fe, fr, gamma(Zd + 2) * fm)
    s, t, o = 17, 4, 3
    dp = v["dpre"][s, t, o].double()
    term = dp * (1 + v["za"][s].double() + v["zb"][t].double())
    tm = dp.abs() * (1 + v["za"][s].double().abs() + v["zb"][t].double().abs())
    bad = (d_fe[t, o].double() - (fr[t, o] - term)).abs() > gamma(Zd + 2) * (fm[t, o] - tm)
    assert bool(bad.any()), "the d_fe bound accepts the sum without one s term"


# ---------------------------------------------------------------------------------------------- table norm
# (R, F, training, affine, running buffers, num_batches_tracked, momentum, rows with count 0, offset data)
TN_CASES = [
    (1, 1, True, True, True, True, 0.1, False, False),
    (5, 33, True, True, True, True, 0.1, True, False),
    (37, 128, True, False, False, False, 0.1, False, False),
    (1369, 1000, True, True, True, True, 1.0, True, False),
    (5000, 128, True, True, True, False, 0.0, True, False),
    (37, 1000, False, True, True, True, 0.1, False, False),
    (5, 128, False, False, True, False, 0.1, False, False),
    (1, 33, True, True, False, False, 0.1, False, False),
    (1369, 33, False, True, True, False, 0.1, True, False),
    (37, 128, True, True, True, True, 0.1, False, True),
    (5000, 1, False, False, True, True, 0.1, True, False),
]
EPS = 1e-5


def _tn_id(c):
    R, F_, tr, aff, run, trk, mom, zero, offs = c
    return (f"k_wbn_fwd+k_wbn_bwd-R{R}-F{F_}-{'train' if tr else 'eval'}{'-affine' if aff else ''}{'-running' if run else ''}"
            f"{'-tracked' if trk else ''}-m{mom}{'-zero-rows' if zero else ''}{'-offset' if offs else ''}")


class NormOps:
    def __init__(self, case, seed, counts=None):
        R, F_, tr, aff, run, trk, mom, zero, offs = case
        g = torch.Generator(device=DEV).manual_seed(seed)
        self.R, self.F, self.training, self.mom = R, F_, tr, mom
        X = 1000 + 0.1 * torch.randn(R, F_, generator=g, device=DEV) if offs else torch.randn(R, F_, generator=g, device=DEV)
        self.xb, self.x = _mat(R, F_, fill=X)
        if counts is None:
            counts = torch.randint(1, 6, (R,), generator=g, device=DEV).float()
            if R == 1:
                counts[0] = 7
            if zero:
                counts[::4] = 0
        self.cb, self.counts = _mat(1, R, fill=counts)
        self.counts = self.counts.view(R)
        f = lambda s: _mat(1, F_, fill=s)   # noqa: E731
        self.gb, self.gam = f(1 + 0.3 * torch.randn(F_, generator=g, device=DEV)) if aff else (None, None)
        self.bb, self.bet = f(torch.randn(F_, generator=g, device=DEV)) if aff else (None, None)
        self.rmb, self.rm = f(0.2 * torch.randn(F_, generator=g, device=DEV)) if run else (None, None)
        self.rvb, self.rv = f(0.5 + torch.rand(F_, generator=g, device=DEV)) if run else (None, None)
        self.tb, self.tracked = _irows(1, torch.tensor([5], device=DEV), torch.int64) if trk else (None, None)
        self.rm0 = self.rm.clone() if run else None
        self.rv0 = self.rv.clone() if run else None
        self.dyb, self.dy = _mat(R, F_, fill=torch.randn(R, F_, generator=g, device=DEV))
        self.inputs = [(q, q.clone()) for q in (self.xb, self.cb, self.gb, self.bb, self.dyb) if q is not None]

    def fwd(self):
        R, F_ = self.R, self.F
        yb, y = _mat(R, F_)
        mb, mean = _mat(1, F_)
        sb, rstd = _mat(1, F_)
        if self.rm is not None:                            # every call starts from the same running statistics
            self.rm.copy_(self.rm0), self.rv.copy_(self.rv0)
        if self.tracked is not None:
            self.tracked.fill_(5)
        _call(["k_wbn_fwd"], "lcao_table_norm_fwd", P_(self.x), P_(self.counts), P_(self.gam), P_(self.bet), R, F_, EPS,
              self.mom, int(self.training), P_(self.rm), P_(self.rv), P_(self.tracked), P_(y), P_(mean), P_(rstd), ST())
        for b_, v, nm in ((yb, y, "y"), (mb, mean, "save_mean"), (sb, rstd, "save_rstd")):
            _padding_untouched(b_, v, nm)
        for b_, v, nm in ((self.rmb, self.rm, "running_mean"), (self.rvb, self.rv, "running_var"),
                          (self.tb, self.tracked, "tracked")):
            if b_ is not None:
                _padding_untouched(b_, v, nm)
        return dict(y=y, mean=mean.view(F_), rstd=rstd.view(F_),
                    rm=None if self.rm is None else self.rm.clone().view(F_),
                    rv=None if self.rv is None else self.rv.clone().view(F_),
                    tracked=None if self.tracked is None else int(self.tracked[0]))

    def bwd(self, mean, rstd):
        R, F_ = self.R, self.F
        xb, dx = _mat(R, F_)
        gb, dg = _mat(1, F_)
        bb, db = _mat(1, F_)
        _call(["k_wbn_bwd"], "lcao_table_norm_bwd", P_(self.dy), P_(self.x), P_(self.counts), P_(self.gam), P_(mean),
              P_(rstd), R, F_, int(self.training), P_(dx), P_(dg), P_(db), ST())
        for b_, v, nm in ((xb, dx, "dx"), (gb, dg, "dgamma"), (bb, db, "dbeta")):
            _padding_untouched(b_, v, nm)
        return dx, dg.view(F_), db.view(F_)

    def inputs_unchanged(self):
        for q, q0 in self.inputs:
            assert _same_bits(q, q0), "an input buffer (operand or padding) was written"


def _tn_fwd_bounds(op, got, counts=None):
    """checks save_mean, save_rstd, y and the running statistics of one forward call"""
    x = op.x.double()
    c = (op.counts if counts is None else counts).double()
    n = c.sum()
    w = (c / n).unsqueeze(1)
    R, F_ = op.R, op.F
    gam = op.gam.view(F_).double() if op.gam is not None else torch.ones(F_, dtype=torch.float64, device=DEV)
    bet = op.bet.view(F_).double() if op.bet is not None else torch.zeros(F_, dtype=torch.float64, device=DEV)
    m_got, r_got = got["mean"].double(), got["rstd"].double()
    lane = math.ceil(R / 32)
    if op.training:
        # mean: a lane's FMA chain (ceil(R / 32)), the 32-lane column sum, the division by n
        nm = lane + 32 + 1
        mean64 = (w * x).sum(0)
        _check("table_norm mean", "save_mean", got["mean"], mean64, gamma(nm) * (w * x.abs()).sum(0))
        # variance two-pass around the kernel's own mean: sum w (x - m)^2 = var + (m - mean)^2 exactly; the kernel adds
        # the roundings of x - m, c d and its FMA chain
        d = x - m_got
        v_ref = (w * d * d).sum(0)
        dv = gamma(nm + 3) * v_ref
        r_ref = 1 / torch.sqrt(v_ref + EPS)
        # rstd: the variance error, the rounding of v + eps and 2 ulp of rsqrtf
        lim_r = r_ref * (0.5 * dv / (v_ref + EPS) + 0.5 * U + 4 * U) * 1.01
        _check("table_norm rstd", "save_rstd", got["rstd"], r_ref, lim_r)
    else:
        assert _same_bits(got["mean"], op.rm0.view(F_)), "eval: save_mean is not running_mean"
        v_ref = op.rv0.view(F_).double()
        r_ref = 1 / torch.sqrt(v_ref + EPS)
        _check("table_norm rstd", "save_rstd (eval)", got["rstd"], r_ref, r_ref * 4.5 * U * 1.01)
    # y from the kernel's own mean and rstd: x - m, gamma * rstd and the FMA
    d = x - m_got
    y_ref = d * (gam * r_got) + bet
    _check("table_norm y", "y", got["y"], y_ref, gamma(3) * (d.abs() * (gam.abs() * r_got) + bet.abs()))
    if op.rm is not None:
        if op.training:
            m32 = float(torch.tensor(op.mom, dtype=torch.float32))
            rm0, rv0 = op.rm0.view(F_).double(), op.rv0.view(F_).double()
            ref = (1 - m32) * rm0 + m32 * m_got
            _check("table_norm running", "running_mean", got["rm"], ref, gamma(4) * ((1 - m32) * rm0.abs() + m32 * m_got.abs()))
            unb = float(n / (n - 1))
            ref = (1 - m32) * rv0 + m32 * v_ref * unb
            _check("table_norm running", "running_var", got["rv"], ref,
                   gamma(6) * ((1 - m32) * rv0 + m32 * v_ref * unb) + m32 * dv * unb)
        else:
            assert _same_bits(got["rm"], op.rm0.view(F_)) and _same_bits(got["rv"], op.rv0.view(F_)), "eval changed the running statistics"
    if op.tracked is not None:
        assert got["tracked"] == (6 if op.training else 5), "num_batches_tracked"


def _tn_vs_batchnorm(op):
    """the FP64 statistics the bounds above are built from are those of nn.BatchNorm1d on the expanded batch (each row
    repeated count times): y of the counted rows and the updated running statistics"""
    F_ = op.F
    c = op.counts.long()
    x = op.x.double()
    w = (op.counts.double() / op.counts.double().sum()).unsqueeze(1)
    gam = op.gam.view(F_).double() if op.gam is not None else 1.0
    bet = op.bet.view(F_).double() if op.bet is not None else 0.0
    if op.training:
        mean = (w * x).sum(0)
        var = (w * (x - mean) ** 2).sum(0)
    else:
        mean, var = op.rm0.view(F_).double(), op.rv0.view(F_).double()
    y64 = (x - mean) / torch.sqrt(var + EPS) * gam + bet
    xe = torch.repeat_interleave(op.x.double(), c, dim=0)
    bn = torch.nn.BatchNorm1d(F_, eps=EPS, momentum=op.mom, affine=op.gam is not None,
                              track_running_stats=op.rm is not None).double().to(DEV)
    with torch.no_grad():
        if op.gam is not None:
            bn.weight.copy_(op.gam.view(F_)), bn.bias.copy_(op.bet.view(F_))
        if op.rm is not None:
            bn.running_mean.copy_(op.rm0.view(F_)), bn.running_var.copy_(op.rv0.view(F_))
    bn.train(op.training)
    if not op.training and op.rm is None:
        return
    ye = bn(xe).detach()
    assert torch.allclose(torch.repeat_interleave(y64, c, dim=0), ye, rtol=1e-9, atol=1e-9), "y differs from nn.BatchNorm1d"
    if op.training and op.rm is not None:
        n = float(op.counts.double().sum())
        rm = (1 - op.mom) * op.rm0.view(F_).double() + op.mom * mean
        rv = (1 - op.mom) * op.rv0.view(F_).double() + op.mom * var * n / (n - 1)
        assert torch.allclose(rm, bn.running_mean, rtol=1e-9, atol=1e-12)
        assert torch.allclose(rv, bn.running_var, rtol=1e-9, atol=1e-12)


def _tn_bwd_bounds(op, got, dx, dg, db):
    """dx, dgamma and dbeta against FP64 given the kernel's save_mean / save_rstd (inputs of the backward)"""
    x, dy = op.x.double(), op.dy.double()
    R, F_ = op.R, op.F
    m, r = got["mean"].double(), got["rstd"].double()
    gam = op.gam.view(F_).double() if op.gam is not None else torch.ones(F_, dtype=torch.float64, device=DEV)
    xh = (x - m) * r
    lane = math.ceil(R / 32)
    db_ref, db_mag = dy.sum(0), dy.abs().sum(0)
    dg_ref, dg_mag = (dy * xh).sum(0), (dy.abs() * xh.abs()).sum(0)
    n_db, n_dg = lane + 32, lane + 32 + 2
    _check("table_norm dbeta", "dbeta", db, db_ref, gamma(n_db) * db_mag)
    _check("table_norm dgamma", "dgamma", dg, dg_ref, gamma(n_dg) * dg_mag)
    sc = (r * gam).abs()
    if op.training:
        c = op.counts.double()
        w = (c / c.sum()).unsqueeze(1)
        ref = r * gam * (dy - w * db_ref - w * xh * dg_ref)
        lim = (gamma(8) * sc * (dy.abs() + w * db_ref.abs() + w * xh.abs() * dg_ref.abs())
               + sc * w * (gamma(n_db) * db_mag + xh.abs() * gamma(n_dg) * dg_mag))
    else:
        ref = r * gam * dy
        lim = gamma(2) * sc * dy.abs()
    _check("table_norm dx", "dx", dx, ref, lim)


@pytest.mark.parametrize("case", TN_CASES, ids=[_tn_id(c) for c in TN_CASES])
def test_table_norm(case):
    op = NormOps(case, seed=sum(case[:2]))
    got = op.fwd()
    again = op.fwd()
    for k in ("y", "mean", "rstd", "rm", "rv"):
        assert _same_bits(got[k], again[k]), f"{k}: two identical calls differ"
    assert got["tracked"] == again["tracked"]
    _tn_fwd_bounds(op, got)
    _tn_vs_batchnorm(op)
    dx, dg, db = op.bwd(got["mean"].view(1, -1), got["rstd"].view(1, -1))
    dx2, dg2, db2 = op.bwd(got["mean"].view(1, -1), got["rstd"].view(1, -1))
    assert _same_bits(dx, dx2) and _same_bits(dg, dg2) and _same_bits(db, db2), "backward: two identical calls differ"
    _tn_bwd_bounds(op, got, dx, dg, db)
    op.inputs_unchanged()


def test_table_norm_offset_data_needs_the_two_pass_variance():
    """x = 1000 + 0.1 N(0, 1): the kernel's rstd passes the two-pass bound, which a one-pass E[x^2] - E[x]^2 in FP32
    (the same data, the same weights) fails"""
    case = (37, 128, True, True, True, True, 0.1, False, True)
    op = NormOps(case, seed=9)
    got = op.fwd()
    _tn_fwd_bounds(op, got)
    w = (op.counts / op.counts.sum()).unsqueeze(1)
    mean1 = (w * op.x).sum(0)
    var1 = ((w * op.x * op.x).sum(0) - mean1 * mean1).clamp_min(0)
    one_pass = dict(got, rstd=torch.rsqrt(var1 + EPS))
    with pytest.raises(AssertionError, match="save_rstd"):
        _tn_fwd_bounds(op, one_pass)


def test_table_norm_bound_single_out_one_row():
    """dropping one counted row of the batch from the reference fails the save_mean bound"""
    case = (37, 128, True, True, True, True, 0.1, False, False)
    op = NormOps(case, seed=11)
    got = op.fwd()
    _tn_fwd_bounds(op, got)
    c = op.counts.clone()
    c[20] = 0
    with pytest.raises(AssertionError, match="save_mean"):
        _tn_fwd_bounds(op, got, counts=c)


def test_table_norm_total_count_one_and_zero():
    """n = 1: the batch statistics are the row itself (var 0, y = beta on it) and running_var becomes NaN (0 * n/(n-1)
    = 0 * inf; nn.BatchNorm1d raises instead).  n = 0: every batch statistic, y and the running statistics are NaN.
    num_batches_tracked still counts both calls."""
    R, F_ = 3, 33
    case = (R, F_, True, True, True, True, 0.1, False, False)
    op = NormOps(case, seed=2, counts=torch.tensor([0.0, 1.0, 0.0], device=DEV))
    got = op.fwd()
    assert _same_bits(got["mean"], op.x[1]), "n = 1: mean is not the row"
    assert _same_bits(got["rstd"], torch.rsqrt(torch.full((F_,), EPS, device=DEV))) or \
        bool(((got["rstd"].double() - EPS ** -0.5).abs() <= 4.5 * U * EPS ** -0.5).all())
    assert _same_bits(got["y"][1], op.bet.view(F_)), "n = 1: y of the row is not beta"
    assert bool(torch.isfinite(got["rm"]).all()) and bool(torch.isnan(got["rv"]).all())
    assert got["tracked"] == 6
    op = NormOps(case, seed=2, counts=torch.zeros(R, device=DEV))
    got = op.fwd()
    for k in ("mean", "rstd", "y", "rm", "rv"):
        assert bool(torch.isnan(got[k]).all()), f"n = 0: {k} is not NaN"
    assert got["tracked"] == 6


# ---------------------------------------------------------------------------------------------- coverage
def _reached():
    ks = set()
    for c in SEG_CASES:
        ks |= set(_seg_case_kernels(c))
    for k in range(10):   # the activation test: vector and scalar segment sums with field k, edge pair, msg_bwd
        ks |= set(segsum_kernels(1, 128, True, 2 | (k << 4))) | set(segsum_kernels(1, 128, False, 2 | (k << 4)))
        ks |= set(edge_pair_kernels(1, k)) | (set(msg_bwd_kernels(1, k)) if k else set())
    for c in EP_CASES:
        ks |= set(edge_pair_kernels(1, c[5]))
    for c in MB_CASES:
        ks |= set(msg_bwd_kernels(1, c[3]))
    for c in GATHER_CASES:
        ks |= set(gather_kernels(c[0], c[1], c[4], _gather_is_vec(c)))
    ks |= {"k_reduce_by_key", "k_act_fwd", "k_wbn_fwd", "k_wbn_bwd", "k_pair_outer_fwd", "k_pair_outer_bwd", "k_hist_f"}
    return ks


def test_cases_reach_every_message_and_table_kernel():
    reached = _reached()
    assert reached == ALL_KERNELS and len(ALL_KERNELS) == 18, reached ^ ALL_KERNELS
    # vector and scalar paths
    assert {_seg_is_vec(c[2], c[3], c[4]) for c in SEG_CASES} == {True, False}
    assert {_gather_is_vec(c) for c in GATHER_CASES} == {True, False}
    assert {c[4] for c in GATHER_CASES} == {True, False}
    # C below, at and above one warp pass in every warp-per-row kernel
    for Cs in ({c[2] for c in SEG_CASES}, {c[1] for c in EP_CASES}, {c[1] for c in MB_CASES}):
        assert min(Cs) < WARP_PASS < max(Cs) and WARP_PASS in Cs
    # both sides of the pair-outer grid cap
    assert {outer_grid_strides(*c) for c in PO_CASES} == {True, False}
    # reduce_by_key: one and several column passes per thread, runs on / before / after a chunk boundary, nkeys = 1
    assert {c[1] <= RBK_PASS for c in RBK_CASES} == {True, False}
    starts = _run_starts(_key_layout("runs")[0])
    assert {(n, s) for n in RUN_SIZES for s in (0, 31, 1)} <= starts
    counts = _key_layout("runs")[0]
    assert int(counts[0]) == 0 and int(counts[-1]) == 0 and (counts == 0).sum() > 10
    assert _key_layout("one")[1] == 1
    # table norm: F a multiple of 32 and not, R < 32 and R > 1024, training and eval, affine and not
    assert {c[1] % 32 == 0 for c in TN_CASES} == {True, False}
    assert min(c[0] for c in TN_CASES) < 32 and max(c[0] for c in TN_CASES) > 1024
    assert {c[2] for c in TN_CASES} == {True, False} and {(c[2], c[3]) for c in TN_CASES} >= {(False, False), (True, False)}
    assert {c[6] for c in TN_CASES} == {0.0, 0.1, 1.0} and {c[0] for c in TN_CASES} >= {1, 5, 37, 1369, 5000}
    assert {c[1] for c in TN_CASES} >= {1, 33, 128, 1000}


# ---------------------------------------------------------------------------------------------- the library's kernels
def _cuobjdump():
    exe = shutil.which("cuobjdump")
    if exe is None:
        home = os.environ.get("CUDA_HOME", os.environ.get("CUDA_PATH", "/usr/local/cuda"))
        exe = os.path.join(home, "bin", "cuobjdump")
    return exe if os.path.exists(exe) else None


_ARG = re.compile(r"L([ib])(\d+)E|([il])")
_TYPES = {"i": "int32_t", "l": "int64_t"}


def _kernel_name(sym):
    """name<args> of a mangled kernel symbol: bool and int literals and the int32 / int64 type arguments"""
    p = 2
    if sym.startswith("_ZN"):   # skip the (anonymous) namespace
        m = re.compile(r"N(\d+)").match(sym, 2)
        p = m.end() + int(m.group(1))
    m = re.compile(r"\d+").match(sym, p)
    L = int(m.group())
    name, p = sym[m.end():m.end() + L], m.end() + L
    args = []
    if sym[p:p + 1] == "I":
        p += 1
        while sym[p] != "E":
            t = _ARG.match(sym, p)
            assert t, sym
            if t.group(3):
                args.append(_TYPES[t.group(3)])
            elif t.group(1) == "b":
                args.append("true" if t.group(2) == "1" else "false")
            else:
                args.append(t.group(2))
            p = t.end()
    return f"{name}<{','.join(args)}>" if args else name


def _library_kernels():
    exe = _cuobjdump()
    if exe is None:
        pytest.skip("cuobjdump not available")
    text = subprocess.run([exe, "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    return {_kernel_name(s) for s in re.findall(r"Function (_Z\w+):", text)}


def test_kernel_list_matches_the_library():
    """the library holds no other kernel of these base names"""
    base = {k.split("<")[0] for k in ALL_KERNELS}
    found = {k for k in _library_kernels() if k.split("<")[0] in base}
    assert found == ALL_KERNELS, found ^ ALL_KERNELS


# Kernels that the ABI files' ALL_KERNELS do not list, each with the test that reaches it.  The dense-layer file restates
# its dispatch per case instead of keeping a list, so its kernels are claimed here.
_LINEAR = "test_gpu_linear_abi.py"
_THREEBODY = "test_gpu_threebody_abi.py (producers of the inputs)"
_INDEX = "test_gpu_parity.py, test_neighbors.py (graph index, bucket sorts, triplets)"
ALLOWLIST = {
    **{k: _INDEX for k in ("k_edge_prep", "k_exscan", "k_scan_block_sums", "k_scan_blocks", "k_hist64", "k_fill64",
                           "k_rank64", "k_ord_hist", "k_ord_scan", "k_ord_fill", "k_tri_count", "k_triplets_fill",
                           "k_validate")},
    "k_nl_count": "test_neighbors.py", "k_nl_fill": "test_neighbors.py",
    "k_geom_cell_partial": "test_gpu_stress.py", "k_geom_cell_final": "test_gpu_stress.py",
    **{f"k_twobody_{d}<{v},{nv}>": _THREEBODY for d in ("fwd", "bwd") for v in ("false", "true") for nv in (1, 2)},
    "k_sigmoid_rows": _THREEBODY, **{f"k_gram<{nl}>": _THREEBODY for nl in range(1, 5)},
    "k_act_bwd<false>": _LINEAR, "k_act_bwd<true>": _LINEAR, "k_act_bwd_any": _LINEAR,
    **{k: _LINEAR for k in ("k_gemm<false,false>", "k_gemm<true,false>", "k_gemm<true,true>", "k_colsum",
                            "k_tiny_rows<false>", "k_tiny_rows<true>", "k_tiny_wgrad", "k_tc_rows<false>",
                            "k_tc_rows<true>", "k_tc_rows_ta", "k_tc_wgrad", "k_wgrad_reduce", "k_wgrad_reduce_batch")},
}


def test_every_library_kernel_is_claimed():
    """every kernel in the library is listed by one of the C-ABI files or claimed by a named test in ALLOWLIST; a new
    kernel fails here until a test claims it"""
    from tests import test_gpu_edge_basis_abi as eb, test_gpu_threebody_abi as tb
    listed = ALL_KERNELS | eb.ALL_KERNELS | tb.ALL_KERNELS
    assert not (listed & set(ALLOWLIST)), listed & set(ALLOWLIST)
    found = _library_kernels()
    assert found == listed | set(ALLOWLIST), found ^ (listed | set(ALLOWLIST))
