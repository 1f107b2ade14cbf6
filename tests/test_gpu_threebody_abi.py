"""Every three-body kernel path of the C ABI, called directly, against an FP64 per-triplet reference.

`lcao_threebody_fwd` / `lcao_threebody_bwd` (threebody.cu) dispatch on C, NL and the forces flag to 36 kernel
instantiations in three files: the 3xTF32 `k_tb_fwd_mma<NL>` (threebody_mma.cu) and the FP32-pipe `k_threebody_fwd<NL>`
forward, the bulk-copy staged `k_tb_bwd_staged<NL, FORCES, CT>` (threebody_staged.cu) and the FP32-pipe
`k_threebody_bwd<NL, FORCES, FULL>` backward.  The helpers below restate that dispatch (and the staged ring depth), so
every case id names the kernels it runs, and one test checks that the cases reach all 36 and that the library holds no
other three-body kernel.

The reference evaluates the chain of the original model per triplet (e = s->t, e' = k->s, e' != e) in FP64:
    cos = u[e].u[e'],  v = sum_l Y_l(cos) B[e',l,:],  y = v / max(|v|, 1e-12),  tbw[e] += y * gate[k]
with the norm taken from v itself (the kernels use the Gram form |v|^2 = Y^T G Y) and an explicit per-triplet backward,
itself checked against torch.autograd.  The error bound is componentwise,
    |out - ref| <= c_kernel * mag,
where mag sums the absolute values of the same per-triplet terms (with |Y_l| + |Y_l'| + |Y_l''| as the angular weight,
so that the FP32 rounding of cos is covered too): one dropped, doubled or misrouted triplet fails even in a
20 000-edge output, and rows that no triplet reaches must be exact.

Every operand is a view into a NaN-filled buffer with NaN rows before and after it; the gate rows have a NaN gap
(ldg = C + 4) and B's groups l >= NL (never read by these kernels) are NaN.  Inputs must be bitwise unchanged and the
padding of every output untouched.
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
from lcaonet_b200.synth import crystal_like_batch
from oracle import lcao_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
P, ST = ops.ptr, ops.stream_ptr
NAN_BITS = 0x7FC00000
PAD = 4          # NaN rows before and after every operand (keeps (E, 3) and FP64 Gram rows 16-byte aligned)
EPS = 1e-12      # F.normalize eps of the three-body and two-body normalisations
KJS = 128        # backward with forces: out-edges per node whose d_unit partials stay in shared memory
Y0, Y1, Y2A, Y2B, Y3 = 0.28209479177387814, 0.4886025119029199, 0.9461746957575601, 0.31539156525252005, 0.3731763325901154

# Componentwise bound per kernel and output, in units of the magnitude above: the largest |out - ref| / mag over every
# case of this file, measured on an NVIDIA B200 (1000 W power limit), times a margin of at most 4
C_TB = {
    ("fwd_mma", "tbw"): 3.2e-6,        # observed 8.22e-7
    ("fwd_fp32", "tbw"): 1.2e-6,       # observed 2.99e-7
    ("bwd_staged", "dB"): 1.35e-6,     # observed 3.38e-7
    ("bwd_staged", "q"): 1.2e-6,       # observed 3.00e-7
    ("bwd_staged", "d_unit"): 2.9e-8,  # observed 7.41e-9
    ("bwd_fp32", "dB"): 1.0e-6,        # observed 2.58e-7
    ("bwd_fp32", "q"): 1.3e-6,         # observed 3.33e-7
    ("bwd_fp32", "d_unit"): 2.9e-8,    # observed 7.49e-9
}
# relative bound of lcao_sigmoid_rows (expf and one division in FP32); observed 1.78e-7
C_SIGMOID = 7.0e-7
# lcao_twobody_fwd / _bwd, in units of the magnitude built by _twobody_mag; observed 1.12e-7 (lw), 1.74e-7 (dB),
# 2.23e-7 (dg)
C_TWOBODY = 8.9e-7
# lcao_coeff_gram (FP64 sums of exact FP32 products), in units of the Gram matrix of |B|; observed 7.24e-16
C_GRAM = 2.9e-15
OBSERVED: dict = {}  # largest ratio per bound over the cases run (what the constants above were calibrated from)


# ---------------------------------------------------------------------------------------------- dispatch restated
def _b(x):
    return "true" if x else "false"


def fwd_kernel(C, NL):
    """lcao_threebody_fwd: the tensor-core forward for C <= 128, the FP32-pipe one above"""
    return f"k_tb_fwd_mma<{NL}>" if C <= 128 else f"k_threebody_fwd<{NL}>"


def bwd_kernel(C, NL, forces):
    """lcao_threebody_bwd: the staged backward for C <= 128 (C = 128 compiled as a constant), the FP32-pipe one above
    (predicate-free FULL variant for C = 256 without forces)"""
    if C <= 128:
        return f"k_tb_bwd_staged<{NL},{_b(forces)},{128 if C == 128 else 0}>"
    return f"k_threebody_bwd<{NL},{_b(forces)},{_b(not forces and C == 256)}>"


def family(kernel):
    return {"k_tb_fwd_mma": "fwd_mma", "k_threebody_fwd": "fwd_fp32", "k_tb_bwd_staged": "bwd_staged",
            "k_threebody_bwd": "bwd_fp32"}[kernel.split("<")[0]]


def staged_nst(C, NL, forces):
    """launch_bwd in threebody_staged.cu: the deepest ring (<= 4 stages) whose bwd_plan fits 55 KB (74 KB with forces)"""
    NP = NL * (NL + 1) // 2

    def total(nst):
        slot = NL * C + C
        o_item = 4 * slot + 4 * 4 + 4 * NP * 2
        stage = o_item + 8
        o_sa = 32 + nst * stage + 2 * (32 * C + 32 * 4)
        t = o_sa + 4 * 33 * 4 + 4 * 32
        return t + (4 * 33 * 4 + 4 * KJS * 3 if forces else 0)

    nst = 4
    while nst > 2 and 4 * total(nst) > (74 if forces else 55) * 1024:
        nst -= 1
    return nst


ALL_KERNELS = ({f"k_tb_fwd_mma<{nl}>" for nl in range(1, 5)} | {f"k_threebody_fwd<{nl}>" for nl in range(1, 5)}
               | {f"k_tb_bwd_staged<{nl},{_b(f)},{ct}>" for nl in range(1, 5) for f in (0, 1) for ct in (0, 128)}
               | {f"k_threebody_bwd<{nl},{f},{full}>" for nl in range(1, 5)
                  for f, full in (("false", "false"), ("false", "true"), ("true", "false"))})

# (graph, C, NL, NG, forces, dP).  NG > NL + 1 runs the forward only (the backward takes at most one valence group).
CASES = [
    # C <= 128: tensor-core forward, staged backward (CT = 128 at C = 128, CT = 0 below; partial consumer warps)
    ("boundary", 128, 1, 1, False, False), ("boundary", 128, 1, 2, True, True),
    ("boundary", 4, 1, 2, False, False), ("boundary", 36, 1, 1, True, True),
    ("boundary", 128, 2, 3, False, True), ("boundary", 128, 2, 2, True, False),
    ("boundary", 12, 2, 2, False, True), ("boundary", 100, 2, 3, True, False),
    ("boundary", 128, 3, 3, False, False), ("boundary", 128, 3, 4, True, True),   # ring depth 2 / 3
    ("boundary", 64, 3, 4, False, True), ("boundary", 64, 3, 3, True, False),     # ring depth 4 / 3
    ("boundary", 128, 4, 5, False, True), ("boundary", 128, 4, 4, True, False),
    ("boundary", 100, 4, 4, False, False), ("boundary", 12, 4, 5, True, True),
    # C > 128: FP32-pipe kernels (FULL = C == 256 without forces; 256 with forces takes FULL = false)
    ("boundary", 256, 1, 1, False, True), ("boundary", 132, 1, 2, False, False), ("boundary", 196, 1, 2, True, True),
    ("boundary", 256, 2, 3, False, False), ("boundary", 196, 2, 2, False, True), ("boundary", 256, 2, 2, True, False),
    ("boundary", 256, 3, 4, False, True), ("boundary", 132, 3, 3, False, False), ("boundary", 132, 3, 4, True, True),
    ("boundary", 256, 4, 4, False, False), ("boundary", 196, 4, 5, False, True), ("boundary", 256, 4, 5, True, False),
    # forward with two groups past NL
    ("boundary", 64, 2, 4, False, False), ("boundary", 196, 3, 5, False, False),
    # past every grid cap, several nodes per CTA; periodic-image duplicate edges
    ("many", 128, 3, 4, True, True), ("many", 196, 2, 2, True, False),
    ("crystal", 128, 3, 3, True, True),
]


def _case_kernels(case):
    _, C, NL, NG, forces, _ = case
    ks = [fwd_kernel(C, NL)]
    if NG <= NL + 1:
        ks.append(bwd_kernel(C, NL, forces))
    return ks


def _case_id(case):
    g, C, NL, NG, forces, dP = case
    names = "+".join(k.replace("<", ".").replace(">", "").replace(",", ".") for k in _case_kernels(case))
    nst = f"-nst{staged_nst(C, NL, forces)}" if C <= 128 and NG <= NL + 1 else ""
    return f"{names}{nst}-C{C}-NL{NL}-NG{NG}{'-forces' if forces else ''}{'-dP' if dP else ''}-{g}"


# ---------------------------------------------------------------------------------------------- graphs
IN_DEG = (1, 3, 4, 5, 8, 9, 31, 32, 33, 64, 65)
OUT_DEG = (1, 7, 8, 9, 15, 16, 17, 31, 32, 33, 129)
ROW_NORMAL, ROW_ZERO, ROW_TINY = 0, 1, 2


def _csr_positions(src, dst, N):
    """position of every edge in its source's out-list (edge id order) and in its target's in-list (source, edge id)"""
    E = src.numel()
    eid = torch.arange(E)
    out_order = torch.argsort(src * E + eid)
    in_order = torch.argsort((dst * N + src) * E + eid)
    out_pos, in_pos = torch.empty(E, dtype=torch.long), torch.empty(E, dtype=torch.long)
    out_first = torch.zeros(N + 1, dtype=torch.long)
    out_first[1:] = torch.bincount(src, minlength=N).cumsum(0)
    in_first = torch.zeros(N + 1, dtype=torch.long)
    in_first[1:] = torch.bincount(dst, minlength=N).cumsum(0)
    out_pos[out_order] = torch.arange(E) - out_first[src[out_order]]
    in_pos[in_order] = torch.arange(E) - in_first[dst[in_order]]
    return out_pos, in_pos


def _finish(src, dst, N, unit_kind, row_kind, g, picks=None):
    """shuffle node and edge ids; returns a dict graph with per-edge unit-vector and B-row kinds"""
    perm = torch.randperm(N, generator=g)
    eperm = torch.randperm(src.numel(), generator=g)
    src, dst = perm[src[eperm]], perm[dst[eperm]]
    unit_kind, row_kind = unit_kind[eperm], row_kind[eperm]
    out_pos, in_pos = _csr_positions(src, dst, N)
    graph = dict(edge_index=torch.stack([src, dst]), N=N, unit_kind=unit_kind, row_kind=row_kind, out_pos=out_pos,
                 in_pos=in_pos)
    if picks is not None:
        graph["picks"] = picks(perm, src, dst, out_pos, in_pos)
    return graph


@functools.lru_cache(None)
def boundary_graph():
    """Centre nodes with every (in, out) degree of IN_DEG x OUT_DEG (the kernels' block sizes 4, 8, 16, 32 and kJS on
    either side), a 300 x 300 hub with a self-loop, in-only / out-only / isolated / self-loop-only nodes, three
    duplicate k->s edges with identical unit vectors (cos = 1 against an out-edge) and an antiparallel pair (cos = -1),
    B rows that are exactly zero (the eps branch) or scaled by 2^-20.  Node and edge ids are shuffled."""
    g = torch.Generator().manual_seed(20261021)
    n_leaf = 400
    src, dst, ukind = [], [], []
    nxt = n_leaf

    def node():
        nonlocal nxt
        nxt += 1
        return nxt - 1

    def edge(s, t, uk=0):
        src.append(s), dst.append(t), ukind.append(uk)

    def leaves(n):
        return torch.randint(0, n_leaf, (n,), generator=g).tolist()

    for di in IN_DEG:
        for do in OUT_DEG:
            c = node()
            for k in leaves(di):
                edge(k, c)
            for t in leaves(do):
                edge(c, t)
    hub = node()
    for k in leaves(299):
        edge(k, hub)
    for t in leaves(299):
        edge(hub, t)
    edge(hub, hub)                       # self-loop on a busy node: 300 in-edges, 300 out-edges
    in_only, out_only, _isolated, loop_only, dup = node(), node(), node(), node(), node()
    for k in leaves(5):
        edge(k, in_only)
    for t in leaves(5):
        edge(out_only, t)
    edge(loop_only, loop_only)
    k0 = n_leaf - 1
    for _ in range(3):
        edge(k0, dup, 1)                 # duplicate k->s edges, unit (1, 0, 0)
    for k in leaves(4):
        edge(k, dup)
    edge(dup, k0, -1)                    # antiparallel to the duplicates: cos = -1
    edge(dup, 0, 1)                      # parallel: cos = 1
    for t in leaves(10):
        edge(dup, t)
    N = nxt
    src, dst = torch.tensor(src), torch.tensor(dst)
    E = src.numel()
    r = torch.rand(E, generator=g)
    row_kind = torch.where(r < 0.03, ROW_ZERO, torch.where(r < 0.06, ROW_TINY, ROW_NORMAL))
    ukind = torch.tensor(ukind)

    def picks(perm, s, d, out_pos, in_pos):
        """three triplets (e, e') at block boundaries whose e' has an ordinary B row"""
        h = int(perm[hub])
        c = int(perm[n_leaf + IN_DEG.index(9) * len(OUT_DEG) + OUT_DEG.index(17)])   # (in 9, out 17) centre

        def first(mask):
            return int(torch.nonzero(mask)[0])

        out_h = (s == h) & (d != h)
        in_h = (d == h) & (s != h)
        return [
            # out-edge 129 of the hub (atomic d_unit row) with its first in-edge
            (first(out_h & (out_pos == 128)), first(in_h & (in_pos == 0))),
            # in-edge 33 of the hub (second panel of 32 in-edges) with out-edge 6
            (first(out_h & (out_pos == 5)), first(in_h & (in_pos == 32))),
            # out-edge 17 of a centre (first row of its second 16-row tile) with in-edge 9
            (first((s == c) & (out_pos == 16)), first((d == c) & (in_pos == 8))),
        ]

    graph = _finish(src, dst, N, ukind, row_kind, g, picks)
    rk = graph["row_kind"]
    for _, ep in graph["picks"]:
        rk[ep] = ROW_NORMAL
    return graph


@functools.lru_cache(None)
def many_graph():
    """20 000 nodes, in- and out-degrees 0..6 (15 % of the nodes without in-edges, 15 % without out-edges) paired at
    random: past every grid cap (148 x {40, 48, 24, 16} CTAs) with several nodes per CTA"""
    g = torch.Generator().manual_seed(7)
    N = 20000
    dout = torch.randint(1, 7, (N,), generator=g) * (torch.rand(N, generator=g) >= 0.15)
    din = torch.randint(1, 7, (N,), generator=g) * (torch.rand(N, generator=g) >= 0.15)
    so = torch.repeat_interleave(torch.arange(N), dout)
    si = torch.repeat_interleave(torch.arange(N), din)
    n = min(so.numel(), si.numel())
    src = so[torch.randperm(so.numel(), generator=g)[:n]]
    dst = si[torch.randperm(si.numel(), generator=g)[:n]]
    z = torch.zeros(n, dtype=torch.long)
    return _finish(src, dst, N, z, z.clone(), g)


@functools.lru_cache(None)
def crystal_graph():
    """one periodic 64-atom cell (~50 neighbours per atom, periodic-image duplicates of the same atom pair)"""
    gb = crystal_like_batch(1, 3)
    ei = gb["edge_index"]
    g = torch.Generator().manual_seed(3)
    z = torch.zeros(ei.shape[1], dtype=torch.long)
    return _finish(ei[0], ei[1], gb["z"].shape[0], z, z.clone(), g)


GRAPHS = {"boundary": boundary_graph, "many": many_graph, "crystal": crystal_graph}


# ---------------------------------------------------------------------------------------------- padded operands
def _rows(M, W, fill=None, dtype=torch.float32):
    """(buffer, view): an (M, W) block of a flat NaN buffer with PAD rows before and after it"""
    buf = torch.full(((M + 2 * PAD) * W,), float("nan"), dtype=dtype, device=DEV)
    v = buf[PAD * W:(PAD + M) * W].view(M, W)
    if fill is not None:
        v.copy_(fill.reshape(M, W))
    return buf, v


def _padding_untouched(buf, view, what):
    mask = torch.ones(buf.numel(), dtype=torch.bool, device=DEV)
    inner = torch.as_strided(torch.arange(buf.numel(), device=DEV), view.shape, view.stride(), view.storage_offset())
    mask[inner.reshape(-1)] = False
    bits = buf.reshape(-1).view(torch.int32)[mask]
    assert bool((bits == NAN_BITS).all()), f"{what}: {int((bits != NAN_BITS).sum())} padding elements written"


def _same_bits(a, b):
    return torch.equal(a.reshape(-1).view(torch.int32 if a.dtype == torch.float32 else torch.int64),
                       b.reshape(-1).view(torch.int32 if b.dtype == torch.float32 else torch.int64))


def _within(got, ref, mag, tol):
    """(ok, max ratio, first bad index): |got - ref| <= tol * mag componentwise, finite"""
    if not bool(torch.isfinite(got).all()):
        bad = torch.nonzero(~torch.isfinite(got))[0].tolist()
        return False, math.inf, bad
    err = (got.double() - ref).abs()
    ratio = float((err / mag.clamp_min(1e-300)).max()) if err.numel() else 0.0
    bad = err > tol * mag
    return (not bool(bad.any())), ratio, (torch.nonzero(bad)[0].tolist() if bool(bad.any()) else None)


def _check(key, what, got, ref, mag):
    tol = C_TB[key] if isinstance(key, tuple) else key
    ok, ratio, first = _within(got, ref, mag, tol)
    name = key if isinstance(key, tuple) else what
    OBSERVED[name] = max(OBSERVED.get(name, 0.0), ratio)
    if not ok:
        idx = tuple(first)
        raise AssertionError(f"{what}: over the bound at {list(idx)} (got {float(got[idx]):.8g}, want {float(ref[idx]):.8g}, "
                             f"mag {float(mag[idx]):.3g}); max ratio {ratio:.3g} > {tol:.3g}")


# ---------------------------------------------------------------------------------------------- FP64 reference
def _sph64(c, NL):
    """Y_l(c), Y_l'(c), Y_l''(c) (shbf.py:41-63), (T, NL) each"""
    z = torch.zeros_like(c)
    Y = [torch.full_like(c, Y0), Y1 * c, Y2A * c * c - Y2B, Y3 * c * (5 * c * c - 3)]
    dY = [z, torch.full_like(c, Y1), 2 * Y2A * c, Y3 * (15 * c * c - 3)]
    d2Y = [z, z, torch.full_like(c, 2 * Y2A), Y3 * 30 * c]
    return torch.stack(Y[:NL], 1), torch.stack(dY[:NL], 1), torch.stack(d2Y[:NL], 1)


class Reference:
    """Sums of the per-triplet terms of the forward and backward chain, and of their magnitudes, in FP64 on the GPU"""

    def __init__(self, B, unit, gate, d_tbw, NL, forces):
        E, C = B.shape[0], B.shape[-1]
        self.NL, self.forces, self.bwd = NL, forces, d_tbw is not None
        self.B = B[:, :NL].double()
        self.u, self.gate = unit.double(), gate.double()
        self.G = d_tbw.double() if d_tbw is not None else None
        z = functools.partial(torch.zeros, dtype=torch.float64, device=DEV)
        self.tbw, self.tbw_m = z(E, C), z(E, C)
        if self.bwd:
            self.dB, self.dB_m, self.gq, self.gq_m = z(E, NL, C), z(E, NL, C), z(E, C), z(E, C)
            self.dks, self.dks_m, self.dst, self.dst_m = z(E, 3), z(E, 3), z(E, 3), z(E, 3)

    def add(self, k, ep, e, sign=1.0, chunk=8192):
        for i in range(0, e.numel(), chunk):
            self._add(k[i:i + chunk], ep[i:i + chunk], e[i:i + chunk], sign)

    def _add(self, k, ep, e, sign):
        ue, up = self.u[e], self.u[ep]
        Y, dY, d2Y = _sph64((ue * up).sum(1), self.NL)
        A = Y.abs() + dY.abs() + d2Y.abs()
        Bp = self.B[ep]
        v = torch.einsum("tl,tlc->tc", Y, Bp)
        nrm = v.norm(dim=1, keepdim=True)
        inv = 1.0 / nrm.clamp_min(EPS)
        y = v * inv
        g = self.gate[k]
        babs = inv * torch.einsum("tl,tlc->tc", A, Bp.abs())
        self.tbw.index_add_(0, e, y * g, alpha=sign)
        self.tbw_m.index_add_(0, e, babs * g.abs(), alpha=sign)
        if not self.bwd:
            return
        G = self.G[e]
        dy = G * g
        live = (nrm > EPS).double()
        dv = (dy - live * y * (y * dy).sum(1, keepdim=True)) * inv
        dvm = (dy.abs() + live * babs * (babs * dy.abs()).sum(1, keepdim=True)) * inv
        self.dB.index_add_(0, ep, Y.unsqueeze(-1) * dv.unsqueeze(1), alpha=sign)
        self.dB_m.index_add_(0, ep, A.unsqueeze(-1) * dvm.unsqueeze(1), alpha=sign)
        self.gq.index_add_(0, ep, y * G, alpha=sign)
        self.gq_m.index_add_(0, ep, babs * G.abs(), alpha=sign)
        if self.forces:
            dc = torch.einsum("tl,tlc,tc->t", dY, Bp, dv).unsqueeze(1)
            dcm = torch.einsum("tl,tlc,tc->t", A, Bp.abs(), dvm).unsqueeze(1)
            self.dst.index_add_(0, e, dc * up, alpha=sign)
            self.dst_m.index_add_(0, e, dcm * up.abs(), alpha=sign)
            self.dks.index_add_(0, ep, dc * ue, alpha=sign)
            self.dks_m.index_add_(0, ep, dcm * ue.abs(), alpha=sign)

    def outputs(self, NG, dP, in_src):
        """{name: (ref, mag)} of the kernel outputs (copies): dB with dP folded in, q with the sigmoid derivative applied"""
        out = {"tbw": (self.tbw.clone(), self.tbw_m.clone())}
        if not self.bwd:
            return out
        E, C = self.tbw.shape
        dB, dB_m = torch.zeros(E, NG, C, dtype=torch.float64, device=DEV), torch.zeros(E, NG, C, dtype=torch.float64, device=DEV)
        dB[:, :self.NL], dB_m[:, :self.NL] = self.dB, self.dB_m
        if dP is not None:
            d = dP.double()
            dB[:, :self.NL] += d[:, :1]
            dB_m[:, :self.NL] += d[:, :1].abs()
            if NG > self.NL:
                dB[:, self.NL], dB_m[:, self.NL] = d[:, 1], d[:, 1].abs()
        s = self.gate[in_src]
        sd = s * (1 - s)
        out.update(dB=(dB, dB_m), q=(self.gq * sd, self.gq_m * sd))
        if self.forces:
            out.update(d_unit_ks=(self.dks.clone(), self.dks_m.clone()), d_unit_st=(self.dst.clone(), self.dst_m.clone()))
        return out


def _triplets(graph):
    k, e_ks, e_st = O.triplets(graph["edge_index"], graph["N"])
    return k.to(DEV), e_ks.to(DEV), e_st.to(DEV)


# ---------------------------------------------------------------------------------------------- the three-body calls
def _inputs(graph, C, NL, NG, dP_given, seed):
    torch.manual_seed(seed)
    ei, N = graph["edge_index"], graph["N"]
    E = ei.shape[1]
    B = torch.randn(E, NG, C, device=DEV)
    rk = graph["row_kind"].to(DEV)
    B[rk == ROW_ZERO] = 0.0
    B[rk == ROW_TINY] *= 2.0 ** -20
    B[:, NL:] = float("nan")                      # valence groups: never read by the three-body kernels
    unit = torch.nn.functional.normalize(torch.randn(E, 3, device=DEV), dim=1)
    uk = graph["unit_kind"].to(DEV)
    ax = torch.tensor([1.0, 0.0, 0.0], device=DEV)
    unit[uk == 1], unit[uk == -1] = ax, -ax
    gate_vals = torch.sigmoid(2 * torch.randn(N, C, device=DEV))
    d_tbw = torch.randn(E, C, device=DEV)
    dP = torch.randn(E, NG - NL + 1, C, device=DEV) if dP_given else None
    return B, unit, gate_vals, d_tbw, dP


class Operands:
    """The padded device operands of one three-body call"""

    def __init__(self, gi, B, unit, gate_vals, d_tbw, dP, NL):
        E, NG, C = B.shape
        self.gi, self.E, self.N, self.NG, self.C, self.NL = gi, E, gi.N, NG, C, NL
        self.Bb, self.B = _rows(E, NG * C, B)
        self.ub, self.unit = _rows(E, 3, unit)
        self.gb = torch.full(((gi.N + 2 * PAD) * (C + 4),), float("nan"), device=DEV)
        self.gate = self.gb[PAD * (C + 4):(PAD + gi.N) * (C + 4)].view(gi.N, C + 4)[:, :C]
        self.gate.copy_(gate_vals)
        NP = NL * (NL + 1) // 2
        self.grb, self.gram = _rows(E, NP, dtype=torch.float64)
        ops._call("lcao_coeff_gram", P(self.B), NG, E, C, NL, P(self.gram), ST())
        self.db, self.d_tbw = _rows(E, C, d_tbw)
        self.dpb, self.dP = _rows(E, (NG - NL + 1) * C, dP) if dP is not None else (None, None)
        torch.cuda.synchronize()
        self.inputs = [(b, b.clone()) for b in (self.Bb, self.ub, self.gb, self.grb, self.db, self.dpb) if b is not None]

    def index_args(self):
        gi = self.gi
        return (P(gi.in_ptr), P(gi.in_edge), P(gi.in_src), P(gi.out_ptr), P(gi.out_edge), self.N, self.E, self.C, self.NL)

    def fwd(self):
        tb, tbw = _rows(self.E, self.C)
        n0 = _lib.launch_count()
        ops._call("lcao_threebody_fwd", P(self.B), self.NG, P(self.gram), P(self.unit), P(self.gate), self.gate.stride(0),
                  *self.index_args(), P(tbw), ST())
        assert _lib.launch_count() - n0 == 1
        torch.cuda.synchronize()
        _padding_untouched(tb, tbw, "tbw")
        return {"tbw": tbw}

    def bwd(self, forces, with_dP=True):
        E, C, NG = self.E, self.C, self.NG
        dBb, dB = _rows(E, NG * C)
        qb, q = _rows(E, C)
        kb, ks = _rows(E, 3) if forces else (None, None)
        sb, st = _rows(E, 3) if forces else (None, None)
        n0 = _lib.launch_count()
        ops._call("lcao_threebody_bwd", P(self.B), NG, P(self.gram), P(self.unit), P(self.gate), self.gate.stride(0),
                  *self.index_args(), P(self.d_tbw), P(self.dP if with_dP else None), P(dB), P(q), P(ks), P(st), ST())
        assert _lib.launch_count() - n0 == 1
        torch.cuda.synchronize()
        out = {"dB": dB.view(E, NG, C), "q": q}
        _padding_untouched(dBb, dB, "dB")
        _padding_untouched(qb, q, "q")
        if forces:
            _padding_untouched(kb, ks, "d_unit_ks")
            _padding_untouched(sb, st, "d_unit_st")
            out.update(d_unit_ks=ks, d_unit_st=st)
        return out

    def inputs_unchanged(self):
        for buf, before in self.inputs:
            assert _same_bits(buf, before), "an input buffer (operand or padding) was written"


def _bound_key(kernel, name):
    return family(kernel), ("d_unit" if name.startswith("d_unit") else name)


def _check_outputs(kernel, got, want, what):
    for name, (ref, mag) in want.items():
        if name in got:
            _check(_bound_key(kernel, name), f"{what} {name}", got[name], ref, mag)


@pytest.mark.parametrize("case", CASES, ids=[_case_id(c) for c in CASES])
def test_threebody_vs_fp64(case):
    gname, C, NL, NG, forces, dP_given = case
    graph = GRAPHS[gname]()
    gi = ops.GraphIndex(graph["edge_index"].to(DEV), graph["N"])
    B, unit, gate_vals, d_tbw, dP = _inputs(graph, C, NL, NG, dP_given, seed=C * 10 + NL * 3 + NG)
    ops_ = Operands(gi, B, unit, gate_vals, d_tbw, dP, NL)
    run_bwd = NG <= NL + 1
    kf = fwd_kernel(C, NL)
    kb = bwd_kernel(C, NL, forces) if run_bwd else None

    got = ops_.fwd()
    if run_bwd:
        got.update(ops_.bwd(forces))
    ops_.inputs_unchanged()

    k, e_ks, e_st = _triplets(graph)
    ref = Reference(ops_.B.view(-1, NG, C), ops_.unit, ops_.gate, ops_.d_tbw if run_bwd else None, NL, forces)
    ref.add(k, e_ks, e_st)
    in_src = graph["edge_index"][0].to(DEV)
    want = ref.outputs(NG, ops_.dP.view(-1, NG - NL + 1, C) if dP_given else None, in_src)
    _check_outputs(kf, {"tbw": got["tbw"]}, {"tbw": want["tbw"]}, kf)
    if run_bwd:
        _check_outputs(kb, {n: v for n, v in got.items() if n != "tbw"}, {n: v for n, v in want.items() if n != "tbw"}, kb)

    # rows no triplet reaches: exactly zero (tbw, q, d_unit) or exactly the two-body gradient (dB)
    E = gi.E
    n_st = torch.bincount(e_st, minlength=E)
    n_ks = torch.bincount(e_ks, minlength=E)
    assert bool((got["tbw"][n_st == 0] == 0).all())
    if run_bwd:
        dead = n_ks == 0
        assert bool((got["q"][dead] == 0).all())
        assert torch.equal(got["dB"][dead].double(), want["dB"][0][dead])
        if forces:
            assert bool((got["d_unit_ks"][dead] == 0).all()) and bool((got["d_unit_st"][n_st == 0] == 0).all())

    # a second identical call agrees bitwise, except the d_unit_st rows past the 128th out-edge of a node (atomics)
    again = ops_.fwd()
    if run_bwd:
        again.update(ops_.bwd(forces))
    for name, v in got.items():
        if name == "d_unit_st":
            keep = graph["out_pos"].to(DEV) < KJS
            assert _same_bits(v[keep], again[name][keep]), name
        else:
            assert _same_bits(v, again[name]), name

    if gname == "boundary":
        # the bound rejects the kernel output against a reference with one triplet at a block boundary removed
        dPv = ops_.dP.view(-1, NG - NL + 1, C) if dP_given else None
        # (not d_unit: its magnitude sums two C-wide dot products per triplet over up to 300 triplets per row, which is
        # too loose to single out one triplet of a busy node)
        names = ["tbw"] + (["dB", "q"] if run_bwd else [])
        for e, ep in graph["picks"]:
            sel = torch.nonzero((e_st == e) & (e_ks == ep)).flatten()
            assert sel.numel() == 1
            ref.add(k[sel], e_ks[sel], e_st[sel], sign=-1.0)
            want1 = ref.outputs(NG, dPv, in_src)
            ref.add(k[sel], e_ks[sel], e_st[sel])
            for name in names:
                kern = kf if name == "tbw" else kb
                row = e if name in ("tbw", "d_unit_st") else ep
                r, m = want1[name]
                ok, _, _ = _within(got[name][row], r[row], m[row], C_TB[_bound_key(kern, name)])
                assert not ok, f"{kern} {name}: the bound accepts the output without triplet ({e}, {ep})"


# ---------------------------------------------------------------------------------------------- scale equivariance
@pytest.mark.parametrize("C,NL,forces", [(128, 3, True), (64, 2, False), (196, 4, True), (256, 1, False)],
                         ids=lambda v: str(v))
def test_threebody_scale_equivariance(C, NL, forces):
    """B -> 2^-20 B (gram recomputed): the coefficients scale by 2^20 and the gated rows by 2^-20, and every step
    (FP64 Gram, sqrtf, the division, the TF32 split, FP32 products and sums) commutes with a power-of-two scaling away
    from the denormal range, so tbw, q and d_unit are bitwise unchanged and dB is multiplied by exactly 2^20"""
    graph = many_graph()
    gi = ops.GraphIndex(graph["edge_index"].to(DEV), graph["N"])
    NG = NL + 1
    B, unit, gate_vals, d_tbw, _ = _inputs(graph, C, NL, NG, False, seed=11 + C + NL)
    a = Operands(gi, B, unit, gate_vals, d_tbw, None, NL)
    b = Operands(gi, B * 2.0 ** -20, unit, gate_vals, d_tbw, None, NL)
    ga, gb = a.fwd(), b.fwd()
    ga.update(a.bwd(forces))
    gb.update(b.bwd(forces))
    for name in ga:
        if name == "dB":
            assert _same_bits(gb[name], ga[name] * 2.0 ** 20), (fwd_kernel(C, NL), bwd_kernel(C, NL, forces), name)
        else:
            assert _same_bits(ga[name], gb[name]), (fwd_kernel(C, NL), bwd_kernel(C, NL, forces), name)


# ---------------------------------------------------------------------------------------------- the reference itself
def test_reference_backward_matches_autograd():
    """The explicit per-triplet backward of `Reference` against torch.autograd of its FP64 forward, with the gate a
    per-in-edge leaf and the unit vectors two leaves (in-edge role, out-edge role), on a small graph with a zero B row"""
    torch.manual_seed(3)
    N, E, C, NL = 12, 60, 8, 4
    ei = torch.randint(0, N, (2, E))
    k, e_ks, e_st = (t.to(DEV) for t in O.triplets(ei, N))
    B = torch.randn(E, NL, C, dtype=torch.float64, device=DEV)
    B[5] = 0.0
    unit = torch.nn.functional.normalize(torch.randn(E, 3, dtype=torch.float64, device=DEV), dim=1)
    gate = torch.sigmoid(torch.randn(N, C, dtype=torch.float64, device=DEV))
    G = torch.randn(E, C, dtype=torch.float64, device=DEV)
    src = ei[0].to(DEV)

    Bl = B.clone().requires_grad_(True)
    g_in = gate[src].clone().requires_grad_(True)      # the gate seen by in-edge e'
    u_ks, u_st = unit.clone().requires_grad_(True), unit.clone().requires_grad_(True)
    cos = (u_st[e_st] * u_ks[e_ks]).sum(1)
    Y = _sph64(cos, NL)[0]
    v = torch.einsum("tl,tlc->tc", Y, Bl[e_ks])
    y = v / v.norm(dim=1, keepdim=True).clamp_min(EPS)
    tbw = torch.zeros(E, C, dtype=torch.float64, device=DEV).index_add(0, e_st, y * g_in[e_ks])
    dB, dg, dks, dst = torch.autograd.grad((tbw * G).sum(), [Bl, g_in, u_ks, u_st])

    ref = Reference(B, unit.float(), gate, G, NL, True)
    ref.u = unit  # the FP64 unit vectors themselves
    ref.add(k, e_ks, e_st)
    assert float((ref.tbw - tbw.detach()).abs().max()) <= 1e-12 * float(ref.tbw_m.max())
    for mine, auto, mag in ((ref.dB, dB, ref.dB_m), (ref.gq, dg, ref.gq_m), (ref.dks, dks, ref.dks_m), (ref.dst, dst, ref.dst_m)):
        assert bool(((mine - auto).abs() <= 1e-12 * mag + 1e-300).all()), float((mine - auto).abs().max())
    assert float(ref.dB[5].abs().max()) > 1e6  # the eps branch: the gradient of v / eps


# ---------------------------------------------------------------------------------------------- coverage of the table
def test_cases_reach_every_threebody_kernel():
    reached = {k for c in CASES for k in _case_kernels(c)}
    assert reached == ALL_KERNELS and len(ALL_KERNELS) == 36, ALL_KERNELS ^ reached
    assert (staged_nst(128, 3, False), staged_nst(128, 3, True), staged_nst(64, 3, False)) == (2, 3, 4)
    assert {staged_nst(c[1], c[2], c[4]) for c in CASES if c[1] <= 128 and c[3] <= c[2] + 1} == {2, 3, 4}
    for fam in ("fwd_mma", "fwd_fp32", "bwd_staged", "bwd_fp32"):  # NG = NL and NL + 1, with and without dP
        cs = [c for c in CASES if any(family(k) == fam for k in _case_kernels(c))]
        assert {c[3] - c[2] for c in cs} >= {0, 1} and {c[5] for c in cs} == {False, True}, fam
        assert "many" in {c[0] for c in cs}, fam
    assert any(c[3] == c[2] + 2 for c in CASES)


def _cuobjdump():
    exe = shutil.which("cuobjdump")
    if exe is None:
        home = os.environ.get("CUDA_HOME", os.environ.get("CUDA_PATH", "/usr/local/cuda"))
        exe = os.path.join(home, "bin", "cuobjdump")
    return exe if os.path.exists(exe) else None


def test_kernel_list_matches_the_library():
    """the restated dispatch lists every three-body kernel the library contains: a new variant needs a case"""
    exe = _cuobjdump()
    if exe is None:
        pytest.skip("cuobjdump not available")
    text = subprocess.run([exe, "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    found = set()
    for name, args in re.findall(r"\d+(k_tb_fwd_mma|k_threebody_fwd|k_tb_bwd_staged|k_threebody_bwd)I((?:L[ib]\d+E)+)E", text):
        vals = [("true" if v == "1" else "false") if t == "b" else v for t, v in re.findall(r"L([ib])(\d+)E", args)]
        found.add(f"{name}<{','.join(vals)}>")
    assert found == ALL_KERNELS, found ^ ALL_KERNELS


# ---------------------------------------------------------------------------------------------- producers of the inputs
@pytest.mark.parametrize("C,NL,NG", [(4, 1, 2), (36, 2, 2), (128, 3, 4), (256, 4, 4), (196, 3, 3)])
def test_coeff_gram_vs_fp64(C, NL, NG):
    """lcao_coeff_gram: FP64 upper-triangle Gram rows of the first NL groups; the groups past NL are NaN (never read)"""
    torch.manual_seed(C + NL)
    E = 5003
    B = torch.randn(E, NG, C, device=DEV) * torch.exp(2 * torch.randn(E, 1, 1, device=DEV))
    B[::17] = 0.0
    B[:, NL:] = float("nan")
    bb, Bv = _rows(E, NG * C, B)
    NP = NL * (NL + 1) // 2
    gb, gram = _rows(E, NP, dtype=torch.float64)
    before = bb.clone()
    ops._call("lcao_coeff_gram", P(Bv), NG, E, C, NL, P(gram), ST())
    torch.cuda.synchronize()
    b64 = Bv.view(E, NG, C)[:, :NL].double()
    iu = torch.triu_indices(NL, NL)
    ref = torch.einsum("elc,emc->elm", b64, b64)[:, iu[0], iu[1]]
    mag = torch.einsum("elc,emc->elm", b64.abs(), b64.abs())[:, iu[0], iu[1]]
    _check(C_GRAM, "coeff_gram", gram, ref, mag)
    assert _same_bits(before, bb)
    mask = torch.ones(gb.numel(), dtype=torch.bool, device=DEV)
    mask[PAD * NP:(PAD + E) * NP] = False
    assert bool(torch.isnan(gb[mask]).all()), "gram padding written"


@pytest.mark.parametrize("M,C", [(20000, 128), (777, 12), (3001, 256)])
def test_sigmoid_rows_strided(M, C):
    """lcao_sigmoid_rows reading the right half of an (M, 2C) buffer (ldx = 2C) into gate rows with ldo = C + 4"""
    torch.manual_seed(M)
    xb = torch.full(((M + 2 * PAD) * 2 * C,), float("nan"), device=DEV)
    x = xb[PAD * 2 * C:(PAD + M) * 2 * C].view(M, 2 * C)[:, C:]
    vals = 4 * torch.randn(M, C, device=DEV)
    vals[0, :4] = torch.tensor([0.0, 30.0, -30.0, -80.0])
    x.copy_(vals)
    ob = torch.full(((M + 2 * PAD) * (C + 4),), float("nan"), device=DEV)
    out = ob[PAD * (C + 4):(PAD + M) * (C + 4)].view(M, C + 4)[:, :C]
    ops._call("lcao_sigmoid_rows", P(x), x.stride(0), P(out), out.stride(0), M, C, ST())
    torch.cuda.synchronize()
    ref = torch.sigmoid(x.double())
    _check(C_SIGMOID, "sigmoid_rows", out, ref, ref)
    _padding_untouched(ob, out, "gate")


def _twobody_mag(B, g, d_lw, NL, valence):
    """magnitudes of lw and of its backward: the same formulas evaluated on absolute values, all differences as sums"""
    b = B.double()
    babs = b[:, :NL].abs().sum(1) + (b[:, NL].abs() if valence else 0)
    C = b.shape[-1]
    gA = g.double()[:, :C].abs()
    pabs = (1 + gA) * babs
    if valence:
        pabs = pabs + (1 + g.double()[:, C:].abs()) * b[:, NL].abs()
    PA = b[:, :NL].sum(1) - (b[:, NL] if valence else 0)
    PV = b[:, NL] if valence else torch.zeros_like(PA)
    p = (1 + g.double()[:, :C]) * PA + ((1 + g.double()[:, C:]) * PV if valence else 0)
    n = p.norm(dim=1, keepdim=True).clamp_min(EPS)
    lw_m = pabs / n + p.abs() * (pabs * p.abs()).sum(1, keepdim=True) / n ** 3
    dl = d_lw.double().abs()
    dp_m = (dl + pabs * (pabs * dl).sum(1, keepdim=True) / n ** 2) / n
    dPA_m = (1 + gA) * dp_m
    return lw_m, dp_m, dPA_m


@pytest.mark.parametrize("C,NL,valence,compact", [(12, 3, 0, 0), (128, 3, 0, 1), (128, 2, 1, 0), (196, 4, 1, 1), (256, 1, 1, 1),
                                                  (64, 4, 0, 0)])
def test_twobody_vs_fp64_autograd(C, NL, valence, compact):
    """lcao_twobody_fwd / _bwd (compact and full dB, with and without the valence slot, zero rows: the eps branch)
    against torch.autograd of the FP64 formula"""
    torch.manual_seed(C + NL + 10 * valence + 100 * compact)
    E = 4099
    NG = NL + valence
    Cg = C * (1 + valence)
    B = torch.randn(E, NG, C, device=DEV)
    B[::23] = 0.0
    g = torch.randn(E, Cg, device=DEV)
    d_lw = torch.randn(E, C, device=DEV)
    bb, Bv = _rows(E, NG * C, B)
    ggb, gv = _rows(E, Cg, g)
    lb, lw = _rows(E, C)
    ops._call("lcao_twobody_fwd", P(Bv), NG, P(gv), E, C, NL, valence, P(lw), ST())
    dlb, dlv = _rows(E, C, d_lw)
    NGo = (1 + valence) if compact else NG
    dbb, dB = _rows(E, NGo * C)
    dgb, dg = _rows(E, Cg)
    ops._call("lcao_twobody_bwd", P(Bv), NG, P(gv), P(dlv), E, C, NL, valence, compact, P(dB), P(dg), ST())
    torch.cuda.synchronize()

    b64 = Bv.view(E, NG, C).double().requires_grad_(True)
    g64 = gv.double().requires_grad_(True)
    PA = b64[:, :NL].sum(1) - (b64[:, NL] if valence else 0)
    p = (1 + g64[:, :C]) * PA + ((1 + g64[:, C:]) * b64[:, NL] if valence else 0)
    lw64 = p / p.norm(dim=1, keepdim=True).clamp_min(EPS)
    dB64, dg64 = torch.autograd.grad((lw64 * dlv.double()).sum(), [b64, g64])
    lw_m, dp_m, dPA_m = _twobody_mag(Bv.view(E, NG, C), gv, dlv, NL, valence)

    _check(C_TWOBODY, "twobody lw", lw, lw64.detach(), lw_m)
    want = dB64.clone()
    mag = dPA_m.unsqueeze(1).expand(E, NG, C).clone()
    if valence:
        mag[:, NL] = dPA_m + (1 + gv.double()[:, C:].abs()) * dp_m
    if compact:
        want = torch.cat([want[:, :1], want[:, NL:]], 1)
        mag = torch.cat([mag[:, :1], mag[:, NL:]], 1)
    _check(C_TWOBODY, "twobody dB", dB.view(E, NGo, C), want, mag)
    PAabs = Bv.view(E, NG, C)[:, :NL].double().abs().sum(1) + (Bv.view(E, NG, C)[:, NL].double().abs() if valence else 0)
    dg_mag = dp_m * PAabs
    if valence:
        dg_mag = torch.cat([dg_mag, dp_m * Bv.view(E, NG, C)[:, NL].double().abs()], 1)
    _check(C_TWOBODY, "twobody dg", dg, dg64, dg_mag)
    for buf, v, what in ((lb, lw, "lw"), (dbb, dB, "dB"), (dgb, dg, "dg")):
        _padding_untouched(buf, v, what)
