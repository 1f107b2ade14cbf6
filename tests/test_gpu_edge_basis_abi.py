"""Every kernel path that builds the per-edge basis, called directly through the C ABI, against exact and high-precision
references.

The chain runs from positions to B:
  - `lcao_geom_basis_fwd` / `_bwd` (geom_basis.cu): distances, unit vectors, the radial basis rb, its derivative drb, and
    the backward to the positions (an edge stage and a node stage);
  - `lcao_coeff_contract_fwd` / `_bwd` (edge_ops.cu): B from per-edge coefficient rows;
  - `lcao_pair_contract_fwd` / `_bwd` (pair_table.cu): B, its Gram matrices and psum from the species-pair table, and the
    keyed reduction of d_tab (k_chunk_ptr -> k_pair_reduce_partial -> k_pair_reduce_final) plus d_rb.
The helpers below restate the dispatch of these entry points (35 kernels), so every case id names the kernels it runs;
one test checks that the cases reach all of them and, where cuobjdump is available, that the library holds no other.

Every contraction case runs twice:
  - exact inputs: small integers in [-4, 4] (vmask in {0, 1}).  Every FP32 product and partial sum is then an integer
    below 2^24, so each output must EQUAL the FP64 reference whatever the summation order (+0 and -0 compare equal):
    one dropped, doubled or misrouted edge, orbital, chunk or key fails.
  - random inputs: normal values, bounded componentwise by |got - ref| <= gamma_n * mag, gamma_n = n u / (1 - n u),
    u = 2^-24, where mag is the same sum over absolute values and n counts the roundings on the longest path through
    the kernel's own summation (the formulas are next to each bound below).
The geometry forward is compared with mpmath at 50 digits (correctly rounded up to FP64 evaluation error); its backward
with an exact dyadic case, a componentwise FP64 bound and torch.autograd of the FP64 oracle.

Every operand is a view into a NaN-filled buffer with NaN rows before and after it (index operands: -1), scratch
buffers start NaN, inputs must stay bitwise unchanged and output padding untouched, two identical calls agree
bitwise (none of these kernels uses atomics), and no output depends on which optional outputs were requested.
"""
from __future__ import annotations

import ctypes
import functools
import math
import os
import re
import shutil
import subprocess

import mpmath
import pytest
import torch

from lcaonet_b200 import _lib, ops
from lcaonet_b200.csrc.build import LIB
from oracle import lcao_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
P_, ST = ops.ptr, ops.stream_ptr
NAN_BITS = 0x7FC00000
PAD = 4            # NaN rows before and after every operand (keeps every row start 16-byte aligned)
U = 2.0 ** -24     # unit roundoff of FP32
U64 = 2.0 ** -53   # unit roundoff of FP64
CHUNK = 256        # k_pair_reduce_partial: sorted edges per stage-1 CTA
FWD_CAP = 148 * 16 * 8   # k_pair_contract_fwd: grid capped at 148 x 16 CTAs of 8 warps (one edge per warp and pass)
SMEM_OPT_IN = 48 * 1024  # dynamic shared memory above this needs cudaFuncSetAttribute


def gamma(n):
    n = torch.as_tensor(n, dtype=torch.float64)
    return n * U / (1 - n * U)


# Largest |got - ref| / bound per bound over every case of this file, measured on an NVIDIA B200 at its 1000 W power
# limit (a ratio <= 1 passes; the bounds are analytic and need no calibration):
#   pair B 0.73, pair gram 0.23, pair d_tab 0.021, pair d_rb 0.25, coeff B 0.53, coeff d_rb 0.28,
#   geometry forward 0.99995 (correct rounding: half an ulp), dvec 0.33, d_pos 0.11, d_pos vs autograd 0.088
OBSERVED: dict = {}


# ---------------------------------------------------------------------------------------------- dispatch restated
def _b(x):
    return "true" if x else "false"


def pair_fwd_kernels(E, NL, val):
    """lcao_pair_contract_fwd: one grid-stride launch per (NL, valence); nothing at E = 0"""
    return [f"k_pair_contract_fwd<{NL},{_b(val)}>"] if E > 0 else []


def pair_bwd_kernels(E, C, val, want_tab, want_rb):
    """lcao_pair_contract_bwd: the keyed reduction for d_tab (stage 1 skipped at E = 0), then d_rb by the pair-sorted
    walk for C <= 128 or one warp per edge above"""
    ks = []
    if want_tab:
        ks += ["k_chunk_ptr"] + ([f"k_pair_reduce_partial<{_b(val)}>"] if E > 0 else []) + ["k_pair_reduce_final"]
    if want_rb and E > 0:
        ks.append(f"k_pair_contract_drb_sorted<{_b(val)}>" if C <= 128 else f"k_pair_contract_drb<{_b(val)}>")
    return ks


def partial_smem(O, val):
    """dynamic shared memory of k_pair_reduce_partial: the chunk's edge ids, rb and (valence) rb * vmask"""
    return 4 * CHUNK + 4 * O * CHUNK * (1 + val)


def fwd_grid_strides(E):
    """k_pair_contract_fwd runs a second grid-stride pass when E exceeds the capped grid"""
    return E > FWD_CAP


def coeff_kernels(NL, val):
    return [f"k_coeff_contract_fwd<{NL},{_b(val)}>", f"k_coeff_contract_bwd<{NL},{_b(val)}>"]


def geom_bwd_kernels(E, N):
    return (["k_geom_edge_bwd"] if E > 0 else []) + (["k_geom_node_bwd"] if N > 0 else [])


ALL_KERNELS = ({f"k_pair_contract_fwd<{nl},{v}>" for nl in range(1, 5) for v in ("false", "true")}
               | {f"k_pair_contract_drb_sorted<{v}>" for v in ("false", "true")}
               | {f"k_pair_contract_drb<{v}>" for v in ("false", "true")}
               | {"k_chunk_ptr", "k_pair_reduce_final"} | {f"k_pair_reduce_partial<{v}>" for v in ("false", "true")}
               | {f"k_coeff_contract_{d}<{nl},{v}>" for d in ("fwd", "bwd") for nl in range(1, 5) for v in ("false", "true")}
               | {"k_geom_basis_fwd", "k_geom_edge_bwd", "k_geom_node_bwd"})
BASE_NAMES = ("k_pair_contract_fwd", "k_pair_contract_drb_sorted", "k_pair_contract_drb", "k_chunk_ptr",
              "k_pair_reduce_partial", "k_pair_reduce_final", "k_coeff_contract_fwd", "k_coeff_contract_bwd",
              "k_geom_basis_fwd", "k_geom_edge_bwd", "k_geom_node_bwd")


def _kid(names):
    return "+".join(k.replace("<", ".").replace(">", "").replace(",", ".") for k in names) or "none"


# ---------------------------------------------------------------------------------------------- padded operands
def _rows(M, W, fill=None, dtype=torch.float32):
    """(buffer, view): an (M, W) block of a flat NaN buffer with PAD rows before and after it"""
    buf = torch.full(((M + 2 * PAD) * W,), float("nan"), dtype=dtype, device=DEV)
    v = buf[PAD * W:(PAD + M) * W].view(M, W)
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
        bits = buf.reshape(-1).view(torch.int32)[mask]
        assert bool((bits == NAN_BITS).all()), f"{what}: {int((bits != NAN_BITS).sum())} padding elements written"
    else:
        assert bool(torch.isnan(buf[mask]).all()), f"{what}: padding written"


def _same_bits(a, b):
    if not a.is_floating_point():
        return torch.equal(a, b)
    return torch.equal(a.reshape(-1).view(torch.int32 if a.dtype == torch.float32 else torch.int64),
                       b.reshape(-1).view(torch.int32 if b.dtype == torch.float32 else torch.int64))


def _within(got, ref, mag, tol):
    """(ok, max ratio, first bad index): |got - ref| <= tol * mag componentwise, finite (tol broadcasts)"""
    if not bool(torch.isfinite(got).all()):
        bad = torch.nonzero(~torch.isfinite(got))[0].tolist()
        return False, math.inf, bad
    err = (got.double() - ref).abs()
    lim = tol * mag
    ratio = float((err / lim.clamp_min(1e-300)).max()) if err.numel() else 0.0
    bad = err > lim
    return (not bool(bad.any())), ratio, (torch.nonzero(bad)[0].tolist() if bool(bad.any()) else None)


def _check(name, what, got, ref, mag, tol):
    ok, ratio, first = _within(got, ref, mag, tol)
    OBSERVED[name] = max(OBSERVED.get(name, 0.0), ratio)
    if not ok:
        idx = tuple(first)
        lim = (torch.as_tensor(tol, dtype=torch.float64, device=DEV).expand_as(mag) * mag)[idx]
        raise AssertionError(f"{what}: over the bound at {list(idx)} (got {float(got[idx]):.9g}, want {float(ref[idx]):.9g}, "
                             f"bound {float(lim):.3g}); max ratio {ratio:.3g}")


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


# ---------------------------------------------------------------------------------------------- contraction inputs
def _lgrp(O, NL, empty):
    """l of each orbital, interleaved and not sorted by l; group `empty` gets no orbital"""
    ls = [l for l in range(NL) if l != empty]
    return torch.tensor([ls[(3 * o + 1) % len(ls)] for o in range(O)], dtype=torch.int32)


DOMINANT_KEY, DOMINANT_N = 7, 19000   # ceil(19000 / 256) = 75 chunks (74 full, one of 56): sub-rows of 10 and 9 chunks
SPECIAL_KEYS = {1: 1, 2: 255, 3: 256, 4: 257, 5: 512}   # key -> edge count: both sides of the 256-edge chunk


@functools.lru_cache(None)
def _keys(kind):
    """(pair (E,) int64 on the host, P): the key layouts of the pair-contraction cases"""
    g = torch.Generator().manual_seed(sum(map(ord, kind)))
    if kind in ("bounds", "big"):
        P = 1369
        n_rand = 3000 if kind == "bounds" else 60000 - DOMINANT_N - sum(SPECIAL_KEYS.values())
        rand = torch.randint(8, P - 1, (n_rand,), generator=g)
        rand = torch.where(rand % 97 == 0, rand + 1, rand)          # keys 0, P - 1 and every 97th key stay absent
        parts = [torch.full((DOMINANT_N,), DOMINANT_KEY)] + [torch.full((n,), k) for k, n in SPECIAL_KEYS.items()]
        pair = torch.cat(parts + [rand])
    elif kind == "P1":
        P, pair = 1, torch.zeros(3000, dtype=torch.long)
    elif kind == "P9":
        P, pair = 9, torch.randint(1, 8, (5000,), generator=g)      # keys 0 and 8 absent
    elif kind == "P5000":
        P, pair = 5000, torch.randint(1, 4999, (20000,), generator=g)
    else:                                                           # "E<n>": a few edges, 9 keys
        P, pair = 9, torch.randint(0, 9, (int(kind[1:]),), generator=g)
    return pair[torch.randperm(pair.numel(), generator=g)], P


def _grouping(pair, P, order):
    """(kptr, kperm): bucket_sort ordered (stable = 2, what the model uses), grouping only (stable = 0), or the ordered
    grouping with a random order inside every key (the ABI only requires grouping)"""
    kptr, kperm = ops.bucket_sort(pair, P, stable=(False if order == "grouped" else "ordered"))
    if order == "shuffled" and pair.numel():
        g = torch.Generator(device=DEV).manual_seed(5)
        perm = kperm[torch.randperm(pair.numel(), generator=g, device=DEV)].long()
        perm = perm[torch.sort(pair[perm], stable=True).indices]
        kperm = perm.int()
    return kptr, kperm


def _values(shape, exact, g, mask=False):
    if mask and exact:
        return torch.randint(0, 2, shape, generator=g, device=DEV).float()
    if exact:
        return torch.randint(-4, 5, shape, generator=g, device=DEV).float()
    return torch.randn(shape, generator=g, device=DEV)


class Contraction:
    """FP64 references of B, d_tab / d_cst1 and d_rb, with the magnitudes of the same sums over absolute values.
    `rows(i, j)` returns the coefficient rows (n, O, Cp) of edges i..j (the pair table gathered, or cst1)."""

    def __init__(self, rows, rb, vmask, lgrp, NL, C):
        self.rows, self.rb, self.vmask, self.NL, self.C = rows, rb.double(), vmask, NL, C
        self.m = vmask.double() if vmask is not None else None
        self.lg = lgrp.long().to(DEV)
        self.onehot = torch.nn.functional.one_hot(self.lg, NL).double()
        self.E, self.O = rb.shape
        self.val = vmask is not None
        self.step = max(1, (1 << 22) // (self.O * C * (1 + self.val)))

    def B(self):
        E, NL, C, val = self.E, self.NL, self.C, self.val
        z = functools.partial(torch.zeros, E, NL + val, C, dtype=torch.float64, device=DEV)
        ref, mag = z(), z()
        for i in range(0, E, self.step):
            j = min(E, i + self.step)
            T = self.rows(i, j).double()
            r = self.rb[i:j]
            for s, (TT, rr) in enumerate(((T, r), (T.abs(), r.abs()))):
                out = (ref, mag)[s]
                w = rr.unsqueeze(-1) * self.onehot
                out[i:j, :NL] = torch.einsum("nol,noc->nlc", w, TT[..., :C])
                if val:
                    mm = self.m[i:j] if s == 0 else self.m[i:j].abs()
                    out[i:j, :NL] += torch.einsum("nol,noc->nlc", w * mm.unsqueeze(-1), TT[..., C:])
                    out[i:j, NL] = torch.einsum("no,noc->nc", rr * mm, TT[..., C:])
        return ref, mag

    def terms(self, dB, i, j, absolute=False):
        """per-edge terms of the table gradient: (n, O, C) of rb dB_l(o), and with valence rb m (dB_l(o) + dB_NL)"""
        d = dB[i:j].double()
        r = self.rb[i:j]
        g = d[:, self.lg]
        if absolute:
            g, r = g.abs(), r.abs()
        A = r.unsqueeze(-1) * g
        if not self.val:
            return A
        m = self.m[i:j].abs() if absolute else self.m[i:j]
        gv = d[:, self.NL].unsqueeze(1)
        s = g + (gv.abs() if absolute else gv)
        return torch.cat([A, (r * m).unsqueeze(-1) * s], -1)

    def d_tab(self, dB, pair, P):
        ref = torch.zeros(P, self.O, self.C * (1 + self.val), dtype=torch.float64, device=DEV)
        mag = torch.zeros_like(ref)
        for i in range(0, self.E, self.step):
            j = min(self.E, i + self.step)
            ref.index_add_(0, pair[i:j], self.terms(dB, i, j))
            mag.index_add_(0, pair[i:j], self.terms(dB, i, j, True))
        return ref, mag

    def d_rb(self, dB):
        ref = torch.zeros(self.E, self.O, dtype=torch.float64, device=DEV)
        mag = torch.zeros_like(ref)
        C = self.C
        for i in range(0, self.E, self.step):
            j = min(self.E, i + self.step)
            T = self.rows(i, j).double()
            d = dB[i:j].double()
            g = d[:, self.lg]
            ref[i:j] = (T[..., :C] * g).sum(-1)
            mag[i:j] = (T[..., :C].abs() * g.abs()).sum(-1)
            if self.val:
                gv = d[:, self.NL].unsqueeze(1)
                m = self.m[i:j]
                ref[i:j] += m * (T[..., C:] * (g + gv)).sum(-1)
                mag[i:j] += m.abs() * (T[..., C:].abs() * (g.abs() + gv.abs())).sum(-1)
        return ref, mag


def _gram64(B, NL):
    b = B[:, :NL].double()
    iu = torch.triu_indices(NL, NL)
    return (torch.einsum("elc,emc->elm", b, b)[:, iu[0], iu[1]],
            torch.einsum("elc,emc->elm", b.abs(), b.abs())[:, iu[0], iu[1]])


# Bounds (n of gamma_n) from the kernels' summation structure:
#   pair B_l: one FMA per orbital of group l into the accumulator (O_l), with valence two (2 O_l) plus the rounding of
#     rb * vmask; the valence slot O FMAs plus that rounding.  A group without orbitals (n = 0) must be exactly 0.
#   coeff B_l: the rounded products rb * A (and rb * m, rb m * V and their sum) added in orbital order: O_l + 1, with
#     valence O_l + 3; the valence slot O + 2.
#   d_tab row of key k: 256 FMAs of one chunk, ceil(chunks_k / 8) adds of a k_pair_reduce_final sub-row, 8 for combining
#     the sub-rows; with valence 2 more (rb * vmask and dB_l + dB_NL).
#   d_rb: per 128-column pass a 4-term dot and its add into the lane's sum (with valence also the dB_l + dB_NL add, the
#     vmask product and a second add), then the 5-level butterfly: (4 + 2 val) ceil(C / 128) + 5 + 2 val.
def _n_pair_B(lgrp, NL, O, val):
    O_l = torch.bincount(lgrp.long(), minlength=NL)[:NL].double()
    n = O_l * (2 if val else 1) + (O_l > 0).double() * val
    return torch.cat([n, torch.tensor([O + 1.0])]) if val else n


def _n_coeff_B(lgrp, NL, O, val):
    O_l = torch.bincount(lgrp.long(), minlength=NL)[:NL].double()
    n = (O_l + (3 if val else 1)) * (O_l > 0)
    return torch.cat([n, torch.tensor([O + 2.0])]) if val else n


def _n_drb(C, val):
    return (4 + 2 * val) * math.ceil(C / 128) + 5 + 2 * val


def _n_dtab(kptr, val):
    cnt = (kptr[1:] - kptr[:-1]).double()
    chunks = torch.ceil(cnt / CHUNK)
    return CHUNK + torch.ceil(chunks / 8) + 8 + 2 * val


# ---------------------------------------------------------------------------------------------- pair contraction
# (NL, valence, C, O, keys, kperm order, forward outputs, backward outputs, empty group)
PAIR_CASES = [
    (1, 0, 128, 8, "bounds", "ordered", "gram+psum", "tab+rb", None),   # C = 128: sorted d_rb, 8 orbitals exactly
    (1, 1, 4, 9, "P1", "ordered", "psum", "tab+rb", None),              # one key; partial lanes; 8-orbital tail
    (2, 0, 12, 23, "P9", "grouped", "gram", "tab", 1),                  # empty group l = 1
    (2, 1, 124, 23, "bounds", "shuffled", "gram+psum", "tab+rb", None),  # valence below the 48 KB opt-in
    (3, 0, 132, 47, "bounds", "ordered", "none", "tab+rb", 2),          # below the opt-in; per-edge d_rb (C > 128)
    (3, 1, 256, 24, "P5000", "ordered", "gram+psum", "tab+rb", None),   # valence opt-in; five keys per k_chunk_ptr thread
    (4, 0, 260, 48, "bounds", "grouped", "gram", "tab+rb", None),       # opt-in; three column passes
    (4, 1, 128, 64, "bounds", "ordered", "psum", "tab+rb", 0),          # 132 KB of shared memory
    (1, 1, 260, 5, "big", "ordered", "gram+psum", "tab+rb", None),      # E = 60 000: past the forward's grid cap
    (3, 0, 128, 9, "big", "shuffled", "gram", "tab", None),
    (2, 0, 256, 64, "P9", "ordered", "none", "rb", None),               # d_rb alone: the positions-only pass
    (4, 1, 12, 1, "E1", "ordered", "gram+psum", "rb", None),
    (1, 0, 124, 5, "E7", "grouped", "psum", "tab+rb", None),
    (2, 1, 128, 8, "E15", "shuffled", "gram", "tab+rb", None),
    (3, 1, 4, 48, "P9", "grouped", "gram+psum", "tab+rb", 1),           # valence, O = 48
    (4, 0, 124, 9, "P1", "ordered", "gram+psum", "tab+rb", 3),
    (1, 1, 132, 47, "P9", "ordered", "gram", "tab+rb", None),           # valence opt-in; per-edge d_rb<true>
    (2, 0, 4, 1, "E0", "ordered", "gram+psum", "tab+rb", None),         # no edges: d_tab written as zeros
]


def _pair_case_kernels(case):
    NL, val, C, O, keys, _, _, bwd_out, _ = case
    E = _keys(keys)[0].numel()
    return pair_fwd_kernels(E, NL, val) + pair_bwd_kernels(E, C, val, "tab" in bwd_out, "rb" in bwd_out)


def _pair_case_id(case):
    NL, val, C, O, keys, order, fwd_out, bwd_out, empty = case
    return (f"{_kid(_pair_case_kernels(case))}-NL{NL}{'-val' if val else ''}-C{C}-O{O}-{keys}-{order}-{fwd_out}-{bwd_out}"
            + (f"-empty{empty}" if empty is not None else ""))


class PairOps:
    """The padded device operands of one pair-contraction case"""

    def __init__(self, case, exact, seed):
        NL, val, C, O, keys, order, _, _, empty = case
        pair, P = _keys(keys)
        E = pair.numel()
        self.NL, self.val, self.C, self.O, self.E, self.P, self.NG = NL, val, C, O, E, P, NL + val
        Cp = C * (1 + val)
        g = torch.Generator(device=DEV).manual_seed(seed)
        self.tb, self.tab = _rows(P * O, Cp, _values((P, O, Cp), exact, g))
        pair = pair.to(DEV)
        self.pb, self.pair = _irows(E, pair, torch.int64)
        self.rbb, self.rb = _rows(E, O, _values((E, O), exact, g))
        self.vb, self.vmask = _rows(E, O, _values((E, O), exact, g, mask=True)) if val else (None, None)
        self.lgrp_cpu = _lgrp(O, NL, empty)
        self.lb, self.lgrp = _irows(O, self.lgrp_cpu, torch.int32)
        self.db, self.dB = _rows(E, self.NG * C, _values((E, self.NG, C), exact, g))
        kptr, kperm = _grouping(pair, P, order)
        self.kpb, self.kptr = _irows(P + 1, kptr, torch.int32)
        self.kmb, self.kperm = _irows(E, kperm, torch.int32)
        torch.cuda.synchronize()
        self.inputs = [(b, b.clone()) for b in (self.tb, self.pb, self.rbb, self.vb, self.lb, self.db, self.kpb, self.kmb)
                       if b is not None]
        self.ref = Contraction(lambda i, j: self.tab.view(P, O, Cp)[self.pair[i:j]], self.rb, self.vmask, self.lgrp, NL, C)

    def fwd(self, want_gram, want_psum):
        E, NG, C, NL, val = self.E, self.NG, self.C, self.NL, self.val
        Bb, B = _rows(E, NG * C)
        gb, gram = _rows(E, NL * (NL + 1) // 2, dtype=torch.float64) if want_gram else (None, None)
        sb, psum = _rows(E, (1 + val) * C) if want_psum else (None, None)
        with Launch() as n:
            ops._call("lcao_pair_contract_fwd", P_(self.tab), P_(self.pair), P_(self.rb), P_(self.vmask), P_(self.lgrp),
                      E, self.O, C, NL, val, P_(B), P_(gram), P_(psum), ST())
        torch.cuda.synchronize()
        assert n.n == len(pair_fwd_kernels(E, NL, val))
        out = {"B": B.view(E, NG, C)}
        _padding_untouched(Bb, B, "B")
        if want_gram:
            _padding_untouched(gb, gram, "gram")
            out["gram"] = gram
        if want_psum:
            _padding_untouched(sb, psum, "psum")
            out["psum"] = psum.view(E, 1 + val, C)
        return out

    def bwd(self, want_tab, want_rb):
        E, P, O, C, val = self.E, self.P, self.O, self.C, self.val
        tb, d_tab = _rows(P * O, C * (1 + val)) if want_tab else (None, None)
        rbb, d_rb = _rows(E, O) if want_rb else (None, None)
        scb = scratch = None
        if want_tab:
            nbytes = int(_lib.load().lcao_pair_contract_bwd_scratch(E, P, O, C, val))
            scb, scratch = _rows((nbytes + 15) // 16, 4)   # NaN: a partial slot that no CTA wrote reads as NaN
        with Launch() as n:
            ops._call("lcao_pair_contract_bwd", P_(self.tab), P_(self.pair), P_(self.kptr), P_(self.kperm), P_(self.rb),
                      P_(self.vmask), P_(self.lgrp), P_(self.dB), E, P, O, C, self.NL, val, P_(d_tab), P_(d_rb),
                      P_(scratch), ST())
        torch.cuda.synchronize()
        assert n.n == len(pair_bwd_kernels(E, C, val, want_tab, want_rb))
        out = {}
        if want_tab:
            _padding_untouched(tb, d_tab, "d_tab")
            _padding_untouched(scb, scratch, "scratch")
            out["d_tab"] = d_tab.view(P, O, C * (1 + val))
        if want_rb:
            _padding_untouched(rbb, d_rb, "d_rb")
            out["d_rb"] = d_rb
        return out

    def inputs_unchanged(self):
        for buf, before in self.inputs:
            assert _same_bits(buf, before), "an input buffer (operand or padding) was written"


def _run_pair(ops_, fwd_out, bwd_out):
    """every call of a case: the full call twice (bitwise the same) and the case's own optional-output combination,
    whose outputs must be bitwise those of the full call"""
    full = ops_.fwd(True, True)
    again = ops_.fwd(True, True)
    mine = ops_.fwd("gram" in fwd_out, "psum" in fwd_out)
    for k, v in full.items():
        assert _same_bits(v, again[k]), f"forward {k}: two identical calls differ"
        if k in mine:
            assert _same_bits(v, mine[k]), f"forward {k} depends on the optional outputs requested"
    bfull = ops_.bwd(True, ops_.E > 0)
    bagain = ops_.bwd(True, ops_.E > 0)
    bmine = ops_.bwd("tab" in bwd_out, "rb" in bwd_out)
    for k, v in bfull.items():
        assert _same_bits(v, bagain[k]), f"backward {k}: two identical calls differ"
        if k in bmine:
            assert _same_bits(v, bmine[k]), f"backward {k} depends on the optional outputs requested"
    ops_.inputs_unchanged()
    full.update(bfull)
    if "d_rb" in bmine:
        full["d_rb"] = bmine["d_rb"]
    return full


def _check_psum(got, NL, val):
    """psum: bitwise the left-to-right FP32 sum of the returned groups 0..NL-1, and the valence slot bitwise B[:, NL]"""
    B = got["B"]
    t = B[:, 0].clone()
    for l in range(1, NL):
        t = t + B[:, l]
    assert _same_bits(got["psum"][:, 0], t), "psum is not the FP32 sum of the returned B groups"
    if val:
        assert _same_bits(got["psum"][:, 1], B[:, NL]), "psum valence slot is not B[:, NL]"


@pytest.mark.parametrize("case", PAIR_CASES, ids=[_pair_case_id(c) for c in PAIR_CASES])
def test_pair_contract_vs_fp64(case):
    NL, val, C, O, keys, order, fwd_out, bwd_out, empty = case
    for exact in (True, False):
        ops_ = PairOps(case, exact, seed=C * 7 + O * 3 + NL + 100 * exact)
        E, P = ops_.E, ops_.P
        got = _run_pair(ops_, fwd_out, bwd_out)
        ref = ops_.ref
        kind = "exact" if exact else "random"
        B_ref, B_mag = ref.B()
        _check_psum(got, NL, val)
        g_ref, g_mag = _gram64(got["B"], NL)
        if empty is not None:
            assert bool((got["B"][:, empty] == 0).all()), "a group without orbitals is not exactly zero"
        dt_ref, dt_mag = ref.d_tab(ops_.dB.view(E, NL + val, C), ops_.pair, P)
        absent = (ops_.kptr[1:] == ops_.kptr[:-1])
        assert bool((got["d_tab"][absent] == 0).all()), "d_tab rows of absent keys are not exactly zero"
        if E:
            dr_ref, dr_mag = ref.d_rb(ops_.dB.view(E, NL + val, C))
        if exact:
            _exact(f"{kind} B", got["B"], B_ref)
            _exact(f"{kind} gram", got["gram"], _gram64(B_ref, NL)[0])
            _exact(f"{kind} d_tab", got["d_tab"], dt_ref)
            if E:
                _exact(f"{kind} d_rb", got["d_rb"], dr_ref)
        else:
            nB = _n_pair_B(ops_.lgrp_cpu, NL, O, val).to(DEV).view(1, -1, 1)
            _check("pair B", f"{kind} B", got["B"], B_ref, B_mag, gamma(nB))
            _check("pair gram", f"{kind} gram", got["gram"], g_ref, g_mag, (C + 5) * U64)
            nk = _n_dtab(ops_.kptr, val).view(-1, 1, 1)
            _check("pair d_tab", f"{kind} d_tab", got["d_tab"], dt_ref, dt_mag, gamma(nk))
            if E:
                _check("pair d_rb", f"{kind} d_rb", got["d_rb"], dr_ref, dr_mag, gamma(_n_drb(C, val)))


def test_pair_bounds_single_out_one_term():
    """The random-case bounds are tight enough to matter: removing from the reference the one edge at sorted position
    256 of the dominant key (19 000 edges) makes the d_tab bound fail for that key, and removing one orbital term makes
    the B bound fail for that edge"""
    case = (2, 1, 128, 9, "bounds", "ordered", "gram+psum", "tab+rb", None)
    NL, val, C, O = 2, 1, 128, 9
    ops_ = PairOps(case, False, seed=77)
    E, P = ops_.E, ops_.P
    got = ops_.fwd(True, False)
    got.update(ops_.bwd(True, False))
    ref = ops_.ref
    dB = ops_.dB.view(E, NL + val, C)
    dt_ref, dt_mag = ref.d_tab(dB, ops_.pair, P)
    nk = _n_dtab(ops_.kptr, val).view(-1, 1, 1)
    _check("pair d_tab", "d_tab", got["d_tab"], dt_ref, dt_mag, gamma(nk))
    k = DOMINANT_KEY
    e = int(ops_.kperm[int(ops_.kptr[k]) + 256])
    assert int(ops_.pair[e]) == k and int(ops_.kptr[k + 1] - ops_.kptr[k]) == DOMINANT_N
    t, ta = ref.terms(dB, e, e + 1)[0], ref.terms(dB, e, e + 1, True)[0]
    ok, _, _ = _within(got["d_tab"][k], dt_ref[k] - t, dt_mag[k] - ta, gamma(nk[k]))
    assert not ok, "the d_tab bound accepts the key's sum without one of its 19 000 edges"

    B_ref, B_mag = ref.B()
    o = 4
    l = int(ops_.lgrp_cpu[o])
    e = 123
    T = ops_.tab.view(P, O, 2 * C)[ops_.pair[e], o].double()
    r, m = float(ops_.rb[e, o]), float(ops_.vmask[e, o])
    term = r * (T[:C] + m * T[C:])
    nB = _n_pair_B(ops_.lgrp_cpu, NL, O, val)
    ok, _, _ = _within(got["B"][e, l], B_ref[e, l] - term, B_mag[e, l] - term.abs(), gamma(nB[l]))
    assert not ok, "the B bound accepts the edge's row without one orbital term"


# ---------------------------------------------------------------------------------------------- coefficient contraction
# (NL, valence, C, O, d_rb given, empty group): every (NL, valence) forward and backward instantiation
COEFF_CASES = [
    (1, 0, 4, 1, True, None), (1, 1, 128, 9, False, None), (2, 0, 124, 5, True, 0), (2, 1, 260, 8, True, None),
    (3, 0, 12, 23, False, None), (3, 1, 132, 24, True, 2), (4, 0, 256, 47, True, None), (4, 1, 12, 48, True, 1),
    (2, 0, 260, 64, True, None), (4, 1, 124, 64, False, None), (3, 0, 128, 8, True, None), (1, 1, 256, 47, True, None),
]


def _coeff_id(case):
    NL, val, C, O, with_drb, empty = case
    return (f"{_kid(coeff_kernels(NL, val))}-NL{NL}{'-val' if val else ''}-C{C}-O{O}{'-drb' if with_drb else ''}"
            + (f"-empty{empty}" if empty is not None else ""))


@pytest.mark.parametrize("case", COEFF_CASES, ids=[_coeff_id(c) for c in COEFF_CASES])
def test_coeff_contract_vs_fp64(case):
    NL, val, C, O, with_drb, empty = case
    Cp, NG = C * (1 + val), NL + val
    E = max(41, min(3001, (1 << 22) // (O * Cp)))
    lgrp_cpu = _lgrp(O, NL, empty)
    for exact in (True, False):
        g = torch.Generator(device=DEV).manual_seed(C + O + NL + 10 * exact)
        cb, cst1 = _rows(E * O, Cp, _values((E, O, Cp), exact, g))
        rbb, rb = _rows(E, O, _values((E, O), exact, g))
        vb, vmask = _rows(E, O, _values((E, O), exact, g, mask=True)) if val else (None, None)
        lb, lgrp = _irows(O, lgrp_cpu, torch.int32)
        db, dB = _rows(E, NG * C, _values((E, NG, C), exact, g))
        torch.cuda.synchronize()
        inputs = [(b, b.clone()) for b in (cb, rbb, vb, lb, db) if b is not None]

        def fwd():
            Bb, B = _rows(E, NG * C)
            with Launch() as n:
                ops._call("lcao_coeff_contract_fwd", P_(cst1), P_(rb), P_(vmask), P_(lgrp), E, O, C, NL, val, P_(B), ST())
            torch.cuda.synchronize()
            assert n.n == 1
            _padding_untouched(Bb, B, "B")
            return B.view(E, NG, C)

        def bwd(want_rb):
            xb, d_cst1 = _rows(E * O, Cp)
            yb, d_rb = _rows(E, O) if want_rb else (None, None)
            with Launch() as n:
                ops._call("lcao_coeff_contract_bwd", P_(cst1), P_(rb), P_(vmask), P_(lgrp), P_(dB), E, O, C, NL, val,
                          P_(d_cst1), P_(d_rb), ST())
            torch.cuda.synchronize()
            assert n.n == 1
            _padding_untouched(xb, d_cst1, "d_cst1")
            if want_rb:
                _padding_untouched(yb, d_rb, "d_rb")
            return d_cst1.view(E, O, Cp), d_rb

        B, B2 = fwd(), fwd()
        dc, d_rb = bwd(True)
        dc2, d_rb2 = bwd(True)
        dc_mine, _ = bwd(with_drb)
        assert _same_bits(B, B2) and _same_bits(dc, dc2) and _same_bits(d_rb, d_rb2), "two identical calls differ"
        assert _same_bits(dc, dc_mine), "d_cst1 depends on whether d_rb is requested"
        for buf, before in inputs:
            assert _same_bits(buf, before), "an input buffer (operand or padding) was written"

        ref = Contraction(lambda i, j: cst1.view(E, O, Cp)[i:j], rb, vmask, lgrp, NL, C)
        B_ref, B_mag = ref.B()
        dB3 = dB.view(E, NG, C)
        dr_ref, dr_mag = ref.d_rb(dB3)
        # d_cst1 is one rounded product per element: fp32(r dB_l), with valence fp32(fp32(r m) fp32(dB_l + dB_NL))
        gl = dB3[:, lgrp.long()]
        assert _same_bits(dc[..., :C], rb.unsqueeze(-1) * gl), "d_cst1 is not fp32(rb * dB_l)"
        if val:
            want = (rb * vmask).unsqueeze(-1) * (gl + dB3[:, NL].unsqueeze(1))
            assert _same_bits(dc[..., C:], want), "d_cst1 valence half is not fp32(fp32(rb m) fp32(dB_l + dB_NL))"
        if empty is not None:
            assert bool((B[:, empty] == 0).all()), "a group without orbitals is not exactly zero"
        if exact:
            _exact("exact B", B, B_ref)
            _exact("exact d_rb", d_rb, dr_ref)
        else:
            nB = _n_coeff_B(lgrp_cpu, NL, O, val).to(DEV).view(1, -1, 1)
            _check("coeff B", "random B", B, B_ref, B_mag, gamma(nB))
            _check("coeff d_rb", "random d_rb", d_rb, dr_ref, dr_mag, gamma(_n_drb(C, val)))


# ---------------------------------------------------------------------------------------------- geometry forward
SHELLS = [(1, 0), (2, 1), (3, 2), (4, 3), (5, 0), (6, 2), (7, 0), (7, 1)]   # every l; 7s has the largest degree (6)
RC, A0 = 5.0, 0.529
RBF = {"hydrogen": 0, "sphericalbessel": 1}
CUT = {"polynomial": 0, "envelope": 1, "cosine": 2}


def _spec(rbf, cut, n_rep):
    sp = _lib.BasisSpec()
    sp.n_unique, sp.n_rep, sp.cutoff_kind, sp.rbf_kind, sp.rc, sp.a0 = len(SHELLS), n_rep, CUT[cut], RBF[rbf], RC, A0
    for u, (n, l) in enumerate(SHELLS):
        coef = O.laguerre_poly(n, l)
        sp.n[u], sp.l[u], sp.deg[u], sp.norm[u] = n, l, len(coef) - 1, O.radial_norm(n, l, A0)
        for i, c in enumerate(coef):
            sp.poly[u][i] = float(c)
    return sp


def _f32_after(x):
    return float(torch.nextafter(torch.tensor(x, dtype=torch.float32), torch.tensor(math.inf)).item())


# edges of graph 0 from the origin along x: (kind, r)
R_SPECIAL = [("r0.05", 0.05), ("rc(1-2^-20)", RC * (1 - 2.0 ** -20)), ("rc", RC), ("past rc", _f32_after(RC))]


@functools.lru_cache(None)
def geom_graph():
    """Three graphs with different (skewed) lattices selected by batch[s], 40 atoms each; edges to every periodic image
    within 1.1 rc (sampled), two self-image edges (s = t, nonzero shift), and in graph 0 the edges of R_SPECIAL."""
    g = torch.Generator().manual_seed(11)
    lat = torch.tensor([[[4.2, 0.0, 0.0], [0.7, 5.1, 0.0], [-0.4, 0.9, 5.6]],
                        [[6.3, 0.0, 0.0], [0.0, 6.0, 0.0], [0.0, 0.0, 4.5]],
                        [[3.9, 1.3, 0.0], [-1.1, 4.4, 0.6], [0.5, -0.8, 6.1]]], dtype=torch.float32)
    n_per = 40
    pos, src, dst, shift, special = [], [], [], [], {}
    for b in range(3):
        frac = torch.rand(n_per, 3, generator=g)
        p = frac @ lat[b]
        base = b * n_per
        if b == 0:   # atoms 0..4: origin and the special distances along x
            p[0] = 0.0
            for k, (_, r) in enumerate(R_SPECIAL):
                p[k + 1] = torch.tensor([r, 0.0, 0.0])
        pos.append(p)
        imgs = torch.tensor([[i, j, k] for i in (-1, 0, 1) for j in (-1, 0, 1) for k in (-1, 0, 1)], dtype=torch.float32)
        vec = (p.double()[None, :, None] - p.double()[:, None, None] + (imgs.double() @ lat[b].double())[None, None])
        r = vec.norm(dim=-1)
        s_, t_, im = torch.nonzero((r < 1.1 * RC) & (r > 0.3), as_tuple=True)
        keep = torch.randperm(s_.numel(), generator=g)[:700]
        src.append(s_[keep] + base), dst.append(t_[keep] + base), shift.append(imgs[im[keep]])
        src.append(torch.tensor([base + 7, base + 9])), dst.append(torch.tensor([base + 7, base + 9]))
        shift.append(torch.tensor([[1.0, 0.0, 0.0], [0.0, 1.0, -1.0]]))
    src.insert(0, torch.zeros(len(R_SPECIAL), dtype=torch.long))
    dst.insert(0, torch.arange(1, len(R_SPECIAL) + 1))
    shift.insert(0, torch.zeros(len(R_SPECIAL), 3))
    for k, (name, _) in enumerate(R_SPECIAL):
        special[name] = k
    src, dst, shift = torch.cat(src), torch.cat(dst), torch.cat(shift)
    batch = torch.arange(3).repeat_interleave(n_per)
    return dict(pos=torch.cat(pos), shift=shift, lattice=lat, batch=batch, edge_index=torch.stack([src, dst]),
                N=3 * n_per, special=special, self_image=[int(i) for i in torch.nonzero(src == dst).flatten()])


mpmath.mp.dps = 50


def _mp_split(x):
    hi = float(x)
    return hi, float(x - hi)


@functools.lru_cache(None)
def geom_reference():
    """per edge, in mpmath from the exact FP32 inputs: dist, unit, the radial functions R_u, dR_u of both bases and the
    cutoffs f, df, as (hi, lo) FP64 pairs; and FP64 magnitudes for the bounds"""
    gr = geom_graph()
    pos, shift, lat, batch = gr["pos"].double(), gr["shift"].double(), gr["lattice"].double(), gr["batch"]
    s, t = gr["edge_index"]
    mpf = mpmath.mpf
    rows = {k: [] for k in ("dist", "unit", "R_h", "dR_h", "R_b", "dR_b", "f", "df")}
    pi = mpmath.pi
    for e in range(s.numel()):
        L = lat[batch[s[e]]]
        v = [mpf(float(pos[t[e], j])) - mpf(float(pos[s[e], j]))
             + sum(mpf(float(shift[e, i])) * mpf(float(L[i, j])) for i in range(3)) for j in range(3)]
        r = mpmath.sqrt(sum(x * x for x in v))
        rows["dist"].append(_mp_split(r))
        rows["unit"].append([_mp_split(x / r) for x in v])
        Rh, dRh, Rb, dRb = [], [], [], []
        for n, l in SHELLS:
            coef = O.laguerre_poly(n, l)
            zs = 2 / (n * mpf(A0))
            z = zs * r
            p = sum(c * z ** i for i, c in enumerate(coef))
            dp = sum(i * c * z ** (i - 1) for i, c in enumerate(coef) if i)
            nrm = mpf(O.radial_norm(n, l, A0))
            ex = mpmath.exp(-z / 2)
            Rh.append(_mp_split(nrm * p * z ** l * ex))
            dRh.append(_mp_split(nrm * ex * zs * (dp * z ** l + (p * l * z ** (l - 1) if l else 0) - p * z ** l / 2)))
            w = pi * n / RC
            Rb.append(_mp_split(mpmath.sin(w * r) / r))
            dRb.append(_mp_split(w * mpmath.cos(w * r) / r - mpmath.sin(w * r) / r ** 2))
        for key, val in (("R_h", Rh), ("dR_h", dRh), ("R_b", Rb), ("dR_b", dRb)):
            rows[key].append(val)
        f, df = [], []
        q = r / RC
        for cut in ("polynomial", "envelope", "cosine"):
            if r > RC:
                fv, dfv = mpf(0), mpf(0)
            elif cut == "polynomial":
                fv, dfv = (1 - q) ** 3 * (1 + 3 * q + 6 * q * q), -30 * q ** 2 * (1 - q) ** 2 / RC
            elif cut == "envelope":
                fv = (1 - q) ** 3 * (1 + 3 * q + 6 * q ** 2 + 10 * q ** 3 + 15 * q ** 4)
                dfv = -105 * q ** 4 * (1 - q) ** 2 / RC
            else:
                fv, dfv = (mpmath.cos(pi * q) + 1) / 2, -pi / RC * mpmath.sin(pi * q) / 2
            f.append(_mp_split(fv))
            df.append(_mp_split(dfv))
        rows["f"].append(f)
        rows["df"].append(df)
    out = {k: torch.tensor(v, dtype=torch.float64, device=DEV) for k, v in rows.items()}   # (..., 2): hi, lo

    # magnitudes (FP64): the terms summed, plus the sensitivity to a relative FP64 error of r (|r d/dr|) and, for sin and
    # cos, of their argument, so that k 2^-53 mag covers every FP64 rounding of the kernel's evaluation
    cell = lat[batch[s]]
    terms = (pos[t].abs() + pos[s].abs() + (shift.abs().unsqueeze(-1) * cell.abs()).sum(1)).to(DEV)
    r = out["dist"][:, 0]
    mag_dist = terms.sum(1)
    u = out["unit"][..., 0]
    mag_unit = terms / r.unsqueeze(1) + u.abs() * (mag_dist / r).unsqueeze(1)
    rr = r.unsqueeze(1)
    Rh = []
    dRh = []
    for n, l in SHELLS:
        coef = O.laguerre_poly(n, l)
        zs = 2.0 / (n * A0)
        z = zs * r
        ex = torch.exp(-z / 2) * abs(O.radial_norm(n, l, A0))
        mR = sum(abs(c) * z ** (i + l) * (2 + i + l + z) for i, c in enumerate(coef)) * ex
        mdR = sum(abs(c) * ((i + l) * z ** max(i + l - 1, 0) + 0.5 * z ** (i + l)) * (3 + i + l + z)
                  for i, c in enumerate(coef)) * ex * zs
        Rh.append(mR), dRh.append(mdR)
    w = torch.tensor([math.pi * n / RC for n, _ in SHELLS], dtype=torch.float64, device=DEV)
    wr = w * rr
    sn, cs = torch.sin(wr).abs(), torch.cos(wr).abs()
    mags = dict(dist=mag_dist, unit=mag_unit, R_h=torch.stack(Rh, 1), dR_h=torch.stack(dRh, 1), R_b=(sn + wr) / rr,
                dR_b=w * (cs + wr) / rr + (sn + wr) / rr ** 2)
    q = (r / RC).unsqueeze(1)
    a = math.pi / RC
    inside = (r <= RC).double().unsqueeze(1)
    fv, dfv = out["f"][..., 0].abs(), out["df"][..., 0].abs()
    uq = (1 - q).abs()
    mf = torch.cat([fv[:, :2] + rr * dfv[:, :2], 0.5 * (1 + torch.cos(a * rr).abs()) + rr * dfv[:, 2:]], 1)
    mdf = torch.cat([dfv[:, :1] + 60 / RC ** 2 * q * uq * rr, dfv[:, 1:2] + 420 / RC ** 2 * q ** 3 * uq * rr,
                     0.5 * a * (torch.sin(a * rr).abs() + a * rr)], 1)
    mags.update(f=mf * inside, df=mdf * inside)
    return out, mags


K_GEOM = 256   # FP64 evaluation error allowance, in units of 2^-53 mag


def _ulp32(x):
    a = x.abs().float()
    return (torch.nextafter(a, torch.full_like(a, math.inf)) - a).double()


def _check_rounded(name, what, got, hl, mag):
    """|got - exact| <= 1/2 ulp32(got) + K 2^-53 mag, with exact = hi + lo"""
    err = ((got.double() - hl[..., 0]) - hl[..., 1]).abs()
    lim = 0.5 * _ulp32(got) + K_GEOM * U64 * mag
    assert bool(torch.isfinite(got).all()), f"{what}: not finite"
    ratio = float((err / lim.clamp_min(1e-300)).max())
    OBSERVED[name] = max(OBSERVED.get(name, 0.0), ratio)
    bad = err > lim
    if bool(bad.any()):
        idx = tuple(torch.nonzero(bad)[0].tolist())
        raise AssertionError(f"{what}: not correctly rounded at {list(idx)}: got {float(got[idx])!r}, exact "
                             f"{float(hl[idx][0])!r}; max ratio {ratio:.3g}")


def _geom_operands(with_batch):
    gr = geom_graph()
    gi = ops.GraphIndex(gr["edge_index"].to(DEV), gr["N"])
    E, N = gi.E, gr["N"]
    posb, pos = _rows(N, 3, gr["pos"].to(DEV))
    shb, shift = _rows(E, 3, gr["shift"].to(DEV))
    lat = gr["lattice"] if with_batch else gr["lattice"][:1]
    latb, lattice = _rows(lat.shape[0], 9, lat.reshape(-1, 9).to(DEV))
    bb, batch = _irows(N, gr["batch"].to(DEV), torch.int64) if with_batch else (None, None)
    sb, src = _irows(E, gi.src32, torch.int32)
    db, dst = _irows(E, gi.dst32, torch.int32)
    return gi, dict(pos=(posb, pos), shift=(shb, shift), lattice=(latb, lattice), batch=(bb, batch), src=(sb, src),
                    dst=(db, dst))


def _geom_fwd(opnds, E, spec, O_, want_drb=True):
    ob = {k: v[1] for k, v in opnds.items()}
    before = [(b, b.clone()) for b, _ in opnds.values() if b is not None]
    distb, dist = _rows(E, 1)
    unitb, unit = _rows(E, 3)
    rbb, rb = _rows(E, O_)
    drbb, drb = _rows(E, O_) if want_drb else (None, None)
    with Launch() as n:
        ops._call("lcao_geom_basis_fwd", P_(ob["pos"]), P_(ob["shift"]), P_(ob["lattice"]), P_(ob["batch"]), P_(ob["src"]),
                  P_(ob["dst"]), E, ctypes.byref(spec), P_(dist), P_(unit), P_(rb), P_(drb), ST())
    torch.cuda.synchronize()
    assert n.n == (1 if E else 0)
    for b, v, w in ((distb, dist, "dist"), (unitb, unit, "unit"), (rbb, rb, "rb"), (drbb, drb, "drb")):
        if b is not None:
            _padding_untouched(b, v, w)
    for b, c in before:
        assert _same_bits(b, c), "an input buffer (operand or padding) was written"
    return dict(dist=dist.view(E), unit=unit, rb=rb, drb=drb)


GEOM_CASES = [(rbf, cut) for rbf in ("hydrogen", "sphericalbessel") for cut in ("polynomial", "envelope", "cosine")]


@pytest.mark.parametrize("rbf,cut", GEOM_CASES, ids=[f"k_geom_basis_fwd-{r}-{c}" for r, c in GEOM_CASES])
def test_geom_basis_fwd_vs_mpmath(rbf, cut):
    gr = geom_graph()
    gi, opnds = _geom_operands(True)
    E, n_u = gi.E, len(SHELLS)
    got = _geom_fwd(opnds, E, _spec(rbf, cut, 2), 2 * n_u)
    ref, mags = geom_reference()
    _check_rounded("geometry", "dist", got["dist"], ref["dist"], mags["dist"])
    _check_rounded("geometry", "unit", got["unit"], ref["unit"], mags["unit"])
    ci = list(CUT).index(cut)
    key = "h" if rbf == "hydrogen" else "b"
    R, dR, mR, mdR = ref["R_" + key], ref["dR_" + key], mags["R_" + key], mags["dR_" + key]
    f, df = ref["f"][:, ci:ci + 1], ref["df"][:, ci:ci + 1]
    mf, mdf = mags["f"][:, ci:ci + 1], mags["df"][:, ci:ci + 1]
    fh, dfh = f[..., 0], df[..., 0]
    # rb = f R and drb = f' R + f R' from the (hi, lo) pairs: the products of two pairs carry ~2^-100 relative error
    rb_hl = torch.stack([fh * R[..., 0], fh * R[..., 1] + f[..., 1] * R[..., 0]], -1)
    drb_hl = torch.stack([dfh * R[..., 0] + fh * dR[..., 0],
                          dfh * R[..., 1] + df[..., 1] * R[..., 0] + fh * dR[..., 1] + f[..., 1] * dR[..., 0]], -1)
    hi = rb_hl[..., 0] + rb_hl[..., 1]
    rb_hl = torch.stack([hi, (rb_hl[..., 0] - hi) + rb_hl[..., 1]], -1)
    hi = drb_hl[..., 0] + drb_hl[..., 1]
    drb_hl = torch.stack([hi, (drb_hl[..., 0] - hi) + drb_hl[..., 1]], -1)
    # the FP64 combination above rounds too: add 8 ulp64 of the products' magnitude to the allowance
    m_rb = mf * mR + 8 * (f[..., 0].abs() * R[..., 0].abs())
    m_drb = mdf * mR + mf * mdR + 8 * (df[..., 0].abs() * R[..., 0].abs() + f[..., 0].abs() * dR[..., 0].abs())
    rb = got["rb"].view(E, n_u, 2)
    drb = got["drb"].view(E, n_u, 2)
    assert _same_bits(rb[..., 0], rb[..., 1]) and _same_bits(drb[..., 0], drb[..., 1]), "n_rep copies differ"
    _check_rounded("geometry", "rb", rb[..., 0], rb_hl, m_rb)
    _check_rounded("geometry", "drb", drb[..., 0], drb_hl, m_drb)

    sp = gr["special"]
    at_rc, past = sp["rc"], sp["past rc"]
    assert float(got["dist"][at_rc]) == RC and float(got["dist"][past]) > RC
    assert bool((rb[at_rc] == 0).all()), "rb at r = rc is not exactly 0"
    assert bool((rb[past] == 0).all()) and bool((drb[past] == 0).all()), "rb / drb past rc are not exactly 0"
    assert float(got["dist"][sp["rc(1-2^-20)"]]) < RC and bool((rb[sp["rc(1-2^-20)"]] != 0).any())
    for e in gr["self_image"]:
        assert float(got["dist"][e]) > 0

    # n_rep = 1 gives the same values; drb = NULL leaves rb bitwise unchanged
    one = _geom_fwd(opnds, E, _spec(rbf, cut, 1), n_u)
    assert _same_bits(one["rb"], rb[..., 0].contiguous()) and _same_bits(one["drb"], drb[..., 0].contiguous())
    nodrb = _geom_fwd(opnds, E, _spec(rbf, cut, 2), 2 * n_u, want_drb=False)
    assert _same_bits(nodrb["rb"], got["rb"]) and _same_bits(nodrb["dist"], got["dist"])

    # batch = NULL selects lattice 0 for every edge: bitwise the batched result on graph 0's edges
    gi0, op0 = _geom_operands(False)
    nob = _geom_fwd(op0, E, _spec(rbf, cut, 2), 2 * n_u)
    g0 = (gr["batch"][gr["edge_index"][0]] == 0).to(DEV)
    for k in ("dist", "unit", "rb", "drb"):
        assert _same_bits(nob[k][g0], got[k][g0]), k
    assert not _same_bits(nob["dist"][~g0], got["dist"][~g0])


def test_geom_reference_matches_the_oracle():
    """the mpmath reference against oracle.lcao_oracle.radial_basis (FP64) away from rc, for both bases and cutoffs"""
    ref, _ = geom_reference()
    r = ref["dist"][:, 0]
    keep = r < 0.99 * RC
    nl = SHELLS
    for rbf, key in (("hydrogen", "h"), ("sphericalbessel", "b")):
        for ci, cut in enumerate(CUT):
            want = O.radial_basis(r[keep].cpu(), nl, RC, cut, rbf, A0).to(DEV)
            mine = ref["f"][keep, ci:ci + 1, 0] * ref["R_" + key][keep, :, 0]
            scale = mine.abs().max(0).values.clamp_min(1e-300)
            assert float(((mine - want).abs() / scale).max()) < 1e-12, (rbf, cut)


def test_geom_basis_fwd_without_edges():
    gi, opnds = _geom_operands(True)
    out = _geom_fwd(opnds, 0, _spec("hydrogen", "polynomial", 1), len(SHELLS))
    assert out["rb"].numel() == 0


# ---------------------------------------------------------------------------------------------- geometry backward
@functools.lru_cache(None)
def bwd_graph():
    """a hub with 320 in- and 310 out-edges (and a self-loop), self-loops elsewhere, isolated nodes (ids 0 and N - 1 among
    them), in 600 nodes"""
    g = torch.Generator().manual_seed(4)
    N = 600
    hub = 300
    src = torch.randint(1, N - 1, (4000,), generator=g)
    dst = torch.randint(1, N - 1, (4000,), generator=g)
    iso = torch.tensor([0, 17, 250, N - 1])
    ok = ~(torch.isin(src, iso) | torch.isin(dst, iso) | (src == hub) | (dst == hub))
    src, dst = src[ok], dst[ok]
    hi = torch.randint(1, N - 1, (320,), generator=g)
    ho = torch.randint(1, N - 1, (310,), generator=g)
    hi, ho = hi[~torch.isin(hi, iso) & (hi != hub)], ho[~torch.isin(ho, iso) & (ho != hub)]
    loops = torch.tensor([hub, 5, 6, 7])
    src = torch.cat([src, hi, torch.full_like(ho, hub), loops])
    dst = torch.cat([dst, torch.full_like(hi, hub), ho, loops])
    perm = torch.randperm(src.numel(), generator=g)
    return torch.stack([src[perm], dst[perm]]), N, hub, iso


def _dyadic(shape, g, lo, hi, den):
    return (torch.randint(lo, hi + 1, shape, generator=g, device=DEV).double() / den).float()


def _dvec64(dist, unit, drb, d_dist, d_unit, d_rb):
    """FP64 dvec = (d_unit - unit (unit . d_unit)) / dist + (d_dist + sum_o d_rb drb) unit, and its magnitude"""
    E = dist.shape[0]
    u, r = unit.double(), dist.double().view(E, 1)
    z = torch.zeros(E, 1, dtype=torch.float64, device=DEV)
    gr = (d_dist.double().view(E, 1) if d_dist is not None else z).clone()
    gm = gr.abs()
    if d_rb is not None:
        gr = gr + (d_rb.double() * drb.double()).sum(1, keepdim=True)
        gm = gm + (d_rb.double() * drb.double()).abs().sum(1, keepdim=True)
    ref, mag = gr * u, gm * u.abs()
    if d_unit is not None:
        a = d_unit.double()
        ref = ref + (a - u * (u * a).sum(1, keepdim=True)) / r
        mag = mag + (a.abs() + u.abs() * (u * a).abs().sum(1, keepdim=True)) / r
    return ref, mag


def _node_sum(dvec, ei, N):
    s, t = ei[0].to(DEV), ei[1].to(DEV)
    out = torch.zeros(N, 3, dtype=dvec.dtype, device=DEV)
    out.index_add_(0, t, dvec)
    out.index_add_(0, s, -dvec)
    return out


def _geom_bwd(gi, O_, dist, unit, drb, d_dist, d_unit, d_rb):
    E, N = gi.E, gi.N
    vb, dvec = _rows(E, 3)             # dvec scratch: NaN
    pb, d_pos = _rows(N, 3)
    with Launch() as n:
        ops._call("lcao_geom_basis_bwd", P_(dist), P_(unit), P_(drb), P_(d_dist), P_(d_unit), P_(d_rb), E, N, O_,
                  P_(gi.in_ptr), P_(gi.in_edge), P_(gi.out_ptr), P_(gi.out_edge), P_(dvec), P_(d_pos), ST())
    torch.cuda.synchronize()
    assert n.n == len(geom_bwd_kernels(E, N))
    _padding_untouched(vb, dvec, "dvec")
    _padding_untouched(pb, d_pos, "d_pos")
    return dvec, d_pos


# d_dist, d_unit, d_rb given (1) or NULL (0)
BWD_COMBOS = [(a, b, c) for a in (0, 1) for b in (0, 1) for c in (0, 1)]


@pytest.mark.parametrize("combo", BWD_COMBOS,
                         ids=[f"k_geom_edge_bwd+k_geom_node_bwd-d_dist{a}-d_unit{b}-d_rb{c}" for a, b, c in BWD_COMBOS])
def test_geom_basis_bwd(combo):
    """exact: dist a power of two and dyadic unit, drb and gradients -> dvec and d_pos equal the FP64 formula;
    random (the forward's outputs): dvec within gamma_{O+8} of its magnitude, d_pos within gamma_{O+8+deg}"""
    ei, N, hub, iso = bwd_graph()
    gi = ops.GraphIndex(ei.to(DEV), N)
    E, O_ = gi.E, len(SHELLS)
    deg = (torch.bincount(ei[0], minlength=N) + torch.bincount(ei[1], minlength=N)).to(DEV).double()
    for exact in (True, False):
        g = torch.Generator(device=DEV).manual_seed(sum(combo) + 10 * exact)
        if exact:
            # every partial sum is then a multiple of 2^-10 below 2^14 in magnitude (630 edges of at most 18 at the hub)
            dist = 2.0 ** torch.randint(-1, 2, (E,), generator=g, device=DEV).float()
            unit, drb = _dyadic((E, 3), g, -8, 8, 8), _dyadic((E, O_), g, -8, 8, 8)
            d_dist, d_unit, d_rb = _dyadic((E,), g, -8, 8, 8), _dyadic((E, 3), g, -8, 8, 8), _dyadic((E, O_), g, -8, 8, 8)
        else:
            fw = _geom_fwd(_bwd_geometry(ei, N), E, _spec("hydrogen", "envelope", 1), O_)
            dist, unit, drb = fw["dist"], fw["unit"], fw["drb"]
            d_dist, d_unit, d_rb = (torch.randn(s, generator=g, device=DEV) for s in ((E,), (E, 3), (E, O_)))
        ins = [_rows(x.shape[0], x[0].numel(), x) for x in (dist, unit, drb, d_dist, d_unit, d_rb)]
        dist, unit, drb, d_dist, d_unit, d_rb = (v.view(x.shape) for (_, v), x in zip(ins, (dist, unit, drb, d_dist, d_unit, d_rb)))
        before = [(b, b.clone()) for b, _ in ins]
        d_dist, d_unit, d_rb = (x if on else None for x, on in zip((d_dist, d_unit, d_rb), combo))
        dvec, d_pos = _geom_bwd(gi, O_, dist, unit, drb, d_dist, d_unit, d_rb)
        dvec2, d_pos2 = _geom_bwd(gi, O_, dist, unit, drb, d_dist, d_unit, d_rb)
        assert _same_bits(dvec, dvec2) and _same_bits(d_pos, d_pos2), "two identical calls differ"
        for b, c in before:
            assert _same_bits(b, c), "an input buffer (operand or padding) was written"
        ref, mag = _dvec64(dist, unit, drb, d_dist, d_unit, d_rb)
        pref, pmag = _node_sum(ref, ei, N), _abs_node_sum(mag, ei, N)
        assert bool((d_pos[iso.to(DEV)] == 0).all()), "isolated nodes: d_pos not exactly 0"
        if exact:
            _exact("exact dvec", dvec, ref)
            _exact("exact d_pos", d_pos, pref)
        else:
            _check("dvec", "random dvec", dvec, ref, mag, gamma(O_ + 8))
            _check("d_pos", "random d_pos", d_pos, pref, pmag, gamma(O_ + 8 + deg).view(N, 1))
            if combo == (1, 1, 1):
                # the bound singles out one out-edge of the hub (310 out-edges, 320 in-edges)
                e = int(torch.nonzero((ei[0] == hub) & (ei[1] != hub))[0])
                ok, _, _ = _within(d_pos[hub], pref[hub] + ref[e], pmag[hub] - mag[e], gamma(O_ + 8 + deg[hub]))
                assert not ok, "the d_pos bound accepts the hub's sum without one of its out-edges"


def _abs_node_sum(mag, ei, N):
    s, t = ei[0].to(DEV), ei[1].to(DEV)
    out = torch.zeros(N, 3, dtype=torch.float64, device=DEV)
    out.index_add_(0, t, mag)
    out.index_add_(0, s, mag)
    return out


@functools.lru_cache(None)
def _bwd_positions(N):
    g = torch.Generator().manual_seed(8)
    return (torch.rand(N, 3, generator=g) * 9.0).to(DEV)


def _bwd_geometry(ei, N):
    """padded forward operands for the backward graph: random positions in a 9 A box, no periodic shift, one graph"""
    gi = ops.GraphIndex(ei.to(DEV), N)
    E = gi.E
    pos = _bwd_positions(N)
    shift = torch.zeros(E, 3, device=DEV)
    shift[(ei[0] == ei[1]).to(DEV), 0] = 1.0   # a self-loop is a self-image edge one lattice vector away (r = 0 is out of scope)
    lat = torch.diag(torch.tensor([3.1, 4.0, 4.5])).reshape(1, 9).to(DEV)
    return dict(pos=_rows(N, 3, pos), shift=_rows(E, 3, shift), lattice=_rows(1, 9, lat), batch=(None, None),
                src=_irows(E, gi.src32, torch.int32), dst=_irows(E, gi.dst32, torch.int32))


def test_geom_basis_bwd_without_edges():
    """E = 0 with N > 0: only the node stage runs, and it writes zeros over the NaN-filled d_pos"""
    ei = torch.zeros(2, 0, dtype=torch.long)
    gi = ops.GraphIndex(ei.to(DEV), 50)
    _, d_pos = _geom_bwd(gi, 4, None, None, None, None, None, None)
    assert bool((d_pos == 0).all())


@pytest.mark.parametrize("rbf,cut", [("hydrogen", "polynomial"), ("sphericalbessel", "cosine")])
def test_geom_basis_bwd_vs_autograd(rbf, cut):
    """forward + backward of the kernels against torch.autograd of the FP64 oracle (edge_geometry + radial_basis)"""
    ei, N, _, _ = bwd_graph()
    gi = ops.GraphIndex(ei.to(DEV), N)
    E, n_u = gi.E, len(SHELLS)
    op = _bwd_geometry(ei, N)
    fw = _geom_fwd(op, E, _spec(rbf, cut, 1), n_u)
    g = torch.Generator(device=DEV).manual_seed(2)
    d_dist, d_unit, d_rb = (torch.randn(s, generator=g, device=DEV) for s in ((E,), (E, 3), (E, n_u)))
    dvec, d_pos = _geom_bwd(gi, n_u, fw["dist"], fw["unit"], fw["drb"], d_dist, d_unit, d_rb)

    pos = op["pos"][1].double().clone().requires_grad_(True)
    lat = op["lattice"][1].view(1, 3, 3).double()
    dist, unit = O.edge_geometry(pos, ei.to(DEV), op["shift"][1].double(), lat, None)
    rb = O.radial_basis(dist, SHELLS, RC, cut, rbf, A0)
    loss = (dist * d_dist.double()).sum() + (unit * d_unit.double()).sum() + (rb * d_rb.double()).sum()
    (want,) = torch.autograd.grad(loss, [pos])
    drb64 = torch.autograd.functional.jacobian(lambda r: O.radial_basis(r, SHELLS, RC, cut, rbf, A0).sum(0),
                                               dist.detach(), vectorize=True).t()
    _, mag = _dvec64(dist.detach(), unit.detach(), drb64, d_dist, d_unit, d_rb)
    pmag = _abs_node_sum(mag, ei, N)
    deg = (torch.bincount(ei[0], minlength=N) + torch.bincount(ei[1], minlength=N)).to(DEV).double()
    # the kernel's own bound plus the FP32 rounding of its inputs dist, unit and drb (4 more)
    _check("d_pos vs autograd", "d_pos vs autograd", d_pos, want, pmag, gamma(n_u + 8 + 4 + deg).view(N, 1))


# ---------------------------------------------------------------------------------------------- coverage of the table
def _reached():
    ks = {k for c in PAIR_CASES for k in _pair_case_kernels(c)}
    ks |= {k for c in COEFF_CASES for k in coeff_kernels(c[0], c[1])}
    ks |= {"k_geom_basis_fwd"} | set(geom_bwd_kernels(1, 1))
    return ks


def test_cases_reach_every_edge_basis_kernel():
    reached = _reached()
    assert reached == ALL_KERNELS and len(ALL_KERNELS) == 35, ALL_KERNELS ^ reached
    # the forward's grid cap and the stage-1 shared-memory opt-in: cases on both sides, with and without valence
    Es = {_keys(c[4])[0].numel() for c in PAIR_CASES}
    assert any(fwd_grid_strides(E) for E in Es) and any(0 < E <= FWD_CAP for E in Es)
    assert (partial_smem(47, 0), partial_smem(48, 0), partial_smem(23, 1), partial_smem(24, 1)) == (49152, 50176, 48128, 50176)
    tab_cases = [c for c in PAIR_CASES if "tab" in c[7] and _keys(c[4])[0].numel() > 0]
    for val in (0, 1):
        sides = {partial_smem(c[3], val) > SMEM_OPT_IN for c in tab_cases if c[1] == val}
        assert sides == {False, True}, val
    assert any(c[1] and c[3] == 64 for c in tab_cases)
    # C at the sorted walk's boundary and past it; every O of the 8-orbital tails; the E of the 16-edge runs
    assert {c[2] for c in PAIR_CASES} == {4, 12, 124, 128, 132, 256, 260}
    assert {c[3] for c in PAIR_CASES} >= {1, 5, 8, 9, 23, 24, 47, 48, 64}
    assert {_keys(c[4])[0].numel() for c in PAIR_CASES} >= {0, 1, 7, 15}
    assert {c[5] for c in PAIR_CASES} == {"ordered", "grouped", "shuffled"}
    assert {_keys(c[4])[1] for c in PAIR_CASES} >= {1, 9, 1369, 5000}


def _cuobjdump():
    exe = shutil.which("cuobjdump")
    if exe is None:
        home = os.environ.get("CUDA_HOME", os.environ.get("CUDA_PATH", "/usr/local/cuda"))
        exe = os.path.join(home, "bin", "cuobjdump")
    return exe if os.path.exists(exe) else None


def test_kernel_list_matches_the_library():
    """the restated dispatch lists every kernel of these eleven base names that the library contains"""
    exe = _cuobjdump()
    if exe is None:
        pytest.skip("cuobjdump not available")
    text = subprocess.run([exe, "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    found = set()
    pat = "|".join(sorted(BASE_NAMES, key=len, reverse=True))
    for name, args in re.findall(r"(" + pat + r")(?:I((?:L[ib]\d+E)+)E|(?=E))", text):
        vals = [("true" if v == "1" else "false") if t == "b" else v for t, v in re.findall(r"L([ib])(\d+)E", args)]
        found.add(f"{name}<{','.join(vals)}>" if vals else name)
    assert found == ALL_KERNELS, found ^ ALL_KERNELS
