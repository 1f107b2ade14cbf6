"""torch.autograd Functions over the C ABI (include/lcao_b200.h).


PyTorch is used for device memory, the current stream and autograd bookkeeping only: every
edge-sized operation of the hot path (forward and backward) is a call into liblcao_b200.so.
All functions require CUDA tensors and raise `LcaoError` otherwise — there is no CPU fallback.
"""
from __future__ import annotations

import ctypes

import torch
from torch import Tensor
from torch.autograd.function import once_differentiable

from . import _lib, second_order
from ._lib import ACT_NONE, ACT_SILU, LcaoError, call, ptr, require_cuda, stream_ptr

# GEMM arithmetic mode for the dense layers: fp32 CUDA cores, 3xTF32 tcgen05 (fp32-equivalent), 1xTF32
GEMM_MODES = {"fp32": _lib.GEMM_FP32, "tf32x3": _lib.GEMM_TF32X3, "tf32": _lib.GEMM_TF32}
# The default is the tcgen05 path in its FP32-equivalent arithmetic (3xTF32 operand split, FP32 accumulation in TMEM):
# it is the mode the parity tests and the benchmark run.  "fp32" selects the CUDA-core kernels (gemm_simt.cu).
_gemm_mode = _lib.GEMM_TF32X3

# launch counter: every C-ABI compute call increments it (bench.py reports it as gpu_launches)
n_calls = 0


def set_gemm_mode(mode: str) -> None:
    global _gemm_mode
    _gemm_mode = GEMM_MODES[mode]


def get_gemm_mode() -> str:
    return {v: k for k, v in GEMM_MODES.items()}[_gemm_mode]


class positions_only:
    """Context for `torch.autograd.grad(energy, pos)` (autograd forces, reference lcaonet.py:310-317): inside it the
    backward kernels skip every PARAMETER gradient — the engine would discard them anyway — and never touch the
    in-place gradient sinks, which belong to the loss's own backward pass.  A plain module-level flag: autograd runs
    CUDA backward nodes on its device thread, so a thread-local would not be seen there."""
    active = False

    def __enter__(self):
        self._prev = positions_only.active
        positions_only.active = True

    def __exit__(self, *exc):
        positions_only.active = self._prev
        return False


def validate_graph(z: Tensor, max_z: int, batch: Tensor | None, n_graph: int, edge_index: Tensor) -> None:
    """Raise IndexError when z, batch or edge_index would index out of range (the reference raises the same from
    nn.Embedding / index_select: embed.py:41,91, base.py:38, lcaonet.py:462).  One small kernel + one host sync."""
    require_cuda(z, edge_index)
    if edge_index.dtype != torch.int64 or edge_index.dim() != 2 or edge_index.shape[0] != 2:
        raise ValueError("edge_index must be an int64 tensor of shape (2, E)")
    if z.dtype != torch.int64 or (batch is not None and batch.dtype != torch.int64):
        raise ValueError("z and batch must be int64 tensors")
    status = torch.empty(1, dtype=torch.int32, device=z.device)
    ei = edge_index.contiguous()
    _call("lcao_validate_graph", ptr(z.contiguous()), z.numel(), int(max_z), ptr(batch.contiguous() if batch is not None else None),
          int(n_graph), ptr(ei), ei.shape[1], ptr(status), stream_ptr())
    bad = int(status.item())
    if bad:
        what = [m for b, m in ((1, f"atomic numbers outside [1, {max_z}]"), (2, f"batch indices outside [0, {n_graph})"),
                               (4, f"edge_index entries outside [0, {z.numel()})")) if bad & b]
        raise IndexError("index out of range in the input batch: " + "; ".join(what))


def _call(name, *args):
    global n_calls
    n_calls += 1
    call(name, *args)


def _rows(x: Tensor, packed: bool = False) -> Tensor:
    """2-D view with unit inner stride and rows that do not overlap (`packed`: no gap between them either); copies only
    if needed.  The launch helpers pass `stride(0)` as the leading dimension, so a single row, whose stride torch leaves
    as it finds it (0 for an expanded gradient), gets the width instead."""
    if x.dim() != 2:
        x = x.reshape(-1, x.shape[-1])
    if packed or x.stride(1) != 1 or (x.shape[0] > 1 and x.stride(0) < x.shape[1]):
        x = x.contiguous()
    if x.shape[0] <= 1 and x.stride(0) != max(x.shape[1], 1):
        x = x.as_strided(x.shape, (max(x.shape[1], 1), 1))
    return x


# ------------------------------------------------------------------------------------------------
# graph indices
# ------------------------------------------------------------------------------------------------
class GraphIndex:
    """int32 CSR views of `edge_index` built on the GPU (bit-exact, deterministic):
    in-CSR by target (ordered by source, then edge id), out-CSR by source, triplet offsets.
    Replaces torch_sparse.SparseTensor in `LCAONet.get_triplets` (reference lcaonet.py:439-486)."""

    def __init__(self, edge_index: Tensor, n_nodes: int):
        require_cuda(edge_index)
        if edge_index.dtype != torch.int64 or edge_index.dim() != 2 or edge_index.shape[0] != 2:
            raise ValueError("edge_index must be an int64 tensor of shape (2, E)")
        ei = edge_index.contiguous()
        E, N, dev = ei.shape[1], int(n_nodes), ei.device
        self.E, self.N, self.edge_index = E, N, ei
        i32 = dict(dtype=torch.int32, device=dev)
        self.src32, self.dst32 = torch.empty(E, **i32), torch.empty(E, **i32)
        self.in_ptr, self.out_ptr = torch.empty(N + 1, **i32), torch.empty(N + 1, **i32)
        self.in_edge, self.in_src, self.out_edge = torch.empty(E, **i32), torch.empty(E, **i32), torch.empty(E, **i32)
        self._tri_ptr = None  # triplet offsets: only the reference's triplet LISTS need them -> built on demand
        scratch = torch.empty(2 * N + 2 * E + 8, **i32)
        _call("lcao_graph_index_build", ptr(ei), E, N, ptr(self.src32), ptr(self.dst32), ptr(self.in_ptr),
              ptr(self.in_edge), ptr(self.in_src), ptr(self.out_ptr), ptr(self.out_edge), None, ptr(scratch), stream_ptr())

    @property
    def tri_ptr(self) -> Tensor:
        if self._tri_ptr is None:
            i32 = dict(dtype=torch.int32, device=self.src32.device)
            self._tri_ptr = torch.empty(self.E + 1, **i32)
            scratch = torch.empty(self.E + self.E // 4096 + 2, **i32)
            _call("lcao_triplet_offsets", ptr(self.src32), ptr(self.dst32), ptr(self.in_ptr), self.E, ptr(self._tri_ptr),
                  ptr(scratch), stream_ptr())
        return self._tri_ptr

    def num_triplets(self) -> int:
        return int(self.tri_ptr[-1].item())  # host sync: T is data dependent

    def triplets(self, unit: Tensor | None = None):
        """(tri_idx_k, edge_idx_ks, edge_idx_st[, cos]) int64 lists in the reference's order."""
        T, dev = self.num_triplets(), self.src32.device
        k, e_ks, e_st = (torch.empty(T, dtype=torch.int64, device=dev) for _ in range(3))
        cos = torch.empty(T, dtype=torch.float32, device=dev) if unit is not None else None
        _call("lcao_triplets_fill", ptr(self.src32), ptr(self.in_ptr), ptr(self.in_edge), ptr(self.tri_ptr), self.E,
              ptr(k), ptr(e_ks), ptr(e_st), ptr(unit), ptr(cos), stream_ptr())
        return (k, e_ks, e_st) if unit is None else (k, e_ks, e_st, cos)


def bucket_sort(keys: Tensor, n_buckets: int, sec: Tensor | None = None, stable: bool | str = True):
    """(ptr int32 (nb+1), perm int32 (n)): items grouped by key; stable=True orders each bucket by
    (sec, id) (small buckets only), stable="ordered" lists the items of a bucket in ascending id (few huge buckets:
    species / species-pair keys; reproducible), stable=False just groups (order inside a bucket unspecified)."""
    require_cuda(keys)
    keys = keys.contiguous()
    n, dev = keys.numel(), keys.device
    p = torch.empty(n_buckets + 1, dtype=torch.int32, device=dev)
    perm = torch.empty(n, dtype=torch.int32, device=dev)
    mode = 2 if stable == "ordered" else (1 if stable else 0)
    scratch = torch.empty(n_buckets + n + 1 + (n_buckets * ((n + 1023) // 1024) if mode == 2 else 0), dtype=torch.int32, device=dev)
    _call("lcao_bucket_sort", ptr(keys), ptr(sec.contiguous() if sec is not None else None), n, n_buckets, ptr(p),
          ptr(perm), ptr(scratch), mode, stream_ptr())
    return p, perm


def histogram(keys: Tensor, n_buckets: int) -> Tensor:
    require_cuda(keys)
    out = torch.empty(n_buckets, dtype=torch.float32, device=keys.device)
    _call("lcao_histogram", ptr(keys.contiguous()), keys.numel(), n_buckets, ptr(out), stream_ptr())
    return out


# ------------------------------------------------------------------------------------------------
# geometry + radial basis
# ------------------------------------------------------------------------------------------------
class _GeomBasis(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pos, shift, lattice, batch, gi: GraphIndex, spec, n_orb: int, strain=None, seg=None, atom_strain=None):
        require_cuda(pos, shift, lattice)
        pos_c, shift_c, lat_c = pos.contiguous().float(), shift.contiguous().float(), lattice.contiguous().float()
        E, dev = gi.E, pos.device
        dist = torch.empty(E, device=dev)
        unit = torch.empty(E, 3, device=dev)
        rb = torch.empty(E, n_orb, device=dev)
        ni = ctx.needs_input_grad
        need_grad = ni[0] or ni[2] or ni[7] or ni[9]
        drb = torch.empty(E, n_orb, device=dev) if need_grad else None
        _call("lcao_geom_basis_fwd", ptr(pos_c), ptr(shift_c), ptr(lat_c), ptr(batch), ptr(gi.src32), ptr(gi.dst32), E,
              ctypes.byref(spec), ptr(dist), ptr(unit), ptr(rb), ptr(drb), stream_ptr())
        ctx.gi, ctx.n_orb, ctx.spec, ctx.seg = gi, n_orb, spec, seg
        ctx.save_for_backward(dist, unit, drb, pos, shift, lattice, batch, strain, atom_strain)
        return dist, unit, rb

    @staticmethod
    def backward(ctx, d_dist, d_unit, d_rb):
        dist, unit, drb, pos, shift, lattice, batch, strain, atom_strain = ctx.saved_tensors
        gi = ctx.gi
        if drb is None:
            return (None,) * 10
        ni = ctx.needs_input_grad
        if torch.is_grad_enabled():  # create_graph=True: this backward is itself differentiated (training on autograd forces)
            with torch.enable_grad():
                pos_, lat_, strain_, astrain_ = second_order.aliases([pos, lattice, strain, atom_strain])
                outs = second_order.geom_basis(pos_, shift, lat_, batch, gi.src32, gi.dst32, ctx.spec, ctx.n_orb, strain_,
                                               astrain_)
                d_pos, d_lat, d_strain, d_astrain = second_order.grads_with_graph(
                    outs, [pos_, lat_, strain_, astrain_], [d_dist, d_unit, d_rb], [ni[0], ni[2], ni[7], ni[9]])
            return d_pos, None, d_lat, None, None, None, None, d_strain, None, d_astrain
        dev = dist.device
        dvec = torch.empty(gi.E, 3, device=dev)
        d_pos = torch.empty(gi.N, 3, device=dev)
        c = lambda t: t.contiguous() if t is not None else None  # noqa: E731
        d_dist, d_unit, d_rb = c(d_dist), c(d_unit), c(d_rb)
        _call("lcao_geom_basis_bwd", ptr(dist), ptr(unit), ptr(drb), ptr(d_dist), ptr(d_unit), ptr(d_rb), gi.E, gi.N,
              ctx.n_orb, ptr(gi.in_ptr), ptr(gi.in_edge), ptr(gi.out_ptr), ptr(gi.out_edge), ptr(dvec), ptr(d_pos),
              stream_ptr())
        d_lat = d_strain = d_astrain = None
        if ni[2] or ni[7]:
            d_lat, d_strain = _cell_grads(dvec, pos, shift, lattice, batch, gi, ctx.seg, ni[2], ni[7])
        if ni[9]:
            d_astrain = _atom_virial(dvec, pos, shift, lattice, batch, gi)
        return d_pos if ni[0] else None, None, d_lat, None, None, None, None, d_strain, None, d_astrain


def _cell_grads(dvec, pos, shift, lattice, batch, gi, seg, want_lattice: bool, want_virial: bool):
    """(d E / d lattice, virial) per graph from dvec = d E / d vec (lcao_geom_cell_bwd); None where not wanted.
    `seg` = (seg_ptr, seg_perm) groups the nodes by graph; built from `batch` here when the caller has none."""
    dev = dvec.device
    if seg is None:
        seg = (torch.tensor([0, gi.N], dtype=torch.int32, device=dev), None) if batch is None else \
            bucket_sort(batch, lattice.shape[0])
    seg_ptr, seg_perm = seg[0], seg[1]
    B = seg_ptr.numel() - 1
    d_lat = torch.empty(B, 3, 3, device=dev) if want_lattice else None
    virial = torch.empty(B, 3, 3, device=dev) if want_virial else None
    scratch = torch.empty((gi.N // _lib.CELL_CHUNK + B) * 18, dtype=torch.float64, device=dev)
    pos_c, shift_c, lat_c = pos.contiguous().float(), shift.contiguous().float(), lattice.contiguous().float()
    _call("lcao_geom_cell_bwd", ptr(pos_c), ptr(shift_c), ptr(lat_c), ptr(batch), ptr(gi.dst32), ptr(dvec), gi.E, gi.N,
          ptr(gi.out_ptr), ptr(gi.out_edge), ptr(seg_ptr), ptr(seg_perm), B, ptr(scratch), ptr(d_lat), ptr(virial),
          stream_ptr())
    if d_lat is not None:
        if lattice.shape[0] > B:  # batch=None: the forward reads lattice[0] only
            d_lat = torch.cat([d_lat, d_lat.new_zeros(lattice.shape[0] - B, 3, 3)])
        d_lat = d_lat.to(lattice.dtype)
    return d_lat, virial


def _atom_virial(dvec, pos, shift, lattice, batch, gi):
    """(N,3,3) per-atom virials W_i = 1/2 sum of vec_e (x) dvec_e over the edges with s_e = i and over those with t_e = i,
    from dvec = d E / d vec (lcao_geom_atom_virial_bwd)."""
    out = torch.empty(gi.N, 3, 3, device=dvec.device)
    pos_c, shift_c, lat_c = pos.contiguous().float(), shift.contiguous().float(), lattice.contiguous().float()
    _call("lcao_geom_atom_virial_bwd", ptr(pos_c), ptr(shift_c), ptr(lat_c), ptr(batch), ptr(gi.dst32), ptr(gi.in_ptr),
          ptr(gi.in_edge), ptr(gi.in_src), ptr(gi.out_ptr), ptr(gi.out_edge), ptr(dvec), gi.E, gi.N, ptr(out), stream_ptr())
    return out


def geom_basis(pos, shift, lattice, batch, gi, spec, n_orb, strain=None, seg=None, atom_strain=None):
    """(dist, unit, rb) of every edge, vec_e = pos[t] - pos[s] + shift_e . lattice[batch[s]] (row vectors, base.py:27-43).
    Differentiable with respect to `pos` and `lattice` (d E / d L_g[i][j] = sum_{e in g} shift_e[i] dvec_e[j]); the
    gradient with respect to `shift` is not computed (None).
    `strain` (internal, not public API: LCAONet.regress_stress creates it) is a (B,3,3) gradient probe: zeros with
    requires_grad whose value the forward never reads, standing for eps_g in pos' = pos (I + eps), L' = L (I + eps).  Its
    gradient is the virial W_g = sum_{e in g} vec_e (x) dvec_e.  `seg` = (seg_ptr, seg_perm), the nodes grouped by
    graph (optional: built from `batch` when a cell gradient is wanted and it is missing).
    `atom_strain` (internal, like `strain`: LCAONet.regress_atom_virial creates it) is an (N,3,3) probe eps_i acting on the
    edges as vec_e -> vec_e + 1/2 vec_e (eps_s + eps_t).  Its gradient is the per-atom virial
    W_i = 1/2 sum_{e: s_e = i} vec_e (x) dvec_e + 1/2 sum_{e: t_e = i} vec_e (x) dvec_e."""
    return _GeomBasis.apply(pos, shift, lattice, batch, gi, spec, n_orb, strain, seg, atom_strain)


# ------------------------------------------------------------------------------------------------
# dense layers
# ------------------------------------------------------------------------------------------------
# Every C-ABI entry point is launched from one place: its only user, or a launch helper (`_lin_*`, `_act_bwd`,
# `_pair_contract_*`, ...) shared by the op-level Functions and `_InteractionLayer`.  A helper allocates the outputs its
# caller does not pass, spells the argument list and sizes the scratch.  Matrices are 2-D tensors with unit inner stride,
# strided views included; their `stride(0)` is the leading dimension.  `st` is the raw CUDA stream.
def _lin_fwd(x, w, bias, st, act=ACT_NONE, need_pre=False):
    """(y, pre): y = act(x W^T + b), and its pre-activation when `need_pre` and there is an activation (else None)."""
    M, (Nout, K) = x.shape[0], w.shape
    y = torch.empty(M, Nout, device=w.device)
    pre = torch.empty(M, Nout, device=w.device) if (need_pre and act != ACT_NONE) else None
    _call("lcao_linear_fwd", ptr(x), x.stride(0), ptr(w), ptr(bias), ptr(y), Nout, ptr(pre), Nout, M, K, Nout, act,
          _gemm_mode, st)
    return y, pre


def _lin_dgrad(dy, w, st, dx=None, accumulate=0):
    """dx = dy W (dx += dy W with `accumulate`); dx is allocated unless the caller passes it."""
    M, (Nout, K) = dy.shape[0], w.shape
    if dx is None:
        dx = torch.empty(M, K, device=w.device)
    _call("lcao_linear_dgrad", ptr(dy), dy.stride(0), None, 0, ACT_NONE, ptr(w), ptr(dx), dx.stride(0), M, K, Nout,
          accumulate, _gemm_mode, None, st)
    return dx


def _lin_dgrad_act(dy, w, pre_in, act, st):
    """dx = (dy W) * act'(pre_in): data gradient chained through the activation that produced the layer's input."""
    M, (Nout, K) = dy.shape[0], w.shape
    dx = torch.empty(M, K, device=w.device)
    _call("lcao_linear_dgrad_act", ptr(dy), dy.stride(0), ptr(w), ptr(pre_in), pre_in.stride(0), act, ptr(dx), K, M, K,
          Nout, _gemm_mode, st)
    return dx


# Weight gradients that go straight into the parameters' .grad buffers (gradient sinks) are only read by the optimizer /
# the all-reduce, so the second stage of the tcgen05 weight-gradient kernel (the sum of its per-CTA partial tiles) is
# deferred: the descriptors pile up here and ONE batched launch at the end of the backward pass (an autograd engine
# callback) finishes them all.
_pending_wgrad = {"desc": [], "keep": [], "queued": False, "stream": None}


def flush_wgrad():
    """Finish the deferred weight gradients (runs by itself at the end of every backward pass that deferred any)."""
    p = _pending_wgrad
    p["queued"] = False
    if p["desc"]:
        arr = (ctypes.c_int64 * len(p["desc"]))(*p["desc"])
        _call("lcao_wgrad_reduce_batch", arr, len(p["desc"]) // 6, p["stream"])
    p["desc"], p["keep"], p["stream"] = [], [], None


def _lin_wgrad(dy, x, w, has_bias, st, dw_sink=None, db_sink=None):
    """dW (+ db) of one layer.  With sinks (the parameters' .grad buffers) the kernels accumulate straight into them
    — the C ABI's `dW +=` contract — and (None, None) is returned: no zero-fill, no separate accumulation pass."""
    M, (Nout, K), ldy, ldx = dy.shape[0], w.shape, dy.stride(0), x.stride(0)
    dw = dw_sink if dw_sink is not None else torch.zeros(Nout, K, device=w.device)
    db = (db_sink if db_sink is not None else torch.zeros(Nout, device=w.device)) if has_bias else None
    n_scr = int(_lib.load().lcao_linear_bwd_scratch(ptr(dy), ldy, None, 0, ACT_NONE, None, ptr(x), ldx, None, 0, M, K, Nout,
                                                    _gemm_mode))
    if dw_sink is not None and (db_sink is not None or not has_bias) and n_scr:
        passes = (Nout + 127) // 128
        scr = torch.empty(n_scr * passes, device=w.device)
        desc, nd = (ctypes.c_int64 * (6 * passes))(), ctypes.c_int32(0)
        _call("lcao_linear_wgrad_deferred", ptr(dy), ldy, ptr(x), ldx, ptr(dw), ptr(db), M, K, Nout, _gemm_mode, ptr(scr),
              desc, ctypes.byref(nd), st)
        if nd.value:
            p = _pending_wgrad
            p["desc"].extend(desc[: 6 * nd.value])
            p["keep"].append((scr, dw, db))  # the partial tiles and their targets stay alive until the flush
            p["stream"] = st
            if not p["queued"]:
                torch.autograd.Variable._execution_engine.queue_callback(flush_wgrad)
                p["queued"] = True
        return None, None
    scr = torch.empty(n_scr, device=w.device) if n_scr else None
    _call("lcao_linear_wgrad", ptr(dy), ldy, None, 0, ACT_NONE, ptr(x), ldx, ptr(dw), ptr(db), M, K, Nout, _gemm_mode,
          ptr(scr), st)
    return (None if dw_sink is not None else dw), (None if (db_sink is not None or not has_bias) else db)


def _act_bwd(dy, pre, act, st):
    """dH = dY * act'(pre)"""
    M, C = dy.shape
    out = torch.empty(M, C, device=dy.device)
    _call("lcao_act_bwd", ptr(dy), dy.stride(0), ptr(pre), pre.stride(0), ptr(out), C, M, C, act, st)
    return out


class _Linear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, act: int):
        require_cuda(x, weight)
        shape = x.shape
        x2 = _rows(x)
        w = weight.contiguous()
        y, pre = _lin_fwd(x2, w, bias, stream_ptr(), act, any(ctx.needs_input_grad))
        ctx.act, ctx.shape, ctx.has_bias = act, shape, bias is not None
        ctx.save_for_backward(x2, w, pre, x, weight, bias)
        return y.reshape(*shape[:-1], w.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, w, pre, x_in, w_in, b_in = ctx.saved_tensors
        if torch.is_grad_enabled():  # create_graph=True (see second_order.py)
            with torch.enable_grad():
                ins = second_order.aliases([x_in, w_in, b_in])
                y = second_order.linear(*ins, ctx.act)
                wanted = list(ctx.needs_input_grad[:3])
                if positions_only.active:
                    wanted[1] = wanted[2] = False
                gx, gw, gb = second_order.grads_with_graph([y], ins, [dy], wanted)
            return gx, gw, gb, None
        dy2 = _rows(dy)
        st = stream_ptr()
        need_dx = ctx.needs_input_grad[0]
        need_dw = (ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2])) and not positions_only.active
        if ctx.act != ACT_NONE:  # dH = dY * act'(pre), shared by the data and the weight gradient
            dy2 = _act_bwd(dy2, pre, ctx.act, st)
        dx = _lin_dgrad(dy2, w, st).reshape(ctx.shape) if need_dx else None
        dw, db = _lin_wgrad(dy2, x2, w, ctx.has_bias, st) if need_dw else (None, None)
        return dx, dw, db, None


def _act_arg(act) -> int:
    """activation argument of the public ops: an LCAO_ACT_* code, or True / False for SiLU / none"""
    return ACT_SILU if act is True else ACT_NONE if act is False or act is None else int(act)


def linear(x: Tensor, weight: Tensor, bias: Tensor | None = None, silu=False) -> Tensor:
    """act(x W^T + b) — nn.Linear semantics (reference nn/base.py:72-81) with an optional fused SiLU.
    Requires the feature sizes to be multiples of 4 only for the vector paths; any size works."""
    return _Linear.apply(x, weight, bias, _act_arg(silu))


# ------------------------------------------------------------------------------------------------
# orbital contraction, three-body, two-body
# ------------------------------------------------------------------------------------------------
class _CoeffContract(torch.autograd.Function):
    @staticmethod
    def forward(ctx, cst1, rb, vmask, lgrp, NL: int, C: int):
        require_cuda(cst1, rb)
        cst1 = cst1.contiguous()
        E, O, Cp = cst1.shape
        valence = 1 if vmask is not None else 0
        assert Cp == C * (1 + valence)
        NG = NL + valence
        B = torch.empty(E, NG, C, device=cst1.device)
        _call("lcao_coeff_contract_fwd", ptr(cst1), ptr(rb), ptr(vmask), ptr(lgrp), E, O, C, NL, valence, ptr(B),
              stream_ptr())
        ctx.dims = (E, O, C, NL, valence)
        ctx.save_for_backward(cst1, rb, vmask, lgrp)
        return B

    @staticmethod
    @once_differentiable
    def backward(ctx, dB):
        cst1, rb, vmask, lgrp = ctx.saved_tensors
        E, O, C, NL, valence = ctx.dims
        dB = dB.contiguous()
        d_cst1 = torch.empty_like(cst1)
        d_rb = torch.empty_like(rb) if ctx.needs_input_grad[1] else None
        _call("lcao_coeff_contract_bwd", ptr(cst1), ptr(rb), ptr(vmask), ptr(lgrp), ptr(dB), E, O, C, NL, valence,
              ptr(d_cst1), ptr(d_rb), stream_ptr())
        return d_cst1, d_rb, None, None, None, None


def coeff_contract(cst1, rb, vmask, lgrp, NL, C):
    """B[e,l,:] = sum_{o in l} rb[e,o] (A[e,o,:] + m V[e,o,:]) (+ valence slot) — the orbital sums of
    lcaonet.py:180-183 and :200-203, grouped by angular momentum so both consumers share them."""
    return _CoeffContract.apply(cst1, rb.contiguous(), vmask, lgrp, NL, C)


def _pair_contract_fwd(tab, pair, rb, vmask, lgrp, NL, C, st, with_psum=False):
    """(B, gram, psum) from the (P, O, C') table: psum = [sum_l B_l | valence slot] only `with_psum` (else None)."""
    E, O, dev = pair.numel(), tab.shape[1], tab.device
    valence = 1 if vmask is not None else 0
    B = torch.empty(E, NL + valence, C, device=dev)
    gram = torch.empty(E, NL * (NL + 1) // 2, dtype=torch.float64, device=dev)
    psum = torch.empty(E, 1 + valence, C, device=dev) if with_psum else None
    _call("lcao_pair_contract_fwd", ptr(tab), ptr(pair), ptr(rb), ptr(vmask), ptr(lgrp), E, O, C, NL, valence, ptr(B),
          ptr(gram), ptr(psum), st)
    return B, gram, psum


def _pair_contract_bwd(tab, pair, grouping, rb, vmask, lgrp, dB, NL, C, need_tab, need_rb, st):
    """(d tab, d rb) of B = pair_contract(tab, rb), None where not needed."""
    (P, O, _), E = tab.shape, pair.numel()
    valence = 1 if vmask is not None else 0
    d_tab = torch.empty_like(tab) if need_tab else None
    d_rb = torch.empty(E, O, device=tab.device) if need_rb else None
    if need_tab or (need_rb and E > 0):  # (an edge-less batch has no d rb to write)
        kptr, kperm = _grouping(grouping, pair, P)
        scratch = None
        if need_tab:
            nbytes = int(_lib.load().lcao_pair_contract_bwd_scratch(E, P, O, C, valence))
            scratch = torch.empty((nbytes + 15) // 16 * 4, dtype=torch.int32, device=tab.device)
        _call("lcao_pair_contract_bwd", ptr(tab), ptr(pair), ptr(kptr), ptr(kperm), ptr(rb), ptr(vmask), ptr(lgrp), ptr(dB),
              E, P, O, C, NL, valence, ptr(d_tab), ptr(d_rb), ptr(scratch), st)
    return d_tab, d_rb


class _PairContract(torch.autograd.Function):
    """B and its Gram matrices from the species-pair coefficient table (see lcao_pair_contract_fwd)."""

    @staticmethod
    def forward(ctx, tab, pair, grouping, rb, vmask, lgrp, NL: int, C: int):
        require_cuda(tab, pair, rb)
        tab = tab.contiguous()
        assert tab.shape[2] == C * (1 + (vmask is not None)) and pair.dtype == torch.int64
        B, gram, _ = _pair_contract_fwd(tab, pair, rb, vmask, lgrp, NL, C, stream_ptr())
        ctx.NL, ctx.C, ctx.grouping = NL, C, grouping
        ctx.save_for_backward(tab, pair, rb, vmask, lgrp)
        ctx.mark_non_differentiable(gram)
        return B, gram

    @staticmethod
    @once_differentiable
    def backward(ctx, dB, _dgram):
        tab, pair, rb, vmask, lgrp = ctx.saved_tensors
        d_tab, d_rb = _pair_contract_bwd(tab, pair, ctx.grouping, rb, vmask, lgrp, dB.contiguous(), ctx.NL, ctx.C, True,
                                         ctx.needs_input_grad[3], stream_ptr())
        return d_tab, None, None, d_rb, None, None, None, None


def _grouping(grouping, pair, P):
    """(kptr, kperm) from whatever the caller supplied: a callable that builds them on demand (PairCoeffs.grouping), a
    ready (kptr, kperm) tuple, or None (built here)."""
    if callable(grouping):
        return grouping()
    if grouping is not None and grouping[0] is not None:
        return grouping
    with torch.no_grad():
        return bucket_sort(pair, P, stable="ordered")


def pair_contract(tab, pair, grouping, rb, vmask, lgrp, NL, C):
    """(B, gram): B[e,l,:] = sum_{o in l} rb[e,o] tab[pair[e],o,:] (+ valence slot) — the orbital sums of
    lcaonet.py:180-183 and :200-203 with f_coeffs (lcaonet.py:170) evaluated on the species-pair table."""
    return _PairContract.apply(tab, pair, grouping, rb.contiguous(), vmask, lgrp, NL, C)


def coeff_gram(B, NL):
    """(E, NL(NL+1)/2) FP64 Gram matrices B[e,l,:].B[e,l',:] of the first NL groups (no autograd: the
    three-body backward differentiates through them itself)."""
    require_cuda(B)
    E, NG, C = B.shape
    gram = torch.empty(E, NL * (NL + 1) // 2, dtype=torch.float64, device=B.device)
    _call("lcao_coeff_gram", ptr(B.detach().contiguous()), NG, E, C, NL, ptr(gram), stream_ptr())
    return gram


class BodyLink:
    """Couples the backward passes of `threebody` and `twobody` on the same B (lcaonet.py:173-204).

    Both consume B, so autograd would add two (E, NG, C) gradients in a separate pass.  The two-body
    gradient is the SAME row for every l < NL, so with a link the two-body backward leaves its compact
    (E, 1 + valence, C) gradient here and the three-body backward kernel folds it into the dB it writes.
    Works whatever order autograd runs the two nodes in: if the three-body backward has already run,
    the two-body one returns its gradient the ordinary way."""

    def __init__(self):
        self.dP = None
        self.consumed = False


def _threebody_fwd(B, gram, unit, xk, gi, NL, st):
    """(tbw, gate): the gate sigmoid(xk) once per node, then the three-body kernel."""
    E, NG, C = B.shape
    gate = torch.empty(gi.N, C, device=B.device)
    _call("lcao_sigmoid_rows", ptr(xk), xk.stride(0), ptr(gate), C, gi.N, C, st)
    tbw = torch.empty(E, C, device=B.device)
    _call("lcao_threebody_fwd", ptr(B), NG, ptr(gram), ptr(unit), ptr(gate), C, ptr(gi.in_ptr), ptr(gi.in_edge),
          ptr(gi.in_src), ptr(gi.out_ptr), ptr(gi.out_edge), gi.N, E, C, NL, ptr(tbw), st)
    return tbw, gate


def _threebody_bwd(B, gram, unit, gate, gi, NL, d_tbw, dP, q, d_xk, forces, st):
    """(dB, d unit) of tbw = threebody(B, unit, xk); d unit is None unless `forces`.  The kernel leaves the gradient of
    the gate's input per edge in `q` (E, C), whose sum over each node's out-edges goes into the caller's `d_xk`."""
    E, NG, C = B.shape
    dB = torch.empty_like(B)
    du_ks = torch.empty(E, 3, device=B.device) if forces else None
    du_st = torch.empty(E, 3, device=B.device) if forces else None
    _call("lcao_threebody_bwd", ptr(B), NG, ptr(gram), ptr(unit), ptr(gate), C, ptr(gi.in_ptr), ptr(gi.in_edge),
          ptr(gi.in_src), ptr(gi.out_ptr), ptr(gi.out_edge), gi.N, E, C, NL, ptr(d_tbw), ptr(dP), ptr(dB), ptr(q),
          ptr(du_ks), ptr(du_st), st)
    _segment_sum(q, gi.out_ptr, gi.out_edge, gi.N, st, out=d_xk)
    return dB, (du_ks + du_st) if forces else None


class _ThreeBody(torch.autograd.Function):
    @staticmethod
    def forward(ctx, B, gram, unit, xk, gi: GraphIndex, NL: int, link):
        require_cuda(B, unit, xk)
        B, unit = B.contiguous(), unit.contiguous()
        assert xk.stride(1) == 1 and gram.dtype == torch.float64 and gram.is_contiguous()
        tbw, gate = _threebody_fwd(B, gram, unit, xk, gi, NL, stream_ptr())
        ctx.gi, ctx.NL, ctx.link = gi, NL, link
        ctx.save_for_backward(B, gram, unit, gate)
        return tbw

    @staticmethod
    @once_differentiable
    def backward(ctx, d_tbw):
        B, gram, unit, gate = ctx.saved_tensors
        gi, link = ctx.gi, ctx.link
        E, _, C = B.shape
        dP = None
        if link is not None:
            dP, link.dP, link.consumed = link.dP, None, True
        q, d_xk = torch.empty(E, C, device=B.device), torch.empty(gi.N, C, device=B.device)
        dB, d_unit = _threebody_bwd(B, gram, unit, gate, gi, ctx.NL, d_tbw.contiguous(), dP, q, d_xk,
                                    ctx.needs_input_grad[2], stream_ptr())
        return dB, None, d_unit, d_xk, None, None, None


def threebody(B, unit, xk, gi, NL, gram=None, link: BodyLink | None = None):
    """Fused gather / angular basis / normalise / gate / triplet->edge sum (lcaonet.py:173-189)."""
    if gram is None:
        gram = coeff_gram(B, NL)
    return _ThreeBody.apply(B, gram, unit, xk, gi, NL, link)


def _twobody_fwd(B, g, NL, valence, st):
    E, NG, C = B.shape
    lw = torch.empty(E, C, device=B.device)
    _call("lcao_twobody_fwd", ptr(B), NG, ptr(g), E, C, NL, valence, ptr(lw), st)
    return lw


def _twobody_bwd(B, g, d_lw, NL, valence, compact, st):
    """(dB, dg); `compact`: dB is the (E, 1 + valence, C) gradient of [sum_l B_l | valence slot]."""
    E, NG, C = B.shape
    dB = torch.empty(E, 1 + valence, C, device=B.device) if compact else torch.empty_like(B)
    dg = torch.empty_like(g)
    _call("lcao_twobody_bwd", ptr(B), NG, ptr(g), ptr(d_lw), E, C, NL, valence, int(compact), ptr(dB), ptr(dg), st)
    return dB, dg


class _TwoBody(torch.autograd.Function):
    @staticmethod
    def forward(ctx, B, g, NL: int, valence: int, link):
        require_cuda(B, g)
        g = g.contiguous()
        lw = _twobody_fwd(B, g, NL, valence, stream_ptr())
        ctx.dims, ctx.link = (NL, valence), link
        ctx.save_for_backward(B, g)
        return lw

    @staticmethod
    @once_differentiable
    def backward(ctx, d_lw):
        B, g = ctx.saved_tensors
        NL, valence = ctx.dims
        link = ctx.link
        compact = link is not None and not link.consumed
        dB, dg = _twobody_bwd(B, g, d_lw.contiguous(), NL, valence, compact, stream_ptr())
        if compact:  # handed to the three-body backward kernel, which adds it to the dB it writes
            link.dP = dB
            return None, dg, None, None, None
        return dB, dg, None, None, None


def twobody(B, g, NL, valence, link: BodyLink | None = None):
    """lw = normalize((1+g_A) P_A + (1+g_V) P_V) with P = sum_l B_l (lcaonet.py:192-204)."""
    return _TwoBody.apply(B, g, NL, valence, link)


# ------------------------------------------------------------------------------------------------
# one interaction block as ONE autograd node
# ------------------------------------------------------------------------------------------------
class _InteractionLayer(torch.autograd.Function):
    """LCAOInteraction.forward (reference lcaonet.py:130-216) as a single autograd node.

    Same kernels, same order and same arithmetic as the op-by-op path (`coeff_contract/pair_contract`,
    `threebody`, `twobody`, `edge_pair`, `mul_segment_sum`, `linear`), but the ~15 forward and ~30
    backward C-ABI calls are issued from one Python frame each: no per-op autograd bookkeeping, no
    gradient-accumulation passes between consumers of the same tensor, strided halves written in place.
    The host cost of a layer drops from ~1.5 ms to ~0.3 ms, which matters once the GPU side of a
    1024-molecule step is ~10 ms."""

    @staticmethod
    def forward(ctx, x, table, rb, unit, w_n, b_n, w_c0, w_c2, w_3, w_b, w_1, b_1, w_2, b_2, w_o, aux):
        pair, grouping, vmask, lgrp, gi, NL, C, sinks, act = aux
        require_cuda(x, table, rb, unit)
        st = stream_ptr()
        N = x.shape[0]
        P, O, _ = table.shape
        valence = 1 if vmask is not None else 0
        grad = any(ctx.needs_input_grad)  # (grad mode is always off inside Function.forward)
        x, table, rb, unit = _rows(x, True), table.contiguous(), rb.contiguous(), unit.contiguous()
        # node side: nw = [xc | xk]
        nw, _ = _lin_fwd(x, w_n, b_n, st)
        # f_coeffs on the species-pair table
        t1, pre1 = _lin_fwd(_rows(table, True), w_c0, None, st, act, grad)
        tab, pre2 = _lin_fwd(t1, w_c2, None, st, act, grad)
        tab = tab.view(P, O, -1)
        # psum = [sum_l B_l | valence slot]: the two-body weight's view of B
        B, gram, psum = _pair_contract_fwd(tab, pair, rb, vmask, lgrp, NL, C, st, with_psum=True)
        # three-body
        xc, xk = nw.chunk(2, 1)
        tbw, gate = _threebody_fwd(B, gram, unit, xk, gi, NL, st)
        g, _ = _lin_fwd(tbw, w_3, None, st)
        # two-body weight and message
        lw = _twobody_fwd(psum, g, 1, valence, st)
        bw, _ = _lin_fwd(lw, w_b, None, st)
        w_1cat = torch.cat([w_1[:, :C], w_1[:, C:]], dim=0)  # (2C, C): [W1a ; W1b] acting on x_s / x_t per NODE
        u, _ = _lin_fwd(xc, w_1cat, None, st)
        a1, pre_a = _edge_pair_fwd(*u.chunk(2, 1), b_1, gi, act, grad, st)
        # h = SiLU(pre_h) is never stored: the message sum and its backward apply the activation on the fly, which takes
        # one E x C write off the f_node GEMM and one E x C read off each consumer
        pre_h, _ = _lin_fwd(a1, w_2, b_2, st)
        agg = _segment_sum(bw, gi.out_ptr, gi.out_edge, N, st, y=pre_h, mode=2 | (act << 4))
        y, _ = _lin_fwd(agg, w_o, None, st)
        out = x + y
        if grad:
            ctx.aux = aux
            ctx.save_for_backward(x, table, rb, unit, w_n, w_c0, w_c2, w_3, w_b, w_1cat, w_2, w_o, xc, t1, pre1, tab, pre2,
                                  B, gram, gate, tbw, g, lw, bw, a1, pre_a, pre_h, agg, psum, b_n, w_1, b_1, b_2)
        return out

    @staticmethod
    def backward(ctx, d_out):
        (x, table, rb, unit, w_n, w_c0, w_c2, w_3, w_b, w_1cat, w_2, w_o, xc, t1, pre1, tab, pre2, B, gram, gate, tbw, g,
         lw, bw, a1, pre_a, pre_h, agg, psum, b_n, w_1, b_1, b_2) = ctx.saved_tensors
        pair, grouping, vmask, lgrp, gi, NL, C, sinks, act = ctx.aux
        if torch.is_grad_enabled():
            # create_graph=True: this backward pass is itself being differentiated (training on autograd forces,
            # lcaonet.py:310-317).  The operator is re-evaluated in its any-order differentiable form (second_order.py) on
            # the saved INPUTS, and autograd returns their gradients together with the graph behind them.
            inputs = second_order.aliases([x, table, rb, unit, w_n, b_n, w_c0, w_c2, w_3, w_b, w_1, b_1, w_2, b_2, w_o])
            wanted = list(ctx.needs_input_grad[:15])
            if positions_only.active:  # only the path to the positions: x, rb, unit
                wanted = [wanted[0], False, wanted[2], wanted[3]] + [False] * 11
            with torch.enable_grad():
                out = second_order.interaction(*inputs, pair, vmask, lgrp, gi, NL, C, act)
                grads = second_order.grads_with_graph([out], inputs, [d_out], wanted)
            return (*grads, None)
        # `positions_only` (autograd forces): no parameter gradient is wanted from this pass, and the sinks are not its to write
        wg = not positions_only.active
        if not wg:
            sinks = None
        # gradient sinks: the parameters' own .grad buffers (order: w_n, b_n, w_c0, w_c2, w_3, w_b, w_1, b_1, w_2, b_2, w_o)
        s_wn, s_bn, s_wc0, s_wc2, s_w3, s_wb, s_w1, s_b1, s_w2, s_b2, s_wo = sinks if sinks is not None else (None,) * 11
        st = stream_ptr()
        (N, _), E = x.shape, gi.E
        P, O, K = table.shape
        valence = 1 if vmask is not None else 0
        need_rb, need_unit = ctx.needs_input_grad[2], ctx.needs_input_grad[3]
        d_out = _rows(d_out, True)
        dw_n = db_n = dw_c0 = dw_c2 = dw_3 = dw_b = dw_1 = db_1 = dw_2 = db_2 = dw_o = d_table = None
        # x_out = x + out_weight(agg)
        if wg:
            dw_o, _ = _lin_wgrad(d_out, agg, w_o, False, st, s_wo)
        d_agg = _lin_dgrad(d_out, w_o, st)
        # agg[s] = sum_{e in out(s)} bw[e] * h[e]
        d_bw, d_preh = torch.empty(E, C, device=x.device), torch.empty(E, C, device=x.device)
        _call("lcao_msg_bwd", ptr(d_agg), C, ptr(gi.src32), None, ptr(bw), ptr(pre_h), E, C, act, ptr(d_bw), ptr(d_preh), st)
        # h = silu(f_node.2(a1)) ; a1 = silu(u_a[s] + u_b[t] + b1)
        if wg:
            dw_2, db_2 = _lin_wgrad(d_preh, a1, w_2, True, st, s_w2, s_b2)
        # d_prea = d_a1 * SiLU'(pre_a) is never materialised: the two segment sums over it apply the factor on the fly
        d_a1 = _lin_dgrad(d_preh, w_2, st)
        d_u = torch.empty(N, 2 * C, device=x.device)
        d_ua, d_ub = d_u.chunk(2, 1)
        _segment_sum(d_a1, gi.out_ptr, gi.out_edge, N, st, y=pre_a, mode=4 | (act << 4), out=d_ua)
        _segment_sum(d_a1, gi.in_ptr, gi.in_edge, N, st, y=pre_a, mode=4 | (act << 4), out=d_ub)
        d_nw = torch.empty(N, 2 * C, device=x.device)
        d_xc, d_xk = d_nw.chunk(2, 1)
        _lin_dgrad(d_u, w_1cat, st, d_xc)
        if wg:
            # the bias b_1 enters once per edge through the u_a half: d b_1 = column sums of d_u[:, :C]
            dw_1cat, db_cat = _lin_wgrad(d_u, xc, w_1cat, True, st)
            dw_1, db_1 = torch.cat([dw_1cat[:C], dw_1cat[C:]], dim=1), db_cat[:C]
            if s_w1 is not None:
                s_w1.add_(dw_1)
                dw_1 = None
            if s_b1 is not None:
                s_b1.add_(db_1)
                db_1 = None
        # bw = basis_weight(lw) ; lw = twobody(B, g) ; g = f_three(tbw) ; tbw = threebody(B, ...)
        if wg:
            dw_b, _ = _lin_wgrad(d_bw, lw, w_b, False, st, s_wb)
        d_lw = _lin_dgrad(d_bw, w_b, st, d_preh)  # (reuses d_preh)
        dP, d_g = _twobody_bwd(psum, g, d_lw, 1, valence, True, st)
        if wg:
            dw_3, _ = _lin_wgrad(d_g, tbw, w_3, False, st, s_w3)
        d_tbw = _lin_dgrad(d_g, w_3, st, d_bw)  # (reuses d_bw)
        dB, d_unit = _threebody_bwd(B, gram, unit, gate, gi, NL, d_tbw, dP, d_a1, d_xk, need_unit, st)  # (q reuses d_a1)
        # B = pair_contract(tab, rb) ; tab = f_coeffs(table)
        need_tab = wg and (ctx.needs_input_grad[1] or any(ctx.needs_input_grad[6:8]))
        d_tab, d_rb = _pair_contract_bwd(tab, pair, grouping, rb, vmask, lgrp, dB, NL, C, need_tab, need_rb, st)
        if need_tab:
            d_pre2 = _act_bwd(d_tab.view(P * O, -1), pre2, act, st)
            dw_c2, _ = _lin_wgrad(d_pre2, t1, w_c2, False, st, s_wc2)
            d_pre1 = _lin_dgrad_act(d_pre2, w_c2, pre1, act, st)
            dw_c0, _ = _lin_wgrad(d_pre1, _rows(table, True), w_c0, False, st, s_wc0)
            if ctx.needs_input_grad[1]:
                d_table = _lin_dgrad(d_pre1, w_c0, st).view(P, O, K)
        # nw = node_weight(x) ; residual
        if wg:
            dw_n, db_n = _lin_wgrad(d_nw, x, w_n, True, st, s_wn, s_bn)
        dx = _lin_dgrad(d_nw, w_n, st, d_out.clone(), accumulate=1)
        return dx, d_table, d_rb, d_unit, dw_n, db_n, dw_c0, dw_c2, dw_3, dw_b, dw_1, db_1, dw_2, db_2, dw_o, None


def interaction_layer(x, table, rb, unit, w_n, b_n, w_c0, w_c2, w_3, w_b, w_1, b_1, w_2, b_2, w_o, pair, grouping, vmask,
                      lgrp, gi, NL, C, grad_sinks=None, act=ACT_SILU):
    """grad_sinks: optional 11-tuple of the weights' / biases' `.grad` buffers (contiguous, same shapes; None entries
    allowed).  The backward pass then ACCUMULATES those gradients in place and returns None for them to autograd —
    what AccumulateGrad would do, without the zero-fills and the per-parameter add kernels.  `grouping`: callable
    returning (kptr, kperm), a ready tuple, or None (see `_grouping`).  Opt-in
    (`LCAOInteraction.grads_in_place`, set by `dist.FlatGradBucket`): parameter hooks do not fire for them."""
    return _InteractionLayer.apply(x, table, rb, unit, w_n, b_n, w_c0, w_c2, w_3, w_b, w_1, b_1, w_2, b_2, w_o,
                                   (pair, grouping, vmask, lgrp, gi, NL, C, grad_sinks, _act_arg(act)))


# ------------------------------------------------------------------------------------------------
# count-weighted BatchNorm over table rows (embedding block)
# ------------------------------------------------------------------------------------------------
class _TableNorm(torch.autograd.Function):
    """nn.BatchNorm1d over a batch given as DISTINCT rows + multiplicities (embed.py:175,194,232,249; DESIGN.md R6)."""

    @staticmethod
    def forward(ctx, x, counts, weight, bias, running_mean, running_var, tracked, training: bool, momentum: float,
                eps: float):
        require_cuda(x)
        x = x.contiguous()
        R, F = x.shape
        y = torch.empty_like(x)
        mean, rstd = torch.empty(F, device=x.device), torch.empty(F, device=x.device)
        _call("lcao_table_norm_fwd", ptr(x), ptr(counts), ptr(weight), ptr(bias), R, F, eps, momentum, 1 if training else 0,
              ptr(running_mean), ptr(running_var), ptr(tracked), ptr(y), ptr(mean), ptr(rstd), stream_ptr())
        ctx.training = training
        ctx.save_for_backward(x, counts, weight, mean, rstd)
        ctx.mark_non_differentiable(*[t for t in (running_mean, running_var, tracked) if t is not None])
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        x, counts, weight, mean, rstd = ctx.saved_tensors
        dy = dy.contiguous()
        R, F = x.shape
        dx = torch.empty_like(x)
        dg = torch.empty(F, device=x.device) if weight is not None else None
        db = torch.empty(F, device=x.device) if weight is not None else None
        _call("lcao_table_norm_bwd", ptr(dy), ptr(x), ptr(counts), ptr(weight), ptr(mean), ptr(rstd), R, F,
              1 if ctx.training else 0, ptr(dx), ptr(dg), ptr(db), stream_ptr())
        return dx, None, dg, db, None, None, None, None, None, None


def table_norm(x, counts, weight, bias, running_mean, running_var, tracked, training, momentum, eps):
    return _TableNorm.apply(x, counts, weight, bias, running_mean, running_var, tracked, training, momentum, eps)


class _PairOuter(torch.autograd.Function):
    """pre[s,t,o,k] = fe[t,o,k] * (1 + za[s,k] + zb[t,k]): the species-pair coefficient table before its BatchNorm
    (embed.py:234-249 on the pair table) as one kernel forward and one backward."""

    @staticmethod
    def forward(ctx, fe, za, zb):
        require_cuda(fe, za, zb)
        fe, za, zb = fe.contiguous(), za.contiguous(), zb.contiguous()
        Zd, O, K = fe.shape
        pre = torch.empty(Zd, Zd, O, K, device=fe.device)
        _call("lcao_pair_outer_fwd", ptr(fe), ptr(za), ptr(zb), Zd, O, K, ptr(pre), stream_ptr())
        ctx.save_for_backward(fe, za, zb)
        return pre

    @staticmethod
    @once_differentiable
    def backward(ctx, dpre):
        fe, za, zb = ctx.saved_tensors
        Zd, O, K = fe.shape
        dpre = dpre.contiguous()
        d_fe, d_za, d_zb = torch.empty_like(fe), torch.empty_like(za), torch.empty_like(zb)
        _call("lcao_pair_outer_bwd", ptr(dpre), ptr(fe), ptr(za), ptr(zb), Zd, O, K, ptr(d_fe), ptr(d_za), ptr(d_zb), stream_ptr())
        return d_fe, d_za, d_zb


def pair_outer(fe, za, zb):
    return _PairOuter.apply(fe, za, zb)


# ------------------------------------------------------------------------------------------------
# gathers / segment sums
# ------------------------------------------------------------------------------------------------
def _segment_sum(x, seg_ptr, seg_perm, R, st, y=None, mode=0, out=None):
    """out[r] = sum of x[i] over the items i of segment r (`mode` bit 0: the mean); with `y`, of x[i] * y[i], or with
    bit 1 / bit 2 set of x[i] * act(y[i]) / x[i] * act'(y[i]) for the activation in bits 4+.  out is allocated (R, C)
    unless the caller passes it."""
    C = x.shape[1]
    if out is None:
        out = torch.empty(R, C, device=x.device)
    _call("lcao_segment_sum", ptr(x), x.stride(0), ptr(y), y.stride(0) if y is not None else 0, ptr(seg_ptr),
          ptr(seg_perm), R, C, mode, ptr(out), out.stride(0), st)
    return out


def _gather_rows(table, idx, st, mul=None):
    """out[i] = table[idx[i]] (* mul[i]) for every entry of idx (int32 or int64)."""
    n, W = idx.numel(), table.shape[1]
    out = torch.empty(n, W, device=table.device)
    _call("lcao_gather_rows", ptr(table), table.stride(0), ptr(idx), 1 if idx.dtype == torch.int64 else 0, ptr(mul),
          mul.stride(0) if mul is not None else 0, n, W, ptr(out), W, st)
    return out


def _edge_pair_fwd(a, b, bias, gi, act, need_pre, st):
    """(out, pre): out = act(pre), pre = a[s_e] + b[t_e] + bias, kept only when `need_pre` (else None)."""
    C = a.shape[1]
    out = torch.empty(gi.E, C, device=a.device)
    pre = torch.empty(gi.E, C, device=a.device) if need_pre else None
    _call("lcao_edge_pair_fwd", ptr(a), a.stride(0), ptr(b), b.stride(0), ptr(bias), ptr(gi.src32), ptr(gi.dst32), gi.E,
          C, act, ptr(out), ptr(pre), st)
    return out, pre


class _EdgePair(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b, bias, gi: GraphIndex, act: int):
        require_cuda(a, b)
        assert a.stride(1) == 1 and b.stride(1) == 1
        out, pre = _edge_pair_fwd(a, b, bias, gi, act, act != ACT_NONE and any(ctx.needs_input_grad), stream_ptr())
        ctx.gi, ctx.act, ctx.has_bias = gi, act, bias is not None
        ctx.save_for_backward(pre)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, d_out):
        (pre,) = ctx.saved_tensors
        gi = ctx.gi
        d_out = _rows(d_out, True)
        st = stream_ptr()
        if ctx.act != ACT_NONE:
            d_out = _act_bwd(d_out, pre, ctx.act, st)
        da = _segment_sum(d_out, gi.out_ptr, gi.out_edge, gi.N, st)
        db = _segment_sum(d_out, gi.in_ptr, gi.in_edge, gi.N, st)
        dbias = da.sum(0) if ctx.has_bias else None
        return da, db, dbias, None, None


def edge_pair(a, b, bias, gi, silu):
    """act(a[s_e] + b[t_e] + bias): `W [x_s ; x_t] + b` with W split per node (lcaonet.py:209, :304)."""
    return _EdgePair.apply(a, b, bias, gi, _act_arg(silu))


class _MulSegSum(torch.autograd.Function):
    """agg[s,:] = sum_{e in out(s)} x[e,:] * y[e,:]   (torch_scatter site lcaonet.py:207-214)."""

    @staticmethod
    def forward(ctx, x, y, gi: GraphIndex):
        require_cuda(x, y)
        x, y = _rows(x, True), _rows(y, True)
        out = _segment_sum(x, gi.out_ptr, gi.out_edge, gi.N, stream_ptr(), y=y)
        ctx.gi = gi
        ctx.save_for_backward(x, y)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, d_out):
        x, y = ctx.saved_tensors
        d_out, st = _rows(d_out, True), stream_ptr()
        return _gather_rows(d_out, ctx.gi.src32, st, mul=y), _gather_rows(d_out, ctx.gi.src32, st, mul=x), None


def mul_segment_sum(x, y, gi):
    return _MulSegSum.apply(x, y, gi)


class _SegmentReduce(torch.autograd.Function):
    """out[r] = sum (or mean) of x over the items of segment r; items listed by (ptr, perm), and
    `seg_of_item` (int64 or int32, n) maps items back to segments for the backward gather."""

    @staticmethod
    def forward(ctx, x, seg_ptr, seg_perm, seg_of_item, mean: bool):
        require_cuda(x)
        out = _segment_sum(_rows(x), seg_ptr, seg_perm, seg_ptr.numel() - 1, stream_ptr(), mode=1 if mean else 0)
        ctx.mean = mean
        ctx.save_for_backward(seg_ptr, seg_of_item, x)
        return out

    @staticmethod
    def backward(ctx, d_out):
        seg_ptr, seg_of_item, x_in = ctx.saved_tensors
        if torch.is_grad_enabled():  # create_graph=True (see second_order.py)
            with torch.enable_grad():
                (x_,) = second_order.aliases([x_in])
                out = second_order.segment_reduce(x_, seg_of_item, seg_ptr.numel() - 1, ctx.mean)
                (gx,) = second_order.grads_with_graph([out], [x_], [d_out], [True])
            return gx, None, None, None, None
        d_out = _rows(d_out, True)
        if ctx.mean:
            cnt = (seg_ptr[1:] - seg_ptr[:-1]).clamp(min=1).to(d_out.dtype)
            d_out = d_out / cnt.unsqueeze(-1)
        return _gather_rows(d_out, seg_of_item, stream_ptr()), None, None, None, None


def segment_reduce(x, seg_ptr, seg_perm, seg_of_item, mean=False):
    return _SegmentReduce.apply(x, seg_ptr, seg_perm, seg_of_item, mean)


class _GatherRows(torch.autograd.Function):
    """out[i,:] = table[idx[i],:]; backward is a keyed reduction over the (ptr, perm) grouping of idx."""

    @staticmethod
    def forward(ctx, table, idx, key_ptr, key_perm):
        require_cuda(table, idx)
        t2 = table.reshape(table.shape[0], -1)
        assert t2.stride(1) == 1
        out = _gather_rows(t2, idx, stream_ptr())
        ctx.tshape = table.shape
        ctx.save_for_backward(key_ptr, key_perm)
        return out.reshape(idx.numel(), *table.shape[1:])

    @staticmethod
    @once_differentiable
    def backward(ctx, d_out):
        key_ptr, key_perm = ctx.saved_tensors
        d2 = d_out.reshape(d_out.shape[0], -1).contiguous()
        n, W = d2.shape
        nkeys = ctx.tshape[0]
        acc = torch.zeros(nkeys, W, device=d_out.device)
        _call("lcao_reduce_by_key", ptr(d2), W, ptr(key_ptr), ptr(key_perm), nkeys, n, W, ptr(acc), stream_ptr())
        return acc.reshape(ctx.tshape), None, None, None


def gather_rows(table, idx, key_ptr, key_perm):
    return _GatherRows.apply(table, idx, key_ptr, key_perm)
