"""Differentiable-to-any-order restatements of the fused operators, used ONLY inside backward passes that were asked to
build a graph (`create_graph=True`): training on autograd forces (reference lcaonet.py:310-317, tests/model/
test_lcaonet.py:219-233) differentiates  F = -dE/dpos  with respect to the parameters, i.e. it back-propagates THROUGH
the backward pass of every operator on the path from `pos` to the energy.

The fused CUDA kernels stay the first-order path: forward always, backward whenever no graph is requested (energy
training, inference, force evaluation).  When a backward is entered with grad mode on, `ops` calls the function of this
module that restates the operator with ordinary torch tensor operations — the same restructured algebra as the kernels
(species-pair table, per-l orbital groups, the `(1+g)` factor outside the orbital sum, `f_node.0` split per node), so no
(T, O, C) tensor appears, only (T, C) ones — re-evaluates it on the saved inputs and lets autograd produce the input
gradients WITH their graph.  Triplet lists come from the GPU index kernels (`GraphIndex.triplets`).

Cost: one extra evaluation of the operator per backward, with triplet-sized (T, C) temporaries kept until the loss has
been back-propagated.  That is the price of the force-training mode only; it is what the reference pays on every step.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F
from torch import Tensor

from . import _lib

_Y = (0.28209479177387814, 0.4886025119029199, 0.9461746957575601, 0.31539156525252005, 0.3731763325901154)


def act_fn(code: int):
    """torch function of an LCAO_ACT_* code (include/lcao_b200.h)."""
    A = _lib.ACT
    return {A["none"]: lambda x: x, A["silu"]: F.silu, A["shiftedsoftplus"]: lambda x: F.softplus(x) - math.log(2.0),
            A["softplus"]: F.softplus, A["relu"]: F.relu, A["tanh"]: torch.tanh, A["sigmoid"]: torch.sigmoid,
            A["gelu"]: F.gelu, A["elu"]: F.elu, A["leakyrelu"]: F.leaky_relu}[int(code)]


def aliases(tensors):
    """Fresh graph nodes for the inputs of a re-evaluated operator.  The saved inputs of one operator are often ANCESTORS
    of one another in the outer graph (the node features of layer i depend on rb and unit through layer i-1), so asking
    autograd for d out / d rb on the tensors themselves would also collect the indirect path through x — which the
    outer backward pass adds a second time.  A view of each input cuts that: gradients are taken at the views, whose
    only way back to the inputs is the view itself."""
    return [t.view_as(t) if (t is not None and t.requires_grad) else t for t in tensors]


def grads_with_graph(outputs, inputs, grad_outputs, wanted):
    """d <grad_outputs, outputs> / d inputs[i] for the wanted i (None elsewhere), with a graph behind every result.
    `inputs` must be the `aliases` the outputs were computed from."""
    outs = [o for o, g in zip(outputs, grad_outputs) if g is not None and o.requires_grad]
    gos = [g for o, g in zip(outputs, grad_outputs) if g is not None and o.requires_grad]
    idx = [i for i, (t, w) in enumerate(zip(inputs, wanted)) if w and t is not None and t.requires_grad]
    res = [None] * len(inputs)
    if outs and idx:
        got = torch.autograd.grad(outs, [inputs[i] for i in idx], gos, create_graph=True, allow_unused=True)
        for i, g in zip(idx, got):
            res[i] = g
    return res


# ------------------------------------------------------------------------------------------------
def linear(x: Tensor, w: Tensor, b: Tensor | None, act: int) -> Tensor:
    return act_fn(act)(F.linear(x, w, b))


def segment_reduce(x: Tensor, seg_of_item: Tensor, n_seg: int, mean: bool) -> Tensor:
    x2 = x.reshape(-1, x.shape[-1])
    out = x2.new_zeros(n_seg, x2.shape[1]).index_add(0, seg_of_item.long(), x2)
    if mean:
        cnt = torch.bincount(seg_of_item.long(), minlength=n_seg).clamp(min=1).to(out.dtype)
        out = out / cnt.unsqueeze(-1)
    return out


def _cutoff(kind: int, r: Tensor, rc: float) -> Tensor:
    q = r / rc
    u = 1 - q
    if kind == _lib.CUT["polynomial"]:
        f = u**3 * (1 + 3 * q + 6 * q * q)
    elif kind == _lib.CUT["envelope"]:
        f = u**3 * (1 + 3 * q + 6 * q**2 + 10 * q**3 + 15 * q**4)
    else:
        f = 0.5 * (torch.cos(math.pi * q) + 1)
    return torch.where(r <= rc, f, torch.zeros_like(f))


def geom_basis(pos: Tensor, shift: Tensor, lattice: Tensor, batch: Tensor | None, src: Tensor, dst: Tensor, spec, n_orb: int,
               strain: Tensor | None = None, atom_strain: Tensor | None = None):
    """(dist, unit, rb) as functions of `pos`, `lattice` and the strain probes (base.py:27-43, rbf.py:92-142,
    cutoff.py:32-67), evaluated in float64 (edge-sized work) and rounded to float32 like the kernel's outputs.
    With `strain` (B,3,3): vec = ((pos[t] - pos[s]) + shift . L) (I + strain[g]); with `atom_strain` (N,3,3) vec gains
    1/2 vec (atom_strain[s] + atom_strain[t]).  Their values are zero, so the result is unchanged and only the derivatives
    (the virial, the per-atom virials) differ from the plain form."""
    s, t = src.long(), dst.long()
    P = pos.double()
    b = batch[s] if batch is not None else torch.zeros_like(s)
    L = lattice.double()[b]
    v = v0 = (P[t] - P[s]) + (shift.double().unsqueeze(-1) * L).sum(1)
    if strain is not None:
        v = v + (v.unsqueeze(-1) * strain.double()[b]).sum(1)
    if atom_strain is not None:
        A = atom_strain.double()
        v = v + 0.5 * (v0.unsqueeze(-1) * (A[s] + A[t])).sum(1)
    r = v.norm(dim=1)
    unit = v / r.unsqueeze(-1)
    fc = _cutoff(spec.cutoff_kind, r, float(spec.rc))
    cols = []
    for u in range(spec.n_unique):
        n, l = spec.n[u], spec.l[u]
        if spec.rbf_kind == _lib.RBF["hydrogen"]:
            zeta = (2.0 / (n * float(spec.a0))) * r
            p = torch.zeros_like(r)
            for i in range(spec.deg[u], -1, -1):
                p = p * zeta + float(spec.poly[u][i])
            R = float(spec.norm[u]) * p * zeta**l * torch.exp(-0.5 * zeta)
        else:
            R = torch.sin((math.pi * n / float(spec.rc)) * r) / r
        cols += [fc * R] * spec.n_rep
    rb = torch.stack(cols, 1)
    assert rb.shape[1] == n_orb
    return r.float(), unit.float(), rb.float()


def _normalize(v: Tensor, eps: float = 1e-12) -> Tensor:
    """F.normalize(v, dim=-1) = v / max(|v|, eps) (lcaonet.py:184,204) written so that rows with |v| <= eps — edges beyond
    the cutoff have all-zero coefficient rows — differentiate to finite values at every order: they take the v / eps
    branch and never see the 0 / 0 of d|v|/dv."""
    sq = (v * v).sum(-1, keepdim=True)
    big = sq > eps * eps
    nrm = torch.sqrt(torch.where(big, sq, torch.ones_like(sq)))
    return torch.where(big, v / nrm, v / eps)


def _sph(c: Tensor, NL: int) -> Tensor:
    y = [torch.full_like(c, _Y[0]), _Y[1] * c, _Y[2] * c * c - _Y[3], _Y[4] * c * (5 * c * c - 3)]
    return torch.stack(y[:NL], 1)


def interaction(x, table, rb, unit, w_n, b_n, w_c0, w_c2, w_3, w_b, w_1, b_1, w_2, b_2, w_o, pair, vmask, lgrp, gi, NL, C, act):
    """LCAOInteraction.forward (reference lcaonet.py:130-216) in the kernels' algebra, with torch operations."""
    f = act_fn(act)
    P, O, K = table.shape
    valence = vmask is not None
    s, t = gi.edge_index[0], gi.edge_index[1]
    tri_k, e_ks, e_st = gi.triplets()
    E = gi.E
    # node side
    nw = F.linear(x, w_n, b_n)
    xc, xk = nw[:, :C], nw[:, C:]
    # f_coeffs on the species-pair table, contracted with the radial basis per edge and grouped by l
    tab = f(F.linear(f(F.linear(table, w_c0)), w_c2))  # (P, O, C')
    G = F.one_hot(lgrp.long(), NL).to(rb.dtype)  # (O, NL)
    B = rb.new_zeros(E, NL, C)
    PV = rb.new_zeros(E, C) if valence else None
    for o in range(O):  # one (E, C) gather per orbital: no (E, O, C) tensor
        row = tab[:, o, :][pair]  # (E, C')
        contrib = rb[:, o:o + 1] * row[:, :C]
        if valence:
            v = (rb[:, o:o + 1] * vmask[:, o:o + 1]) * row[:, C:]
            contrib = contrib + v
            PV = PV + v
        B = B + contrib.unsqueeze(1) * G[o].view(1, NL, 1)
    # three-body: per-triplet chain (lcaonet.py:173-189)
    cos = (unit[e_st] * unit[e_ks]).sum(-1)
    Y = _sph(cos, NL)
    v3 = (Y.unsqueeze(-1) * B[e_ks]).sum(1)  # (T, C)
    v3 = _normalize(v3)
    v3 = v3 * torch.sigmoid(xk)[tri_k]
    tbw = x.new_zeros(E, C).index_add(0, e_st, v3)
    g = F.linear(tbw, w_3)
    # two-body weight (lcaonet.py:192-204) and message (lcaonet.py:207-214)
    S = B.sum(1)
    if valence:
        p2 = (1 + g[:, :C]) * (S - PV) + (1 + g[:, C:]) * PV
    else:
        p2 = (1 + g) * S
    lw = _normalize(p2)
    bw = F.linear(lw, w_b)
    u = F.linear(xc, torch.cat([w_1[:, :C], w_1[:, C:]], dim=0))  # (N, 2C)
    a1 = f(u[:, :C][s] + u[:, C:][t] + b_1)
    h = f(F.linear(a1, w_2, b_2))
    agg = x.new_zeros(x.shape[0], C).index_add(0, s, bw * h)
    return x + F.linear(agg, w_o)
