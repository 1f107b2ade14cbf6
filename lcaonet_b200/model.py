"""`LCAONet`: drop-in for `lcaonet.model.LCAONet` (reference lcaonet/model/lcaonet.py:322-540) whose
forward pass runs on the B200-native kernels of liblcao_b200.so.

Same constructor keywords, same `forward(graph)` contract (input keys, output shapes, side-effect
keys written into `graph`), same parameter / buffer names and shapes (reference checkpoints load with
`load_state_dict(strict=True)`), same initialisers.  What differs is the execution: no triplet-sized
tensor is ever built, every edge-sized step is one fused CUDA kernel (see DESIGN.md), and the only
PyTorch ops left are O(#species^2) table algebra for the embedding block and O(N) glue.

There is no CPU path: tensors must live on a CUDA (sm_100a) device.
"""
from __future__ import annotations

import math
import weakref
from fractions import Fraction

import torch
import torch.nn as nn
from torch import Tensor

from . import _lib, ops
from .keys import GraphKeys
from .orbitals import ElecInfo
from .resolve import activation_code, activation_resolver, cutoff_kind, init_params, init_resolver, rbf_kind, swish_beta


# ----------------------------------------------------------------------------------------------
# parameter holders (names/shapes/initialisers of the reference modules)
# ----------------------------------------------------------------------------------------------
class Dense(nn.Linear):
    """nn.Linear with the reference's initialisation protocol (nn/base.py:11-81): `weight_init`
    (default scale=2.0 / gain=1.0) on the weight, zeros on the bias; evaluated by `ops.linear`."""

    def __init__(self, in_dim, out_dim, bias=True, weight_init=None, bias_init=nn.init.zeros_, **kwargs):
        if bias and bias_init is None:
            raise ValueError("bias_init must not be None if set bias")
        self.bias_init, self.weight_init = bias_init, weight_init
        if weight_init is not None:
            for p in init_params(weight_init):
                if p not in kwargs and p == "gain":
                    kwargs[p] = 1.0
                elif p not in kwargs and p == "scale":
                    kwargs[p] = 2.0
        self.kwargs = kwargs
        super().__init__(in_dim, out_dim, bias)
        self.reset_parameters()

    def reset_parameters(self):
        if self.weight_init is not None:
            self.weight_init(self.weight, **self.kwargs)
        if self.bias is not None and self.bias_init is not None:
            self.bias_init(self.bias)

    def forward(self, x: Tensor, silu=False) -> Tensor:
        """`silu`: activation fused into the epilogue — False / True (SiLU) or an LCAO_ACT_* code."""
        return ops.linear(x, self.weight, self.bias, silu)


def _mlp(seq: nn.Sequential, x: Tensor) -> Tensor:
    """Dense layers of an nn.Sequential with the activation that follows each one fused into its epilogue."""
    mods = list(seq)
    i = 0
    while i < len(mods):
        fused = i + 1 < len(mods) and not isinstance(mods[i + 1], Dense)
        beta = swish_beta(mods[i + 1]) if fused else None
        if beta is not None:  # Swish: SiLU kernel on beta-scaled weights, then 1 / beta (see resolve.swish_beta)
            d = mods[i]
            x = ops.linear(x, d.weight * beta, d.bias * beta if d.bias is not None else None, True) / beta
        else:
            x = mods[i](x, silu=activation_code(mods[i + 1]) if fused else False)
        i += 2 if fused else 1
    return x


def _weighted_batch_norm(bn: nn.BatchNorm1d, table: Tensor, counts: Tensor, training: bool) -> Tensor:
    """BatchNorm1d over a batch given as DISTINCT rows + multiplicities.

    The reference normalises (N, F) node rows and (E, O*K) edge rows (embed.py:194,249); both are
    functions of the species (pair) only, so the batch statistics are the count-weighted statistics of
    the distinct rows — same numbers, O(#species^2) work.  Updates the running statistics exactly like
    nn.BatchNorm1d (momentum, unbiased running variance, num_batches_tracked)."""
    stats = training or not bn.track_running_stats  # normalise with batch statistics
    if table.dtype == torch.float32 and (bn.momentum is not None or not stats) and (bn.weight is None) == (bn.bias is None):
        # one kernel forward, one backward (lcao_table_norm_*): statistics, running buffers, normalisation, affine
        upd = training and bn.track_running_stats
        return ops.table_norm(table, counts.to(torch.float32), bn.weight, bn.bias,
                              bn.running_mean if (upd or not stats) else None, bn.running_var if (upd or not stats) else None,
                              bn.num_batches_tracked if upd else None, stats, float(bn.momentum or 0.0), float(bn.eps))
    if training or not bn.track_running_stats:
        n = counts.sum()
        w = (counts / n).unsqueeze(1)
        mean = (w * table).sum(0)
        var = (w * (table - mean) ** 2).sum(0)
        if training and bn.track_running_stats:
            with torch.no_grad():
                bn.num_batches_tracked += 1
                m = bn.momentum if bn.momentum is not None else 1.0 / float(bn.num_batches_tracked)
                bn.running_mean.mul_(1 - m).add_(m * mean)
                bn.running_var.mul_(1 - m).add_(m * var * (n / (n - 1)))
    else:
        mean, var = bn.running_mean, bn.running_var
    out = (table - mean) * torch.rsqrt(var + bn.eps)
    if bn.affine:
        out = out * bn.weight + bn.bias
    return out


class EmbedZ(nn.Module):
    def __init__(self, emb_size: int, max_z: int = 94):
        super().__init__()
        self.emb_size = emb_size
        self.z_embed = nn.Embedding(max_z, emb_size)
        self.z_embed.weight.data.uniform_(-math.sqrt(3), math.sqrt(3))

    def table(self) -> Tensor:
        """(max_z+1, emb): row z = embedding of element z (the reference indexes with z-1, embed.py:41)."""
        w = self.z_embed.weight
        return torch.cat([w.new_zeros(1, w.shape[1]), w], dim=0)


class EmbedElec(nn.Module):
    def __init__(self, emb_size: int, elec_info: ElecInfo, extend_orb: bool = False):
        super().__init__()
        self.register_buffer("elec", elec_info.elec_table)
        self.n_orb, self.emb_size, self.extend_orb = elec_info.n_orb, emb_size, extend_orb
        self.e_embeds = nn.ModuleList()
        min_idx = elec_info.min_orb_idx if elec_info.min_orb_idx else -1
        for i, max_e in enumerate(elec_info.max_elec_idx):
            pad = None if (i <= min_idx or extend_orb) else 0
            self.e_embeds.append(nn.Embedding(int(max_e), emb_size, padding_idx=pad))
        for ee in self.e_embeds:
            ee.weight.data.uniform_(-math.sqrt(2), math.sqrt(2))
            ee._fill_padding_idx_with_zero()

    def table(self) -> Tensor:
        """(max_z+1, n_orb, emb): electron-count embedding of every orbital of every element."""
        return torch.stack([ee(self.elec[:, o]) for o, ee in enumerate(self.e_embeds)], dim=1)


class ValenceMask(nn.Module):
    def __init__(self, emb_size: int, elec_info: ElecInfo):
        super().__init__()
        self.register_buffer("valence", elec_info.valence_table)
        self.n_orb, self.emb_size = elec_info.n_orb, emb_size

    def forward(self, z: Tensor, idx_t: Tensor) -> Tensor:
        """(E, n_orb) 0/1 floats (the reference expands this to (E, n_orb, C), embed.py:132-133)."""
        return self.valence[z[idx_t]].to(torch.float32).contiguous()


class EmbedNode(nn.Module):
    def __init__(self, emb_size, emb_size_z, use_elec, emb_size_e=None, activation=nn.SiLU(), weight_init=None):
        super().__init__()
        self.emb_size, self.emb_size_z, self.use_elec = emb_size, emb_size_z, use_elec
        self.emb_size_e = emb_size_e if use_elec else 0
        hid = max(emb_size, (emb_size_z + self.emb_size_e) // 2)
        self.f_enc = nn.Sequential(Dense(emb_size_z + self.emb_size_e, hid, True, weight_init), activation,
                                   Dense(hid, emb_size, True, weight_init), activation)
        self.bn = nn.BatchNorm1d(emb_size)


class EmbedCoeffs(nn.Module):
    def __init__(self, emb_size, emb_size_z, emb_size_e, n_orb, activation=nn.SiLU(), weight_init=None):
        super().__init__()
        self.emb_size, self.emb_size_z, self.emb_size_e = emb_size, emb_size_z, emb_size_e
        self.f_z = nn.Sequential(Dense(2 * emb_size_z, emb_size, False, weight_init))
        self.f_e = nn.Sequential(Dense(emb_size_e, emb_size, False, weight_init), activation,
                                 Dense(emb_size, emb_size, False, weight_init), activation)
        self.bn = nn.BatchNorm1d(emb_size * n_orb)


class PairCoeffs:
    """The reference's coefficient tensor `cst` (E, O, K) (embed.py:234-249) in factored form.

    cst[e] depends on the element pair (z_s, z_t) of the edge only, so it is kept as the P = (max_z+1)^2
    row table plus the pair index of every edge.  The interaction blocks apply their bias-free,
    row-wise f_coeffs MLP to the table rows and contract against the radial basis per edge
    (`ops.pair_contract`): the (E, O, K) tensor and the E*O-row GEMMs of the reference never exist.
    `materialize()` returns the reference-shaped tensor for callers that want it."""

    def __init__(self, table: Tensor, pair: Tensor, kptr: Tensor | None = None, kperm: Tensor | None = None):
        self.table, self.pair, self.kptr, self.kperm = table, pair, kptr, kperm

    def grouping(self) -> tuple[Tensor, Tensor]:
        """(kptr, kperm): edges grouped by species pair.  Built on
        first use — every backward through the pair table needs it (d table: keyed reduction; d rb: pair-sorted walk),
        whichever of the embedding / interaction parameters or the positions is being differentiated."""
        if self.kptr is None:
            with torch.no_grad():
                self.kptr, self.kperm = ops.bucket_sort(self.pair, self.table.shape[0], stable="ordered")
        return self.kptr, self.kperm

    def materialize(self) -> Tensor:
        P, O, K = self.table.shape
        return ops.gather_rows(self.table.reshape(P, O * K), self.pair, *self.grouping()).reshape(-1, O, K)


class LCAOEmbedding(nn.Module):
    """Embedding block (reference lcaonet.py:30-74, embed.py).  Everything here depends on the atomic
    numbers only: x[n] on z_n, cst[e] on the pair (z_s, z_t).  The dense layers and both BatchNorms
    therefore run on the (max_z+1)- and (max_z+1)^2-row tables (count-weighted statistics); the
    coefficient tensor is returned in factored form (`PairCoeffs`), so no edge-sized work happens here."""

    def __init__(self, emb_size, emb_size_coeff, elec_info, max_z, use_elec, extend_orb, activation=nn.SiLU(),
                 weight_init=None):
        super().__init__()
        self.emb_size, self.emb_size_coeff, self.use_elec, self.max_z = emb_size, emb_size_coeff, use_elec, max_z
        self.z_embed = EmbedZ(emb_size + emb_size_coeff, max_z)
        self.emb_size_node_e = emb_size if use_elec else 0
        self.e_embed = EmbedElec(self.emb_size_node_e + emb_size_coeff, elec_info, extend_orb)
        self.node_embed = EmbedNode(emb_size, emb_size, use_elec, self.emb_size_node_e, activation, weight_init)
        self.coeff_embed = EmbedCoeffs(emb_size_coeff, emb_size_coeff, emb_size_coeff, elec_info.n_orb, activation,
                                       weight_init)
        # training steps replay the static-shape table arithmetic (`_tables`) as CUDA graphs: ~220 launches of a few
        # microseconds each become two graph launches (1.35 ms -> see profiles/r01_notes.md).  Opt-in.
        self.graph_tables = False

    def _tables(self, cnt_z: Tensor, cnt_pair: Tensor) -> tuple[Tensor, Tensor]:
        """The static-shape part of the block: parameters + species / species-pair counts -> the normalised node table
        (Zd, H) and coefficient table (Zd^2, O*K).  Its ~80 forward and ~140 backward launches work on rows of a few
        hundred floats; `graph_tables` replays them as two CUDA graphs."""
        H, K, Zd = self.emb_size, self.emb_size_coeff, self.max_z + 1
        ztab = self.z_embed.table()  # (Zd, H+K)
        etab = self.e_embed.table()  # (Zd, O, He+K)
        O = etab.shape[1]
        node_z, coeff_z = ztab[:, :H], ztab[:, H:]
        if self.use_elec:
            node_e, coeff_e = etab[..., : self.emb_size_node_e], etab[..., self.emb_size_node_e:]
            enc_in = torch.cat([node_z, node_e.sum(1) / math.sqrt(O)], dim=-1)
        else:
            coeff_e, enc_in = etab, node_z
        # node embedding: species table -> BN with species counts
        xtab = _mlp(self.node_embed.f_enc, enc_in.contiguous())
        xtab = _weighted_batch_norm(self.node_embed.bn, xtab, cnt_z, self.training)
        # coefficient embedding: pair table (z_s, z_t) -> BN with pair counts
        wz = self.coeff_embed.f_z[0].weight  # (K, 2K) acting on [z_s ; z_t]
        za = ops.linear(coeff_z.contiguous(), wz[:, :K].contiguous())
        zb = ops.linear(coeff_z.contiguous(), wz[:, K:].contiguous())
        fe = _mlp(self.coeff_embed.f_e, coeff_e.contiguous())  # (Zd, O, K), orbitals of the TARGET element
        if fe.dtype == torch.float32 and K % 4 == 0:
            pre = ops.pair_outer(fe, za, zb)  # (Zd_s, Zd_t, O, K): one kernel forward, one backward
        else:
            pre = fe.unsqueeze(0) * (1.0 + za[:, None, None, :] + zb[None, :, None, :])
        ctab = _weighted_batch_norm(self.coeff_embed.bn, pre.reshape(Zd * Zd, O * K), cnt_pair, self.training)
        return xtab.contiguous(), ctab

    def _graphed_tables(self, cnt_z: Tensor, cnt_pair: Tensor):
        """`_tables` captured (forward and backward) by torch.cuda.make_graphed_callables, built on first use per
        device.  Capture runs the function a few times, so the BatchNorm buffers are restored afterwards."""
        # the graphs hold raw pointers: key them on the storage of every parameter and buffer (`.to()`, `.float()` ... move them)
        key = (cnt_z.device, cnt_z.shape, cnt_pair.shape,
               tuple(t.data_ptr() for t in list(self.parameters()) + list(self.buffers())))
        cache = self.__dict__.setdefault("_graph_cache", {})
        if key not in cache:
            cache.clear()  # a stale capture is never valid again
            bufs = [b for bn in (self.node_embed.bn, self.coeff_embed.bn)
                    for b in (bn.running_mean, bn.running_var, bn.num_batches_tracked) if b is not None]
            saved = [b.clone() for b in bufs]
            holder = _EmbedTables(self)
            # (capture runs on a side stream: the AccumulateGrad nodes of the parameters then live on another stream
            # than the replayed backward, which autograd reports once per process; the accumulation itself is ordered)
            quiet = getattr(torch.autograd.graph, "set_warn_on_accumulate_grad_stream_mismatch", None)
            if quiet is not None:
                quiet(False)
            cache[key] = torch.cuda.make_graphed_callables(holder, (cnt_z.clone(), cnt_pair.clone()),
                                                           allow_unused_input=True)
            with torch.no_grad():
                for b, v in zip(bufs, saved):
                    b.copy_(v)
        return cache[key]

    def forward(self, z: Tensor, idx_s: Tensor, idx_t: Tensor) -> tuple[Tensor, Tensor]:
        H, Zd = self.emb_size, self.max_z + 1
        pair = z[idx_s] * Zd + z[idx_t]
        cnt_z, cnt_pair = ops.histogram(z, Zd), ops.histogram(pair, Zd * Zd)
        grad = torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
        use_graph = self.graph_tables and self.training and grad and z.is_cuda and all(p.requires_grad for p in self.parameters())
        if use_graph:
            # a captured forward/backward pair serves ONE outstanding forward: its outputs and saved activations are static
            # buffers.  If the previous graphed forward is still alive and has not been back-propagated (two forwards
            # before a backward), this call takes the eager path instead of overwriting them.
            last = self.__dict__.get("_graph_last")
            if last is not None and last[0]() is not None and not last[1][0]:
                use_graph = False
        graphed = None
        if use_graph:
            try:
                graphed = self._graphed_tables(cnt_z, cnt_pair)
            except RuntimeError as e:  # capture refused (driver / allocator state): stay on the eager path, once and for all
                import warnings
                warnings.warn(f"LCAOEmbedding.graph_tables: CUDA graph capture failed ({e}); using the eager path")
                self.graph_tables = False
                use_graph = False
        if use_graph:
            xtab, ctab = graphed(cnt_z, cnt_pair)
            done = [False]
            ctab.register_hook(lambda g, d=done: d.__setitem__(0, True))
            self.__dict__["_graph_last"] = (weakref.ref(ctab), done)
        else:
            xtab, ctab = self._tables(cnt_z, cnt_pair)
        need_bwd = torch.is_grad_enabled() and xtab.requires_grad
        if H % 4 == 0:
            x = ops.gather_rows(xtab, z, *(ops.bucket_sort(z, Zd, stable="ordered") if need_bwd else (None, None)))
        else:
            x = xtab[z]
        O = ctab.shape[1] // self.emb_size_coeff
        return x, PairCoeffs(ctab.reshape(Zd * Zd, O, self.emb_size_coeff), pair)


class _EmbedTables(nn.Module):
    """LCAOEmbedding._tables as a module of its own (what torch.cuda.make_graphed_callables wants: the parameters are
    found through `.parameters()`).  Never registered on the embedding block, so no state_dict entry and no cycle."""

    def __init__(self, emb: "LCAOEmbedding"):
        super().__init__()
        self.emb = emb

    def forward(self, cnt_z: Tensor, cnt_pair: Tensor):
        return self.emb._tables(cnt_z, cnt_pair)


class LCAOInteraction(nn.Module):
    """Message-passing block (reference lcaonet.py:77-216) on the fused kernels."""

    def __init__(self, emb_size, emb_size_coeff, emb_size_conv, add_valence=False, activation=nn.SiLU(),
                 weight_init=None):
        super().__init__()
        self.emb_size, self.emb_size_coeff, self.emb_size_conv = emb_size, emb_size_coeff, emb_size_conv
        self.add_valence = add_valence
        C = emb_size_conv
        Cp = 2 * C if add_valence else C
        self.node_weight = Dense(emb_size, 2 * C, True, weight_init)
        self.f_coeffs = nn.Sequential(Dense(emb_size_coeff, C, False, weight_init), activation,
                                      Dense(C, Cp, False, weight_init), activation)
        self.f_three = nn.Sequential(Dense(C, Cp, False, weight_init))
        self.basis_weight = Dense(C, C, False, weight_init)
        self.f_node = nn.Sequential(Dense(2 * C, C, True, weight_init), activation,
                                    Dense(C, C, True, weight_init), activation)
        self.out_weight = Dense(C, emb_size, False, weight_init)
        # run the block as ONE autograd node (ops.interaction_layer); False = one node per kernel (same arithmetic)
        self.fused_node = True
        # accumulate parameter gradients straight into existing `.grad` buffers (see ops.interaction_layer); switched
        # on by dist.FlatGradBucket, whose flat buffer backs every .grad
        self.grads_in_place = False

    def forward(self, x, cst, vmask, rb, unit, gi, lgrp, NL) -> Tensor:
        if self.add_valence and vmask is None:
            raise ValueError("valence_mask must be provided when add_valence=True")
        C = self.emb_size_conv
        if isinstance(cst, PairCoeffs) and self.fused_node and x.shape[1] % 4 == 0:
            fc, fn = self.f_coeffs, self.f_node
            params = (self.node_weight.weight, self.node_weight.bias, fc[0].weight, fc[2].weight, self.f_three[0].weight,
                      self.basis_weight.weight, fn[0].weight, fn[0].bias, fn[2].weight, fn[2].bias, self.out_weight.weight)
            sinks = None
            beta = swish_beta(fn[1])
            if beta is not None:
                # Swish: every activation site becomes SiLU on beta-scaled weights (resolve.swish_beta).  The factors that are
                # left over cancel or fold into the next layer: tab comes out as beta * tab, which both of its consumers
                # normalise away (lcaonet.py:184,204); a1 and h come out times beta -> f_node.2 keeps its weight, its bias
                # and out_weight absorb the rest.
                w_n, b_n, w_c0, w_c2, w_3, w_b, w_1, b_1, w_2, b_2, w_o = params
                params = (w_n, b_n, w_c0 * beta, w_c2, w_3, w_b, w_1 * beta, b_1 * beta, w_2, b_2 * beta, w_o / beta)
            elif self.grads_in_place and torch.is_grad_enabled():
                sinks = tuple(p.grad if (p.requires_grad and p.grad is not None and p.grad.is_contiguous()) else None
                              for p in params)
            return ops.interaction_layer(x, cst.table, rb, unit, *params, cst.pair, cst.grouping, vmask, lgrp, gi, NL, C,
                                         sinks, activation_code(fn[1]))
        nw = self.node_weight(x)  # (N, 2C): [:, :C] feeds f_node, [:, C:] is the three-body gate
        xc, xk = nw[:, :C], nw[:, C:]
        if isinstance(cst, PairCoeffs):  # f_coeffs on the species-pair table, contracted per edge
            tab = _mlp(self.f_coeffs, cst.table)  # (P, O, C')
            B, gram = ops.pair_contract(tab, cst.pair, cst.grouping, rb, vmask, lgrp, NL, C)  # (E, NL(+1), C)
        else:  # a materialised (E, O, K) coefficient tensor, as in the reference signature
            cst1 = _mlp(self.f_coeffs, cst)  # (E, O, C')
            B, gram = ops.coeff_contract(cst1, rb, vmask, lgrp, NL, C), None
        link = ops.BodyLink()  # the two consumers of B share one gradient pass
        tbw = ops.threebody(B, unit, xk, gi, NL, gram, link)  # (E, C)
        g = self.f_three[0](tbw)  # (E, C')
        lw = ops.twobody(B, g, NL, 1 if self.add_valence else 0, link)  # (E, C)
        bw = self.basis_weight(lw)
        w1 = self.f_node[0].weight  # (C, 2C) acting on [x_s ; x_t]  ->  W1a x_s + W1b x_t, per NODE
        act, beta = activation_code(self.f_node[1]), swish_beta(self.f_node[1])
        b1, w2, b2 = self.f_node[0].bias, self.f_node[2].weight, self.f_node[2].bias
        if beta is not None:  # Swish = SiLU on beta-scaled weights (resolve.swish_beta); a1 comes out times beta
            w1, b1, b2 = w1 * beta, b1 * beta, b2 * beta
        u = ops.linear(xc, torch.cat([w1[:, :C], w1[:, C:]], dim=0))  # (N, 2C)
        a1 = ops.edge_pair(u[:, :C], u[:, C:], b1, gi, silu=act)  # (E, C)
        h = ops.linear(a1, w2, b2, act)
        agg = ops.mul_segment_sum(bw, h, gi)  # (N, C) sum over out-edges of each centre
        if beta is not None:
            agg = agg / beta
        return x + self.out_weight(agg)


class LCAOOut(nn.Module):
    """Output block (reference lcaonet.py:219-319)."""

    def __init__(self, emb_size, out_size, is_extensive=True, regress_forces=False, direct_forces=True,
                 activation=nn.SiLU(), weight_init=None):
        super().__init__()
        self.emb_size, self.out_size, self.is_extensive = emb_size, out_size, is_extensive
        self.regress_forces, self.direct_forces = regress_forces, direct_forces
        # autograd forces: None = differentiable forces (double backward) in training mode, first-order kernels in eval
        # mode; True / False force either.  False is the fast choice for a training loop whose loss is on the energy only.
        self.force_training = None
        self.out_lin = nn.Sequential(Dense(emb_size, emb_size, True, weight_init), activation,
                                     Dense(emb_size, emb_size // 2, True, weight_init), activation,
                                     Dense(emb_size // 2, out_size, False, weight_init))
        if regress_forces and direct_forces:
            self.out_lin_force = nn.Sequential(Dense(2 * emb_size, emb_size, True, weight_init), activation,
                                               Dense(emb_size, emb_size // 2, True, weight_init), activation,
                                               Dense(emb_size // 2, 1, False, weight_init))

    def forward(self, x, seg, gi, unit, pos, strain=None, lattice=None):
        prop = ops.segment_reduce(_mlp(self.out_lin, x), *seg, mean=not self.is_extensive)
        if not self.regress_forces:
            return prop
        if self.direct_forces:
            H = self.emb_size
            w1, b1 = self.out_lin_force[0].weight, self.out_lin_force[0].bias
            w2, b2 = self.out_lin_force[2].weight, self.out_lin_force[2].bias
            act, beta = activation_code(self.out_lin_force[1]), swish_beta(self.out_lin_force[1])
            if beta is not None:  # Swish = SiLU on beta-scaled weights (resolve.swish_beta): a comes out times beta, twice
                w1, b1, b2 = w1 * beta, b1 * beta, b2 * beta
            u = ops.linear(x, torch.cat([w1[:, :H], w1[:, H:]], dim=0))
            a = ops.edge_pair(u[:, :H], u[:, H:], b1, gi, silu=act)
            a = ops.linear(a, w2, b2, act)
            if beta is not None:
                a = a / beta
            f_st = self.out_lin_force[4](a) * unit  # (E, 3)
            return prop, ops.segment_reduce(f_st, gi.out_ptr, gi.out_edge, gi.src32, mean=False)
        # F = -dE/dpos (lcaonet.py:310-317).  The reference always builds the graph of this backward pass (create_graph=True)
        # so that a loss on the forces can be trained; here that graph is what switches the operators from their fused
        # backward kernels to the re-evaluated differentiable form (second_order.py), so it is built only when the forces can
        # be trained on: in training mode, unless `force_training` says otherwise.  Only d E / d pos is wanted from this
        # pass: the backward kernels skip every parameter gradient inside it (ops.positions_only).
        graph = self.training if self.force_training is None else bool(self.force_training)
        graph = graph and torch.is_grad_enabled()
        if strain is None:
            with ops.positions_only():
                cols = [-torch.autograd.grad(prop[:, i].sum(), pos, create_graph=graph, retain_graph=True)[0]
                        for i in range(self.out_size)]
            return prop, (cols[0] if len(cols) == 1 else torch.stack(cols, dim=1).squeeze(1))
        # stress (LCAONet.regress_stress): the same backward pass also yields d E / d strain = the virial W (ops.geom_basis)
        with ops.positions_only():
            grads = [torch.autograd.grad(prop[:, i].sum(), [pos, strain], create_graph=graph, retain_graph=True)
                     for i in range(self.out_size)]
        cols = [-g[0] for g in grads]
        L = lattice[: strain.shape[0]].double()
        vol = (L[:, 0] * torch.linalg.cross(L[:, 1], L[:, 2], dim=-1)).sum(-1).abs().to(grads[0][1].dtype)
        sig = [g[1] / vol.view(-1, 1, 1) for g in grads]
        return (prop, (cols[0] if len(cols) == 1 else torch.stack(cols, dim=1).squeeze(1)),
                (sig[0] if len(sig) == 1 else torch.stack(sig, dim=1)))


class PostProcess(nn.Module):
    """atomref / mean offsets (reference nn/post.py:8-89)."""

    def __init__(self, out_dim, is_extensive=True, atomref=None, mean=None):
        super().__init__()
        self.out_dim, self.is_extensive = out_dim, is_extensive
        self.register_buffer("atomref", atomref)
        self.register_buffer("mean", mean)

    def forward(self, out, z, seg):
        out, *rest = out if isinstance(out, tuple) else (out,)
        if self.atomref is not None:
            out = out + ops.segment_reduce(self.atomref[z].to(torch.float32), *seg, mean=not self.is_extensive)
        if self.mean is not None:
            m = self.mean.unsqueeze(0)
            if self.is_extensive:
                cnt = (seg[0][1:] - seg[0][:-1]).to(m.dtype).unsqueeze(1)
                m = cnt * m
            out = out + m
        return (out, *rest) if rest else out


# ----------------------------------------------------------------------------------------------
# basis descriptors (no parameters; evaluated inside the geometry / three-body kernels)
# ----------------------------------------------------------------------------------------------
def _laguerre(n: int, l: int) -> list[int]:
    """ascending integer coefficients of -(n+l)! L_{n-l-1}^{(2l+1)}(x) (reference rbf.py:82-87)."""
    k, a = n - l - 1, 2 * l + 1
    return [int(Fraction((-1) ** i * math.comb(k + a, k - i), math.factorial(i)) * (-math.factorial(n + l)))
            for i in range(k + 1)]


def _cutoff_value(kind: int, r: float, rc: float) -> float:
    """host-side cutoff functions (cutoff.py:32-67) for the constructor-time quadrature of `integral_norm`"""
    if r > rc:
        return 0.0
    q = r / rc
    if kind == _lib.CUT["polynomial"]:
        return (1.0 - q) ** 3 * (1.0 + 3.0 * q + 6.0 * q * q)  # = 1 - 10 q^3 + 15 q^4 - 6 q^5
    if kind == _lib.CUT["envelope"]:
        return (1.0 - q) ** 3 * (1.0 + 3.0 * q + 6.0 * q**2 + 10.0 * q**3 + 15.0 * q**4)  # p = 5: 1 - 21 q^5 + 35 q^6 - 15 q^7
    return 0.5 * (math.cos(math.pi * q) + 1.0)


def _radial_norm_integral(sp, u: int) -> float:
    """int_0^rc (r R_u(r))^2 dr of the spec's orbital u in float64 (reference: scipy.integrate.quad, rbf.py:122-126);
    composite Gauss-Legendre on 64 panels x 16 points — the integrand is a polynomial times exp(-zeta) times a smooth
    cutoff, so this agrees with quad to ~1e-14 relative."""
    import numpy as np
    n, l, rc, a0 = sp.n[u], sp.l[u], float(sp.rc), float(sp.a0)
    xs, ws = np.polynomial.legendre.leggauss(16)
    total = 0.0
    edges = np.linspace(0.0, rc, 65)
    for a, b in zip(edges[:-1], edges[1:]):
        for x, w in zip(xs, ws):
            r = 0.5 * (b - a) * x + 0.5 * (a + b)
            zeta = 2.0 / n / a0 * r
            poly = 0.0
            for i in range(sp.deg[u], -1, -1):
                poly = poly * zeta + sp.poly[u][i]
            f = _cutoff_value(sp.cutoff_kind, r, rc) * sp.norm[u] * poly * zeta**l * math.exp(-0.5 * zeta)
            total += 0.5 * (b - a) * w * (r * f) ** 2
    return total


class RadialBasis(nn.Module):
    """Hydrogen-like R_nl(r) x cutoff (reference nn/rbf.py:34-142; spherical-Bessel variant :145-182),
    described by an `lcao_basis_spec` that the geometry kernel evaluates."""

    def __init__(self, cutoff: float, elec_info: ElecInfo, cutoff_net: str, rbf_type: str = "hydrogen",
                 bohr_radius: float = 0.529, integral_norm: bool = False):
        super().__init__()
        self.cutoff, self.elec_info, self.n_orb = cutoff, elec_info, elec_info.n_orb
        self.cutoff_net, self.rbf_type, self.bohr_radius = cutoff_net, rbf_type, bohr_radius
        self.integral_norm = integral_norm
        nl = elec_info.nl_list[:: elec_info.n_per_orb].tolist()
        if len(nl) > _lib.MAX_UNIQUE_ORB:
            raise ValueError("too many orbitals")
        sp = _lib.BasisSpec()
        sp.n_unique, sp.n_rep = len(nl), elec_info.n_per_orb
        sp.cutoff_kind, sp.rbf_kind = _lib.CUT[cutoff_net], _lib.RBF[rbf_type]
        sp.rc, sp.a0 = float(cutoff), float(bohr_radius)
        for u, (n, l) in enumerate(nl):
            coef = _laguerre(n, l)
            sp.n[u], sp.l[u], sp.deg[u] = n, l, len(coef) - 1
            sp.norm[u] = -math.sqrt((2.0 / n / bohr_radius) ** 3 * math.factorial(n - l - 1) / 2.0 / n
                                    / math.factorial(n + l) ** 3)
            for i, c in enumerate(coef):
                sp.poly[u][i] = float(c)
            if integral_norm and sp.rbf_kind == _lib.RBF["hydrogen"]:
                # rbf.py:92-93,107-127: prefactor -2/(n a0), then scaled so that int_0^rc (r R(r))^2 dr = 1 (cutoff included)
                sp.norm[u] = -2.0 / n / bohr_radius
                sp.norm[u] = sp.norm[u] / (math.sqrt(_radial_norm_integral(sp, u)) + 1e-12)
        self.spec = sp

    def extra_repr(self) -> str:
        return f"cutoff={self.cutoff}, cutoff_net={self.cutoff_net}, rbf_type={self.rbf_type}, n_orb={self.n_orb}"

    def forward(self, r: Tensor) -> Tensor:
        """(E,) distances -> (E, n_orb); standalone entry (the model fuses this with the geometry)."""
        _lib.require_cuda(r)
        n = r.numel()
        pos = torch.zeros(2 * n, 3, device=r.device)
        pos[1::2, 0] = r.reshape(-1).float()
        ei = torch.arange(2 * n, device=r.device).reshape(n, 2).t().contiguous()
        gi = ops.GraphIndex(ei, 2 * n)
        shift = torch.zeros(n, 3, device=r.device)
        lat = torch.eye(3, device=r.device).unsqueeze(0)
        return ops.geom_basis(pos, shift, lat, None, gi, self.spec, self.n_orb)[2]


class SphericalHarmonicsBasis(nn.Module):
    """Y_l^0(cos theta) per orbital (reference nn/shbf.py:14-87).  Inside the model the three-body kernel
    evaluates these in registers; this module is the standalone (T,) -> (T, n_orb) entry."""

    _COEF = (0.28209479177387814, 0.4886025119029199, 0.9461746957575601, 0.31539156525252005, 0.3731763325901154)

    def __init__(self, elec_info: ElecInfo):
        super().__init__()
        self.elec_info = elec_info
        self.l_list = elec_info.nl_list[:, 1].tolist()

    def forward(self, c: Tensor) -> Tensor:
        y0, y1, y2a, y2b, y3 = self._COEF
        y = [torch.full_like(c, y0), y1 * c, y2a * c * c - y2b, y3 * c * (5 * c * c - 3)]
        return torch.stack([y[l] for l in self.l_list], dim=1)


# ----------------------------------------------------------------------------------------------
# the model
# ----------------------------------------------------------------------------------------------
class LCAONet(nn.Module):
    """LCAONet on B200 kernels.  Constructor identical to the reference (lcaonet.py:327-351)."""

    def __init__(self, emb_size: int = 128, emb_size_coeff: int = 128, emb_size_conv: int = 128, out_size: int = 1,
                 n_interaction: int = 3, n_per_orb: int = 1, cutoff: float = 6.0, rbf_type="hydrogen",
                 cutoff_net="envelope", max_z: int = 36, min_orb: str | None = None, max_orb: str | None = None,
                 elec_to_node: bool = True, add_valence: bool = False, extend_orb: bool = False,
                 is_extensive: bool = True, activation: str = "SiLU", weight_init: str | None = "glorotorthogonal",
                 atomref: Tensor | None = None, mean: Tensor | None = None, regress_forces: bool = False,
                 direct_forces: bool = True):
        super().__init__()
        wi = init_resolver(weight_init) if weight_init is not None else None
        act = activation_resolver(activation)
        activation_code(act)  # raises for activations the kernels do not fuse
        if emb_size_conv % 4 or emb_size_coeff % 4 or emb_size_conv > 256:
            raise NotImplementedError("the B200 kernels need emb_size_conv and emb_size_coeff to be multiples of 4 "
                                      f"and emb_size_conv <= 256 (got {emb_size_conv}, {emb_size_coeff})")
        self.emb_size, self.emb_size_coeff, self.emb_size_conv = emb_size, emb_size_coeff, emb_size_conv
        self.out_size, self.n_interaction, self.cutoff, self.cutoff_net = out_size, n_interaction, cutoff, cutoff_net
        self.elec_to_node, self.add_valence = elec_to_node, add_valence
        self.regress_forces, self.direct_forces = regress_forces, direct_forces
        self.max_z = max_z
        # write the reference's triplet side-effect keys (idx_k_3b, edge_idx_*_3b, angles_3b) into the
        # batch; costs one host sync (T is data dependent) — set False for a fully asynchronous forward
        self.side_effect_keys = True
        # range-check z / batch / edge_index on the device before they index anything (IndexError like the reference's
        # nn.Embedding / index_select); costs one host sync per forward — set False when the caller vouches for the batch
        self.validate_inputs = True
        # also return the stress  sigma_g = (1 / |det L_g|) d E / d eps_g  (B,3,3) (ASE's get_stress convention before Voigt
        # packing; eps_g a strain of cell g acting as pos (I + eps), L (I + eps)), computed in the same backward pass as the
        # autograd forces: forward returns (energy, forces, stress), stress in energy units per A^3, not symmetrised; a cell
        # of zero volume gives non-finite rows.  Needs regress_forces=True, direct_forces=False.
        self.regress_stress = False

        elec_info = ElecInfo(max_z, max_orb, min_orb, n_per_orb)
        if elec_info.n_orb > 64:
            raise NotImplementedError("more than 64 orbitals")
        self.rbf = RadialBasis(cutoff, elec_info, cutoff_kind(cutoff_net), rbf_kind(rbf_type))
        self.shbf = SphericalHarmonicsBasis(elec_info)
        l_list = elec_info.nl_list[:, 1].to(torch.int32)
        self.register_buffer("_lgrp", l_list.contiguous(), persistent=False)
        self._n_l = int(l_list.max()) + 1

        self.emb_layer = LCAOEmbedding(emb_size, emb_size_coeff, elec_info, max_z, elec_to_node, extend_orb, act, wi)
        if add_valence:
            self.valence_mask = ValenceMask(emb_size_conv, elec_info)
        self.int_layers = nn.ModuleList([LCAOInteraction(emb_size, emb_size_coeff, emb_size_conv, add_valence, act, wi)
                                         for _ in range(n_interaction)])
        self.out_layer = LCAOOut(emb_size, out_size, is_extensive, regress_forces, direct_forces, act, wi)
        self.pp_layer = PostProcess(out_size, is_extensive, atomref, mean)

    @property
    def n_param(self) -> int:
        return sum(p.numel() for p in self.parameters() if p.requires_grad)

    # -- reference helper API (lcaonet.py:417-486, base.py:15-43), kept for callers that use it ------
    def get_triplets(self, graph):
        ei = graph[GraphKeys.Edge_idx]
        gi = ops.GraphIndex(ei, graph[GraphKeys.Z].shape[0])
        k, e_ks, e_st = gi.triplets()
        graph[GraphKeys.Idx_k_3b], graph[GraphKeys.Edge_idx_ks_3b], graph[GraphKeys.Edge_idx_st_3b] = k, e_ks, e_st
        return graph

    @staticmethod
    def calc_atomic_distances(graph, return_vec: bool = False):
        pos = graph[GraphKeys.Pos]
        s, t = graph[GraphKeys.Edge_idx]
        b = graph.get(GraphKeys.Batch_idx)
        b = b if b is not None else torch.zeros(pos.shape[0], dtype=torch.long, device=pos.device)
        vec = pos[t] - pos[s] + torch.einsum("ni,nij->nj", graph[GraphKeys.Edge_shift], graph[GraphKeys.Lattice][b[s]])
        graph[GraphKeys.Edge_dist] = vec.norm(dim=1)
        if return_vec:
            graph[GraphKeys.Edge_vec_st] = vec / graph[GraphKeys.Edge_dist].unsqueeze(-1)
        return graph

    def calc_3body_angles(self, graph):
        vec = graph.get(GraphKeys.Edge_vec_st)
        if vec is None:
            raise ValueError("edge_vec_st is not calculated. Please run calc_atomic_distances(return_vec=True) first.")
        e_st, e_ks = graph[GraphKeys.Edge_idx_st_3b], graph[GraphKeys.Edge_idx_ks_3b]
        graph[GraphKeys.Angles_3b] = (vec[e_st] * vec[e_ks]).sum(-1)
        return graph

    # -- forward ------------------------------------------------------------------------------------
    def forward(self, graph):
        autograd_forces = self.regress_forces and not self.direct_forces
        if self.regress_stress and not autograd_forces:
            raise ValueError("regress_stress needs autograd forces: construct the model with regress_forces=True, "
                             "direct_forces=False")
        if autograd_forces:
            graph[GraphKeys.Pos].requires_grad_(True)
        batch_idx = graph.get(GraphKeys.Batch_idx)
        z, pos = graph[GraphKeys.Z], graph[GraphKeys.Pos]
        edge_index = graph[GraphKeys.Edge_idx]
        lattice, shift = graph[GraphKeys.Lattice], graph[GraphKeys.Edge_shift]
        _lib.require_cuda(z, pos, edge_index, lattice, shift)
        N, n_graph = z.shape[0], lattice.shape[0]
        idx_s, idx_t = edge_index[0], edge_index[1]
        if self.validate_inputs:
            ops.validate_graph(z, self.max_z, batch_idx, n_graph, edge_index)

        # indices: CSR by target / by source built on the GPU (replaces torch_sparse, lcaonet.py:462-477)
        gi = ops.GraphIndex(edge_index, N)
        # nodes -> graphs segments
        if batch_idx is None:
            seg = (torch.tensor([0, N], dtype=torch.int32, device=z.device), None,
                   torch.zeros(N, dtype=torch.int64, device=z.device))
        else:
            seg = (*ops.bucket_sort(batch_idx, n_graph), batch_idx)
        # stress: a zero strain per graph whose gradient is the virial (ops.geom_basis)
        strain = (torch.zeros(seg[0].numel() - 1, 3, 3, device=pos.device, requires_grad=True) if self.regress_stress
                  else None)
        # geometry + radial basis in one kernel (base.py:27-43, rbf.py:129-142)
        dist, unit, rb = ops.geom_basis(pos, shift, lattice, batch_idx, gi, self.rbf.spec, self.rbf.n_orb, strain, seg[:2])
        graph[GraphKeys.Edge_dist], graph[GraphKeys.Edge_vec_st] = dist, unit
        if self.side_effect_keys:
            k, e_ks, e_st, cos = gi.triplets(unit.detach())
            graph[GraphKeys.Idx_k_3b], graph[GraphKeys.Edge_idx_ks_3b], graph[GraphKeys.Edge_idx_st_3b] = k, e_ks, e_st
            graph[GraphKeys.Angles_3b] = cos

        x, cst = self.emb_layer(z, idx_s, idx_t)
        vmask = self.valence_mask(z, idx_t) if self.add_valence else None
        for layer in self.int_layers:
            x = layer(x, cst, vmask, rb, unit, gi, self._lgrp, self._n_l)
        out = self.out_layer(x, seg, gi, unit, pos, strain, lattice)
        return self.pp_layer(out, z, seg)
