"""CPU oracle for the LCAONet hot path — TEST INFRASTRUCTURE, never the product path.

A plain, un-fused restatement of the reference algorithm (nmdl-mizo/lcaonet v0.0.3) written as
pure functions over a parameter dict that uses the reference's `state_dict` names.  It is dtype
generic (run it in float64 for parity checks) and device generic, materialises every triplet-sized
tensor exactly like the reference does, and gets its gradients from torch autograd.

Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s `cpu_baseline` / `--impl reference` legs
may import this module, and only as the checker / the timed CPU baseline.  `lcaonet_b200/` never
imports it.

Parity pinning (see tests/test_oracle_golden.py):
  * against the UNMODIFIED reference imported in the build container through `oracle/_shims`
    (all interaction / embedding / output numerics, triplet indices) -> committed golden vectors
    in tests/golden/ made by oracle/make_golden.py;
  * against the known-answer vectors the reference's own tests hold: closed-form R_nl
    (tests/nn/test_rbf.py:37-48), scipy Y_l^0 (tests/nn/test_shbf.py:46), cutoff properties
    (tests/nn/test_cutoff.py), the 3-atom periodic fixture (tests/model/conftest.py:6-35).
  * third-party pieces absent from /root/reference: torch_scatter / torch_sparse (versions
    un-pinned: requirements.txt:7-8) are restated from their published behaviour; the triplet
    ORDER among periodic-image duplicates of one (k, s) pair is implementation-defined in the
    reference (non-stable argsort) — "parity unpinned" there; the canonical order here is the
    stable one (ascending edge id).

Each function cites the reference lines it follows.
"""
from __future__ import annotations

import math
from fractions import Fraction

import torch
import torch.nn.functional as F

# --------------------------------------------------------------------------------------------
# orbital bookkeeping (reference: lcaonet/atomistic/elec.py:6-29, info.py:39-127)
# --------------------------------------------------------------------------------------------
_ORB = ("1s", "2s", "2p", "3s", "3p", "4s", "3d", "4p", "5s", "4d", "5p", "6s", "4f", "5d", "6p", "7s", "5f", "6d")
_LQ = {"s": 0, "p": 1, "d": 2, "f": 3}
_Z_TO_LAST = ((2, 0), (4, 1), (10, 2), (12, 3), (18, 4), (20, 5), (30, 6), (36, 7), (38, 8), (48, 9), (54, 10),
              (56, 11), (80, 13), (86, 14), (88, 15), (96, 17))


def orbital_quantum_numbers(max_z: int, max_orb: str | None = None, n_per_orb: int = 1) -> list[tuple[int, int]]:
    """(n, l) for each of the model's orbitals, in order (info.py:25-31,124-127)."""
    last = next(i for zmax, i in _Z_TO_LAST if max_z <= zmax)
    if max_orb is not None:
        last = max(last, _ORB.index(max_orb))
    out = []
    for name in _ORB[: last + 1]:
        out += [(int(name[0]), _LQ[name[1]])] * n_per_orb
    return out


def min_orb_index(min_orb: str | None, n_per_orb: int = 1) -> int:
    """Last orbital column that is always embedded with a trainable row 0 (info.py:110-114; the
    reference treats index 0 as "unset", embed.py:64), or -1."""
    if not min_orb:
        return -1
    idx = _ORB.index(min_orb) * n_per_orb + (n_per_orb - 1)
    return idx if idx else -1


# --------------------------------------------------------------------------------------------
# index construction (reference: lcaonet.py:439-486 through torch_sparse)
# --------------------------------------------------------------------------------------------
def triplets(edge_index: torch.Tensor, n_nodes: int):
    """For every edge e=(s->t), in edge order, every edge e'=(k->s) INTO s, ordered by k ascending
    and (canonical tie-break) by edge id ascending; only e'==e (a self-loop) is dropped — the
    reference's mask compares edge ids (lcaonet.py:470), so back-tracking k==t triplets stay.

    Returns (tri_idx_k, edge_idx_ks, edge_idx_st), int64, length T = sum_e indeg(s_e) - #self-loops.
    """
    idx_s, idx_t = edge_index[0].cpu(), edge_index[1].cpu()
    E = idx_s.numel()
    order = torch.argsort(idx_t * n_nodes + idx_s, stable=True)  # by (target, source, edge id)
    indeg = torch.bincount(idx_t, minlength=n_nodes)
    ptr = torch.zeros(n_nodes + 1, dtype=torch.long)
    ptr[1:] = indeg.cumsum(0)
    cnt = indeg[idx_s]
    e_st = torch.arange(E).repeat_interleave(cnt)
    first = (cnt.cumsum(0) - cnt).repeat_interleave(cnt)
    pos = ptr[idx_s].repeat_interleave(cnt) + (torch.arange(e_st.numel()) - first)
    e_ks = order[pos]
    keep = e_ks != e_st
    e_ks, e_st = e_ks[keep], e_st[keep]
    dev = edge_index.device
    return idx_s[e_ks].to(dev), e_ks.to(dev), e_st.to(dev)


# --------------------------------------------------------------------------------------------
# geometry (reference: base.py:27-43, lcaonet.py:417-437)
# --------------------------------------------------------------------------------------------
def edge_geometry(pos, edge_index, edge_shift, lattice, batch):
    """vec = pos[t] - pos[s] + shift @ lattice[batch[s]];  dist = |vec|;  unit = vec / dist."""
    s, t = edge_index
    if batch is None:
        batch = torch.zeros(pos.shape[0], dtype=torch.long, device=pos.device)
    cell = lattice[batch[s]]  # (E, 3, 3)
    vec = pos[t] - pos[s] + (edge_shift.unsqueeze(-1) * cell).sum(1)
    dist = vec.norm(dim=1)
    return dist, vec / dist.unsqueeze(-1)


def triplet_cosines(unit, e_st, e_ks):
    return (unit[e_st] * unit[e_ks]).sum(-1)


# --------------------------------------------------------------------------------------------
# cutoffs (reference: cutoff.py:28-67)
# --------------------------------------------------------------------------------------------
def cutoff_fn(kind: str, r, rc: float):
    kind = kind.lower().replace("-", "").replace("_", "").replace(" ", "")
    if kind.endswith("cutoff"):
        kind = kind[: -len("cutoff")]
    q = r / rc
    if kind == "polynomial":
        val = 1 - 6 * q**5 + 15 * q**4 - 10 * q**3
    elif kind == "cosine":
        val = 0.5 * (torch.cos(r * math.pi / rc) + 1.0)
    elif kind == "envelope":  # p = 5: a=-21, b=35, c=-15
        val = 1 - 21.0 * q**5 + 35.0 * q**6 - 15.0 * q**7
    else:
        raise ValueError(f"{kind} not found")
    return torch.where(r <= rc, val, torch.zeros_like(val))


# --------------------------------------------------------------------------------------------
# radial basis (reference: rbf.py:67-105,129-142; spherical Bessel variant rbf.py:164-182)
# --------------------------------------------------------------------------------------------
def laguerre_poly(n: int, l: int) -> list[int]:
    """Ascending integer coefficients of  -(n+l)! * L_{n-l-1}^{(2l+1)}(x)  (rbf.py:82-87; the
    reference's factor (-1)^(2l+1) is always -1)."""
    k, a = n - l - 1, 2 * l + 1
    coef = []
    for i in range(k + 1):
        c = Fraction((-1) ** i * math.comb(k + a, k - i), math.factorial(i)) * (-math.factorial(n + l))
        assert c.denominator == 1
        coef.append(int(c))
    return coef


def radial_norm(n: int, l: int, a0: float = 0.529) -> float:
    """-sqrt((2/(n a0))^3 (n-l-1)! / (2n (n+l)!^3))  (rbf.py:92-94)."""
    return -math.sqrt((2.0 / n / a0) ** 3 * math.factorial(n - l - 1) / 2.0 / n / math.factorial(n + l) ** 3)


def radial_basis(dist, nl, rc: float, cutoff_kind: str, rbf_type: str = "hydrogen", a0: float = 0.529):
    """(E,) -> (E, n_orb):  fc(r) * s_nl * Lag(zeta) * zeta^l * exp(-zeta/2),  zeta = 2 r / (n a0)."""
    fc = cutoff_fn(cutoff_kind, dist, rc)
    cols = []
    kind = rbf_type.lower().replace("radialbasis", "").replace("_", "").replace("-", "")
    for n, l in nl:
        if kind == "hydrogen":
            zeta = 2.0 / n / a0 * dist
            poly = torch.zeros_like(dist)
            for c in reversed(laguerre_poly(n, l)):
                poly = poly * zeta + c
            cols.append(fc * radial_norm(n, l, a0) * poly * zeta**l * torch.exp(-zeta / 2.0))
        elif kind == "sphericalbessel":
            cols.append(fc * torch.sin(math.pi * n * dist / rc) / dist)
        else:
            raise ValueError(f"{rbf_type} not found")
    return torch.stack(cols, dim=1)


# --------------------------------------------------------------------------------------------
# angular basis (reference: shbf.py:28-87; only m = 0)
# --------------------------------------------------------------------------------------------
def legendre(l: int, c):
    if l == 0:
        return torch.ones_like(c)
    if l == 1:
        return c
    if l == 2:
        return 1.5 * c * c - 0.5
    if l == 3:
        return 2.5 * c**3 - 1.5 * c
    raise ValueError(l)


def angular_basis(cos_theta, nl):
    """(T,) -> (T, n_orb):  Y_l^0 = sqrt((2l+1)/(4 pi)) P_l(cos theta)."""
    return torch.stack([math.sqrt((2 * l + 1) / (4 * math.pi)) * legendre(l, cos_theta) for _, l in nl], dim=1)


# --------------------------------------------------------------------------------------------
# small helpers
# --------------------------------------------------------------------------------------------
def _lin(p, name, x):
    return F.linear(x, p[name + ".weight"], p.get(name + ".bias"))


# activations `activation_resolver` can return without parameters (utils/resolve.py:65-76, nn/activation.py:36-65);
# names normalised like the reference does (lower case, no '-', '_', ' ')
_ACTIVATIONS = {"silu": F.silu, "shiftedsoftplus": lambda x: F.softplus(x) - math.log(2.0), "softplus": F.softplus,
                "relu": F.relu, "tanh": torch.tanh, "sigmoid": torch.sigmoid, "gelu": F.gelu, "elu": F.elu,
                "leakyrelu": F.leaky_relu}


def _act(cfg, p=None):
    name = str(cfg.get("activation", "SiLU")).lower().replace("-", "").replace("_", "").replace(" ", "")
    if name == "swish":
        # nn/activation.py:7-33: x sigmoid(beta x); the reference shares ONE Swish module (one trainable beta) between all
        # its blocks, so every site uses the first `.beta` entry of the state dict (where its gradient accumulates)
        beta = p[next(k for k in p if k.endswith(".beta"))]
        return lambda x: x * torch.sigmoid(beta * x)
    return _ACTIVATIONS[name]


def _batch_norm(p, name, x, training: bool, new_stats: dict | None):
    """nn.BatchNorm1d semantics (embed.py:175,232): batch statistics + running-stat update
    (momentum 0.1, unbiased running variance) in training, running statistics in eval."""
    rm, rv = p[name + ".running_mean"], p[name + ".running_var"]
    if training and new_stats is not None:
        rm, rv = rm.clone(), rv.clone()
        new_stats[name + ".running_mean"], new_stats[name + ".running_var"] = rm, rv
    elif training:
        rm = rv = None
    return F.batch_norm(x, rm, rv, p[name + ".weight"], p[name + ".bias"], training, 0.1, 1e-5)


def _segment_sum(src, index, size):
    out = src.new_zeros((size,) + tuple(src.shape[1:]))
    return out.index_add(0, index, src)


# --------------------------------------------------------------------------------------------
# embedding block (reference: lcaonet.py:59-74, embed.py:32-41,81-99,177-194,234-249)
# --------------------------------------------------------------------------------------------
def embedding(p, cfg, z, idx_s, idx_t, training, new_stats=None):
    H, K = cfg["emb_size"], cfg["emb_size_coeff"]
    n_orb = p["emb_layer.e_embed.elec"].shape[1]
    zemb = p["emb_layer.z_embed.z_embed.weight"][z - 1]  # EmbedZ indexes with z-1
    node_z, coeff_z = zemb[:, :H], zemb[:, H:]
    occ = p["emb_layer.e_embed.elec"][z]  # (N, n_orb) electron counts, indexed with z
    # row 0 ("no electrons") is a frozen zero row (padding_idx=0, no gradient) unless the basis is
    # extended or the orbital is at/below min_orb (embed.py:64-71)
    min_idx = cfg.get("_min_orb_idx", -1)
    eemb = torch.stack([
        F.embedding(occ[:, o], p[f"emb_layer.e_embed.e_embeds.{o}.weight"],
                    padding_idx=None if (o <= min_idx or cfg.get("extend_orb", False)) else 0)
        for o in range(n_orb)], dim=1)
    if cfg["elec_to_node"]:
        node_e, coeff_e = eemb[..., :H], eemb[..., H:]
        enc_in = torch.cat([node_z, node_e.sum(1) / math.sqrt(n_orb)], dim=-1)
    else:
        coeff_e = eemb
        enc_in = node_z
    h = _act(cfg, p)(_lin(p, "emb_layer.node_embed.f_enc.0", enc_in))
    h = _act(cfg, p)(_lin(p, "emb_layer.node_embed.f_enc.2", h))
    x = _batch_norm(p, "emb_layer.node_embed.bn", h, training, new_stats)

    fz = _lin(p, "emb_layer.coeff_embed.f_z.0", torch.cat([coeff_z[idx_s], coeff_z[idx_t]], dim=-1))  # (E, K)
    fe = _act(cfg, p)(_lin(p, "emb_layer.coeff_embed.f_e.0", coeff_e))
    fe = _act(cfg, p)(_lin(p, "emb_layer.coeff_embed.f_e.2", fe))[idx_t]  # (E, n_orb, K): orbitals of the TARGET
    pre = fe + fe * fz.unsqueeze(1)
    cst = _batch_norm(p, "emb_layer.coeff_embed.bn", pre.reshape(pre.shape[0], -1), training, new_stats)
    return x, cst.reshape(pre.shape)


# --------------------------------------------------------------------------------------------
# interaction block (reference: lcaonet.py:130-216)
# --------------------------------------------------------------------------------------------
def interaction(p, pre, cfg, x, cst, vmask, rb, shb, idx_s, idx_t, tri_k, e_ks, e_st, trace=None):
    C = cfg["emb_size_conv"]
    x_in = x
    nw = _lin(p, pre + "node_weight", x)
    xc, xk = nw[:, :C], nw[:, C:]
    c1 = _act(cfg, p)(_lin(p, pre + "f_coeffs.0", cst))
    c1 = _act(cfg, p)(_lin(p, pre + "f_coeffs.2", c1))  # (E, O, C')
    # three-body: gather the coefficient rows of the incoming edge (k->s) of every triplet
    w3 = rb[e_ks] * shb  # (T, O)
    if cfg["add_valence"]:
        gathered = c1[e_ks]
        v = torch.einsum("to,toc->tc", w3, gathered[..., :C])
        v = v + torch.einsum("to,toc->tc", w3, gathered[..., C:] * vmask[e_ks].unsqueeze(-1))
    else:
        v = torch.einsum("to,toc->tc", w3, c1[e_ks])
    v = F.normalize(v, dim=-1) * torch.sigmoid(xk[tri_k])
    tbw = _segment_sum(v, e_st, rb.shape[0])  # triplets -> edges
    c2 = c1 + c1 * _lin(p, pre + "f_three.0", tbw).unsqueeze(1)
    # two-body
    if cfg["add_valence"]:
        lw = torch.einsum("eo,eoc->ec", rb, c2[..., :C]) + torch.einsum(
            "eo,eoc->ec", rb, c2[..., C:] * vmask.unsqueeze(-1))
    else:
        lw = torch.einsum("eo,eoc->ec", rb, c2)
    lw = F.normalize(lw, dim=-1)
    h = _act(cfg, p)(_lin(p, pre + "f_node.0", torch.cat([xc[idx_s], xc[idx_t]], dim=-1)))
    h = _act(cfg, p)(_lin(p, pre + "f_node.2", h))
    msg = _lin(p, pre + "basis_weight", lw) * h
    agg = _segment_sum(msg, idx_s, x.shape[0])  # edges -> source/centre nodes
    if trace is not None:
        trace[pre + "cst1"], trace[pre + "tbw"], trace[pre + "lw"], trace[pre + "agg"] = c1, tbw, lw, agg
    return x_in + _lin(p, pre + "out_weight", agg)


# --------------------------------------------------------------------------------------------
# output block + post-processing (reference: lcaonet.py:271-319, post.py:44-89)
# --------------------------------------------------------------------------------------------
def _mlp3(p, pre, x, cfg):
    x = _act(cfg, p)(_lin(p, pre + ".0", x))
    x = _act(cfg, p)(_lin(p, pre + ".2", x))
    return _lin(p, pre + ".4", x)


def _per_graph(val, batch, n_graph, extensive: bool):
    if batch is None:
        return val.sum(0, keepdim=True) if extensive else val.mean(0, keepdim=True)
    out = _segment_sum(val, batch, n_graph)
    if not extensive:
        cnt = torch.bincount(batch, minlength=n_graph).clamp(min=1).to(val.dtype)
        out = out / cnt.unsqueeze(-1)
    return out


def forward(params: dict, cfg: dict, graph, training: bool = True, trace: dict | None = None,
            new_stats: dict | None = None):
    """LCAONet.forward (lcaonet.py:488-540).  `cfg` holds the constructor keyword arguments.
    Returns energies (B, out) or (energies, forces (N, 3))."""
    p = params
    z, pos = graph["z"], graph["pos"]
    ei = graph["edge_index"]
    idx_s, idx_t = ei[0], ei[1]
    batch = graph.get("batch")
    lattice, shift = graph["lattice"], graph["edge_shift"]
    n_graph = lattice.shape[0]
    autograd_forces = cfg.get("regress_forces", False) and not cfg.get("direct_forces", True)
    if autograd_forces and not pos.requires_grad:
        pos = pos.detach().requires_grad_(True)
    nl = orbital_quantum_numbers(cfg["max_z"], cfg.get("max_orb"), cfg.get("n_per_orb", 1))
    cfg = dict(cfg)
    cfg["_min_orb_idx"] = min_orb_index(cfg.get("min_orb"), cfg.get("n_per_orb", 1))

    tri_k, e_ks, e_st = triplets(ei, z.shape[0])
    dist, unit = edge_geometry(pos, ei, shift, lattice, batch)
    cos_t = triplet_cosines(unit, e_st, e_ks)
    rb = radial_basis(dist, nl, cfg["cutoff"], cfg["cutoff_net"], cfg.get("rbf_type", "hydrogen"))
    shb = angular_basis(cos_t, nl)
    x, cst = embedding(p, cfg, z, idx_s, idx_t, training, new_stats)
    vmask = p["valence_mask.valence"][z][idx_t].to(cst.dtype) if cfg["add_valence"] else None  # (E, O)
    if trace is not None:
        trace.update(tri_k=tri_k, e_ks=e_ks, e_st=e_st, dist=dist, unit=unit, cos=cos_t, rb=rb, shb=shb, x0=x, cst=cst)
    for i in range(cfg["n_interaction"]):
        x = interaction(p, f"int_layers.{i}.", cfg, x, cst, vmask, rb, shb, idx_s, idx_t, tri_k, e_ks, e_st, trace)
        if trace is not None:
            trace[f"x{i + 1}"] = x
    ext = cfg.get("is_extensive", True)
    energy = _per_graph(_mlp3(p, "out_layer.out_lin", x, cfg), batch, n_graph, ext)
    forces = None
    if cfg.get("regress_forces", False):
        if cfg.get("direct_forces", True):
            f_e = _mlp3(p, "out_layer.out_lin_force", torch.cat([x[idx_s], x[idx_t]], dim=-1), cfg) * unit
            forces = _segment_sum(f_e, idx_s, x.shape[0])
        else:
            cols = [-torch.autograd.grad(energy[:, i].sum(), pos, create_graph=True)[0] for i in range(energy.shape[1])]
            forces = cols[0] if len(cols) == 1 else torch.stack(cols, dim=1).squeeze(1)
    if p.get("pp_layer.atomref") is not None:
        energy = energy + _per_graph(p["pp_layer.atomref"][z], batch, n_graph, ext)
    if p.get("pp_layer.mean") is not None:
        m = p["pp_layer.mean"].unsqueeze(0)
        if ext:
            m = _per_graph(m.expand(z.shape[0], -1), batch, n_graph, True)
        energy = energy + m
    return energy if forces is None else (energy, forces)


def cast_params(state_dict: dict, dtype=torch.float64, device="cpu", requires_grad: bool = False) -> dict:
    """Copy a reference-named state_dict into a parameter dict of `dtype` (integer buffers kept)."""
    out = {}
    for k, v in state_dict.items():
        if v is None:
            continue
        if v.is_floating_point():
            t = v.detach().to(device=device, dtype=dtype).clone()
            if requires_grad and "running_" not in k and not k.startswith("pp_layer."):
                t.requires_grad_(True)
            out[k] = t
        else:
            out[k] = v.detach().to(device).clone()
    return out
