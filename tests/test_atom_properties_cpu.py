"""Per-atom energies and per-atom virials (LCAONet.regress_atom_energy / regress_atom_virial) checked on CPU through the
torch emulator of the C ABI (tests/cpu_abi.py, plus the restatement of lcao_geom_atom_virial_bwd below), against FP64
autograd of the oracle:
  W_i = d E / d eps_i  for a per-atom strain acting on the edge vectors as  vec_e -> vec_e + 1/2 vec_e (eps_s + eps_t),
  e_i = out_lin(x_i) + atomref[z_i] + mean  from the oracle's last node features."""
import pytest
import torch

from lcaonet_b200 import LCAONet  # (import the package before the emulator is installed)
from lcaonet_b200.keys import GraphKeys
from lcaonet_b200.synth import GraphBatch, reference_fixture_graph
from oracle import lcao_oracle as O
from tests._util import full_cfg, graph_as, load_golden, rel_l2
from tests.test_stress_cpu import lcao_geom_cell_bwd

F32, I32, I64, F64 = torch.float32, torch.int32, torch.int64, torch.float64


def lcao_geom_atom_virial_bwd(pos, shift, lattice, batch, dst32, in_ptr, in_edge, in_src, out_ptr, out_edge, dvec, E, N,
                              atom_virial, stream):
    """torch restatement of the C-ABI entry point (include/lcao_b200.h), in the style of tests/cpu_abi.py: 1/2 vec (x) dvec
    of every edge added to its source and to its target, vec in FP64 as the forward forms it"""
    from tests.cpu_abi import view
    W = torch.zeros(N, 3, 3, dtype=F64)
    if E:
        op = view(out_ptr, N + 1, dtype=I32).long()
        s = torch.empty(E, dtype=I64)
        s[view(out_edge, E, dtype=I32).long()] = torch.repeat_interleave(torch.arange(N), op[1:] - op[:-1])
        t = view(dst32, E, dtype=I32).long()
        b = view(batch, N, dtype=I64)[s] if batch else torch.zeros(E, dtype=I64)
        L = view(lattice, (int(b.max()) + 1) * 3, 3).double().reshape(-1, 3, 3)[b]
        P, sh, dv = view(pos, N, 3).double(), view(shift, E, 3).double(), view(dvec, E, 3).double()
        v = (P[t] - P[s]) + (sh.unsqueeze(-1) * L).sum(1)
        half = 0.5 * v.unsqueeze(2) * dv.unsqueeze(1)
        W.index_add_(0, s, half).index_add_(0, t, half)
    if N:
        view(atom_virial, N * 9).copy_(W.reshape(-1).float())


def _install(monkeypatch):
    """the C-ABI emulator of tests/cpu_abi.py, with the per-atom and the per-graph virial entry points added to its table"""
    from tests import cpu_abi
    cpu_abi.install(monkeypatch)
    monkeypatch.setitem(cpu_abi._TABLE, "lcao_geom_atom_virial_bwd", lcao_geom_atom_virial_bwd)
    monkeypatch.setitem(cpu_abi._TABLE, "lcao_geom_cell_bwd", lcao_geom_cell_bwd)


def oracle_atom_terms(p, cfg, g, monkeypatch, training=False, create_graph=False, pos=None):
    """FP64 (or `p`'s dtype) oracle: (energy, e_i, W_i[, d E / d pos]).  W_i is the gradient with respect to a zero per-atom
    strain that a wrapper of `oracle.lcao_oracle.edge_geometry` injects into the edge vectors; e_i is out_lin of the
    oracle's last node features plus atomref[z] and mean.  `pos` (a leaf with requires_grad) also returns d E / d pos."""
    cfg = dict(cfg, regress_forces=False)  # energy only: the derivatives are taken here
    g = dict(g)
    if pos is not None:
        g["pos"] = pos
    N = g["pos"].shape[0]
    eps = torch.zeros(N, 3, 3, dtype=g["pos"].dtype, requires_grad=True)
    geometry = O.edge_geometry

    def strained(pos_, edge_index, edge_shift, lattice, batch):
        dist, unit = geometry(pos_, edge_index, edge_shift, lattice, batch)
        s, t = edge_index
        vec = unit * dist.unsqueeze(-1)
        vec = vec + 0.5 * (vec.unsqueeze(-1) * (eps[s] + eps[t])).sum(1)
        d = vec.norm(dim=1)
        return d, vec / d.unsqueeze(-1)

    trace = {}
    with monkeypatch.context() as m:
        m.setattr(O, "edge_geometry", strained)
        energy = O.forward(p, cfg, g, training=training, trace=trace)
    wrt = [eps] if pos is None else [eps, pos]
    grads = [torch.autograd.grad(energy[:, i].sum(), wrt, create_graph=create_graph, retain_graph=True)
             for i in range(energy.shape[1])]
    W = grads[0][0] if len(grads) == 1 else torch.stack([gr[0] for gr in grads], dim=1)
    e = O._mlp3(p, "out_layer.out_lin", trace[f"x{cfg['n_interaction']}"], cfg)
    if p.get("pp_layer.atomref") is not None:
        e = e + p["pp_layer.atomref"][g["z"]]
    if p.get("pp_layer.mean") is not None:
        e = e + p["pp_layer.mean"].unsqueeze(0)
    if pos is None:
        return energy, e, W
    return energy, e, W, grads[0][1]


def oracle_atom_properties(kwargs, state_dict, graph, monkeypatch, training=False):
    """(energy, e_i, W_i) of the FP64 oracle for a golden-style case"""
    p = O.cast_params(state_dict, F64)
    return oracle_atom_terms(p, full_cfg(kwargs), graph_as(graph, F64), monkeypatch, training)


def graph_virial_sums(atom_virial, graph):
    """sum_{i in g} W_i per graph, in FP64"""
    b = graph.get("batch")
    b = torch.zeros(atom_virial.shape[0], dtype=I64, device=atom_virial.device) if b is None else b.to(atom_virial.device)
    B = graph["lattice"].shape[0]
    return torch.zeros(B, *atom_virial.shape[1:], dtype=F64, device=atom_virial.device).index_add_(0, b, atom_virial.double())


def graph_energy_sums(atom_energy, graph, extensive):
    b = graph.get("batch")
    b = torch.zeros(atom_energy.shape[0], dtype=I64, device=atom_energy.device) if b is None else b.to(atom_energy.device)
    B = graph["lattice"].shape[0]
    out = torch.zeros(B, atom_energy.shape[1], dtype=F64, device=atom_energy.device).index_add_(0, b, atom_energy.double())
    if not extensive:
        out = out / torch.bincount(b, minlength=B).clamp(min=1).double().unsqueeze(1)
    return out


def _fixture_case():
    """the 3-atom periodic fixture (duplicate images, a self-image edge, edges beyond the cutoff) with the model of the
    reference's force test"""
    torch.manual_seed(0)
    kw = dict(emb_size=16, emb_size_coeff=16, emb_size_conv=16, out_size=1, n_interaction=2, cutoff=2.0,
              cutoff_net="envelope", max_z=5, regress_forces=True, direct_forces=False)
    model = LCAONet(**kw)
    return kw, {k: v.detach().clone() for k, v in model.state_dict().items()}, dict(reference_fixture_graph())


def _case(name):
    if name == "fixture":
        return _fixture_case()
    gold = load_golden(name)
    return gold["kwargs"], gold["state_dict"], gold["graph"]


def _model(kwargs, state_dict, energy=True, virial=True, stress=False):
    model = LCAONet(**kwargs)
    model.load_state_dict(state_dict, strict=True)
    model.eval()
    model.regress_atom_energy, model.regress_atom_virial, model.regress_stress = energy, virial, stress
    return model


@pytest.mark.parametrize("name", ["crystal_autograd_forces", "cfg4_crystal_width128", "fixture"])
def test_atom_virials_and_energies_match_oracle(name, monkeypatch):
    _install(monkeypatch)
    kwargs, sd, graph = _case(name)
    ref_energy, ref_e, ref_W = oracle_atom_properties(kwargs, sd, graph, monkeypatch)
    g = GraphBatch({k: v.clone() for k, v in graph.items()})
    energy, forces, stress = _model(kwargs, sd, stress=True)(g)
    W, e = g[GraphKeys.Atom_virial], g[GraphKeys.Atom_energy]
    N = graph["pos"].shape[0]
    assert W.shape == (N, 3, 3) and W.dtype == F32 and e.shape == (N, 1)
    assert rel_l2(W, ref_W) < 2e-5, rel_l2(W, ref_W)
    assert rel_l2(e, ref_e) < 2e-5, rel_l2(e, ref_e)
    # sum rules: the per-atom virials of a graph add up to its virial W_g = stress_g |det L_g|, the per-atom energies to
    # its energy
    vol = torch.linalg.det(graph["lattice"].double()).abs().view(-1, 1, 1)
    assert rel_l2(graph_virial_sums(W, graph), stress.double() * vol) < 1e-6
    assert rel_l2(graph_virial_sums(ref_W, graph), graph_virial_sums(W, graph)) < 2e-5
    assert rel_l2(graph_energy_sums(e, graph, True), energy) < 1e-6


@pytest.mark.parametrize("extensive", [True, False])
def test_atom_energies_with_atomref_and_mean_match_oracle(extensive, monkeypatch):
    """the reference's cosine / min-max-orbital fixture with atomref and mean (energy only: no autograd forces)"""
    _install(monkeypatch)
    gold = load_golden("fixture_cosine_minmaxorb_atomref")
    kwargs, sd, graph = dict(gold["kwargs"], is_extensive=extensive), gold["state_dict"], gold["graph"]
    ref_energy, ref_e, _ = oracle_atom_properties(kwargs, sd, graph, monkeypatch)
    g = GraphBatch({k: v.clone() for k, v in graph.items()})
    energy = _model(kwargs, sd, virial=False)(g)
    e = g[GraphKeys.Atom_energy]
    assert GraphKeys.Atom_virial not in g
    assert rel_l2(e, ref_e) < 2e-5, rel_l2(e, ref_e)
    assert rel_l2(energy, ref_energy) < 2e-5
    assert rel_l2(graph_energy_sums(e, graph, extensive), energy) < 1e-6


@pytest.mark.parametrize("out_size", [1, 2])
def test_shapes_and_unchanged_outputs(out_size, monkeypatch):
    _install(monkeypatch)
    gold = load_golden("crystal_autograd_forces")
    g = dict(gold["graph"])
    N = g["pos"].shape[0]
    two = {"z": g["z"].repeat(2), "pos": g["pos"].repeat(2, 1), "edge_shift": g["edge_shift"].repeat(2, 1),
           "edge_index": torch.cat([g["edge_index"], g["edge_index"] + N], 1), "lattice": g["lattice"].repeat(2, 1, 1),
           "batch": torch.cat([g["batch"], g["batch"] + 1])}
    torch.manual_seed(0)
    kw = dict(emb_size=16, emb_size_coeff=16, emb_size_conv=16, n_interaction=1, cutoff=6.0, cutoff_net="polynomial",
              out_size=out_size, regress_forces=True, direct_forces=False)
    model = LCAONet(**kw).eval()
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    plain_batch = GraphBatch({k: v.clone() for k, v in two.items()})
    plain = model(plain_batch)
    assert GraphKeys.Atom_energy not in plain_batch and GraphKeys.Atom_virial not in plain_batch
    model.regress_atom_energy = model.regress_atom_virial = True
    b = GraphBatch({k: v.clone() for k, v in two.items()})
    out = model(b)
    assert isinstance(out, tuple) and len(out) == 2  # the return value keeps its shape
    assert torch.equal(out[0], plain[0]) and torch.equal(out[1], plain[1])
    W, e = b[GraphKeys.Atom_virial], b[GraphKeys.Atom_energy]
    assert e.shape == (2 * N, out_size)
    assert W.shape == ((2 * N, 3, 3) if out_size == 1 else (2 * N, out_size, 3, 3))
    assert torch.allclose(W[:N], W[N:], rtol=1e-5, atol=1e-7)  # identical cells
    ref_energy, ref_e, ref_W = oracle_atom_properties(kw, sd, two, monkeypatch)
    assert rel_l2(W, ref_W) < 2e-5 and rel_l2(e, ref_e) < 2e-5, (rel_l2(W, ref_W), rel_l2(e, ref_e))
    model.regress_stress = True
    energy, forces, stress = model(GraphBatch({k: v.clone() for k, v in two.items()}))
    vol = torch.linalg.det(two["lattice"].double()).abs().view(-1, *([1] * (stress.dim() - 1)))
    assert rel_l2(graph_virial_sums(W, two), stress.double() * vol) < 1e-6
    if out_size == 2:  # one virial per output column
        assert not torch.allclose(W[:, 0], W[:, 1])


@pytest.mark.parametrize("kwargs", [dict(regress_forces=True, direct_forces=True), dict(regress_forces=False)])
def test_atom_virial_needs_autograd_forces(kwargs, monkeypatch):
    _install(monkeypatch)
    model = LCAONet(emb_size=16, emb_size_coeff=16, emb_size_conv=16, n_interaction=1, cutoff=2.0, max_z=5, **kwargs).eval()
    model.regress_atom_virial = True
    with pytest.raises(ValueError, match="regress_atom_virial"):
        model(reference_fixture_graph())
    model.regress_atom_virial, model.regress_atom_energy = False, True  # per-atom energies work with any configuration
    g = reference_fixture_graph()
    model(g)
    assert g[GraphKeys.Atom_energy].shape == (3, 1)
