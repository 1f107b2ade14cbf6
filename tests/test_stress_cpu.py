"""Stress and lattice gradients of periodic structures (LCAONet.regress_stress, ops.geom_basis) checked on CPU through the
torch emulator of the C ABI (tests/cpu_abi.py, plus the restatement of lcao_geom_cell_bwd below), against FP64
autograd of the oracle:
  stress = (1 / |det L|) d E / d eps  with  pos' = pos (I + eps),  L' = L (I + eps)  at eps = 0."""
import pytest
import torch

from lcaonet_b200 import LCAONet  # (import the package before the emulator is installed)
from lcaonet_b200.synth import GraphBatch, reference_fixture_graph
from oracle import lcao_oracle as O
from tests._util import full_cfg, graph_as, load_golden, rel_l2

F32, I32, I64, F64 = torch.float32, torch.int32, torch.int64, torch.float64


def lcao_geom_cell_bwd(pos, shift, lattice, batch, dst32, dvec, E, N, out_ptr, out_edge, seg_ptr, seg_perm, B, scratch,
                       d_lattice, virial, stream):
    """torch restatement of the C-ABI entry point (include/lcao_b200.h), in the style of tests/cpu_abi.py: per graph,
    d E / d L = sum_e shift_e (x) dvec_e and the virial sum_e vec_e (x) dvec_e, vec in FP64 as the forward forms it"""
    from tests.cpu_abi import view
    sp = view(seg_ptr, B + 1, dtype=I32).long()
    n_items = int(sp[-1])
    perm = view(seg_perm, n_items, dtype=I32).long() if seg_perm else torch.arange(n_items)
    graph_of = torch.zeros(N, dtype=I64)
    graph_of[perm] = torch.repeat_interleave(torch.arange(B), sp[1:] - sp[:-1])
    lat_g, vir_g = torch.zeros(B, 3, 3, dtype=F64), torch.zeros(B, 3, 3, dtype=F64)
    if E:
        op = view(out_ptr, N + 1, dtype=I32).long()
        s = torch.empty(E, dtype=I64)
        s[view(out_edge, E, dtype=I32).long()] = torch.repeat_interleave(torch.arange(N), op[1:] - op[:-1])
        t = view(dst32, E, dtype=I32).long()
        b = view(batch, N, dtype=I64)[s] if batch else torch.zeros(E, dtype=I64)
        L = view(lattice, (int(b.max()) + 1) * 3, 3).double().reshape(-1, 3, 3)[b]
        P, sh, dv = view(pos, N, 3).double(), view(shift, E, 3).double(), view(dvec, E, 3).double()
        v = (P[t] - P[s]) + (sh.unsqueeze(-1) * L).sum(1)
        lat_g.index_add_(0, graph_of[s], sh.unsqueeze(2) * dv.unsqueeze(1))
        vir_g.index_add_(0, graph_of[s], v.unsqueeze(2) * dv.unsqueeze(1))
    if d_lattice:
        view(d_lattice, B * 9).copy_(lat_g.reshape(-1).float())
    if virial:
        view(virial, B * 9).copy_(vir_g.reshape(-1).float())


def _install(monkeypatch):
    """the C-ABI emulator of tests/cpu_abi.py, with the cell-gradient entry point added to its table for this test"""
    from tests import cpu_abi
    cpu_abi.install(monkeypatch)
    monkeypatch.setitem(cpu_abi._TABLE, "lcao_geom_cell_bwd", lcao_geom_cell_bwd)


def _fixture_case():
    """the 3-atom periodic fixture (duplicate images, edges beyond the cutoff) with the model of the reference's force test"""
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


def oracle_cell_grads(kwargs, state_dict, graph):
    """FP64 oracle (eval mode): stress W / |det L| from a zero strain, and d E / d pos, d E / d lattice."""
    cfg = full_cfg(kwargs)
    cfg["regress_forces"] = False  # energy only: the derivatives are taken here
    p = O.cast_params(state_dict, torch.float64)
    g = graph_as(graph, torch.float64)
    B = g["lattice"].shape[0]
    b = g.get("batch")
    b = torch.zeros(g["pos"].shape[0], dtype=torch.long) if b is None else b
    eye = torch.eye(3, dtype=torch.float64)
    eps = torch.zeros(B, 3, 3, dtype=torch.float64, requires_grad=True)
    gs = dict(g)
    gs["pos"] = (g["pos"].unsqueeze(1) @ (eye + eps[b])).squeeze(1)
    gs["lattice"] = g["lattice"] @ (eye + eps)
    (W,) = torch.autograd.grad(O.forward(p, cfg, gs, training=False).sum(), eps)
    stress = W / torch.linalg.det(g["lattice"]).abs().view(-1, 1, 1)
    pos, lat = g["pos"].clone().requires_grad_(True), g["lattice"].clone().requires_grad_(True)
    gp = dict(g)
    gp["pos"], gp["lattice"] = pos, lat
    d_pos, d_lat = torch.autograd.grad(O.forward(p, cfg, gp, training=False).sum(), [pos, lat])
    return stress, W, d_pos, d_lat


def _model(kwargs, state_dict, stress=True):
    model = LCAONet(**kwargs)
    model.load_state_dict(state_dict, strict=True)
    model.eval()
    model.regress_stress = stress
    return model


@pytest.mark.parametrize("name", ["crystal_autograd_forces", "cfg4_crystal_width128", "fixture"])
def test_stress_and_cell_gradient_match_oracle(name, monkeypatch):
    _install(monkeypatch)
    kwargs, sd, graph = _case(name)
    ref_stress, ref_W, ref_dpos, ref_dlat = oracle_cell_grads(kwargs, sd, graph)
    energy, forces, stress = _model(kwargs, sd)(GraphBatch({k: v.clone() for k, v in graph.items()}))
    assert stress.shape == ref_stress.shape and stress.dtype == torch.float32
    assert rel_l2(stress, ref_stress) < 2e-5, rel_l2(stress, ref_stress)
    assert rel_l2(forces, -ref_dpos) < 2e-5
    # the user recipe: d E / d (pos, lattice) by autograd
    g = GraphBatch({k: v.clone() for k, v in graph.items()})
    pos, lat = g["pos"].requires_grad_(True), g["lattice"].requires_grad_(True)
    energy = _model(kwargs, sd, stress=False)(g)[0]
    d_pos, d_lat = torch.autograd.grad(energy.sum(), [pos, lat])
    assert d_lat.shape == lat.shape
    assert rel_l2(d_pos, ref_dpos) < 2e-5 and rel_l2(d_lat, ref_dlat) < 2e-5, (rel_l2(d_pos, ref_dpos), rel_l2(d_lat, ref_dlat))
    # the virial identity behind the kernel's edge form: W = sum_n pos_n (x) dpos_n + L^T dE/dL (one cell here)
    if ref_W.shape[0] == 1:
        W = pos.detach().double().T @ d_pos.double() + lat.detach()[0].double().T @ d_lat[0].double()
        assert rel_l2(W, ref_W[0]) < 2e-5


@pytest.mark.parametrize("kwargs", [dict(regress_forces=True, direct_forces=True), dict(regress_forces=False)])
def test_stress_needs_autograd_forces(kwargs, monkeypatch):
    _install(monkeypatch)
    model = LCAONet(emb_size=16, emb_size_coeff=16, emb_size_conv=16, n_interaction=1, cutoff=2.0, max_z=5, **kwargs).eval()
    model.regress_stress = True
    with pytest.raises(ValueError, match="regress_stress"):
        model(reference_fixture_graph())


@pytest.mark.parametrize("out_size", [1, 2])
def test_output_shapes_and_unchanged_outputs_without_stress(out_size, monkeypatch):
    _install(monkeypatch)
    gold = load_golden("crystal_autograd_forces")
    g = dict(gold["graph"])
    B = 2  # two copies of the cell in one batch
    N = g["pos"].shape[0]
    two = {"z": g["z"].repeat(2), "pos": g["pos"].repeat(2, 1), "edge_shift": g["edge_shift"].repeat(2, 1),
           "edge_index": torch.cat([g["edge_index"], g["edge_index"] + N], 1), "lattice": g["lattice"].repeat(2, 1, 1),
           "batch": torch.cat([g["batch"], g["batch"] + 1])}
    torch.manual_seed(0)
    kw = dict(emb_size=16, emb_size_coeff=16, emb_size_conv=16, n_interaction=1, cutoff=6.0, cutoff_net="polynomial",
              out_size=out_size, regress_forces=True, direct_forces=False)
    model = LCAONet(**kw).eval()
    plain = model(GraphBatch({k: v.clone() for k, v in two.items()}))
    assert isinstance(plain, tuple) and len(plain) == 2
    model.regress_stress = True
    energy, forces, stress = model(GraphBatch({k: v.clone() for k, v in two.items()}))
    assert energy.shape == (B, out_size)
    assert forces.shape == ((2 * N, 3) if out_size == 1 else (2 * N, out_size, 3))
    assert stress.shape == ((B, 3, 3) if out_size == 1 else (B, out_size, 3, 3))
    assert torch.equal(energy, plain[0]) and torch.equal(forces, plain[1])
    assert torch.allclose(stress[0], stress[1], rtol=1e-5, atol=1e-7)  # identical cells
    if out_size == 2:  # one stress per output column
        assert not torch.allclose(stress[:, 0], stress[:, 1])
