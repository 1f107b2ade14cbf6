"""Per-atom energies and per-atom virials on the B200: the lcao_geom_atom_virial_bwd kernel against an FP64 torch
restatement, and the model's values (LCAONet.regress_atom_energy / regress_atom_virial) against FP64 autograd of the oracle
with respect to a zero per-atom strain (vec_e -> vec_e + 1/2 vec_e (eps_s + eps_t); W_i = d E / d eps_i)."""
import pytest
import torch

from lcaonet_b200 import LCAONet, ops
from lcaonet_b200.dist import FlatGradBucket
from lcaonet_b200.keys import GraphKeys
from lcaonet_b200.synth import GraphBatch, qm9_like_batch
from oracle import lcao_oracle as O
from tests._util import full_cfg, graph_as, load_golden, rel_l2
from tests.test_atom_properties_cpu import graph_energy_sums, graph_virial_sums, oracle_atom_properties, oracle_atom_terms
from tests.test_gpu_stress import _sheared_batch

pytestmark = pytest.mark.gpu
DEV = "cuda"


# ---------------------------------------------------------------------------------------------------------------------
# the kernel
# ---------------------------------------------------------------------------------------------------------------------
def _atom_inputs(seed=0):
    """random geometry: 7 graphs whose atoms are interleaved (an empty graph, a graph without edges, a lone atom), one
    structure of 20 000 atoms x 55 out-edges (1.1 M edges), a hub atom with 3000 out- and 3000 in-edges, and 10 periodic
    self-image edges (s = t, non-zero shift)"""
    gen = torch.Generator().manual_seed(seed)
    sizes = [40, 0, 7, 300, 1, 20000, 64]  # graph 1 empty; graphs 2 and 4 get no edges
    B = len(sizes)
    batch = torch.cat([torch.full((n,), g, dtype=torch.long) for g, n in enumerate(sizes)])
    batch = batch[torch.randperm(batch.numel(), generator=gen)]  # atoms of a graph are NOT contiguous
    N = batch.numel()
    nodes_of = [torch.nonzero(batch == g).flatten() for g in range(B)]
    src, dst = [], []
    for g, nodes in enumerate(nodes_of):
        if g in (2, 4) or nodes.numel() == 0:
            continue
        deg = 55 if g == 5 else 9
        s = nodes.repeat_interleave(deg)
        src.append(s)
        dst.append(nodes[torch.randint(nodes.numel(), (s.numel(),), generator=gen)])
    hub, g3 = nodes_of[3][0], nodes_of[3]
    src += [hub.repeat(3000), g3[torch.randint(g3.numel(), (3000,), generator=gen)]]
    dst += [g3[torch.randint(g3.numel(), (3000,), generator=gen)], hub.repeat(3000)]
    n_rand = sum(s.numel() for s in src)
    selfs = nodes_of[0][:10]
    src.append(selfs)
    dst.append(selfs)
    ei = torch.stack([torch.cat(src), torch.cat(dst)])
    E = ei.shape[1]
    shift = torch.randint(-2, 3, (E, 3), generator=gen).float()
    shift[n_rand:] = torch.tensor([1.0, 0.0, -1.0])  # the self-image edges
    order = torch.randperm(E, generator=gen)
    ei, shift = ei[:, order], shift[order]
    lattice = 10 * torch.eye(3).repeat(B, 1, 1) + 2 * torch.rand(B, 3, 3, generator=gen)  # triclinic cells
    pos = 10 * torch.rand(N, 3, generator=gen)
    dvec = torch.randn(E, 3, generator=gen)
    return pos, shift, lattice, batch, ei, dvec


def _atom_reference(pos, shift, lattice, batch, ei, dvec):
    """FP64: 1/2 vec (x) dvec of every edge added to its source and to its target"""
    s, t = ei
    b = batch[s] if batch is not None else torch.zeros_like(s)
    P = pos.double()
    v = (P[t] - P[s]) + (shift.double().unsqueeze(-1) * lattice.double()[b]).sum(1)
    half = 0.5 * v.unsqueeze(2) * dvec.double().unsqueeze(1)
    W = torch.zeros(pos.shape[0], 3, 3, dtype=torch.float64, device=pos.device)
    return W.index_add_(0, s, half).index_add_(0, t, half)


def _run_kernel(pos, shift, lattice, batch, ei, dvec):
    gi = ops.GraphIndex(ei, pos.shape[0])
    return ops._atom_virial(dvec, pos, shift, lattice, batch, gi)


def _check_rows(W, ref, ei):
    deg = torch.bincount(ei.flatten(), minlength=W.shape[0])
    lone = deg == 0
    assert int(lone.sum()) > 0 and torch.equal(W[lone], torch.zeros_like(W[lone]))  # atoms without edges: exact zeros
    err = (W[~lone].double() - ref[~lone]).flatten(1).norm(dim=1)
    nrm = ref[~lone].flatten(1).norm(dim=1)
    worst = float((err / nrm).max())
    assert worst <= 1e-6, worst


def test_atom_kernel_matches_fp64_restatement():
    inputs = [x.to(DEV) for x in _atom_inputs()]
    pos, shift, lattice, batch, ei, dvec = inputs
    assert ei.shape[1] >= 10**6
    W = _run_kernel(*inputs)
    ref = _atom_reference(*inputs)
    assert W.shape == (pos.shape[0], 3, 3) and W.dtype == torch.float32
    _check_rows(W, ref, ei)
    W2 = _run_kernel(*inputs)
    assert torch.equal(W, W2)  # bitwise reproducible
    # graph sums: the cell kernel's virial
    seg = ops.bucket_sort(batch, lattice.shape[0])
    gi = ops.GraphIndex(ei, pos.shape[0])
    _, vir = ops._cell_grads(dvec, pos, shift, lattice, batch, gi, seg, False, True)
    assert rel_l2(graph_virial_sums(W, {"batch": batch, "lattice": lattice}), vir) <= 1e-6


def test_atom_kernel_single_graph_and_without_edges():
    pos, shift, lattice, batch, ei, dvec = _atom_inputs(seed=3)
    # the 300-atom graph with its hub as a structure of its own with batch=None, plus an atom without edges and an atom
    # whose only edge is a periodic self-image
    keep = batch[ei[0]] == 3
    nodes = torch.nonzero(batch == 3).flatten()
    M = nodes.numel()
    new_id = torch.full((batch.numel(),), -1, dtype=torch.long)
    new_id[nodes] = torch.arange(M)
    ins = [torch.cat([pos[nodes], torch.tensor([[1.0, 2.0, 3.0], [4.0, 5.0, 6.0]])]),
           torch.cat([shift[keep], torch.tensor([[0.0, 1.0, 0.0]])]), lattice[3:4], None,
           torch.cat([new_id[ei[:, keep]], torch.tensor([[M + 1], [M + 1]])], 1), torch.cat([dvec[keep], dvec[:1]])]
    ins = [x.to(DEV) if x is not None else None for x in ins]
    W = _run_kernel(*ins)
    _check_rows(W, _atom_reference(*ins), ins[4])
    # a self-image edge gives its atom 1/2 + 1/2: vec (x) dvec, vec = the second cell vector
    v, dv = ins[2][0, 1].double(), ins[5][-1].double()
    assert torch.allclose(W[M + 1].double(), torch.outer(v, dv), rtol=1e-6, atol=0)
    # E = 0: zeros
    W0 = _run_kernel(pos.to(DEV), shift[:0].to(DEV), lattice.to(DEV), batch.to(DEV), ei[:, :0].to(DEV), dvec[:0].to(DEV))
    assert torch.equal(W0, torch.zeros(pos.shape[0], 3, 3, device=DEV))


# ---------------------------------------------------------------------------------------------------------------------
# the model against the FP64 oracle
# ---------------------------------------------------------------------------------------------------------------------
def _graphs():
    out = {n: (load_golden(n)["kwargs"], load_golden(n)["state_dict"], load_golden(n)["graph"])
           for n in ("crystal_autograd_forces", "cfg4_crystal_width128")}
    kw, sd, _ = out["crystal_autograd_forces"]
    out["sheared_2cells"] = (kw, sd, _sheared_batch())
    # molecules with every edge at least 0.05 A inside the cutoff (the cutoff shell is ill-conditioned in FP32: SURVEY
    # Appendix B)
    out["qm9_molecules"] = (kw, sd, dict(qm9_like_batch(8, seed=3, cutoff=6.0, margin=0.05)))
    return out


def _model(kwargs, sd, energy=True, virial=True, stress=False, train=False):
    model = LCAONet(**kwargs)
    model.load_state_dict(sd, strict=True)
    model = model.to(DEV).train(train)
    model.regress_atom_energy, model.regress_atom_virial, model.regress_stress = energy, virial, stress
    return model


@pytest.mark.parametrize("name", ["crystal_autograd_forces", "cfg4_crystal_width128", "sheared_2cells", "qm9_molecules"])
def test_model_atom_properties_match_oracle(name, monkeypatch):
    kwargs, sd, graph = _graphs()[name]
    ref_energy, ref_e, ref_W = oracle_atom_properties(kwargs, sd, graph, monkeypatch)
    g = GraphBatch(graph).to(DEV)
    energy, forces, stress = _model(kwargs, sd, stress=True)(g)
    W, e = g[GraphKeys.Atom_virial], g[GraphKeys.Atom_energy]
    assert rel_l2(W, ref_W) <= 1e-5, rel_l2(W, ref_W)
    assert rel_l2(e, ref_e) <= 1e-5, rel_l2(e, ref_e)
    # sum rules against the same forward: sum_{i in g} W_i = stress_g |det L_g|, sum_{i in g} e_i = E_g
    vol = torch.linalg.det(graph["lattice"].double()).abs().view(-1, 1, 1).to(DEV)
    assert rel_l2(graph_virial_sums(W, g), stress.double() * vol) <= 1e-6, rel_l2(graph_virial_sums(W, g), stress.double() * vol)
    assert rel_l2(graph_energy_sums(e, g, True), energy) <= 1e-6


@pytest.mark.parametrize("extensive", [True, False])
def test_atom_energies_with_atomref_and_mean_match_oracle(extensive, monkeypatch):
    gold = load_golden("fixture_cosine_minmaxorb_atomref")
    kwargs, sd, graph = dict(gold["kwargs"], is_extensive=extensive), gold["state_dict"], gold["graph"]
    _, ref_e, _ = oracle_atom_properties(kwargs, sd, graph, monkeypatch)
    g = GraphBatch(graph).to(DEV)
    energy = _model(kwargs, sd, virial=False)(g)
    e = g[GraphKeys.Atom_energy]
    assert rel_l2(e, ref_e) <= 1e-5, rel_l2(e, ref_e)
    assert rel_l2(graph_energy_sums(e, g, extensive), energy) <= 1e-6


def test_out_size_two_matches_oracle(monkeypatch):
    kw, _, graph = _graphs()["sheared_2cells"]
    kw = dict(kw, out_size=2)
    torch.manual_seed(0)
    sd = {k: v.clone() for k, v in LCAONet(**kw).state_dict().items()}
    _, ref_e, ref_W = oracle_atom_properties(kw, sd, graph, monkeypatch)
    g = GraphBatch(graph).to(DEV)
    energy, forces, stress = _model(kw, sd, stress=True)(g)
    W, e = g[GraphKeys.Atom_virial], g[GraphKeys.Atom_energy]
    N = graph["pos"].shape[0]
    assert W.shape == (N, 2, 3, 3) and e.shape == (N, 2)
    assert rel_l2(W, ref_W) <= 1e-5 and rel_l2(e, ref_e) <= 1e-5, (rel_l2(W, ref_W), rel_l2(e, ref_e))
    vol = torch.linalg.det(graph["lattice"].double()).abs().view(-1, 1, 1, 1).to(DEV)
    assert rel_l2(graph_virial_sums(W, g), stress.double() * vol) <= 1e-6


def test_permutation_and_translation_invariance():
    kwargs, sd, graph = _graphs()["sheared_2cells"]
    model = _model(kwargs, sd)
    g = GraphBatch(graph).to(DEV)
    model(g)
    W, e = g[GraphKeys.Atom_virial], g[GraphKeys.Atom_energy]
    N = graph["pos"].shape[0]
    perm = torch.randperm(N, generator=torch.Generator().manual_seed(11))
    inv = torch.argsort(perm)
    gp = dict(graph)
    gp["z"], gp["pos"], gp["batch"] = graph["z"][perm], graph["pos"][perm], graph["batch"][perm]
    gp["edge_index"] = inv[graph["edge_index"]]
    gp = GraphBatch(gp).to(DEV)
    model(gp)
    assert rel_l2(gp[GraphKeys.Atom_virial], W[perm.to(DEV)]) <= 1e-5
    assert rel_l2(gp[GraphKeys.Atom_energy], e[perm.to(DEV)]) <= 1e-5
    gt = dict(graph)
    gt["pos"] = graph["pos"] + torch.tensor([0.37, -1.21, 2.93])
    gt = GraphBatch(gt).to(DEV)
    model(gt)
    assert rel_l2(gt[GraphKeys.Atom_virial], W) <= 1e-5, rel_l2(gt[GraphKeys.Atom_virial], W)
    assert rel_l2(gt[GraphKeys.Atom_energy], e) <= 1e-5


def test_switches_off_change_nothing():
    kwargs, sd, graph = _graphs()["sheared_2cells"]
    model = _model(kwargs, sd, energy=False, virial=False)

    def run():
        g = GraphBatch(graph).to(DEV)
        n0 = ops.n_calls
        out = model(g)
        return out, ops.n_calls - n0, g

    (e0, f0), calls0, g0 = run()
    assert GraphKeys.Atom_energy not in g0 and GraphKeys.Atom_virial not in g0
    model.regress_atom_energy = True
    (e1, f1), calls1, g1 = run()
    assert calls1 == calls0 and torch.equal(e1, e0) and torch.equal(f1, f0)
    assert GraphKeys.Atom_virial not in g1
    model.regress_atom_virial = True
    (e2, f2), calls2, g2 = run()
    assert calls2 == calls0 + 1  # the per-atom virial kernel, in the forces pass
    assert torch.equal(e2, e0) and torch.equal(f2, f0)
    assert not g2[GraphKeys.Atom_virial].requires_grad


# ---------------------------------------------------------------------------------------------------------------------
# training mode
# ---------------------------------------------------------------------------------------------------------------------
def test_training_mode_values_carry_a_graph_and_match_first_order():
    kwargs, sd, graph = _graphs()["sheared_2cells"]
    model = _model(kwargs, sd, train=True)
    # the differentiable backward scatters with torch's index_add, whose CUDA atomics move results by a few 1e-7 from run
    # to run: compare with torch's deterministic algorithms
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True, warn_only=True)
    try:
        g = GraphBatch(graph).to(DEV)
        model(g)
    finally:
        torch.use_deterministic_algorithms(prev)
    W, e = g[GraphKeys.Atom_virial], g[GraphKeys.Atom_energy]
    assert W.requires_grad and e.requires_grad
    model.out_layer.force_training = False  # same batch statistics, first-order kernels
    g1 = GraphBatch(graph).to(DEV)
    model(g1)
    assert not g1[GraphKeys.Atom_virial].requires_grad
    # the same forward kernels give the per-atom energies.  The differentiable backward evaluates every operator with
    # torch operations instead of the fused kernels, which moves W_i by 6e-6 rel-L2 on a B200: the bar of the same
    # comparison for the stress (test_stress_paths_and_reproducibility)
    assert rel_l2(e, g1[GraphKeys.Atom_energy]) <= 1e-6
    assert rel_l2(W, g1[GraphKeys.Atom_virial]) <= 1e-5, rel_l2(W, g1[GraphKeys.Atom_virial])


def _oracle_loss_grads(sd, kwargs, graph, dtype, monkeypatch):
    p = O.cast_params(sd, dtype, requires_grad=True)
    g = graph_as(graph, dtype)
    pos = g["pos"].clone().requires_grad_(True)
    energy, _, W, d_pos = oracle_atom_terms(p, full_cfg(kwargs), g, monkeypatch, training=True, create_graph=True, pos=pos)
    loss = (energy**2).mean() + (d_pos**2).mean() + (W**2).sum()
    names = [n for n, v in p.items() if v.requires_grad]
    grads = torch.autograd.grad(loss, [p[n] for n in names], allow_unused=True)
    return {n: gr for n, gr in zip(names, grads)}


@pytest.mark.parametrize("bucket", [False, True])
def test_atom_virial_loss_gradients_match_oracle(bucket, monkeypatch):
    gold = load_golden("crystal_autograd_forces")
    kwargs, sd, graph = gold["kwargs"], gold["state_dict"], gold["graph"]
    ref64 = _oracle_loss_grads(sd, kwargs, graph, torch.float64, monkeypatch)
    ref32 = _oracle_loss_grads(sd, kwargs, graph, torch.float32, monkeypatch)
    model = _model(kwargs, sd, energy=False, train=True)
    b = FlatGradBucket(model) if bucket else None
    for _ in range(2):  # (second step: graphed embedding tables replay)
        if b is not None:
            b.zero()
        else:
            model.zero_grad(set_to_none=True)
        g = GraphBatch(graph).to(DEV)
        energy, forces = model(g)
        W = g[GraphKeys.Atom_virial]
        assert W.requires_grad
        ((energy**2).mean() + (forces**2).mean() + (W**2).sum()).backward()
    checked = 0
    for n, q in model.named_parameters():
        ref = ref64.get(n)
        if ref is None or float(ref.norm()) == 0.0:
            continue
        bar = max(1e-4, 3 * rel_l2(ref32[n], ref))
        assert rel_l2(q.grad, ref) <= bar, (n, rel_l2(q.grad, ref), bar)
        checked += 1
    assert checked > 10


@pytest.mark.parametrize("kwargs", [dict(regress_forces=True, direct_forces=True), dict(regress_forces=False)])
def test_atom_virial_needs_autograd_forces(kwargs):
    model = LCAONet(emb_size=16, emb_size_coeff=16, emb_size_conv=16, n_interaction=1, cutoff=5.0, **kwargs).to(DEV).eval()
    model.regress_atom_virial = True
    with pytest.raises(ValueError, match="regress_atom_virial"):
        model(qm9_like_batch(2, seed=1, margin=0.05).to(DEV))
