"""Stress and lattice gradients on the B200: the lcao_geom_cell_bwd kernel against an FP64 torch restatement, and the model's
stress (LCAONet.regress_stress) against FP64 autograd of the oracle with respect to a zero strain
(pos' = pos (I + eps), L' = L (I + eps); stress = (d E / d eps) / |det L|)."""
import pytest
import torch

from lcaonet_b200 import LCAONet, ops
from lcaonet_b200.dist import FlatGradBucket
from lcaonet_b200.neighbors import build_neighbor_list
from lcaonet_b200.synth import GraphBatch, crystal_like_batch, qm9_like_batch, reference_fixture_graph
from oracle import lcao_oracle as O
from tests._util import full_cfg, graph_as, load_golden, rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda"


# ---------------------------------------------------------------------------------------------------------------------
# the kernel
# ---------------------------------------------------------------------------------------------------------------------
def _cell_inputs(seed=0):
    """random geometry: 6 graphs (a triclinic cell, an empty graph, a graph without edges, interleaved atoms) + one
    structure of 20 000 atoms x 55 out-edges (1.1 M edges, 157 chunks of LCAO_CELL_CHUNK nodes)"""
    gen = torch.Generator().manual_seed(seed)
    sizes = [40, 0, 7, 300, 1, 20000, 64]  # graph 1 empty; graph 2 gets no edges
    B = len(sizes)
    batch = torch.cat([torch.full((n,), g, dtype=torch.long) for g, n in enumerate(sizes)])
    batch = batch[torch.randperm(batch.numel(), generator=gen)]  # atoms of a graph are NOT contiguous
    N = batch.numel()
    nodes_of = [torch.nonzero(batch == g).flatten() for g in range(B)]
    src, dst = [], []
    for g, nodes in enumerate(nodes_of):
        if g == 2 or nodes.numel() == 0:
            continue
        deg = 55 if g == 5 else 9
        s = nodes.repeat_interleave(deg)
        src.append(s)
        dst.append(nodes[torch.randint(nodes.numel(), (s.numel(),), generator=gen)])
    ei = torch.stack([torch.cat(src), torch.cat(dst)])
    ei = ei[:, torch.randperm(ei.shape[1], generator=gen)]
    E = ei.shape[1]
    lattice = 10 * torch.eye(3).repeat(B, 1, 1) + 2 * torch.rand(B, 3, 3, generator=gen)  # triclinic cells
    pos = 10 * torch.rand(N, 3, generator=gen)
    shift = torch.randint(-2, 3, (E, 3), generator=gen).float()
    dvec = torch.randn(E, 3, generator=gen)
    return pos, shift, lattice, batch, ei, dvec


def _cell_reference(pos, shift, lattice, batch, ei, dvec):
    s, t = ei
    b = batch[s]
    P = pos.double()
    v = (P[t] - P[s]) + (shift.double().unsqueeze(-1) * lattice.double()[b]).sum(1)
    B = lattice.shape[0]
    dv = dvec.double()
    d_lat = torch.zeros(B, 3, 3, dtype=torch.float64, device=pos.device).index_add_(0, b, shift.double().unsqueeze(2) * dv.unsqueeze(1))
    vir = torch.zeros(B, 3, 3, dtype=torch.float64, device=pos.device).index_add_(0, b, v.unsqueeze(2) * dv.unsqueeze(1))
    return d_lat, vir


def _run_kernel(pos, shift, lattice, batch, ei, dvec):
    gi = ops.GraphIndex(ei, pos.shape[0])
    seg = ops.bucket_sort(batch, lattice.shape[0])
    return ops._cell_grads(dvec, pos, shift, lattice, batch, gi, seg, True, True)


def test_cell_kernel_matches_fp64_restatement():
    inputs = [x.to(DEV) for x in _cell_inputs()]
    pos, shift, lattice, batch, ei, dvec = inputs
    assert ei.shape[1] >= 10**6
    d_lat, vir = _run_kernel(*inputs)
    ref_lat, ref_vir = _cell_reference(*inputs)
    for g in range(lattice.shape[0]):
        for out, ref in ((d_lat, ref_lat), (vir, ref_vir)):
            if g == 1 or g == 2:  # empty graph, graph without edges
                assert torch.equal(out[g], torch.zeros_like(out[g]))
            else:
                assert rel_l2(out[g], ref[g]) <= 1e-6, (g, rel_l2(out[g], ref[g]))
    d_lat2, vir2 = _run_kernel(*inputs)
    assert torch.equal(d_lat, d_lat2) and torch.equal(vir, vir2)  # bitwise reproducible


def test_cell_kernel_without_edges_writes_zeros():
    pos, shift, lattice, batch, ei, dvec = _cell_inputs()
    B = lattice.shape[0]
    d_lat, vir = _run_kernel(pos.to(DEV), shift[:0].to(DEV), lattice.to(DEV), batch.to(DEV), ei[:, :0].to(DEV),
                             dvec[:0].to(DEV))
    assert torch.equal(d_lat, torch.zeros(B, 3, 3, device=DEV)) and torch.equal(vir, torch.zeros(B, 3, 3, device=DEV))


# ---------------------------------------------------------------------------------------------------------------------
# the model against the FP64 oracle
# ---------------------------------------------------------------------------------------------------------------------
def _oracle_stress(kwargs, state_dict, graph, training=False):
    cfg = full_cfg(kwargs)
    cfg["regress_forces"] = False
    p = O.cast_params(state_dict, torch.float64)
    g = graph_as(graph, torch.float64)
    b = g.get("batch")
    b = torch.zeros(g["pos"].shape[0], dtype=torch.long) if b is None else b
    eye = torch.eye(3, dtype=torch.float64)
    eps = torch.zeros(g["lattice"].shape[0], 3, 3, dtype=torch.float64, requires_grad=True)
    gs = dict(g)
    gs["pos"] = (g["pos"].unsqueeze(1) @ (eye + eps[b])).squeeze(1)
    gs["lattice"] = g["lattice"] @ (eye + eps)
    (W,) = torch.autograd.grad(O.forward(p, cfg, gs, training=training).sum(), eps)
    pos, lat = g["pos"].clone().requires_grad_(True), g["lattice"].clone().requires_grad_(True)
    gp = dict(g)
    gp["pos"], gp["lattice"] = pos, lat
    d_pos, d_lat = torch.autograd.grad(O.forward(p, cfg, gp, training=training).sum(), [pos, lat])
    return W / torch.linalg.det(g["lattice"]).abs().view(-1, 1, 1), d_pos, d_lat


def _sheared_batch(seed=7):
    """two cells sheared into triclinic ones, edges rebuilt (all ~50 neighbours kept), edges within 0.05 A of the cutoff
    dropped (the cutoff shell is ill-conditioned in FP32: SURVEY Appendix B)"""
    g = crystal_like_batch(2, seed, margin=0.05)
    S = torch.tensor([[1.0, 0.06, -0.03], [0.02, 0.97, 0.05], [-0.04, 0.01, 1.03]])
    pos, lat = g["pos"] @ S, g["lattice"] @ S
    ei, sh, _ = build_neighbor_list(pos.to(DEV), g["batch"].to(DEV), lat.to(DEV), torch.ones(2, 3, device=DEV), 6.0,
                                    max_neighbors=512)
    ei, sh = ei.cpu(), sh.cpu()
    b = g["batch"][ei[0]]
    d = (pos[ei[1]].double() - pos[ei[0]].double() + (sh.double().unsqueeze(-1) * lat.double()[b]).sum(1)).norm(dim=1)
    keep = d <= 6.0 - 0.05
    return {"z": g["z"], "pos": pos, "edge_index": ei[:, keep], "edge_shift": sh[keep], "lattice": lat, "batch": g["batch"]}


def _graphs():
    out = {n: (load_golden(n)["kwargs"], load_golden(n)["state_dict"], load_golden(n)["graph"])
           for n in ("crystal_autograd_forces", "cfg4_crystal_width128")}
    kw, sd, _ = out["crystal_autograd_forces"]
    out["sheared_2cells"] = (kw, sd, _sheared_batch())
    return out


def _model(kwargs, sd, stress=True, train=False):
    model = LCAONet(**kwargs)
    model.load_state_dict(sd, strict=True)
    model = model.to(DEV).train(train)
    model.regress_stress = stress
    return model


@pytest.mark.parametrize("name", ["crystal_autograd_forces", "cfg4_crystal_width128", "sheared_2cells"])
def test_model_stress_matches_oracle(name):
    kwargs, sd, graph = _graphs()[name]
    ref_stress, ref_dpos, ref_dlat = _oracle_stress(kwargs, sd, graph)
    energy, forces, stress = _model(kwargs, sd)(GraphBatch(graph).to(DEV))
    assert rel_l2(stress, ref_stress) <= 1e-5, rel_l2(stress, ref_stress)
    assert rel_l2(forces, -ref_dpos) <= 1e-5
    s = stress.double()
    assert float((s - s.transpose(-1, -2)).norm() / s.norm()) <= 1e-5
    # the user recipe: d E / d (pos, lattice)
    g = GraphBatch(graph).to(DEV)
    pos, lat = g["pos"].requires_grad_(), g["lattice"].requires_grad_()
    energy = _model(kwargs, sd, stress=False)(g)[0]
    d_pos, d_lat = torch.autograd.grad(energy.sum(), [pos, lat])
    assert rel_l2(d_pos, ref_dpos) <= 1e-5 and rel_l2(d_lat, ref_dlat) <= 1e-5, (rel_l2(d_pos, ref_dpos), rel_l2(d_lat, ref_dlat))


def test_stress_paths_and_reproducibility():
    kwargs, sd, graph = _graphs()["sheared_2cells"]
    g = GraphBatch(graph)
    # first-order kernels: eval mode, or training mode with force_training=False
    for train in (False, True):
        model = _model(kwargs, sd, train=train)
        model.out_layer.force_training = False if train else None
        e1, f1, s1 = model(g.to(DEV))
        e2, f2, s2 = model(g.to(DEV))
        assert not s1.requires_grad and torch.equal(s1, s2)
        model.regress_stress = False
        e0, f0 = model(g.to(DEV))
        assert torch.equal(e0, e1) and torch.equal(f0, f1)
    # training mode: differentiable path, same energy and forces with the switch on and off.  The differentiable backward
    # scatters with torch's index_add, whose CUDA atomics alone move the forces by a few 1e-6 from run to run: compare
    # with torch's deterministic algorithms
    model = _model(kwargs, sd, train=True)
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True, warn_only=True)
    try:
        e1, f1, s1 = model(g.to(DEV))
        assert s1.requires_grad
        model.regress_stress = False
        e0, f0 = model(g.to(DEV))
    finally:
        torch.use_deterministic_algorithms(prev)
    assert rel_l2(e1, e0) <= 1e-6 and rel_l2(f1, f0) <= 1e-6, (rel_l2(e1, e0), rel_l2(f1, f0))
    model.regress_stress = True
    model.out_layer.force_training = False  # same batch statistics, first-order kernels
    assert rel_l2(s1, model(g.to(DEV))[2]) <= 1e-5


def _oracle_loss_grads(sd, kwargs, graph, dtype):
    cfg = full_cfg(kwargs)
    cfg["regress_forces"] = False
    p = O.cast_params(sd, dtype, requires_grad=True)
    g = graph_as(graph, dtype)
    eye = torch.eye(3, dtype=dtype)
    eps = torch.zeros(g["lattice"].shape[0], 3, 3, dtype=dtype, requires_grad=True)
    b = g["batch"]
    pos = (g["pos"].unsqueeze(1) @ (eye + eps[b])).squeeze(1)
    gs = dict(g)
    gs["pos"], gs["lattice"] = pos, g["lattice"] @ (eye + eps)
    energy = O.forward(p, cfg, gs, training=True)
    d_pos, W = torch.autograd.grad(energy.sum(), [pos, eps], create_graph=True)
    stress = W / torch.linalg.det(g["lattice"]).abs().view(-1, 1, 1)
    loss = (energy**2).mean() + (d_pos**2).mean() + (stress**2).mean()
    names = [n for n, v in p.items() if v.requires_grad]
    grads = torch.autograd.grad(loss, [p[n] for n in names], allow_unused=True)
    return {n: gr for n, gr in zip(names, grads)}


@pytest.mark.parametrize("bucket", [False, True])
def test_stress_loss_gradients_match_oracle(bucket):
    gold = load_golden("crystal_autograd_forces")
    kwargs, sd, graph = gold["kwargs"], gold["state_dict"], gold["graph"]
    ref64 = _oracle_loss_grads(sd, kwargs, graph, torch.float64)
    ref32 = _oracle_loss_grads(sd, kwargs, graph, torch.float32)
    model = _model(kwargs, sd, train=True)
    b = FlatGradBucket(model) if bucket else None
    for _ in range(2):  # (second step: graphed embedding tables replay)
        if b is not None:
            b.zero()
        else:
            model.zero_grad(set_to_none=True)
        energy, forces, stress = model(GraphBatch(graph).to(DEV))
        assert stress.requires_grad
        ((energy**2).mean() + (forces**2).mean() + (stress**2).mean()).backward()
    checked = 0
    for n, q in model.named_parameters():
        ref = ref64.get(n)
        if ref is None or float(ref.norm()) == 0.0:
            continue
        bar = max(1e-4, 3 * rel_l2(ref32[n], ref))
        assert rel_l2(q.grad, ref) <= bar, (n, rel_l2(q.grad, ref), bar)
        checked += 1
    assert checked > 10


def test_degenerate_batches_give_finite_stress():
    """isolated atoms, a batch without edges, batch=None (cf. test_degenerate_graphs_match_oracle)"""
    kwargs = dict(emb_size=32, emb_size_coeff=32, emb_size_conv=32, cutoff=5.0, cutoff_net="polynomial",
                  regress_forces=True, direct_forces=False)
    torch.manual_seed(5)
    model = LCAONet(**kwargs).to(DEV).eval()
    model.regress_stress = True
    g = qm9_like_batch(3, seed=12, margin=0.05)
    g2 = GraphBatch(z=torch.cat([g["z"], torch.tensor([1, 8])]), pos=torch.cat([g["pos"], torch.tensor([[0.0, 0, 0], [30.0, 0, 0]])]),
                    edge_index=g["edge_index"], edge_shift=g["edge_shift"], lattice=torch.cat([g["lattice"], g["lattice"][:1]]),
                    batch=torch.cat([g["batch"], torch.tensor([3, 3])]))
    _, _, stress = model(g2.to(DEV))
    assert stress.shape == (4, 3, 3) and torch.isfinite(stress).all()
    assert torch.equal(stress[3], torch.zeros(3, 3, device=DEV)) and float(stress[:3].abs().sum()) > 0
    g3 = GraphBatch(z=torch.tensor([1, 6, 8]), pos=torch.tensor([[0.0, 0, 0], [20.0, 0, 0], [0, 20.0, 0]]),
                    edge_index=torch.zeros(2, 0, dtype=torch.long), edge_shift=torch.zeros(0, 3), lattice=50 * torch.eye(3).unsqueeze(0),
                    batch=torch.zeros(3, dtype=torch.long))
    _, forces, stress = model(g3.to(DEV))
    assert torch.equal(stress, torch.zeros(1, 3, 3, device=DEV)) and torch.equal(forces, torch.zeros(3, 3, device=DEV))
    g1 = qm9_like_batch(1, seed=13, margin=0.05)
    g1n = GraphBatch({k: v for k, v in g1.items() if k != "batch"})
    _, _, s1 = model(g1n.to(DEV))
    _, _, s1b = model(g1.to(DEV))
    assert s1.shape == (1, 3, 3) and torch.isfinite(s1).all() and torch.equal(s1, s1b)


def test_trainability_with_a_stress_term():
    """the reference's force-training test on the 3-atom periodic fixture with a stress term added to the loss"""
    torch.manual_seed(0)
    model = LCAONet(emb_size=16, emb_size_coeff=16, emb_size_conv=16, out_size=1, n_interaction=2, cutoff=2.0,
                    cutoff_net="envelope", max_z=5, regress_forces=True, direct_forces=False).to(DEV)
    model.regress_stress = True
    opt = torch.optim.Adam(model.parameters(), lr=0.001)
    g0 = reference_fixture_graph().to(DEV)
    mse = torch.nn.functional.mse_loss
    losses = []
    for _ in range(100):
        opt.zero_grad()
        energy, forces, stress = model(GraphBatch(g0))
        # (the fixture's 15 A box makes stresses ~1e-6 eV/A^3: the stress term is scaled to the size of the others)
        loss = (0.001 * mse(energy, torch.ones(1, 1, device=DEV)) + 0.999 * mse(forces, torch.ones(3, 3, device=DEV))
                + mse(1e4 * stress, torch.ones(1, 3, 3, device=DEV)))
        loss.backward()
        opt.step()
        losses.append(float(loss))
    assert all(x == x for x in losses) and losses[-1] < losses[0]
