"""Neighbour list (SURVEY.md §8 a-12 / f-1): the brute-force oracle against the synthetic generators' own edge sets
(CPU), the host wrapper through the emulator (CPU), and the CUDA kernels against the oracle, bit-exact (GPU)."""
import numpy as np
import pytest
import torch

from lcaonet_b200.synth import crystal_like_batch, qm9_like_batch
from oracle import neighbor_oracle as NO


def _as_set(src, dst, shift):
    return sorted(zip(np.asarray(src).tolist(), np.asarray(dst).tolist(), *[np.asarray(shift)[:, k].tolist() for k in range(3)]))


def _structures():
    q = qm9_like_batch(5, seed=4, cutoff=5.0, margin=0.05)
    q["pbc"] = torch.zeros(5, 3, dtype=torch.long)
    x = crystal_like_batch(2, seed=3, cutoff=6.0, margin=0.05)
    x["pbc"] = torch.ones(2, 3, dtype=torch.long)
    return {"qm9": (q, 5.0 - 0.05), "crystal": (x, 6.0 - 0.05)}  # the generators keep d <= cutoff - margin


@pytest.mark.parametrize("kind", ["qm9", "crystal"])
def test_oracle_reproduces_generator_edge_sets(kind):
    g, rc = _structures()[kind]
    gptr = np.concatenate([[0], np.bincount(g["batch"].numpy()).cumsum()])
    s, t, sh, cnt = NO.batch_neighbor_list(g["pos"].numpy(), gptr, g["lattice"].numpy(), g["pbc"].numpy(), rc, 10**6)
    assert _as_set(s, t, sh) == _as_set(g["edge_index"][0], g["edge_index"][1], g["edge_shift"].numpy())
    assert cnt.sum() == g["edge_index"].shape[1]
    # grouped by centre ascending, each centre sorted by distance
    assert (np.diff(s) >= 0).all()


def test_oracle_order_truncation_and_fallback():
    # perfect simple-cubic cell: 6 equidistant first neighbours per atom -> the canonical tie-break decides the order
    pos = np.zeros((1, 3), dtype=np.float32)
    cell = (2.0 * np.eye(3)).astype(np.float32)
    s, t, sh = NO.neighbor_list(pos, cell, [True] * 3, 2.5, 32)
    assert len(s) == 6 and sh.tolist() == sorted(sh.tolist())     # periodic self-images, (S0,S1,S2) ascending
    s, t, sh = NO.neighbor_list(pos, cell, [True] * 3, 2.5, 4)
    assert len(s) == 4 and sh.tolist() == sorted(sh.tolist())
    s, t, sh = NO.neighbor_list(pos, cell, [True, False, False], 2.5, 32)
    assert sh.tolist() == [[-1, 0, 0], [1, 0, 0]]
    # isolated atoms: fully linked graph in (i, j) order with zero shifts
    pos = np.array([[0, 0, 0], [10, 0, 0], [0, 10, 0]], dtype=np.float32)
    s, t, sh = NO.neighbor_list(pos, (50 * np.eye(3)).astype(np.float32), [False] * 3, 3.0, 32)
    assert s.tolist() == [0, 0, 1, 1, 2, 2] and t.tolist() == [1, 2, 0, 2, 0, 1] and not sh.any()
    # small cell, cutoff > cell: several images per direction
    s, t, sh = NO.neighbor_list(np.zeros((1, 3), np.float32), np.eye(3, dtype=np.float32), [True] * 3, 2.01, 10**6)
    assert len(s) == sum(1 for a in range(-3, 4) for b in range(-3, 4) for c in range(-3, 4)
                         if 0 < a * a + b * b + c * c < 2.01**2)


def _run_wrapper(g, rc, max_nb, dev):
    from lcaonet_b200.neighbors import build_neighbor_list
    ei, sh, nb = build_neighbor_list(g["pos"].to(dev), g["batch"].to(dev), g["lattice"].to(dev), g["pbc"].to(dev), rc, max_nb)
    return ei.cpu(), sh.cpu(), nb.cpu()


def _check_vs_oracle(g, rc, max_nb, dev):
    ei, sh, nb = _run_wrapper(g, rc, max_nb, dev)
    gptr = np.concatenate([[0], np.bincount(g["batch"].numpy(), minlength=g["lattice"].shape[0]).cumsum()])
    s, t, osh, cnt = NO.batch_neighbor_list(g["pos"].numpy(), gptr, g["lattice"].numpy(), g["pbc"].numpy(), rc, max_nb)
    assert ei.shape[1] == len(s)
    assert torch.equal(ei[0], torch.from_numpy(s)) and torch.equal(ei[1], torch.from_numpy(t))   # bit-exact, same order
    assert torch.equal(sh, torch.from_numpy(osh)) and nb.tolist() == cnt.tolist()


def _cases():
    st = _structures()
    cases = [(st["qm9"][0], st["qm9"][1], 32), (st["qm9"][0], st["qm9"][1], 6), (st["crystal"][0], st["crystal"][1], 32),
             (st["crystal"][0], st["crystal"][1], 1000)]
    # perfect lattice (ties everywhere), a tiny cell (cutoff spans 3 images), isolated atoms (fallback), one atom
    lat = dict(pos=torch.tensor(np.stack(np.meshgrid(*[np.arange(3.0)] * 3, indexing="ij"), -1).reshape(-1, 3) * 2.0, dtype=torch.float32),
               batch=torch.zeros(27, dtype=torch.long), lattice=(6.0 * torch.eye(3)).unsqueeze(0), pbc=torch.ones(1, 3, dtype=torch.long))
    cases.append((lat, 3.0, 32))
    tiny = dict(pos=torch.tensor([[0.1, 0.2, 0.3], [0.6, 0.5, 0.4]]), batch=torch.zeros(2, dtype=torch.long),
                lattice=torch.tensor([[[1.0, 0.0, 0.0], [0.3, 1.1, 0.0], [0.0, 0.2, 0.9]]]), pbc=torch.tensor([[1, 1, 0]]))
    cases.append((tiny, 2.5, 32))
    iso = dict(pos=torch.tensor([[0.0, 0, 0], [10, 0, 0], [0, 10, 0], [1.0, 1, 1], [1.5, 1, 1]]),
               batch=torch.tensor([0, 0, 0, 1, 1]), lattice=(50 * torch.eye(3)).repeat(2, 1, 1), pbc=torch.zeros(2, 3, dtype=torch.long))
    cases.append((iso, 3.0, 32))
    return cases


@pytest.mark.parametrize("idx", range(7))
def test_wrapper_through_emulator(idx, monkeypatch):
    # imported before the emulator is installed: the module binds `call`, `require_cuda` and `stream_ptr` at import, and
    # bound to the emulator's stand-ins they would outlive this test and route the CUDA tests below to the emulator
    from lcaonet_b200 import neighbors
    from tests import cpu_abi
    cpu_abi.install(monkeypatch)
    monkeypatch.setattr(neighbors, "require_cuda", lambda *a: None)
    monkeypatch.setattr(neighbors, "stream_ptr", lambda: 0)
    monkeypatch.setattr(neighbors, "call", lambda name, *a: cpu_abi._TABLE[name](*a))
    g, rc, max_nb = _cases()[idx]
    _check_vs_oracle(g, rc, max_nb, "cpu")


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(7))
def test_cuda_neighbor_list_bit_exact_vs_oracle(idx):
    g, rc, max_nb = _cases()[idx]
    _check_vs_oracle(g, rc, max_nb, "cuda")


@pytest.mark.gpu
def test_model_on_gpu_built_neighbor_list_matches_generator_graph():
    """the hot path fed by the GPU-built neighbour list gives the energies of the generator's graph (edge order differs)"""
    from lcaonet_b200 import LCAONet
    from lcaonet_b200.neighbors import attach_neighbor_list
    from tests._util import rel_l2
    g, rc = _structures()["crystal"]
    torch.manual_seed(0)
    model = LCAONet(emb_size=32, emb_size_coeff=32, emb_size_conv=32, cutoff=6.0, cutoff_net="polynomial").cuda().eval()
    with torch.no_grad():
        e_ref = model(g.to("cuda"))
        g2 = g.to("cuda")
        attach_neighbor_list(g2, rc, max_neighbors=10**6)
        assert g2["edge_index"].shape == g["edge_index"].shape
        e_new = model(g2)
    assert rel_l2(e_new, e_ref) < 1e-5
