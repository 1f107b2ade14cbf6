"""Cost of the per-atom energies and virials (LCAONet.regress_atom_energy / regress_atom_virial) on the crystal workload of
bench.py (config 4: 64 cells x 64 atoms per GPU, cutoff 6.0, polynomial cutoff, autograd forces), one GPU.

    python scripts/bench_atom_properties.py --out DIR [--cells 64] [--steps 20] [--repeats 5]

Two step kinds, both bench.py's step (energy + forces by the first-order kernels, force_training=False, energy-loss
backward, optimizer step), timed with CUDA events in the same process, alternating kind by kind for `--repeats` rounds:
  off   the switches off (the default)
  on    regress_atom_energy and regress_atom_virial on
and lcao_geom_atom_virial_bwd alone (events around `--kernel-reps` back-to-back calls on the step's dvec-sized inputs;
the inputs are L2 resident at this size).  Writes DIR/bench_atom_properties.json with the card's name and power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from lcaonet_b200 import LCAONet, _lib, ops  # noqa: E402
from lcaonet_b200.dist import FlatGradBucket  # noqa: E402
from lcaonet_b200.synth import crystal_like_batch, graph_sizes  # noqa: E402
from scripts.bench_stress import card  # noqa: E402

KINDS = ("off", "on")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--cells", type=int, default=64)
    ap.add_argument("--steps", type=int, default=20, help="steps per timed window")
    ap.add_argument("--repeats", type=int, default=5, help="alternating rounds over the two kinds")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--kernel-reps", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_atom_properties.py measures on a CUDA device; none found")
    dev = torch.device("cuda")
    _lib.load()
    torch.manual_seed(0)
    model = LCAONet(cutoff=6.0, cutoff_net="polynomial", regress_forces=True, direct_forces=False).to(dev).train()
    model.out_layer.force_training = False
    bucket = FlatGradBucket(model)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4, fused=True)
    host = crystal_like_batch(args.cells, seed=1000, cutoff=6.0)
    sizes = graph_sizes(host)
    batch = host.to(dev)
    mse = torch.nn.functional.mse_loss

    def step(kind):
        model.regress_atom_energy = model.regress_atom_virial = kind == "on"
        bucket.zero()
        out = model(dict(batch))
        mse(out[0], batch["y"]).backward()
        opt.step()

    def window(kind):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step(kind)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    launches = {}
    for kind in KINDS:
        for _ in range(args.warmup):
            step(kind)
        torch.cuda.synchronize()
        l0 = _lib.launch_count()
        step(kind)
        torch.cuda.synchronize()
        launches[kind] = _lib.launch_count() - l0
    ms = {k: [] for k in KINDS}
    t_start = time.time()
    for _ in range(args.repeats):
        for kind in KINDS:
            ms[kind].append(window(kind))
    wall = time.time() - t_start

    # the kernel alone, on the inputs of one step of this batch
    gi = ops.GraphIndex(batch["edge_index"], batch["z"].shape[0])
    dvec = torch.randn(gi.E, 3, device=dev)
    args_k = (dvec, batch["pos"], batch["edge_shift"], batch["lattice"], batch["batch"], gi)
    for _ in range(10):
        ops._atom_virial(*args_k)
    kern = []
    for _ in range(5):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.kernel_reps):
            ops._atom_virial(*args_k)
        e1.record()
        torch.cuda.synchronize()
        kern.append(e0.elapsed_time(e1) * 1e3 / args.kernel_reps)
    E, N = sizes["E"], sizes["N"]
    # algorithmic bytes: every edge is read twice, once from each end: per visit edge id + dst or src (8), shift + dvec +
    # pos of the other end (36); per node both CSR pointers (16), batch + pos (20), the 3x3 output (36)
    kbytes = 2 * 44 * E + 72 * N

    def summary(v):
        return {"median": statistics.median(v), "min": min(v), "max": max(v), "all": v}

    med = {k: statistics.median(v) for k, v in ms.items()}
    res = {
        "what": "scripts/bench_atom_properties.py: per-atom energy + virial cost on the crystal workload "
                "(bench.py --workload crystal)",
        "card": card(),
        "sizes": sizes, "cells": args.cells, "steps_per_window": args.steps, "repeats": args.repeats, "timed_wall_s": wall,
        "step_ms": {k: summary(v) for k, v in ms.items()},
        "launches_per_step": launches,
        "overhead_first_order": med["on"] / med["off"] - 1.0,
        "atom_kernel_us": summary(kern),
        "atom_kernel_bytes": kbytes,
        "atom_kernel_GBps_median": kbytes / (statistics.median(kern) * 1e-6) / 1e9,
        "atom_kernel_note": "one launch per call (warp per atom); inputs L2 resident (< 126 MB)",
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_atom_properties.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "overhead_first_order", "launches_per_step")}
                     | {"step_ms_median": med, "atom_kernel_us_median": statistics.median(kern)}))


if __name__ == "__main__":
    main()
