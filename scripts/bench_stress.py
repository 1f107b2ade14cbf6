"""Cost of the stress (LCAONet.regress_stress) on the crystal workload of bench.py (config 4: 64 cells x 64 atoms per GPU,
cutoff 6.0, polynomial cutoff, autograd forces), one GPU.

    python scripts/bench_stress.py --out DIR [--cells 64] [--steps 20] [--repeats 5]

Four step kinds, timed with CUDA events in the same process, alternating kind by kind for `--repeats` rounds:
  fo_forces     energy + forces by the first-order kernels (force_training=False), energy-loss step (bench.py's step)
  fo_stress     the same with the stress
  train_forces  training step on energy and forces (differentiable backward: loss = mse(E) + mse(F))
  train_stress  training step on energy, forces and stress (loss = mse(E) + mse(F) + mse(sigma))
and lcao_geom_cell_bwd alone (events around `--kernel-reps` back-to-back calls on the step's dvec-sized inputs; the
inputs are L2 resident at this size).  Writes DIR/bench_stress.json with the card's name and power limit.

The two training kinds run on `--train-cells` cells (default 4): the differentiable backward keeps triplet-sized (T, C)
tensors alive until the loss is back-propagated, and at width 128 those of 64 cells (T = 9.8 M) do not fit in 180 GB,
with or without the stress.  If the warm-up runs out of memory the count is halved (down to 1) and the JSON says so.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from lcaonet_b200 import LCAONet, _lib, ops  # noqa: E402
from lcaonet_b200.dist import FlatGradBucket  # noqa: E402
from lcaonet_b200.synth import crystal_like_batch, graph_sizes  # noqa: E402

KINDS = ("fo_forces", "fo_stress", "train_forces", "train_stress")


def card() -> dict:
    q = "name,power.limit,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        vals = [v.strip() for v in r.stdout.strip().splitlines()[torch.cuda.current_device()].split(",")]
        return dict(zip(q.split(","), vals))
    except (OSError, IndexError, subprocess.SubprocessError) as e:
        return {"name": torch.cuda.get_device_name(), "error": f"nvidia-smi: {e}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--cells", type=int, default=64)
    ap.add_argument("--train-cells", type=int, default=4)
    ap.add_argument("--steps", type=int, default=20, help="steps per timed window")
    ap.add_argument("--repeats", type=int, default=5, help="alternating rounds over the four kinds")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--kernel-reps", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_stress.py measures on a CUDA device; none found")
    dev = torch.device("cuda")
    _lib.load()
    torch.manual_seed(0)
    model = LCAONet(cutoff=6.0, cutoff_net="polynomial", regress_forces=True, direct_forces=False).to(dev).train()
    bucket = FlatGradBucket(model)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4, fused=True)
    host = crystal_like_batch(args.cells, seed=1000, cutoff=6.0)
    sizes = graph_sizes(host)
    batch = host.to(dev)
    mse = torch.nn.functional.mse_loss
    batches = {"fo": batch}

    def set_train_cells(n):
        h = crystal_like_batch(n, seed=1000, cutoff=6.0)
        batches["train"] = h.to(dev)
        return graph_sizes(h)

    train_sizes = set_train_cells(args.train_cells)

    def step(kind):
        model.regress_stress = kind.endswith("stress")
        model.out_layer.force_training = False if kind.startswith("fo") else None
        bucket.zero()
        b = batches[kind.split("_")[0]]
        out = model(dict(b))
        loss = mse(out[0], b["y"])
        if kind.startswith("train"):
            loss = loss + (out[1] ** 2).mean()
            if model.regress_stress:
                loss = loss + (out[2] ** 2).mean()
        loss.backward()
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

    launches, oom = {}, []
    for kind in KINDS:
        while True:
            try:
                for _ in range(args.warmup):
                    step(kind)
                break
            except torch.OutOfMemoryError:
                n = train_sizes["B"]
                if not kind.startswith("train") or n == 1:
                    raise
                oom.append(n)
                bucket.zero()
                torch.cuda.empty_cache()
                train_sizes = set_train_cells(n // 2)
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
    seg = ops.bucket_sort(batch["batch"], batch["lattice"].shape[0])
    dvec = torch.randn(gi.E, 3, device=dev)
    args_k = (dvec, batch["pos"], batch["edge_shift"], batch["lattice"], batch["batch"], gi, seg, True, True)
    for _ in range(10):
        ops._cell_grads(*args_k)
    kern = []
    for _ in range(5):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.kernel_reps):
            ops._cell_grads(*args_k)
        e1.record()
        torch.cuda.synchronize()
        kern.append(e0.elapsed_time(e1) * 1e3 / args.kernel_reps)
    E, N, B = sizes["E"], sizes["N"], sizes["B"]
    # algorithmic bytes: per edge out_edge + dst (8), shift + dvec + pos[t] (36); per node out_ptr + perm + batch + pos (28);
    # partials (18 doubles per chunk, written and read) and outputs are negligible
    kbytes = 44 * E + 28 * N

    def summary(v):
        return {"median": statistics.median(v), "min": min(v), "max": max(v), "all": v}

    med = {k: statistics.median(v) for k, v in ms.items()}
    res = {
        "what": "scripts/bench_stress.py: stress cost on the crystal workload (bench.py --workload crystal)",
        "card": card(),
        "sizes": sizes, "train_sizes": train_sizes, "train_cells_out_of_memory": oom,
        "cells": args.cells, "steps_per_window": args.steps, "repeats": args.repeats, "timed_wall_s": wall,
        "step_ms": {k: summary(v) for k, v in ms.items()},
        "launches_per_step": launches,
        "overhead_first_order": med["fo_stress"] / med["fo_forces"] - 1.0,
        "overhead_training": med["train_stress"] / med["train_forces"] - 1.0,
        "cell_kernel_us": summary(kern),
        "cell_kernel_bytes": kbytes,
        "cell_kernel_GBps_median": kbytes / (statistics.median(kern) * 1e-6) / 1e9,
        "cell_kernel_note": "two launches (chunk partials + per-graph sum) per call; inputs L2 resident (< 126 MB)",
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_stress.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "overhead_first_order", "overhead_training")}
                     | {"step_ms_median": med, "cell_kernel_us_median": statistics.median(kern)}))


if __name__ == "__main__":
    main()
