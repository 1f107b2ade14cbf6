#!/usr/bin/env python
"""Benchmark of the LCAONet hot path on B200 (BASELINE.json metric: molecules/s forward+backward on
QM9-shape synthetic batches) — see DESIGN.md §Measurement for every definition used here.

    python bench.py --gpus N --steps K --warmup W            # our arm (torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/*.npy

One "step" = one training step over one batch of 1024 synthetic QM9-shaped molecules per GPU
(index build + forward + backward of the energy MSE loss + gradient all-reduce for N > 1 + fused
Adam update).  `value` times it with the batch already resident in HBM; `e2e` times the same step
through the public API starting from pinned HOST tensors (H2D copy of the batch and D2H read of the
loss inside the timed region).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MODEL_KW = dict(cutoff=5.0, cutoff_net="polynomial")  # BASELINE.json configs[1]: default model, hydrogen rbf, poly cutoff 5.0
WORKLOAD = "QM9-shape synthetic, {m} molecules/GPU (~18 atoms, cutoff 5.0), default LCAONet 128/128/128 x3, energy MSE training step"


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines, self.t0 = index, None, [], 0.0

    def mark(self):
        """the timed region starts now: only samples taken from here on are reported (nvidia-smi itself is started
        well before, during warm-up, because it needs up to a second to deliver its first sample)"""
        self.t0 = time.time()

    def count(self) -> int:
        return sum(1 for t, _ in self.lines if t >= self.t0)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if ts < self.t0:
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def _ncu_traffic(call: str):
    """(bytes, note): MEASURED DRAM bytes (read + write) of one launch of `call` from profiles/ncu_traffic.json, which
    scripts/ncu_traffic.py writes from an ncu capture of this same bench step and stamps with the digest of the CUDA
    sources.  A stamp that does not match the sources in the tree means the numbers belong to other kernels: refused."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(path):
        return None, "profiles/ncu_traffic.json absent"
    from lcaonet_b200.csrc.build import _digest
    data = json.load(open(path))
    if data.get("csrc_digest") != _digest():
        return None, "profiles/ncu_traffic.json was measured on other CUDA sources (digest mismatch): regenerate with scripts/ncu_traffic.py"
    return data.get(call, {}).get("dram_bytes_per_launch"), "ncu dram__bytes_read.sum + dram__bytes_write.sum, scripts/ncu_traffic.py"


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return p["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs, STREAM-style copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------
def cpu_oracle_step_time(n_mol: int, reps: int, threads: int | None = None):
    """fwd+bwd of the oracle (CPU port of the reference) on `n_mol` QM9-shape molecules; best of reps."""
    from lcaonet_b200 import LCAONet
    from lcaonet_b200.synth import qm9_like_batch
    from oracle import lcao_oracle as O

    if threads:
        torch.set_num_threads(threads)
    cfg = dict(emb_size=128, emb_size_coeff=128, emb_size_conv=128, out_size=1, n_interaction=3, n_per_orb=1, cutoff=6.0,
               rbf_type="hydrogen", cutoff_net="envelope", max_z=36, min_orb=None, max_orb=None, elec_to_node=True,
               add_valence=False, extend_orb=False, is_extensive=True, regress_forces=False, direct_forces=True)
    cfg.update(MODEL_KW)
    torch.manual_seed(0)
    sd = LCAONet(**MODEL_KW).state_dict()
    p = O.cast_params(sd, torch.float32, requires_grad=True)
    g = qm9_like_batch(n_mol, seed=0, cutoff=5.0)
    y = g["y"]
    times = []
    for _ in range(max(reps, 1) + 1):  # first one is the warm-up
        for v in p.values():
            if v.grad is not None:
                v.grad = None
        t0 = time.perf_counter()
        out = O.forward(p, cfg, g, training=True)
        torch.nn.functional.mse_loss(out, y).backward()
        times.append(time.perf_counter() - t0)
    return min(times[1:]), times


def gpu_oracle_sweep(batches, reps: int, dev):
    """The reference algorithm (oracle port: materialises the (T,O,C) tensors like lcaonet.py:173-189) run by
    PyTorch eager ON THE GPU — the denominator of BASELINE.json's ">= 20x reference-PyTorch-on-B200" target.
    The eager reference gets more efficient with the batch until it runs out of memory, so every batch size in
    `batches` is timed (best of `reps` after a warm-up) and the BEST throughput is the one quoted.  Baseline only."""
    from lcaonet_b200 import LCAONet
    from lcaonet_b200.synth import qm9_like_batch
    from oracle import lcao_oracle as O

    cfg = dict(emb_size=128, emb_size_coeff=128, emb_size_conv=128, out_size=1, n_interaction=3, n_per_orb=1, cutoff=6.0,
               rbf_type="hydrogen", cutoff_net="envelope", max_z=36, min_orb=None, max_orb=None, elec_to_node=True,
               add_valence=False, extend_orb=False, is_extensive=True, regress_forces=False, direct_forces=True)
    cfg.update(MODEL_KW)
    torch.manual_seed(0)
    sd = {k: v.to(dev) for k, v in LCAONet(**MODEL_KW).state_dict().items()}
    results = []
    for n_mol in batches:
        p = g = out = None
        try:
            p = O.cast_params(sd, torch.float32, device=dev, requires_grad=True)
            g = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in qm9_like_batch(n_mol, seed=0, cutoff=5.0).items()}
            times = []
            for _ in range(reps + 1):
                for v in p.values():
                    v.grad = None
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = O.forward(p, cfg, g, training=True)
                torch.nn.functional.mse_loss(out, g["y"]).backward()
                torch.cuda.synchronize()
                times.append(time.perf_counter() - t0)
            results.append({"molecules": n_mol, "molecules_per_s": n_mol / min(times[1:]),
                            "peak_mem_gib": round(torch.cuda.max_memory_allocated() / 2**30, 1)})
        except torch.OutOfMemoryError:
            results.append({"molecules": n_mol, "molecules_per_s": None, "note": "out of memory"})
        del p, g, out
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        if results[-1]["molecules_per_s"] is None:
            break
    return results


def run_reference(args):
    """`--impl reference`: the reference's own CPU algorithm (oracle port; the reference tree itself is
    Python and does not travel to the GPU box) timed on the host cores, same metric and config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_mol = 32  # BASELINE.json configs[0]: the reference's CPU-runnable case; a bounded sample of the workload
    t0 = time.perf_counter()
    steps = max(1, args.steps)
    best, times = cpu_oracle_step_time(n_mol, reps=max(steps, 1) + max(args.warmup - 1, 0), threads=cores)
    timed = times[-steps:]
    dt = sum(timed) / len(timed)
    val = n_mol / dt
    line = {
        "impl": "reference", "metric": "molecules/sec fwd+bwd (QM9-shape)", "value": val, "unit": "molecules/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD.format(m=args.mol_per_gpu), "sample": f"{n_mol} molecules per step on host CPU"},
        "cpu_baseline": {"value": val, "unit": "molecules/s", "cores": cores, "kind": "port",
                         "sample": f"{n_mol} QM9-shape molecules, fwd+bwd, mean of {steps} steps"},
        "e2e": {"value": val, "unit": "molecules/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def algorithmic_bytes(name, shp):
    """Compulsory HBM bytes of one launch (FP32), per DESIGN.md §Kernels / SURVEY.md §8d."""
    E, N, O, C, K, NL = shp["E"], shp["N"], shp["O"], shp["C"], shp["K"], shp["NL"]
    NP = NL * (NL + 1) // 2
    if name == "lcao_threebody_fwd":  # read B (E,NL,C) + Gram + unit + CSR + xk rows; write tbw (E,C)
        return E * (4 * NL * C + 8 * NP + 12 + 8 + 4 * C) + N * (4 * C + 8)
    if name == "lcao_threebody_bwd":  # read B, Gram, d_tbw, unit, CSR, xk; write dB (E,NL,C), q (E,C)
        return E * (4 * NL * C + 8 * NP + 4 * C + 12 + 8 + 4 * NL * C + 4 * C) + N * (4 * C + 8)
    if name == "lcao_pair_contract_fwd":  # read rb + pair id (table is L2 resident); write B + Gram + two-body sums
        return E * (4 * O + 8 + 4 * NL * C + 8 * NP + 4 * C)
    if name == "lcao_pair_contract_bwd":  # read dB + rb + perm; the (P,O,C) result is L2 sized
        return E * (4 * NL * C + 4 * O + 4)
    if name == "lcao_coeff_contract_fwd":  # read cst' (E,O,C) + rb; write B
        return E * (4 * O * C + 4 * O + 4 * NL * C)
    if name == "lcao_coeff_contract_bwd":  # read dB + rb; write d_cst' (E,O,C)
        return E * (4 * NL * C + 4 * O + 4 * O * C)
    if name == "lcao_twobody_fwd":  # read sum_l B_l and g; write lw
        return E * 3 * 4 * C
    if name == "lcao_twobody_bwd":  # read sum_l B_l, g, d_lw; write the compact dP and d_g
        return E * 5 * 4 * C
    return None


def run_ours(args):
    import torch.distributed as dist

    from lcaonet_b200 import LCAONet, _lib, ops
    from lcaonet_b200.dist import FlatGradBucket, broadcast_module
    from lcaonet_b200.synth import graph_sizes, qm9_like_batch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()  # fail loudly when the CUDA library is missing
    ops.set_gemm_mode(args.gemm)

    # --workload: the headline config (BASELINE.json configs[1]) or one of the other named configs (not bench lines:
    # used to report their throughput in profiles/)
    model_kw, workload, make_batch = MODEL_KW, WORKLOAD.format(m=args.mol_per_gpu), None
    if args.workload == "valence":  # configs[2]
        model_kw = dict(MODEL_KW, add_valence=True, extend_orb=True, n_per_orb=2, max_z=36)
        workload = (f"QM9-shape synthetic, {args.mol_per_gpu} molecules/GPU, LCAONet add_valence extend_orb n_per_orb=2 "
                    "(16 orbitals, C'=256), energy MSE training step")
    elif args.workload == "crystal":  # configs[3]: energy + autograd forces (first order), energy-loss gradients
        from lcaonet_b200.synth import crystal_like_batch
        model_kw = dict(cutoff=6.0, cutoff_net="polynomial", regress_forces=True, direct_forces=False)
        workload = (f"periodic crystals, {args.mol_per_gpu} cells/GPU x 64 atoms, cutoff 6.0 (~49 neighbours/atom), energy + "
                    "autograd forces + energy-loss gradients (units = cells)")
        make_batch = lambda seed: crystal_like_batch(args.mol_per_gpu, seed=seed, cutoff=6.0)  # noqa: E731
    torch.manual_seed(0)
    model = LCAONet(**model_kw).to(dev).train()
    model.side_effect_keys = not args.no_side_effect_keys
    model.out_layer.force_training = False  # (crystal workload: forces are evaluated, the loss is on the energy)
    broadcast_module(model)
    bucket = FlatGradBucket(model)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4, fused=True)

    stream_note = None
    if args.stream:
        # BASELINE.json configs[4]: a STREAM of molecules — every step sees a fresh batch.  A pool of `stream_pool` batches
        # of synthetic molecules per rank stands in for the data set (the stream wraps around it in a new random order);
        # `value`: the pool lives in HBM and each step's batch is collated on the GPU (SamplePool.batch);
        # `e2e`: the pool lives in pinned host memory, each step copies its next window and finishes the collation on the GPU.
        from lcaonet_b200.data import SamplePool, collate_window
        B_ = args.mol_per_gpu
        src = make_batch(1000 + rank) if make_batch else qm9_like_batch(B_ * args.stream_pool, seed=1000 + rank, cutoff=5.0)
        pool_host = SamplePool.from_batch(src).pin_memory()
        pool_dev = pool_host.to(dev)
        n_pool = len(pool_host)
        B_ = min(B_, n_pool)
        gen = torch.Generator(device=dev)
        gen.manual_seed(1234 + rank)
        win_k = [0]

        def next_resident():
            ids = torch.randperm(n_pool, device=dev, generator=gen)[:B_]
            return pool_dev.batch(ids)

        def next_window_host():
            lo = (win_k[0] * B_) % max(n_pool - B_ + 1, 1)
            win_k[0] += 1
            return pool_host.window(lo, lo + B_)

        first = next_resident()
        sizes = graph_sizes(first)
        w0 = next_window_host()
        h2d = sum(v.numel() * v.element_size() for v in w0.values() if torch.is_tensor(v))
        stream_note = (f"stream: pool of {n_pool} molecules per rank, a fresh batch of {B_} every step (device collation); "
                       "N/E/T are those of the first batch")
        get_batch = lambda: (lambda b: (b, b["y"]))(next_resident())  # noqa: E731
    else:
        host = (make_batch(1000 + rank) if make_batch else qm9_like_batch(args.mol_per_gpu, seed=1000 + rank, cutoff=5.0)).pin_memory()
        sizes = graph_sizes(host)
        resident = host.to(dev)
        y_dev = resident["y"]
        h2d = sum(v.numel() * v.element_size() for v in host.values() if torch.is_tensor(v))
        get_batch = lambda: (GraphClone(resident), y_dev)  # noqa: E731

    # --dump-outputs: the outputs of the latest step, detached (a reference to the graph would keep it alive)
    last = {} if args.dump_outputs else None

    def step(batch, y):
        bucket.zero()
        out = model(batch)
        if last is not None:
            last["out"] = tuple(t.detach() for t in out) if isinstance(out, tuple) else out.detach()
        if isinstance(out, tuple):  # (energy, forces): the forces are evaluated, the loss is on the energy
            out = out[0]
        loss = torch.nn.functional.mse_loss(out, y)
        loss.backward()
        bucket.all_reduce_mean()
        opt.step()
        if last is not None:
            last["loss"] = loss.detach()
        return loss

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    host_ms = [0.0]

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        host_ms[0] = (time.perf_counter() - t0) * 1e3 / steps  # CPU time to ENQUEUE one step (no sync inside)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / steps

    # ---- device-resident timing (value)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # (started before the warm-up: see ClockSampler.mark)
    for _ in range(max(args.warmup, 3)):
        step(*get_batch())
    sampler.mark()
    l0 = _lib.launch_count()
    ms_dev = timed(lambda: step(*get_batch()), args.steps)
    launches = (_lib.launch_count() - l0) // max(args.steps, 1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, last["out"], last["loss"])
    # CPU time to enqueue ONE step into an empty stream (median of 5): if it approaches ms_per_step the host is the limit
    hs = []
    for _ in range(5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        step(*get_batch())
        hs.append((time.perf_counter() - t0) * 1e3)
    torch.cuda.synchronize()
    host_enqueue_ms = sorted(hs)[2]

    # ---- end-to-end timing (e2e): pinned host batch -> H2D -> step -> D2H loss
    def e2e_step():
        if args.stream:
            b = collate_window(next_window_host().to(dev, non_blocking=True))
        else:
            b = host.to(dev, non_blocking=True)
        loss = step(b, b["y"])
        return float(loss.detach())  # D2H read of the step's result (synchronises)

    for _ in range(2):
        e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    if rank == 0 and sampler.proc is not None:
        # the timed regions last a few hundred ms: keep the same step running (untimed) until nvidia-smi has delivered
        # a handful of samples under this load
        t_end = time.time() + 3.0
        while sampler.count() < 5 and time.time() < t_end:  # (rank 0 only: forward + backward, no collective)
            bucket.zero()
            b_, y_ = get_batch()
            o = model(b_)
            torch.nn.functional.mse_loss(o[0] if isinstance(o, tuple) else o, y_).backward()
            torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None

    if args.profile_host and rank == 0:  # where does the CPU time of one step go?
        import cProfile
        import pstats
        pr = cProfile.Profile()
        torch.cuda.synchronize()
        pr.enable()
        for _ in range(5):
            step(*get_batch())
        pr.disable()
        torch.cuda.synchronize()
        st_ = pstats.Stats(pr, stream=sys.stderr)
        st_.sort_stats("tottime").print_stats(35)
        st_.sort_stats("cumtime").print_stats(45)

    # ---- per-kernel profile of one step (CUDA events around every C-ABI call on the launching stream)
    prof = profile_step(ops, lambda: step(*get_batch()), reps=3)
    total_mols = args.mol_per_gpu * world
    if rank == 0:
        peak, peak_src = _peaks()
        shp = dict(E=sizes["E"], N=sizes["N"], O=model.rbf.n_orb, C=model.emb_size_conv, K=model.emb_size_coeff,
                   NL=model._n_l)
        kernels = []
        step_sum = sum(v["ms"] for v in prof.values())
        for name, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"]):
            ent = {"call": name, "calls_per_step": v["calls"], "ms_per_step": round(v["ms"], 4),
                   "share": round(v["ms"] / step_sum, 4)}
            ab = algorithmic_bytes(name, shp)
            if ab is not None:
                gbs = ab / (v["ms"] / v["calls"] * 1e-3) / 1e9
                ent.update(bytes_per_launch=ab, achieved_gbs=round(gbs, 1), frac=round(gbs / peak, 4))
            elif name.startswith("lcao_linear"):
                ent.update(bytes_per_step=v["bytes"], achieved_gbs=round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1),
                           tflops=round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 2))
                ent["frac"] = round(ent["achieved_gbs"] / peak, 4)
            kernels.append(ent)
        dom = next((k for k in kernels if "frac" in k), None)
        roofline = None
        if dom is not None:
            per_launch = dom.get("bytes_per_launch", dom.get("bytes_per_step", 0) / max(dom["calls_per_step"], 1))
            traffic, traffic_src = (_ncu_traffic(dom["call"]) if args.workload == "qm9" and args.mol_per_gpu == 1024 and not args.stream
                                    else (None, "measured for the default workload only"))
            roofline = {"kernel": dom["call"], "bound": "hbm", "achieved": dom["achieved_gbs"], "peak": peak, "unit": "GB/s",
                        "frac": dom["frac"], "traffic": traffic, "traffic_source": traffic_src,
                        "peak_source": peak_src, "algorithmic_bytes_per_launch": per_launch,
                        "share_of_step": dom["share"]}
        cpu = None
        if world == 1:
            best, _ = cpu_oracle_step_time(32, reps=args.cpu_reps, threads=os.cpu_count())
            cpu = {"value": 32 / best, "unit": "molecules/s", "cores": os.cpu_count(), "kind": "port",
                   "sample": f"32 QM9-shape molecules (BASELINE configs[0]), fwd+bwd, best of {args.cpu_reps}, oracle port of the reference"}
        ref_gpu = None
        sek = model.side_effect_keys
        if world == 1 and args.ref_gpu_mols and args.workload == "qm9":
            del model, opt, bucket, get_batch  # the eager reference needs the memory (its (T,O,C) tensors are ~15 GB each at 1024)
            torch.cuda.empty_cache()
            sampler2 = ClockSampler(local)
            sampler2.start()
            sampler2.mark()
            sweep = gpu_oracle_sweep([int(x) for x in args.ref_gpu_mols.split(",")], 3, dev)
            clocks2 = sampler2.stop()
            ok = [r for r in sweep if r["molecules_per_s"]]
            if ok:
                best = max(ok, key=lambda r: r["molecules_per_s"])
                ref_gpu = {"value": best["molecules_per_s"], "unit": "molecules/s",
                           "kind": "oracle port of the reference, PyTorch eager on cuda:0 (FP32)",
                           "sample": f"batch sweep {[r['molecules'] for r in sweep]} QM9-shape molecules, fwd+bwd, best of 3 each; "
                                     f"best at {best['molecules']} molecules", "sweep": sweep, "clocks": clocks2,
                           "ours_over_reference": round(total_mols / (ms_dev * 1e-3) / best["molecules_per_s"], 1)}
        line = {
            "metric": "molecules/sec fwd+bwd (QM9-shape)", "value": total_mols / (ms_dev * 1e-3), "unit": "molecules/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_dev,
            "host_enqueue_ms_per_step": round(host_enqueue_ms, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "N": sizes["N"], "E": sizes["E"], "T": sizes["T"],
                       "gemm_mode": ops.get_gemm_mode(), "side_effect_keys": sek, **({"stream": stream_note} if stream_note else {}),
                       "parallelism": f"dp{world}", "l2": "per-step working set (>1 GB) exceeds the 126 MB L2; no explicit flush"},
            "e2e": {"value": total_mols / (ms_e2e * 1e-3), "unit": "molecules/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
            "gpu_launches": int(launches), "roofline": roofline,
            "kernels": kernels if os.environ.get("LCAO_BENCH_SHAPES") else kernels[:12], "cpu_baseline": cpu,
            "reference_on_gpu": ref_gpu,
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_ROWS_BYTES = 16 << 20  # per model output: energies and forces together stay well inside 64 MB with the parameters


def dump_outputs(path, model, out, loss):
    """Write what one training step computed as float32 DIR/<name>.npy: the model outputs (`energy`, and `forces` for
    the crystal workload), the `loss`, every parameter's gradient (`grad.<name>`), every parameter after the optimizer
    step (`param.<name>`) and the floating-point buffers the step updates (`buffer.<name>`, BatchNorm statistics).  A
    model output larger than DUMP_ROWS_BYTES is replaced by the same rows every run (sorted, drawn with seed 0), so that
    two builds run with the same arguments can be compared file for file."""
    import numpy as np

    outputs = dict(zip(("energy", "forces"), out)) if isinstance(out, tuple) else {"energy": out}
    arrays = {"loss": loss}
    for name, t in outputs.items():
        rows = max(1, DUMP_ROWS_BYTES // (4 * max(1, t[0].numel())))
        if t.shape[0] > rows:
            keep = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:rows].sort().values
            t = t[keep.to(t.device)]
        arrays[name] = t
    arrays.update((f"grad.{n}", p.grad) for n, p in model.named_parameters() if p.grad is not None)
    arrays.update((f"param.{n}", p) for n, p in model.named_parameters())
    arrays.update((f"buffer.{n}", b) for n, b in model.named_buffers() if b.is_floating_point())
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())


class GraphClone(dict):
    """Fresh shallow copy of the resident batch per step (forward writes side-effect keys into it)."""

    def __init__(self, src):
        super().__init__(src)

    def get(self, k, default=None):
        return super().get(k, default)


def profile_step(ops, fn, reps=3):
    """CUDA-event duration of every C-ABI call of one step, averaged over `reps` steps."""
    import torch

    records = []
    orig = ops._call

    def timed_call(name, *a):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig(name, *a)
        e1.record()
        meta = None
        if name == "lcao_linear_fwd":
            M, K, Nout = a[8], a[9], a[10]
            meta = (4 * M * (K + Nout), 2 * M * K * Nout)
        elif name == "lcao_linear_dgrad":
            M, K, Nout = a[8], a[9], a[10]
            meta = (4 * M * (K + Nout), 2 * M * K * Nout)
        elif name == "lcao_linear_wgrad":
            M, K, Nout = a[9], a[10], a[11]
            meta = (4 * M * (K + Nout), 2 * M * K * Nout)
        elif name == "lcao_linear_wgrad_deferred":  # stage 1 of a weight gradient whose reduction is batched at the end
            M, K, Nout = a[6], a[7], a[8]
            name, meta = "lcao_linear_wgrad", (4 * M * (K + Nout), 2 * M * K * Nout)
        elif name == "lcao_wgrad_reduce_batch":  # ... and that batched second stage: time of the family, not a call of its own
            name, meta = "lcao_linear_wgrad", "extra"
        if meta and meta != "extra" and os.environ.get("LCAO_BENCH_SHAPES"):
            name = f"{name}[M={M},K={K},N={Nout}]"
        records.append((name, e0, e1, meta))

    ops._call = timed_call
    try:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    finally:
        ops._call = orig
    out = {}
    for name, e0, e1, meta in records:
        d = out.setdefault(name, {"ms": 0.0, "calls": 0, "bytes": 0, "flops": 0})
        d["ms"] += e0.elapsed_time(e1) / reps
        if meta == "extra":
            continue
        d["calls"] += 1
        if meta:
            d["bytes"] += meta[0] / reps
            d["flops"] += meta[1] / reps
    for d in out.values():
        d["calls"] = max(d["calls"] // reps, 1)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mol-per-gpu", type=int, default=1024)
    ap.add_argument("--workload", default="qm9", choices=["qm9", "valence", "crystal"],
                    help="qm9 = BASELINE.json configs[1] (the bench line); valence / crystal = configs[2] / configs[3]")
    ap.add_argument("--gemm", default="tf32x3", choices=["fp32", "tf32x3", "tf32"],
                    help="dense-layer arithmetic: tf32x3 = tcgen05 3xTF32 split (FP32-equivalent, parity-tested), fp32 = CUDA cores")
    ap.add_argument("--no-side-effect-keys", action="store_true")
    ap.add_argument("--stream", action="store_true",
                    help="BASELINE configs[4]: a fresh batch every step, collated on the GPU from a resident pool (value) or "
                         "streamed from pinned host memory (e2e)")
    ap.add_argument("--stream-pool", type=int, default=4, help="--stream: batches of molecules in the pool per rank")
    ap.add_argument("--cpu-reps", type=int, default=3)
    ap.add_argument("--ref-gpu-mols", default="128,256,512,1024",
                    help="also time the oracle port with PyTorch eager on the GPU at these batch sizes and quote the best "
                         "(empty string = skip)")
    ap.add_argument("--profile-host", action="store_true", help="cProfile of 5 steps (host side) to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
