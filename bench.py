#!/usr/bin/env python
"""Benchmark of the hot path on BASELINE.json's metric.

metric : time-steps/s  (one time-step = one 1-ns sampling interval, the
         granularity the reference forces QuTiP to, SURVEY.md 0.6 / 8d)
workload (N=1 and per GPU for N>1): BASELINE configs[1] = C2, 20-atom random 2D
         register (AnalogDevice limits), Rydberg-blockade sweep, 4000 ns,
         Schroedinger fp64, Hilbert dim 2^20.
step   : one pass of the hot path over the whole 4000-step sequence.

    python bench.py --gpus N --steps K --warmup W          # this repo
    python bench.py --impl reference ...                   # CPU arm (oracle port)
    python bench.py ... --dump-outputs DIR                 # + what the last timed step computed, as DIR/*.npy

The run writes nothing into the repository tree: it loads libpulser_b200.so as
build() left it and keeps Python from caching bytecode next to the sources.

N > 1: one process per GPU (torchrun).  `value` stays C2: the single-state path
does not shard ("replicas only", DESIGN.md), every GPU evolves the same Sequence,
one NCCL all-reduce of the final observables; weak scaling.

Every run also carries
  "c4": BASELINE configs[3], the path that DOES shard: the 16-atom doppler +
        amplitude noise trajectories (1024 of them for N >= 2, 128 at N = 1)
        striped over the N ranks, sampled on the device, ONE NCCL all-reduce of
        the bitstring histogram + Rydberg densities; trajectories/s and the
        speed-up against a 1-GPU reference leg measured in the same job;
  "c5": BASELINE configs[4] (N = 1 only): the 24-atom anneal end to end,
        steps/s, H-applies/ns, us per apply, achieved GB/s;
  "c3": BASELINE configs[2] (N = 1 only): the 14-atom three-level sequence.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

N_ATOMS = int(os.environ.get("PB200_BENCH_ATOMS", "20"))
INTEGRATOR_NAMES = {1: "chebyshev-clenshaw (Richardson-CF4 Magnus)", 2: "lanczos (Richardson-CF4 Magnus)", 3: "time-dependent taylor"}
METRIC = "time-steps/s (1 ns sampling intervals of the Sequence evolved per second)"
UNIT = "steps/s"
DUMP_BYTES = 48 << 20   # at most this much of the final state in --dump-outputs (a seeded sample above it)


def workload(seed: int):
    from pulser_b200 import workloads as W

    return W.config_c2(n=N_ATOMS, seed=seed)


def config_dict(n_gpus: int) -> dict:
    return {
        "workload": f"C2: {N_ATOMS}-atom random 2D register (disc R=38um, min dist 5um, AnalogDevice C6), "
                    "Rydberg-blockade sweep 500+2500+1000 ns, ground-rydberg basis, Schroedinger fp64",
        "hilbert_dim": 2**N_ATOMS,
        "time_steps_per_sequence": 4000,
        "accuracy": "time-dependent Taylor propagator (integrator 3): QobjEvo splines fitted by polynomials per step, one H-apply per "
                    "Taylor order, a-priori 2-norm error budget 1e-8 (fit residuals + remainders); state error <= 1e-8 against the "
                    "DOP853 oracle and against the Richardson-CF4 Magnus path (tests/test_gpu_taylor.py)",
        "parallelism": "single GPU" if n_gpus == 1 else f"{n_gpus} replicas (the same C2 Sequence on every GPU, no collective in the time loop), 1 all-reduce of the final densities",
        "l2": "L2 flushed between timed iterations (256 MiB write); the 16 MiB state is L2-resident within a step",
    }


# --------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples: list[list[str]] = []
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(
                    ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                    capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self) -> dict:
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples)}


def measured_peak() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic_per_launch() -> float | None:
    """dram bytes per launch of the dominant kernel from the committed ncu summary."""
    for name in ("r02_taylor_stage_kernel_summary.json", "r02_stage_kernel_summary.json", "r01_stage_kernel_summary.json"):
        try:
            return float(json.load(open(os.path.join(ROOT, "profiles", name)))["dram_bytes_per_launch"])
        except Exception:
            continue
    return None


# --------------------------------------------------------------------------
def cpu_reference_run(spec, n_sample_steps: int, t_begin_us: float = 1.0) -> dict:
    """The reference's CPU path (oracle port of QobjEvo + qutip.sesolve at
    QuTiP-default options, zvode Adams, max_step 1 ns) on a bounded sample of
    the workload: `n_sample_steps` consecutive 1-ns steps starting mid-sweep."""
    from oracle import evolve
    from oracle.fast_terms import global_ising_hamiltonian

    H = global_ising_hamiltonian(spec)
    psi0 = evolve.all_ground_state(spec)
    # warm the integrator / caches with 2 steps, then time the sample
    evolve.sesolve(H, psi0, [t_begin_us, t_begin_us + 2e-3], method="zvode-adams", rtol=1e-6, atol=1e-8,
                   max_step=1e-3, nsteps=10**6)
    t0 = time.perf_counter()
    _, stats = evolve.sesolve(H, psi0, [t_begin_us, t_begin_us + n_sample_steps * 1e-3], method="zvode-adams",
                              rtol=1e-6, atol=1e-8, max_step=1e-3, nsteps=10**6, return_stats=True)
    dt = time.perf_counter() - t0
    return {"value": n_sample_steps / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"{n_sample_steps} consecutive 1-ns steps of the same {N_ATOMS}-atom sequence from t={t_begin_us} us, "
                      f"scipy CSR (5 QobjEvo terms) + zvode Adams atol 1e-8 rtol 1e-6 max_step 1 ns "
                      f"(QuTiP defaults as pulser sets them), {stats['rhs_calls']} RHS calls, {dt:.1f} s; "
                      "QuTiP's CSR matvec is single-threaded, host has %d cores" % (os.cpu_count() or 1)}


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    spec = workload(N_ATOMS)
    n_sample = int(os.environ.get("PB200_REF_SAMPLE_STEPS", "50" if N_ATOMS >= 20 else "400"))
    vals = []
    for i in range(args.warmup + args.steps):
        r = cpu_reference_run(spec, n_sample)
        if i >= args.warmup:
            vals.append(r)
    value = float(np.mean([v["value"] for v in vals]))
    cb = dict(vals[-1]); cb["value"] = value
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * n_sample / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64 (complex128)",
        "data": "synthetic", "config": config_dict(args.gpus), "cpu_baseline": cb,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))



# --------------------------------------------------------------------------
C4_BATCH = int(os.environ.get("PB200_BENCH_C4_BATCH", "64"))


def c4_stripe_run(local: int, rank: int, world: int, n_total: int, stream) -> dict:
    """This rank's stripe of the C4 trajectories (BASELINE configs[3], reference loop simulation.py:885-915):
    device batches, one shot per trajectory drawn on the device (pb200_state_sample), per-atom Rydberg densities
    reduced on the device.  Returns the local histogram / sums and the device time of the stripe."""
    import torch

    from pulser_b200 import engine, parallel, workloads as W

    mine = set(parallel.stripe(n_total, rank, world))
    n = 16
    hist = np.zeros(1 << n, dtype=np.float64)
    dens = np.zeros(n)
    stats = {"n_applies": 0, "n_launches": 0, "gpu_ms": 0.0, "batches": 0, "traj_applies": 0}
    np.random.seed(4000 + rank)  # sampling uniforms of this rank (plan.sample draws from np.random)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    chunk = []

    def flush():
        if not chunk:
            return
        with engine.DevicePlan(chunk, device=local) as plan:
            plan.set_stream(stream.cuda_stream)
            plan.set_state("all-ground")
            st = plan.propagate(0.0, chunk[0].sampling_times[-1])
            for k in ("n_applies", "n_launches", "gpu_ms"):
                stats[k] += st[k]
            stats["batches"] += 1
            stats["traj_applies"] += st["n_applies"] * len(chunk)   # n_applies counts per trajectory of the batch
            stats["integrator"] = int(st["integrator"])
            stats["taylor_batches"] = stats.get("taylor_batches", 0) + (1 if int(st["integrator"]) == 3 else 0)
            r = chunk[0].eigenbasis.index("r")
            dens[:] += plan.occupation(r).sum(axis=0)
            for i in range(len(chunk)):
                (bits, cnt), = plan.sample(1, "r", traj=i).items()
                hist[int(bits, 2)] += cnt
        chunk.clear()

    for _, spec in W.config_c4_stream(n_total, keep=mine):
        chunk.append(spec)
        if len(chunk) == C4_BATCH:
            flush()
    flush()
    e1.record(stream)
    torch.cuda.synchronize()
    return {"hist": hist, "dens": dens, "ms": e0.elapsed_time(e1), "n_local": len(mine), **stats}


def c4_warmup(local: int) -> None:
    from pulser_b200 import engine, workloads as W

    specs = W.config_c4(C4_BATCH, seed=99)
    with engine.DevicePlan(specs, device=local) as plan:
        plan.set_state("all-ground")
        plan.propagate(0.0, 0.25)
        plan.sample(1, "r", traj=0)


def c3_leg(local: int, stream) -> dict:
    """BASELINE configs[2]: 14-atom 'all' basis (3 levels, Raman + Rydberg channels), whole 2000-ns sequence."""
    import torch

    from pulser_b200 import engine, workloads as W

    n = int(os.environ.get("PB200_BENCH_C3_ATOMS", "14"))
    spec = W.config_c3(n=n)
    with engine.DevicePlan(spec, device=local) as plan:
        plan.set_stream(stream.cuda_stream)
        plan.set_state("all-ground")
        plan.propagate(0.0, 0.05)   # warm-up
        plan.set_state("all-ground")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        st = plan.propagate(0.0, spec.sampling_times[-1])
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        norm2 = float(plan.norm2()[0])
    T = spec.total_duration_ns
    return {"workload": f"C3: {n}-atom random 2D register, basis 'all' (r, g, h), raman_global Blackman pi/2 - rydberg_global "
                        f"Blackman pi - raman_global Blackman pi/2, {T} ns, fp64",
            "hilbert_dim": spec.hilbert_dim, "steps_per_s": T / (ms * 1e-3), "seconds": ms * 1e-3,
            "h_applies_per_time_step": st["n_applies"] / T, "integrator": INTEGRATOR_NAMES.get(int(st["integrator"]), "?"),
            "gpu_launches": int(st["n_launches"]), "norm2_final": norm2}


def c4_leg(local: int, rank: int, world: int, dist, barrier, stream) -> dict | None:
    import torch

    n_total = int(os.environ.get("PB200_BENCH_C4_TRAJ", "1024" if world > 1 else "128"))
    # untimed warm-up: one full-size device batch over a short stretch, so that the buffer pool and the kernels of this
    # path exist before the timed stripe (the 1-GPU reference leg below runs warm too)
    c4_warmup(local)
    barrier()
    r = c4_stripe_run(local, rank, world, n_total, stream)
    # THE collective of the path: histogram + density sums + (max) time in one packed tensor pair
    packed = torch.from_numpy(np.concatenate([r["hist"], r["dens"], [r["traj_applies"], r["n_launches"]]])).to("cuda")
    tmax = torch.tensor([r["ms"]], dtype=torch.float64, device="cuda")
    # diagnostics only (not part of the path): every rank's device time, device-batch count and how many of its batches
    # ran on the Taylor propagator, placed in its own slot of a zero vector that rides on a second SUM
    diag = torch.zeros(3 * world, dtype=torch.float64, device="cuda")
    diag[3 * rank: 3 * rank + 3] = torch.tensor([r["ms"] * 1e-3, r["batches"], r.get("taylor_batches", 0)], dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(packed, op=dist.ReduceOp.SUM)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(diag, op=dist.ReduceOp.SUM)
    barrier()
    diag = diag.cpu().numpy().reshape(world, 3)
    tot = packed.cpu().numpy()
    hist, dens = tot[: 1 << 16], tot[1 << 16: (1 << 16) + 16]
    seconds = float(tmax.item()) * 1e-3
    out = {
        "workload": "C4: 16-atom 4x4 square (6 um, MockDevice C6), blockade sweep 4000 ns, SimConfig(doppler 50 uK + amplitude "
                    "sigma 0.05, waist 175 um) noise trajectories, ground-rydberg, fp64",
        "n_trajectories": n_total, "n_gpus": world, "trajectories_per_rank": r["n_local"], "device_batch": C4_BATCH,
        "seconds": seconds, "trajectories_per_s": n_total / seconds, "traj_steps_per_s": n_total * 4000 / seconds,
        "h_applies_per_traj_step": float(tot[-2]) / (4000.0 * n_total), "gpu_launches": int(tot[-1]),
        "integrator": INTEGRATOR_NAMES.get(r.get("integrator", 0), "?"),
        "per_rank": {"seconds": [round(float(x), 3) for x in diag[:, 0]], "device_batches": [int(x) for x in diag[:, 1]],
                     "taylor_batches": [int(x) for x in diag[:, 2]]},
        "shots": int(round(hist.sum())), "mean_rydberg_density": float(dens.sum() / (16 * n_total)),
        "collective": "1 all_reduce(SUM) of [2^16 histogram | 16 densities | counters] + 1 all_reduce(MAX) of the time "
                      "(+ 1 diagnostic SUM of the per-rank timings, outside the timed region)",
        "timing": "CUDA events on the stream of the plans around the whole stripe (host-side spec building, plan "
                  "creation and sampling included), max over ranks",
    }
    if world > 1:
        # 1-GPU reference leg in the same job: rank 0 alone evolves 64 of the same trajectories
        barrier()
        ref = c4_stripe_run(local, 0, 1, C4_BATCH, stream) if rank == 0 else None
        barrier()
        if rank == 0:
            n1 = C4_BATCH / (ref["ms"] * 1e-3)
            out["n1_reference_trajectories_per_s"] = n1
            out["n1_reference_sample"] = f"{C4_BATCH} trajectories on rank 0 alone, same code path"
            out["speedup_vs_n1"] = out["trajectories_per_s"] / n1
    else:
        out["speedup_vs_n1"] = 1.0
    return out if rank == 0 else None


def c5_leg(local: int, stream, peak: float) -> dict:
    """BASELINE configs[4]: 24-atom adiabatic anneal, whole 4000-ns sequence on one GPU (auto integrator)."""
    import torch

    from pulser_b200 import engine, workloads as W

    n = int(os.environ.get("PB200_BENCH_C5_ATOMS", "24"))
    spec = W.config_c5(n=n)
    D = spec.hilbert_dim
    with engine.DevicePlan(spec, device=local) as plan:
        plan.set_stream(stream.cuda_stream)
        plan.set_state("all-ground")
        ms_apply, launches = plan.bench_apply(1.0, 20)
        plan.set_state("all-ground")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        st = plan.propagate(0.0, spec.sampling_times[-1])
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        norm2 = float(plan.norm2()[0])
    T = spec.total_duration_ns
    per_apply = st["gpu_ms"] * 1e-3 / max(st["n_applies"], 1)
    bare = ms_apply * 1e-3 / 20
    return {
        "workload": f"C5: {n}-atom random 2D register, adiabatic anneal 0 -> Omega -> 0 with a detuning ramp, {T} ns, "
                    "ground-rydberg, fp64, " + INTEGRATOR_NAMES.get(int(st["integrator"]), "?") + " propagator "
                    "(the Krylov / Lanczos path of round 1 is integrator=2: tests/test_gpu_full_size.py compares the two)",
        "integrator": INTEGRATOR_NAMES.get(int(st["integrator"]), "?"),
        "hilbert_dim": D, "steps_per_s": T / (ms * 1e-3), "seconds": ms * 1e-3,
        "h_applies_per_time_step": st["n_applies"] / T, "us_per_h_apply_in_sequence": per_apply * 1e6,
        "us_per_bare_h_apply": bare * 1e6, "gpu_launches": int(st["n_launches"]), "norm2_final": norm2,
        "roofline": {"bound": "hbm", "unit": "GB/s", "peak": peak,
                     "achieved_bare_apply": 40.0 * D / bare / 1e9, "frac_bare_apply": 40.0 * D / bare / 1e9 / peak,
                     "achieved_sequence": 40.0 * D / per_apply / 1e9, "frac_sequence": 40.0 * D / per_apply / 1e9 / peak,
                     "note": "40 B/amplitude algorithmic per H-apply (psi 16 + Dint 8 + out 16); a Taylor order moves 72-104 "
                             "B/amplitude of own-element traffic (history term, accumulator), a Lanczos iteration 88 (DESIGN.md)"},
    }


# --------------------------------------------------------------------------
def dump_outputs(out_dir: str, psi: np.ndarray, dens: np.ndarray) -> None:
    """What the last timed step computed: the final C2 state as float64 (re, im) pairs (c2_state.npy, [D, 2]) and the
    per-atom Rydberg densities derived from it (c2_rydberg_density.npy).  Above DUMP_BYTES the state is a fixed,
    seeded sample of amplitudes, whose indices go to c2_state_index.npy (float64, exact below 2^53)."""
    os.makedirs(out_dir, exist_ok=True)
    state = np.ascontiguousarray(psi).view(np.float64).reshape(-1, 2)
    if state.nbytes > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(len(state), size=DUMP_BYTES // 16, replace=False))
        state = state[idx]
        np.save(os.path.join(out_dir, "c2_state_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "c2_state.npy"), state)
    np.save(os.path.join(out_dir, "c2_rydberg_density.npy"), np.asarray(dens, dtype=np.float64))


def run_gpu(args) -> None:
    import torch

    from pulser_b200 import engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if engine.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device (the hot path has no CPU fallback)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist  # type: ignore
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{local}"))

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # every replica evolves the same C2 Sequence (same register): equal work per GPU, so that the driver's
    # weak-scaling ratio measures the machine and not the spread of step counts between random registers
    spec = workload(N_ATOMS)
    T = spec.total_duration_ns
    tf = spec.sampling_times[-1]
    D = spec.hilbert_dim
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream()

    # ---- device-resident: plan + tables + psi0 already in HBM ----
    plan = engine.DevicePlan(spec, device=local)
    plan.set_stream(stream.cuda_stream)
    launches = applies = 0
    kernel_ms = 0.0
    for _ in range(args.warmup):
        plan.set_state("all-ground")
        plan.propagate(0.0, tf)
    times_ms = []
    with ClockSampler(local) as clocks:
        for _ in range(args.steps):
            plan.set_state("all-ground")
            flush.fill_(1)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            st = plan.propagate(0.0, tf)
            e1.record(stream)
            barrier()
            times_ms.append(e0.elapsed_time(e1))
            launches += st["n_launches"]; applies += st["n_applies"]; kernel_ms += st["gpu_ms"]
    psi_final = plan.get_state()[0] if args.dump_outputs and rank == 0 else None
    norm2 = float(plan.norm2()[0])
    # final observable of this replica: Rydberg density per atom (host side, from |psi|^2)
    probs = plan.probabilities()[0]
    idx = np.arange(D)
    dens = np.array([probs[((idx >> (N_ATOMS - 1 - k)) & 1) == 0].sum() for k in range(N_ATOMS)])
    total_ms = float(np.sum(times_ms))
    t_all = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    obs = torch.tensor(dens, dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX)  # max over ranks
        dist.all_reduce(obs, op=dist.ReduceOp.SUM)    # THE collective of the path: final expectation values
    total_ms = float(t_all.item())
    value = world * T * args.steps / (total_ms * 1e-3)
    if psi_final is not None:
        dump_outputs(args.dump_outputs, psi_final, dens)

    # ---- end to end through the public API with host buffers ----
    psi0_host = np.zeros(D, dtype=np.complex128)
    psi0_host[D - 1] = 1.0
    psi0_pinned = torch.from_numpy(psi0_host).pin_memory().numpy()
    h2d = psi0_host.nbytes + sum(d.coef[:1].nbytes + d.det[:1].nbytes for d in spec.drives) \
        + spec.interaction_matrix.nbytes + spec.sampling_times.nbytes
    d2h = psi0_host.nbytes
    plan.close()
    e2e_times = []
    for i in range(args.warmup + args.steps):
        barrier()
        t0 = time.perf_counter()
        with engine.DevicePlan(spec, device=local) as p2:   # uploads tables + U, builds Dint on device
            p2.set_state(psi0_pinned)                        # H2D of the initial state
            p2.propagate(0.0, tf)
            final = p2.get_state()[0]                        # D2H of the result
        barrier()
        if i >= args.warmup:
            e2e_times.append(time.perf_counter() - t0)
    assert abs(np.vdot(final, final).real - 1.0) < 1e-8
    e2e_t = torch.tensor([float(np.sum(e2e_times))], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_value = world * T * args.steps / float(e2e_t.item())

    peak, peak_src = measured_peak()
    c4 = None
    if os.environ.get("PB200_BENCH_SKIP_C4", "0") != "1":
        c4 = c4_leg(local, rank, world, dist, barrier, stream)
    c5 = None
    if world == 1 and os.environ.get("PB200_BENCH_SKIP_C5", "0") != "1":
        c5 = c5_leg(local, stream, peak)
    c3 = None
    if world == 1 and os.environ.get("PB200_BENCH_SKIP_C3", "0") != "1":
        c3 = c3_leg(local, stream)
    if rank == 0:
        per_launch_s = (kernel_ms * 1e-3) / max(launches, 1)
        # 16 (psi) + 8 (Dint) + 16 (out) per amplitude per H-apply (SURVEY 8d); a launch of the Taylor stage kernel
        # carries one H-apply (the history / accumulator traffic of the order is NOT counted as algorithmic)
        applies_per_launch = applies / max(launches, 1)
        alg_bytes = 40.0 * D * applies_per_launch
        achieved = alg_bytes / per_launch_s / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64 (complex128)", "data": "synthetic",
            "config": config_dict(world),
            "steps_x_dim": value * D,
            "h_applies_per_time_step": applies / (T * args.steps),
            "integrator": INTEGRATOR_NAMES.get(int(st.get("integrator", 1)), "?"),
            "norm2_final": norm2,
            "clocks": clocks.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "api": "pulser_b200.engine.DevicePlan(spec).set_state/propagate/get_state (C-ABI, host buffers)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic_per_launch(), "peak_source": peak_src,
                         "kernel": "stage_d2_taylor_kernel (fused H-apply + Taylor-order update + accumulation; one order per launch)",
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "h_applies_per_launch": applies_per_launch,
                         "avg_launch_us": per_launch_s * 1e6,
                         "note": "achieved = algorithmic bytes / (CUDA-event time of the propagation / launches), launch "
                                 "gaps included; traffic = dram read+write per launch from the committed ncu --set full "
                                 "capture (profiles/r02_taylor_stage_kernel_summary.json), cold L2 at every ncu replay; in the "
                                 "timed run the 16 MiB state and its ring buffers stay L2-resident"},
        }
        if c4 is not None:
            line["c4"] = c4
        if c5 is not None:
            line["c5"] = c5
        if c3 is not None:
            line["c3"] = c3
        if os.environ.get("PB200_BENCH_SKIP_CPU", "0") != "1":
            n_sample = int(os.environ.get("PB200_REF_SAMPLE_STEPS", "50" if N_ATOMS >= 20 else "400"))
            line["cpu_baseline"] = cpu_reference_run(workload(N_ATOMS), n_sample) if world == 1 else None
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def _count(minimum: int):
    def parse(text: str) -> int:
        v = int(text)
        if v < minimum:
            raise argparse.ArgumentTypeError(f"must be >= {minimum}, got {v}")
        return v
    return parse


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=_count(1), default=1)
    ap.add_argument("--steps", type=_count(1), default=5, help="timed steps (passes over the whole sequence)")
    ap.add_argument("--warmup", type=_count(0), default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/*.npy (b200 arm)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
