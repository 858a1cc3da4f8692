#!/usr/bin/env python
"""bench.py — headline benchmark of the WVA optimization hot path on B200.

Metric (BASELINE.json): (model,variant,replica) evals/sec + solver wall-ms at 1/2/4/8 B200, next to the reference
algorithm on the box's host cores.

Workload = BASELINE.json configs[2], the largest single-GPU configuration: 100 k models x 32 accelerator variants x 256
replica levels (N = 256, K = 2816 chain states), 3 service classes with per-class latency SLOs, per-type GPU-count cap at
60 % of the unconstrained demand.  One "step" = one pass of the hot path over that system with its inputs resident in HBM:

    System.Calculate   sizing of every (server, accelerator) candidate          pkg/core/system.go:258-268
    Manager.Optimize   unlimited (per-server argmin + AllocateByType) AND limited (SolveGreedy, policy None,
                       + AllocateByType) on the same candidates                  pkg/solver/solver.go:32-60, greedy.go:35-105
    replica grid       QueueAnalyzer.Analyze(totalRate / r), r = 1..R, materialised  pkg/analyzer/queueanalyzer.go:127-167

`value` = S*A*R grid evaluations / time of the WHOLE step (sizing + both allocators + grid): the bisection solves of the
sizer make it smaller, never larger.  With --gpus N the SAME system is strong-scaled over N ranks (one process per GPU):
every rank sizes and grids its block of servers, the candidate arena is all-gathered and the by-type partials all-reduced
over NCCL inside the C-ABI library (include/wva_b200.h, wva_comm_*), the greedy sweep runs on every rank.

A second timed leg runs BASELINE configs[3], the one HBM-bound kernel of the path: V1 saturation analysis of 1 M models x
32 variants (~1.44e8 replicas), model-sharded over the ranks with an all-reduce of the partials (`saturation` block and
`roofline_hbm`).  The queueing kernels are FP64-pipe bound (SURVEY 0.4): `roofline` reports the dominant kernel (the
sizer) against the HBM peak as the contract asks — meaningless by construction — and against the measured FP64 peak.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

--steps K sets the number of timed steps of every leg (resident step, end-to-end call, saturation kernel).
--dump-outputs DIR writes, after the timed steps, what the last step of each timed leg computed as DIR/<name>.npy
(float32 stays float32, everything else becomes float64): the candidates, the limited solution, the replica grid
(frontier and per-level arrays) and the saturation outputs.  An output of more than 2^18 entries is written as the same
seeded sample of its entries on every run, so two builds can be compared array by array.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True      # the tree may be read-only: nothing is cached next to the sources

# Rank 0 prints ONE JSON line on stdout.  Libraries (NCCL's version banner, torchrun notices) write to file descriptor 1
# too, so the descriptor is pointed at stderr for the whole run and the line goes out through a saved copy of it.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)
sys.stdout = os.fdopen(os.dup(2), "w", buffering=1)


def emit(line: dict):
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
PKG = "llm-d-workload-variant-autoscaler_b200"

S_TOTAL, A, NB, R = 100_000, 32, 256, 256
SAT_MODELS, SAT_VARIANTS = 1_000_000, 32
CAP_FRACTION = 0.6
ALG_BYTES_PER_EVAL = 17.9                 # SURVEY.md 8(d): 16 B written + amortised inputs per grid evaluation
ALG_BYTES_PER_PAIR = 24 + 36.0 / A + 37   # sizing: 24 B + 36 B/A in, 37 B out per (server, accelerator)
FP64_OPS_PER_STATE = 9.0                  # 5 FP64-pipe ops per pass-1 state, 13 per pass-2 state (DESIGN.md 4)
METRIC = "(model,variant,replica) evals/sec"
DUMP_SAMPLE = 1 << 18                     # --dump-outputs: entries kept of a larger output
DUMP_BYTES = 64 << 20                     # --dump-outputs: size cap of all written arrays together


def workload(scale: float = 1.0):
    synth = importlib.import_module(PKG + ".synth")
    return synth.baseline_config(3, scale=scale)          # stream 3 = BASELINE config 3 (100k x 32 x 256, limited)


def config_dict(world, S):
    return {"workload": f"BASELINE configs[2]: {S} models x {A} variants x {R} replica levels, state-dependent M/M/1/K "
                        f"sizing + unlimited and limited (greedy, policy None, capacity {int(CAP_FRACTION * 100)} % of demand) "
                        f"allocator + materialised replica grid, N={NB}, K={11 * NB}, 3 service classes; second leg "
                        f"configs[3]: V1 saturation, {SAT_MODELS} models x {SAT_VARIANTS} variants",
            "models": S, "variants": A, "replica_levels": R, "max_batch": NB, "chain_states": 11 * NB + 1,
            "parallelism": f"model-sharded x{world} (strong scaling of the same system; NCCL all-gather of candidates, "
                           "all-reduce of by-type partials inside the C-ABI)",
            "l2": "flushed between steps (256 MiB write inside the timed region); the working set (0.3 GB system + "
                  "14 GB grid) exceeds L2 anyway",
            "evaluation": "value = S*A*R grid Analyze evaluations / time of the whole step (sizing + both allocators + "
                          "grid); the sizer's own chain solves are not counted"}


def effective_cores():
    """threads this process may really use: min(affinity mask, cgroup CPU quota)"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(p)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    eff = n if quota is None else max(1, min(n, int(quota)))
    return eff, n, quota


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (profiling recipe)."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, smax, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); smax = max(smax, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---- --dump-outputs ---------------------------------------------------------------------------------------------------
def _pick(n, seed):
    """sorted indices into an output of n entries: all of them, or the same seeded sample of DUMP_SAMPLE draws"""
    if n <= DUMP_SAMPLE:
        return np.arange(n)
    return np.unique(np.random.default_rng(seed).integers(0, n, DUMP_SAMPLE))


def step_outputs(eng, R):
    """What the last resident step left for its caller: the candidates and the limited solution of the whole system,
    the replica grid of this rank's block of servers (frontier + per-level arrays, fetched one array at a time)."""
    out = {}
    cand = eng.candidates()
    pick = _pick(cand["state"].size, 1)
    out.update({"candidates_" + k: v.reshape(-1)[pick] for k, v in cand.items() if k != "n_solves"})   # a work count
    sol = eng.solution()
    pick = _pick(sol["state"].size, 4)
    out.update({"solution_" + k: v if k.startswith("type_") else v[pick] for k, v in sol.items()})
    front = eng.grid_fetch_frontier().reshape(-1)
    out["grid_frontier"] = front[_pick(front.size, 2)]
    n = front.size * R
    pick = _pick(n, 3)
    for i, (k, dt) in enumerate((("ok", np.uint8), ("ttft", np.float32), ("itl", np.float32), ("rho", np.float32),
                                 ("tput", np.float32))):
        buf = np.empty(max(n, 1), dt)
        ptrs = [None] * 6
        ptrs[i] = buf.ctypes.data
        eng._check(eng.lib.wva_grid_fetch(eng.ctx, *ptrs), "wva_grid_fetch")
        out["grid_" + k] = buf[pick]
        del buf
    return out


def write_outputs(path, arrays):
    arrays = {k: np.asarray(v, np.float32 if np.asarray(v).dtype == np.float32 else np.float64)
              for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES} byte cap")
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v)


# ---- the reference algorithm on the host cores ------------------------------------------------------------------------
def _oracle():
    # thread placement must be fixed before libgomp starts: spread-free, pinned (the round-1 numbers swung 6x between boxes
    # with unpinned threads over a cgroup-limited core set)
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    from tests import oracle_lib
    return oracle_lib.load()


def _cpu_step(orc, d, threads):
    """one pass of the reference path on a sample system: Calculate + Optimize (greedy, None) + the replica grid"""
    t0 = time.perf_counter()
    cand = orc.calculate(d, nthreads=threads)
    t1 = time.perf_counter()
    orc.solve(d, cand)
    t2 = time.perf_counter()
    orc.analyze_grid(d, R, nthreads=threads, full=True)
    t3 = time.perf_counter()
    return {"calculate_ms": (t1 - t0) * 1e3, "solve_ms": (t2 - t1) * 1e3, "grid_ms": (t3 - t2) * 1e3, "seconds": t3 - t0,
            "evals": int(d["n_servers"]) * A * R}


def _sample_system(n_servers):
    synth = importlib.import_module(PKG + ".synth")
    d = synth.queue_system(n_servers, A, NB, n_classes=3, stream=3, unlimited=False, R=R)
    d["type_count"] = np.full(d["n_types"], max(1, n_servers), np.int32)      # a cap that binds on the sample too
    return d


_ONE_THREAD = None
_EFF = None


def cpu_reference_leg(target_seconds: float, fixed_sample: int = 0):
    """The reference algorithm (oracle port: the reference is Go and no Go toolchain exists on the box) on a bounded
    sample of the same workload: first one thread on a few servers (also the calibration), then every usable thread on a
    sample sized for ~target_seconds."""
    # before libgomp starts: with OMP_PROC_BIND set it pins the calling thread to its first place, and the affinity mask
    # read afterwards would be that one core (final1 evidence run: "2 pinned threads" in the reference arm)
    global _EFF
    if _EFF is None:
        _EFF = effective_cores()
    eff, aff, quota = _EFF
    orc = _oracle()
    global _ONE_THREAD
    if _ONE_THREAD is None:
        _ONE_THREAD = _cpu_step(orc, _sample_system(4), 1)
    one = _ONE_THREAD
    per_server_1t = one["seconds"] / 4
    n = fixed_sample or int(max(eff * 2, min(20_000, target_seconds * eff / max(per_server_1t, 1e-6))))
    n = max(8, (n // eff) * eff if n >= eff else n)
    allt = _cpu_step(orc, _sample_system(n), eff)
    return {"value": allt["evals"] / allt["seconds"], "unit": "evals/s", "cores": eff, "kind": "port",
            "sample": f"{n} of {S_TOTAL} models x {A} variants x {R} levels (N={NB}), oracle C++ restatement of the "
                      f"reference (every bisection step, stored p[]), OpenMP over servers, {eff} pinned threads",
            "one_thread": {"value": one["evals"] / one["seconds"], "unit": "evals/s", "sample_models": 4,
                           "seconds": one["seconds"]},
            "affinity_cpus": aff, "cgroup_cpu_quota": quota, "sample_models": n,
            "calculate_ms": allt["calculate_ms"], "solve_ms": allt["solve_ms"], "grid_ms": allt["grid_ms"],
            "evals": allt["evals"], "seconds": allt["seconds"]}


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    args.ref_seconds = min(args.ref_seconds, 150.0 / (args.steps + args.warmup))   # the whole arm ends within minutes
    first = cpu_reference_leg(args.ref_seconds)
    n = first["sample_models"]
    legs = [first] + [cpu_reference_leg(args.ref_seconds, fixed_sample=n) for _ in range(args.warmup + args.steps - 1)]
    legs = legs[args.warmup:]
    secs, evals, last = sum(v["seconds"] for v in legs), sum(v["evals"] for v in legs), legs[-1]
    value = evals / secs
    emit({
        "metric": METRIC, "value": value, "unit": "evals/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": secs / len(legs) * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_dict(args.gpus, S_TOTAL),
        "impl": "reference",
        "cpu_baseline": {"value": value, "unit": "evals/s", "cores": last["cores"], "kind": "port",
                         "sample": last["sample"], "one_thread": last["one_thread"],
                         "affinity_cpus": last["affinity_cpus"], "cgroup_cpu_quota": last["cgroup_cpu_quota"]},
        "e2e": {"value": value, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "solver_wall_ms": {"calculate": last["calculate_ms"], "solve": last["solve_ms"], "grid": last["grid_ms"],
                           "note": f"on the bounded sample of {n} models"},
        "host": {"nproc": os.cpu_count()}})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-seconds", type=float, default=8.0, help="CPU seconds per step of the bounded reference sample")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the system (development only; 1.0 = configs[2])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-saturation", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; the reference arm has none")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    pkg = importlib.import_module(PKG)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (there is no CPU fallback); --impl reference runs on the host")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    eng = pkg.Engine(device=local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        # the library's own communicator: the 128-byte id travels through the host-side process group
        idt = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(pkg.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        eng.comm_init(world, rank, bytes(idt.cpu().numpy().tobytes()))
    sysd = workload(args.scale)
    S, T = sysd["n_servers"], sysd["n_types"]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- setup (untimed): the GPU-count cap = 60 % of the unconstrained demand of this very system -----------------------
    eng.load_system(sysd)
    eng.calculate()
    eng.set_optimizer(True)
    eng.solve()
    un = eng.solution()
    cap = np.maximum(1, np.floor(np.asarray(un["type_count"], np.float64) * CAP_FRACTION)).astype(np.int32)
    eng.set_capacity(cap)
    sysd = dict(sysd); sysd["type_count"] = cap; sysd["unlimited"] = False; sysd["saturation_policy"] = "None"
    S_loc = eng.hi - eng.lo

    def resident_step():
        """inputs already in HBM: sizing of the rank's block, both allocators (with their NCCL exchange), grid of the block"""
        flush.zero_()
        eng.calculate()
        t = eng.timing()
        info = dict(size_solves=t["chain_solves"], size_states=t["chain_states"], calc_ms=t["calculate_ms"], sizer_kernel=t["sizer_kernel"])
        eng.set_optimizer(True)
        eng.solve()
        t = eng.timing()
        info.update(solve_unlimited_ms=t["solve_ms"], exch_unlimited_ms=t["exchange_ms"])
        eng.set_optimizer(False, False, "None")
        eng.solve()
        t = eng.timing()
        info.update(solve_limited_ms=t["solve_ms"], exch_limited_ms=t["exchange_ms"],
                    greedy_events=t["greedy_events"], greedy_heap_pushes=t["greedy_heap_pushes"])
        eng.grid_run(R, full=True)
        t = eng.timing()
        info.update(grid_ms=t["grid_ms"], grid_solves=t["chain_solves"], grid_states=t["chain_states"])
        return info

    sysd_pinned = pkg.pinned_copy(sysd)     # the step's inputs in page-locked host memory (wva_host_alloc)

    def e2e_step():
        """the call a user makes: host buffers in, host results out (H2D and D2H inside the timed region)"""
        sol = eng.optimize(sysd_pinned)     # SetFromSpec -> Calculate -> Optimize (limited) -> solution on the host
        eng.grid_run(R, full=False)
        fr = eng.grid_fetch_frontier()
        return sol, fr

    h2d = sum(np.asarray(v).nbytes for v in sysd.values() if isinstance(v, np.ndarray))
    d2h = S * (1 + 9 * 4) + T * 16 + S_loc * A * 4

    for _ in range(args.warmup):
        resident_step()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.25)
    launches0 = eng.launch_count()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    infos = [resident_step() for _ in range(args.steps)]
    e1.record()
    barrier()
    launches = eng.launch_count() - launches0 + args.steps      # + the L2 flush kernel of every step
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    evals_total = float(S) * A * R * len(infos)                 # all ranks together evaluate the whole grid once per step
    value = evals_total / (total_ms * 1e-3)

    # per-phase device times: max over ranks (the step waits for the slowest rank)
    keys = ["calc_ms", "solve_unlimited_ms", "solve_limited_ms", "grid_ms", "exch_unlimited_ms", "exch_limited_ms"]
    ph = torch.tensor([float(np.mean([i[k] for i in infos])) for k in keys], dtype=torch.float64, device=dev)
    cnt = torch.tensor([float(infos[-1]["size_solves"]), float(infos[-1]["size_states"]), float(infos[-1]["grid_solves"]),
                        float(infos[-1]["grid_states"])], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ph, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt)
    ph = dict(zip(keys, ph.tolist()))
    size_solves, size_states, grid_solves, grid_states = cnt.tolist()
    dump = step_outputs(eng, R) if args.dump_outputs and rank == 0 else None    # before the e2e arm replaces the grid

    # ---- end-to-end arm ---------------------------------------------------------------------------------------------------
    for _ in range(2):
        e2e_step()
    barrier()
    e0.record()
    e2e_steps = args.steps
    for _ in range(e2e_steps):
        sol, fr = e2e_step()
    e1.record()
    barrier()
    ms2 = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_value = float(S) * A * R * e2e_steps / (float(ms2.item()) * 1e-3)
    clocks = sampler.stop() if sampler else None
    # (reported beside the step, not part of it) the same limited solve under a best-effort policy
    rr = []
    for _ in range(3):
        eng.set_optimizer(False, False, "RoundRobin")
        eng.solve()
        rr.append(eng.timing()["solve_ms"])
    eng.set_optimizer(False, False, "None")
    rr_t = torch.tensor([float(min(rr))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(rr_t, op=dist.ReduceOp.MAX)
    sizer_id = int(infos[-1]["sizer_kernel"])

    # ---- second leg: configs[3], V1 saturation (the HBM-bound kernel), model-sharded ---------------------------------------
    sat = None
    if not args.no_saturation:
        M_loc = int(SAT_MODELS * args.scale) // world
        batch = pkg.synth.saturation_batch(M_loc, SAT_VARIANTS, stream=4 + 1000 * rank)
        t0 = time.perf_counter()
        eng.saturation_upload(batch)
        up_ms = (time.perf_counter() - t0) * 1e3
        for _ in range(3):
            eng.saturation_run(False)
        ks, xs = [], []
        barrier()
        for _ in range(args.steps):
            flush.zero_()
            torch.cuda.synchronize()      # the flush runs on torch's stream, the kernel on the library's: no overlap
            eng.saturation_run(False)
            t = eng.timing()
            ks.append(t["saturation_ms"]); xs.append(t["exchange_ms"])
        res = eng.saturation_fetch(fields=("partials", "partials_all") + (("var_target", "mod_flags") if dump is not None else ()))
        if dump is not None:
            dump["saturation_partials_all"] = res["partials_all"]
            for k in ("var_target", "mod_flags"):
                dump["saturation_" + k] = res[k][_pick(res[k].size, 5)]
        alg_loc = batch["n_replicas"] * 16 + batch["n_variants"] * 32 + M_loc * 40      # SURVEY 8(d)
        v = torch.tensor([float(np.mean(ks)), float(np.min(ks)), float(np.mean(xs))], dtype=torch.float64, device=dev)
        tot = torch.tensor([float(alg_loc), float(batch["n_replicas"])], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(v, op=dist.ReduceOp.MAX)
            dist.all_reduce(tot)
        sat = {"kernel_ms_mean": v[0].item(), "kernel_ms_min": v[1].item(), "allreduce_ms": v[2].item(),
               "alg_bytes": tot[0].item(), "replicas": int(tot[1].item()), "models": M_loc * world,
               "upload_ms_host_wall": up_ms, "alg_bytes_local": alg_loc,
               "partials_all": [int(x) for x in res["partials_all"]]}

    if rank == 0:
        peaks, traffic = {}, {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
        calc_ms, grid_ms = ph["calc_ms"], ph["grid_ms"]
        dominant = {1: "sizer_warp_kernel", 2: "sizer_lane_kernel", 3: "sizer_lane_kernel", 4: "sizer_pool_kernel"}.get(sizer_id, "sizer_lane_kernel")
        alg_bytes = S_loc * A * ALG_BYTES_PER_PAIR
        achieved = alg_bytes / (calc_ms * 1e-3) / 1e9
        dfma, ddiv = eng.microbench_fp64()
        fp64_rate = FP64_OPS_PER_STATE * (size_states / world) / (calc_ms * 1e-3)
        line = {
            "metric": METRIC, "value": value, "unit": "evals/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(world, S),
            "solver_wall_ms": {"calculate": calc_ms, "solve_unlimited": ph["solve_unlimited_ms"],
                               "solve_limited_none": ph["solve_limited_ms"], "grid": grid_ms,
                               "solve_limited_round_robin_not_in_step": float(rr_t.item()),
                               "nccl_exchange_unlimited": ph["exch_unlimited_ms"], "nccl_exchange_limited": ph["exch_limited_ms"],
                               "calculate_plus_solve_limited": calc_ms + ph["solve_limited_ms"],
                               "note": "device time per phase, max over ranks; solve_* include their NCCL exchange"},
            "evals_per_step": {"grid": S * A * R, "grid_admitted_solves": int(grid_solves),
                               "sizing_solves": int(size_solves), "states_grid": int(grid_states),
                               "states_sizing": int(size_states),
                               "admitted_solves_per_s": grid_solves / (total_ms / args.steps * 1e-3),
                               "note": "grid = S*A*R levels; levels whose rate exceeds RateRange.Max are rejected without a "
                                       "chain solve (as QueueAnalyzer.Analyze does): grid_admitted_solves ran a chain"},
            "greedy": {"events": int(infos[-1]["greedy_events"]), "heap_pushes": int(infos[-1]["greedy_heap_pushes"])},
            "roofline": {"bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved / hbm_peak, "traffic": traffic.get(dominant), "peak_source": peak_src,
                         "note": "dominant kernel of the step; algorithmic bytes / kernel time as the contract asks, but "
                                 "this kernel is FP64-pipe bound (1e3-1e5 flop/B): see `fp64`; the HBM-bound kernel of "
                                 "the path is reported in `roofline_hbm`",
                         "fp64": {"achieved_ops_per_s": fp64_rate, "peak_dfma_per_s": dfma, "peak_ddiv_per_s": ddiv,
                                  "frac_of_dfma_peak": fp64_rate / dfma,
                                  "pipe_active_pct_ncu": (traffic.get("fp64_pipe_active_pct") or {}).get(dominant),
                                  "note": "ALGORITHMIC FP64-pipe ops (9 x live states) / kernel time on rank 0's share; "
                                          "peaks measured in this run by wva_microbench_fp64"}},
            "e2e": {"value": e2e_value, "unit": "evals/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": float(ms2.item()) / e2e_steps,
                    "note": "Engine.optimize (load_system from pinned host buffers -> calculate -> limited solve -> "
                            "solution to the host) + frontier-only grid + frontier to the host"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "decisions": {"allocated_limited": int((sol["state"] == 1).sum()),
                          "gpus_by_type_limited": np.asarray(sol["type_count"]).tolist(), "cap_by_type": cap.tolist()},
            "host": {"nproc": os.cpu_count()},
        }
        if sat:
            a = sat["alg_bytes"] / (sat["kernel_ms_mean"] * 1e-3) / 1e9
            line["saturation"] = sat
            line["roofline_hbm"] = {"bound": "hbm", "kernel": "saturation_kernel", "achieved": a,
                                    "peak": hbm_peak * world, "unit": "GB/s", "frac": a / (hbm_peak * world),
                                    "traffic": traffic.get("saturation_kernel"), "peak_source": peak_src,
                                    "note": "configs[3]: algorithmic bytes of all ranks (16 B/replica + 32 B/variant + "
                                            "40 B/model) / mean kernel time (max over ranks, CUDA events on the library's "
                                            "stream, L2 flushed before every launch); peak = per-GPU copy bandwidth x ranks"}
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = {k: v for k, v in cpu_reference_leg(args.ref_seconds).items()
                                    if k in ("value", "unit", "cores", "kind", "sample", "one_thread", "affinity_cpus",
                                             "cgroup_cpu_quota")}
        if dump is not None:
            write_outputs(args.dump_outputs, dump)
        emit(line)
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
