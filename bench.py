#!/usr/bin/env python
"""bench.py — MPC QP solves/sec of the batched B200 tracking step (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (libcudampc.so)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path, restated (oracle/), all host cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results as DIR/<name>.npy

Headline (`value`, `e2e`, `roofline`): BASELINE.json configs[2] - 65,536 independent horizon-50 tracking QPs with the
steering-rate limit +-0.02 rad/step PER GPU; a "step" is one pass of the hot path over that batch.  Under torchrun every rank
solves its own shard of one seeded global batch (weak scaling, no collective on the data path); torch.distributed only gathers
the per-rank times and counters.  The same JSON line carries a `configs` block with the other BASELINE configurations as the
driver's default invocation measures them:
  config2  4,096 x horizon 20 (default limits), L2 flushed between launches                          (rank 0)
  config4  closed-loop roll-out of 8,192 vehicles x 500 steps, warm start, per-step p50 / p99 latency   (rank 0)
  config5  the 1,048,576-problem horizon-50 sweep (seed 5) split over the N ranks: STRONG scaling       (all ranks)
One JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only; nothing is cached in it

METRIC = "MPC QP solves/sec (horizon 50, batched)"
UNIT = "solves/s"
HORIZON = 50
BATCH = 65536
SEED = 3
DU_DELTA = 0.02            # rad/step, configs[2] "tight steering-rate limits"
EPS = 1e-6                 # parity setting of BASELINE.json (u0 within 1e-5 at eps_abs = eps_rel = 1e-6)
POLISH_PASSES = 5
POLISH_RETRY = 4           # with 4, every problem of the bench batch ends on a polished KKT point (2 leaves 1 of 65,536)
EARLY_POLISH = 1           # finish as soon as a polish certifies a KKT point of a settled active set (DESIGN.md §2)
EARLY_CHECK = 50           # with early polish: termination checks / polish probes every 50 iterations = the rho-adaptation interval, i.e. ONE
                           # driver event per block of 50 iterations (measured 368k -> 431k; the OSQP-literal arm keeps OSQP's 25)
SWEEP_BATCH = 1 << 20      # configs[4]: 1,048,576 problems, seed 5
FP64_NOMINAL_TFLOPS = 37.2  # B200 data-sheet non-tensor fp64 rate (the live DFMA probe measures ~34)

# canonical flop model of BASELINE.md §2 / SURVEY.md §8d (n = 11N+5, m = 19N+7, nnz(A) = 43N+5)
_NNZ_L = {15: 706, 20: 941, 50: 2349}
# DRAM traffic per solve of K_solve: dram__bytes_read.sum + dram__bytes_write.sum of the ncu --set full capture committed under
# profiles/ (see profiles/README.md for the file and launch it comes from); a constant from that capture, not measured live.
TRAFFIC_BYTES_PER_SOLVE = None     # filled from profiles/traffic.json when present


def flop_model(N: int):
    n, m, nnzA = 11 * N + 5, 19 * N + 7, 43 * N + 5
    nnzL = _NNZ_L.get(N, int(round(47 * N + 1)))
    f_iter = 4 * nnzL + 4 * nnzA + 8 * n + 10 * m
    f_chol = 121 * n
    return dict(f_iter=f_iter, f_chol=f_chol, f_solve=4 * nnzL, f_lin=40 * N)


def flops_of_batch(N, iters, n_fac, n_solves):
    """flops = n_fac*F_chol + iters*F_iter + (polish triangular solves)*4 nnz(L) + F_lin, from the kernel's counters."""
    fm = flop_model(N)
    it, nf, ns = float(np.sum(iters)), float(np.sum(n_fac)), float(np.sum(n_solves))
    return nf * fm["f_chol"] + it * fm["f_iter"] + max(ns - it, 0.0) * fm["f_solve"] + len(iters) * fm["f_lin"]


def io_bytes(N, B):
    """algorithmic bytes per solve (SURVEY §8d): in 32N+80, out 48N+56."""
    return B * (32 * N + 80), B * (48 * N + 56)


DUMP_BYTES = 60_000_000     # --dump-outputs stays under 64 MB: a fixed sample of the problems when the whole batch does not fit
DUMP_FIELDS = ("u0", "Xp", "Up", "status", "iters", "pri_res", "dua_res", "info")


def dump_outputs(out_dir: str, res) -> None:
    """Every array of the BatchResult the timed path returns, as float64 (the int32 counters are exact in it), so that two builds
    can be compared output for output.  All problems when they fit DUMP_BYTES, else the same seeded sample of problems from every
    array; `problem_index.npy` holds the sampled problems' positions in the batch."""
    import torch
    B = res.u0.shape[0]
    row_bytes = 8 * (1 + sum(int(np.prod(getattr(res, k).shape[1:])) for k in DUMP_FIELDS))
    n = min(B, DUMP_BYTES // row_bytes)
    idx = np.arange(B) if n == B else np.sort(np.random.default_rng(0).choice(B, n, replace=False))
    sel = torch.as_tensor(idx, device=res.u0.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "problem_index.npy"), idx.astype(np.float64))
    for k in DUMP_FIELDS:
        np.save(os.path.join(out_dir, f"{k}.npy"), getattr(res, k)[sel].double().cpu().numpy())


def shard_range(rank: int, world: int, total: int):
    """Static contiguous split of a global batch of `total` problems over `world` ranks (SURVEY §8e): (start, count)."""
    base, rem = divmod(total, world)
    start = rank * base + min(rank, rem)
    return start, base + (1 if rank < rem else 0)


def product_params(N=HORIZON, du=DU_DELTA):
    from rrt_mpc_b200 import MPCConfig
    p = MPCConfig(horizon=N).to_parameters(0.8)
    return dataclasses.replace(p, du_bounds=((-12.0, 12.0), (-du, du)))


def gather_metrics(local: dict, world: int):
    """All-gather a flat dict of floats (summary metrics only)."""
    if world == 1:
        return [local]
    import torch
    import torch.distributed as dist
    keys = sorted(local)
    dev = "cuda" if dist.get_backend() == "nccl" else "cpu"
    t = torch.tensor([float(local[k]) for k in keys], dtype=torch.float64, device=dev)
    out = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return [dict(zip(keys, o.cpu().tolist())) for o in out]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        # under load = upper half of the samples (the sampler also sees the idle gaps between steps)
        load = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------
# CPU baseline: the oracle's restatement of the reference path, one process per host core
# ----------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    lo, hi, N, du, seed, batch, eps, scaling = args
    from oracle import c_oracle as CO
    from oracle import mpc_numpy as O
    from rrt_mpc_b200.synthetic import make_batch
    p = dataclasses.replace(O.Params(horizon=N), du_bounds=((-12.0, 12.0), (-du, du)))
    x0, ref, up = make_batch(batch, N, seed, start=lo, count=hi - lo)
    CO.lib()
    t = time.perf_counter()
    r = CO.solve_batch(p, x0, ref, up, eps_abs=eps, eps_rel=eps, scaling=scaling, polish_passes=1, z0_projected=int(scaling == 0))
    dt = time.perf_counter() - t
    return dt, int((r["status"] == 1).sum()), float(r["iters"].mean())


def cpu_baseline(sample: int, N=HORIZON, eps=EPS, scaling=10, cores=None):
    """Cold solves (the reference rebuilds its problem every call, mpc_controller.py:119) of the first `sample`
    problems of the bench batch with the restated OSQP path; input generation excluded.  scaling = 10: OSQP's default
    (what the reference runs); scaling = 0: the unscaled iteration the CUDA kernel runs (same algorithm, for the split
    of the GPU/CPU ratio into hardware and iteration count)."""
    import multiprocessing as mp
    cores = cores or os.cpu_count() or 1
    per = max(1, sample // cores)
    jobs = [(i * per, (i + 1) * per, N, DU_DELTA, SEED, BATCH, eps, scaling) for i in range(cores)]
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, jobs)
    tmax = max(r[0] for r in res)
    n = per * cores
    return {"value": n / tmax, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"first {n} of the {BATCH} bench problems, cold start each, eps {eps:g}, OSQP-equivalent C restatement "
                      f"(Ruiz scaling {scaling}, polish), one process per core, {tmax:.1f} s",
            "solved": int(sum(r[1] for r in res)), "mean_iters": float(np.mean([r[2] for r in res]))}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (restated; cvxpy/osqp are absent offline)."""
    if rank != 0:
        return
    vals = []
    sample = args.cpu_sample
    for i in range(args.warmup + args.steps):
        cb = cpu_baseline(sample)
        if i >= args.warmup:
            vals.append(cb)
    v = float(np.mean([c["value"] for c in vals]))
    ms = 1e3 * sample / v
    cb = dict(vals[-1]); cb["value"] = v
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{BATCH} independent tracking QPs, horizon {HORIZON}, steering-rate +-{DU_DELTA} (BASELINE configs[2]); "
                                   f"each step = a bounded sample of {sample} problems on all host cores", "eps": EPS},
            "cpu_baseline": cb,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------
# The other BASELINE configurations
# ----------------------------------------------------------------------------------------------------
def timed_launches(torch, dev, stream, flush, fn, reps):
    """CUDA-event time of `reps` launches of fn() with an L2 flush (untimed) before each."""
    out = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); res = fn(); e1.record(stream)
        torch.cuda.synchronize(dev)
        out.append(e0.elapsed_time(e1))
    return np.array(out), res


def run_config2(torch, dev, stream, flush, local_rank, peak_tf, reps=30):
    """BASELINE configs[1]: 4,096 independent QPs, horizon 20, default limits, one launch (7 MB of I/O: L2 flushed)."""
    from rrt_mpc_b200 import MPCController, SolverSettings
    from rrt_mpc_b200.synthetic import make_batch
    N, B = 20, 4096
    x0, ref, up = make_batch(B, N, 2)
    d = [torch.as_tensor(a).to(dev) for a in (x0, ref, up)]
    out = {"workload": "4,096 independent tracking QPs, horizon 20, default limits (BASELINE.json configs[1]), seed 2; one launch, "
                       "256 MB written between launches to flush L2", "batch": B, "horizon": N}
    for name, early in (("early_polish", True), ("osqp_literal", False)):
        ctl = MPCController(product_params(N, 0.15), SolverSettings(eps_abs=EPS, eps_rel=EPS, polish_passes=POLISH_PASSES, polish_retry=POLISH_RETRY, keep_iterate=False,
                                                                      early_polish=early, check_termination=EARLY_CHECK if early else 25), device=local_rank, max_batch=B)
        for _ in range(3):
            ctl.solve_batch(d[0], d[1], u_prev=d[2])
        ms, res = timed_launches(torch, dev, stream, flush, lambda: ctl.solve_batch(d[0], d[1], u_prev=d[2]), reps)
        it, info = res.iters.cpu().numpy(), res.info.cpu().numpy()
        tf = flops_of_batch(N, it, info[:, 1], info[:, 3]) / (ms.mean() * 1e-3) / 1e12
        out[name] = {"value": B / (ms.mean() * 1e-3), "unit": UNIT, "ms_per_step": float(ms.mean()), "p50_ms": float(np.percentile(ms, 50)),
                     "p99_ms": float(np.percentile(ms, 99)), "launches": reps, "iters_mean": float(it.mean()),
                     "solved_frac": float((res.status == 1).double().mean().item()), "polished_frac": float((info[:, 2] > 0).mean()),
                     "problems_per_sm": ctl.problems_per_sm(),
                     "roofline": {"bound": "fp64", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf if peak_tf > 0 else None}}
        ctl.close()
    return out


def run_config4(torch, dev, local_rank, vehicles=8192, steps=500):
    """BASELINE configs[3]: closed-loop roll-out of 8,192 vehicles along perturbed copies of the default RRT* path for 500 steps,
    per-step relinearisation, warm start, everything on the device (one launch of K_rollout; goals placed out of reach so that
    every vehicle runs all steps).  Per-step latency: %globaltimer around every closed-loop step of every vehicle."""
    from rrt_mpc_b200 import MPCConfig, SolverSettings, TrajectoryTracker
    d = np.load(os.path.join(ROOT, "tests", "golden", "default_scenario.npz"))
    path = np.array(d["path"])
    rng = np.random.default_rng(4)
    noise = rng.normal(size=(vehicles,) + path.shape) * 0.15
    noise[:, 0] = 0.0
    paths = [path + noise[b] for b in range(vehicles)]
    starts = path[0] + rng.normal(size=(vehicles, 2)) * 0.5
    goals = np.full((vehicles, 2), 1e9)
    tr = TrajectoryTracker(MPCConfig(sim_steps=steps), None, device=local_rank,
                           settings=SolverSettings(eps_abs=EPS, eps_rel=EPS, polish_passes=POLISH_PASSES, polish_retry=2, early_polish=False))
    tr.track_batch(paths[:512], starts[:512], goals[:512], map_resolution=0.8, warm_start=True, sim_steps=50)      # warm-up
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t = time.perf_counter()
    e0.record()
    res = tr.track_batch(paths, starts, goals, map_resolution=0.8, warm_start=True, record_step_time=True)
    e1.record()
    torch.cuda.synchronize(dev)
    wall = time.perf_counter() - t
    n = int(res.n_steps.sum())
    ns = res.step_ns[res.step_status != 0].astype(np.float64)
    # A vehicle's steps are sequential, so the launch ends with its slowest vehicle.  A few of the perturbed vehicles lose the
    # path (spinning, |yaw| of several turns) and need 10-20x the iterations of the others at every step: report what the
    # device sustains while all its slots are busy next to the wall-clock rate.
    per_vehicle_s = res.step_ns.astype(np.float64).sum(axis=1) / 1e9
    slots = min(vehicles, tr._controller(tr.mpc.to_parameters(0.8), key="rollout").rollout_resident())
    busy_s = float(per_vehicle_s.sum())
    speed = np.abs(res.states[:, :, 3])
    return {"workload": f"{vehicles} vehicles x {steps} closed-loop steps along perturbed copies of the default RRT* path (BASELINE.json configs[3]), "
                        "horizon 15, warm start, OSQP-literal termination + polish, references built on the device, one K_rollout launch",
            "vehicles": vehicles, "sim_steps": steps, "vehicle_steps": n, "value": n / wall, "unit": "vehicle-steps/s (= closed-loop MPC solves/s)",
            "wall_s": wall, "device_ms_incl_reference_build_and_d2h": float(e0.elapsed_time(e1)), "aborted": int(res.aborted.sum()),
            "relaxed": int(res.relaxed.sum()), "iters_mean_per_step": float(res.step_iters[res.step_status != 0].mean()),
            "settings": "eps 1e-6, polish_passes 5, polish_retry 2 (the closed-loop tests' settings), warm start",
            "resident_vehicles": int(slots),
            "value_all_slots_busy": n / (busy_s / slots) if busy_s > 0 else None,
            "slowest_vehicle_s": float(per_vehicle_s.max()), "median_vehicle_s": float(np.median(per_vehicle_s)),
            "moving_steps_frac": float(np.nanmean(speed > 0.5)),
            "note": "wall clock = slowest vehicle: the launch ends when the last sequential 500-step chain ends; value_all_slots_busy = steps / "
                    "(sum of all step times / resident vehicles); vehicles reach the end of the 45-point path after ~100 steps and hold "
                    "position for the rest (moving_steps_frac)",
            "step_latency_us": {"p50": float(np.percentile(ns, 50)) / 1e3, "p99": float(np.percentile(ns, 99)) / 1e3, "max": float(ns.max()) / 1e3,
                                "mean": float(ns.mean()) / 1e3, "samples": int(ns.size),
                                "note": "one closed-loop step of one vehicle (window gather, solve, f_discrete, path-index rule) while "
                                        "all vehicles share the GPU"}}


def run_config5(torch, dist, dev, stream, rank, world, local_rank):
    """BASELINE configs[4]: the 1,048,576-problem horizon-50 sweep (seed 5), split contiguously over the ranks - STRONG scaling.
    One warm-up and one timed step per rank (device resident); time = max over ranks."""
    from rrt_mpc_b200 import MPCController, SolverSettings
    from rrt_mpc_b200.synthetic import make_batch
    start, count = shard_range(rank, world, SWEEP_BATCH)
    x0, ref, up = make_batch(SWEEP_BATCH, HORIZON, 5, start=start, count=count)
    ctl = MPCController(product_params(), SolverSettings(eps_abs=EPS, eps_rel=EPS, polish_passes=POLISH_PASSES, polish_retry=POLISH_RETRY, keep_iterate=False,
                                                         early_polish=bool(EARLY_POLISH), check_termination=EARLY_CHECK if EARLY_POLISH else 25), device=local_rank, max_batch=count)
    d = [torch.as_tensor(a).to(dev) for a in (x0, ref, up)]
    ctl.solve_batch(d[0][:BATCH], d[1][:BATCH], u_prev=d[2][:BATCH])
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream); res = ctl.solve_batch(d[0], d[1], u_prev=d[2]); e1.record(stream)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    info = res.info.cpu().numpy()
    local = {"ms": ms, "count": float(count), "solved": float((res.status == 1).sum().item()), "polished": float((info[:, 2] > 0).sum()),
             "iters": float(res.iters.double().sum().item())}
    ctl.close()
    return local


# ----------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH, help="problems per GPU per step")
    ap.add_argument("--cpu-sample", type=int, default=2048, help="problems in the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--latency-launches", type=int, default=100, help="launches of one resident wave for the latency percentiles")
    ap.add_argument("--skip-configs", action="store_true", help="headline only: skip the config2 / config4 / config5 blocks")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (rank 0) as DIR/<name>.npy, float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the MPC hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from rrt_mpc_b200 import MPCController, SolverSettings
    from rrt_mpc_b200.synthetic import make_batch

    N, B = HORIZON, args.batch
    warmup = max(3, args.warmup)
    params = product_params()
    settings = SolverSettings(eps_abs=EPS, eps_rel=EPS, polish_passes=POLISH_PASSES, polish_retry=POLISH_RETRY, keep_iterate=False, early_polish=bool(EARLY_POLISH),
                              check_termination=EARLY_CHECK if EARLY_POLISH else 25)
    start, count = rank * B, B                      # weak scaling: every rank its own B problems of the seeded global batch
    x0, ref, up = make_batch(B * world, N, SEED, start=start, count=count)
    ctl = MPCController(params, settings, device=local_rank, max_batch=B)
    dev = torch.device("cuda", local_rank)
    d_x0, d_ref, d_up = (torch.as_tensor(a).to(dev) for a in (x0, ref, up))
    pin = lambda a: torch.as_tensor(a).pin_memory().numpy()
    h_x0, h_ref, h_up = pin(x0), pin(ref), pin(up)
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream(dev)
    peak_tf = ctl.fp64_peak_tflops()

    def sync():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    for _ in range(warmup):
        res = ctl.solve_batch(d_x0, d_ref, u_prev=d_up)
    sync()

    # ---- device-resident timing (value) ----------------------------------------------------------
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    launches0 = ctl.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sync()
    t_wall = time.perf_counter()
    for e0, e1 in ev:
        flush.zero_()                       # L2 flush between timed iterations (untimed)
        e0.record(stream)
        res = ctl.solve_batch(d_x0, d_ref, u_prev=d_up)
        e1.record(stream)
    sync()
    t_wall = time.perf_counter() - t_wall
    launches = ctl.launch_count() - launches0
    step_ms = [e0.elapsed_time(e1) for e0, e1 in ev]
    clk = clocks.stop() if rank == 0 else None

    iters = res.iters.cpu().numpy(); info = res.info.cpu().numpy(); status = res.status.cpu().numpy()
    flops = flops_of_batch(N, iters, info[:, 1], info[:, 3])

    # ---- same batch, OSQP-literal termination (polish only after the ADMM residual test; no early polish) -----------
    lit = SolverSettings(eps_abs=EPS, eps_rel=EPS, polish_passes=POLISH_PASSES, polish_retry=POLISH_RETRY, keep_iterate=False, early_polish=False)
    ctl.solve_batch(d_x0, d_ref, u_prev=d_up, settings=lit)
    sync()
    lit_ms = []
    for _ in range(max(2, min(args.steps, 3))):
        l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        flush.zero_()
        l0.record(stream); lres = ctl.solve_batch(d_x0, d_ref, u_prev=d_up, settings=lit); l1.record(stream)
        sync()
        lit_ms.append(l0.elapsed_time(l1))
    lit_ms_all = [float(x) for x in lit_ms]
    lit_ms = float(np.median(lit_ms))
    lit_iters = lres.iters.cpu().numpy(); lit_info = lres.info.cpu().numpy()
    lit_flops = flops_of_batch(N, lit_iters, lit_info[:, 1], lit_info[:, 3])
    u0_gap = float((lres.u0 - res.u0).abs().max().item())

    # ---- per-launch latency of one resident wave (BASELINE metric: p99 per-step latency) -----------------------------
    wave = min(B, 148 * ctl.problems_per_sm())          # (SMs x problems/SM)
    lat = []
    for i in range(args.latency_launches):
        o = (i * wave) % max(1, B - wave + 1)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(stream); ctl.solve_batch(d_x0[o:o + wave], d_ref[o:o + wave], u_prev=d_up[o:o + wave]); a1.record(stream)
        torch.cuda.synchronize(dev)
        lat.append(a0.elapsed_time(a1))
    lat = np.array(lat[5:]) if len(lat) > 10 else np.array(lat)

    # ---- end-to-end through the public API with host buffers, EVERY step timed ------------------------------------------
    ctl.pinned_outputs = True            # page-locked result arrays, reused per call (inputs are pinned above)
    for _ in range(2):
        ctl.solve_batch(h_x0, h_ref, u_prev=h_up)
    sync()
    e2e_t = []
    for _ in range(args.steps):
        t = time.perf_counter()
        hres = ctl.solve_batch(h_x0, h_ref, u_prev=h_up)
        e2e_t.append(time.perf_counter() - t)
    sync()
    h2d = B * (4 + 4 * (N + 1) + 2) * 8
    d2h = B * (2 + 4 * (N + 1) + 2 * N + 2) * 8 + B * 6 * 4
    assert np.array_equal(hres.status, status)
    per_sm, ws_doubles = ctl.problems_per_sm(), ctl.workspace_doubles()
    ctl.close()

    local = {"ms_total": float(np.sum(step_ms)), "ms_max_step": float(np.max(step_ms)), "solves": float(B * args.steps), "flops": flops,
             "solved": float((status == 1).sum()), "iters_mean": float(iters.mean()), "iters_max": float(iters.max()),
             "e2e_total_s": float(np.sum(e2e_t)), "e2e_max_s": float(np.max(e2e_t)), "launches": float(launches), "polished": float((info[:, 2] > 0).sum()),
             "n_fac_mean": float(info[:, 1].mean()), "wall_s": t_wall, "lit_ms": lit_ms, "lit_solves": float(B),
             "lit_polished": float((lit_info[:, 2] > 0).sum())}
    allm = gather_metrics(local, world)

    # ---- the other BASELINE configurations ------------------------------------------------------------------------------
    configs = {}
    c5 = None
    if not args.skip_configs:
        del d_x0, d_ref, d_up
        torch.cuda.empty_cache()
        c5 = gather_metrics(run_config5(torch, dist, dev, stream, rank, world, local_rank), world)
        if rank == 0:
            configs["config2"] = run_config2(torch, dev, stream, flush, local_rank, peak_tf)
            configs["config4"] = run_config4(torch, dev, local_rank)
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    if c5 is not None:
        t5 = max(m["ms"] for m in c5) * 1e-3
        n5 = sum(m["count"] for m in c5)
        configs["config5"] = {"workload": f"{SWEEP_BATCH} independent tracking QPs, horizon {HORIZON}, steering-rate +-{DU_DELTA}, seed 5 (BASELINE.json configs[4]), "
                                          f"split contiguously over {world} GPU(s), device resident, one timed step, time = max over ranks",
                              "scaling": "strong", "global_batch": int(n5), "n_gpus": world, "ms_per_step": t5 * 1e3, "value": n5 / t5, "unit": UNIT,
                              "solved_frac": sum(m["solved"] for m in c5) / n5, "polished_frac": sum(m["polished"] for m in c5) / n5,
                              "iters_mean": sum(m["iters"] for m in c5) / n5, "per_rank_ms": [m["ms"] for m in c5]}

    t_ms = max(m["ms_total"] for m in allm)                     # max over ranks
    total_solves = sum(m["solves"] for m in allm)
    value = total_solves / (t_ms * 1e-3)
    ms_per_step = t_ms / args.steps
    e2e_value = (B * world * args.steps) / max(m["e2e_total_s"] for m in allm)
    # roofline of the dominant (only) kernel, per launch on rank 0: canonical flops / CUDA-event duration
    ach_tf = flops / (float(np.mean(step_ms)) * 1e-3) / 1e12
    inb, outb = io_bytes(N, B)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_ach = (inb + outb) / (float(np.mean(step_ms)) * 1e-3) / 1e9
    cb = cb0 = None
    if not args.no_cpu_baseline:
        cb = cpu_baseline(args.cpu_sample)
        cb0 = cpu_baseline(max(args.cpu_sample // 2, os.cpu_count() or 1), scaling=0)
        cb["same_algorithm"] = {"value": cb0["value"], "unit": UNIT, "mean_iters": cb0["mean_iters"], "sample": cb0["sample"],
                                "note": "the C port run as the kernel runs OSQP (scaling 0, z0 = clip(0)): compare with value_literal - "
                                        "that ratio is hardware + implementation; the rest of the headline ratio is iteration count"}
    lit_value = sum(m["lit_solves"] for m in allm) / (max(m["lit_ms"] for m in allm) * 1e-3)
    lit_tf = lit_flops / (lit_ms * 1e-3) / 1e12

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
        "ms_per_step": ms_per_step, "p99_ms_per_step": float(np.percentile(step_ms, 99)), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "value_literal": lit_value,
        "config": {"workload": f"{B} independent tracking QPs per GPU, horizon {N}, 4 states / 2 controls, steering-rate +-{DU_DELTA} rad/step "
                               f"(BASELINE.json configs[2]), seed {SEED}", "batch_per_gpu": B, "horizon": N, "eps_abs": EPS, "eps_rel": EPS,
                   "polish_passes": POLISH_PASSES, "polish_retry": POLISH_RETRY, "early_polish": EARLY_POLISH, "check_termination": EARLY_CHECK if EARLY_POLISH else 25, "parallelism": f"{world} x independent shards, no data-path collective",
                   "termination": "value: early certified polish (finishes as soon as a polish ends on a KKT point of a settled active set); "
                                  "value_literal: the same kernel with OSQP's own termination (residual test at eps 1e-6, then polish)",
                   "l2": "working set per step (inputs 112 MB + outputs 161 MB) exceeds the 126 MB L2 (stateless solves: keep_iterate=False, no per-problem warm-start state is written); "
                         "a 256 MB write flushes L2 between timed steps"},
        "solve_stats": {"solved_frac": sum(m["solved"] for m in allm) / (B * world), "iters_mean": float(np.mean([m["iters_mean"] for m in allm])),
                        "iters_max": max(m["iters_max"] for m in allm), "polished_frac": sum(m["polished"] for m in allm) / (B * world),
                        "factorisations_mean": float(np.mean([m["n_fac_mean"] for m in allm])),
                        "problems_per_sm": per_sm, "smem_doubles_per_problem": ws_doubles},
        "roofline": {"bound": "fp64", "achieved": ach_tf, "peak": peak_tf, "peak_nominal": FP64_NOMINAL_TFLOPS, "unit": "TFLOP/s",
                     "frac": ach_tf / peak_tf if peak_tf > 0 else None, "frac_of_nominal": ach_tf / FP64_NOMINAL_TFLOPS,
                     "traffic": (traffic["bytes_per_solve"] * B) if traffic else None,
                     "traffic_unit": "bytes per launch" + (f" ({traffic['source']})" if traffic else ""),
                     "note": "binding roofline is the non-tensor fp64 pipe (SURVEY.md 8d); achieved = canonical flops (BASELINE.md model, from the "
                             "kernel's own iteration/factorisation counters) / CUDA-event time of one launch; peak = DFMA throughput measured "
                             "live by cudampc_fp64_peak_tflops (MEASURED_PEAKS.json has no fp64 figure), peak_nominal = data sheet",
                     "hbm": {"achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                             "algorithmic_bytes_per_launch": inb + outb, "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}},
        "osqp_literal": {"value": lit_value, "unit": UNIT, "ms_per_step": lit_ms, "ms_per_step_all": lit_ms_all,
                         "iters_mean": float(lit_iters.mean()), "achieved_tflops": lit_tf,
                         "frac": lit_tf / peak_tf if peak_tf > 0 else None, "frac_of_nominal": lit_tf / FP64_NOMINAL_TFLOPS,
                         "polished_frac": sum(m["lit_polished"] for m in allm) / (B * world), "max_abs_u0_gap_vs_early_polish": u0_gap,
                         "note": "same kernel with early_polish off: ADMM runs until the eps 1e-6 residual test passes, then polishes; median of the timed launches"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps_timed": args.steps,
                "ms_per_step_mean": 1e3 * float(np.mean(e2e_t)), "ms_per_step_p99": 1e3 * float(np.percentile(e2e_t, 99)),
                "ms_per_step_max_over_ranks": 1e3 * max(m["e2e_max_s"] for m in allm),
                "note": "MPCController.solve_batch on pinned host arrays: H2D, solve, D2H inside every timed call"},
        "latency": {"batch": int(wave), "launches": int(len(lat)), "p50_ms": float(np.percentile(lat, 50)), "p99_ms": float(np.percentile(lat, 99)),
                    "note": "one launch of exactly one resident wave of problems (SMs x problems/SM), device-resident, rank 0"},
        "configs": configs,
        "gpu_launches": int(sum(m["launches"] for m in allm)),
        "clocks": clk,
        "cpu_baseline": cb,
        "wall_s_timed_region": max(m["wall_s"] for m in allm),
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res)            # res: the last timed step of the headline
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
