"""Closed loop with the plant outside the library: BASELINE.json configs[3]'s shape (8,192 vehicles along perturbed copies of
the default RRT* path, horizon 15, eps 1e-6, polish_retry 2, warm start, 500 steps, goals out of reach) driven one step per
call through TrajectoryTracker.start_batch / TrackingSession.step, with cudampc_f_discrete_batch as the plant on device
tensors (nothing crosses PCIe between steps).  Reports the per-step time (CUDA events around every step), vehicle-steps/s,
and track_batch's wall time on the same inputs in the same process.  Prints one JSON line.
usage: python tools/step_bench.py [--vehicles B] [--steps T]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, check=True).stdout.strip()
    except Exception as e:  # noqa: BLE001 - reported, not fatal
        return f"not read ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--vehicles", type=int, default=8192)
    ap.add_argument("--steps", type=int, default=500)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("step_bench needs a CUDA device")
    from rrt_mpc_b200 import MPCConfig, SolverSettings, TrajectoryTracker
    B, T = args.vehicles, args.steps
    d = np.load(os.path.join(ROOT, "tests", "golden", "default_scenario.npz"))
    path = np.array(d["path"])
    rng = np.random.default_rng(4)                     # the vehicles of bench.py's config 4
    noise = rng.normal(size=(B,) + path.shape) * 0.15
    noise[:, 0] = 0.0
    paths = [path + noise[b] for b in range(B)]
    starts = path[0] + rng.normal(size=(B, 2)) * 0.5
    goals = np.full((B, 2), 1e9)
    tr = TrajectoryTracker(MPCConfig(sim_steps=T), None,
                           settings=SolverSettings(eps_abs=1e-6, eps_rel=1e-6, polish_passes=5, polish_retry=2, early_polish=False))
    dev = torch.device("cuda", 0)

    def run_session(n, steps, timed):
        sess = tr.start_batch(paths[:n], starts[:n], goals[:n], map_resolution=0.8, warm_start=True)
        h = sess._h
        x = torch.as_tensor(sess.states0).to(dev)
        xn = torch.empty_like(x)
        stream = torch.cuda.current_stream(dev)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)] if timed else None
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for k in range(steps):
            if timed:
                ev[k][0].record(stream)
            r = sess.step(x)
            if timed:
                ev[k][1].record(stream)
            rc = h.lib.cudampc_f_discrete_batch(h.ptr, n, C.c_void_p(x.data_ptr()), C.c_void_p(r.u0.data_ptr()), None,
                                                C.c_void_p(xn.data_ptr()), C.c_void_p(stream.cuda_stream))
            assert rc == 0, h.lib.cudampc_last_error(h.ptr)
            x = torch.where(torch.isfinite(r.u0[:, :1]), xn, x)     # stopped vehicles keep their state
        torch.cuda.synchronize(dev)
        wall = time.perf_counter() - t0
        ms = np.array([a.elapsed_time(b) for a, b in ev]) if timed else None
        n_steps = int(sess.n_steps.sum())
        aborted = int(sess.aborted.sum())
        sess.close()
        return wall, ms, n_steps, aborted

    run_session(512, 20, False)                         # warm-up: modules, allocator
    wall, ms, n_steps, aborted = run_session(B, T, True)
    tr.track_batch(paths[:512], starts[:512], goals[:512], map_resolution=0.8, warm_start=True, sim_steps=50)   # warm-up
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    res = tr.track_batch(paths, starts, goals, map_resolution=0.8, warm_start=True)
    torch.cuda.synchronize(dev)
    tb_wall = time.perf_counter() - t0
    tb_steps = int(res.n_steps.sum())
    print(json.dumps({
        "gpu": torch.cuda.get_device_name(dev), "power_limit": gpu_power_limit(),
        "workload": f"{B} vehicles x {T} steps, horizon 15, eps 1e-6, polish_passes 5, polish_retry 2, warm start, goals out of reach",
        "session": {"vehicle_steps": n_steps, "aborted": aborted, "wall_s_incl_plant": wall,
                    "vehicle_steps_per_s": n_steps / wall, "step_ms_p50": float(np.percentile(ms, 50)),
                    "step_ms_p99": float(np.percentile(ms, 99)), "step_ms_max": float(ms.max()), "step_ms_sum": float(ms.sum())},
        "track_batch": {"vehicle_steps": tb_steps, "aborted": int(res.aborted.sum()), "wall_s": tb_wall,
                        "vehicle_steps_per_s": tb_steps / tb_wall},
    }))


if __name__ == "__main__":
    main()
