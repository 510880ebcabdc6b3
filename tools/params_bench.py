"""Per-problem parameters against the shared-parameter kernels, in one process on one GPU.  Prints one JSON line.
(a) bench.py's headline batch (65,536 x horizon 50, seed 3, steering-rate +-0.02, SolverSettings.early_certified()): the
    shared-parameter solve against cudampc_solve_batch_params with every record equal to the handle's, alternated, 3 rounds each;
(b) a sweep of the same problems under 8 du_bounds / weight settings: one per-problem launch of 8 x B problems against 8
    set_params launches of B problems;
(c) bench.py's config-4 shape (8,192 vehicles x 500 steps, horizon 15): track_batch with and without all-equal vehicle_params.
Device times are CUDA events around each launch, inputs and records already on the device.
usage: python tools/params_bench.py [--batch B] [--vehicles V] [--steps T]"""
import argparse
import ctypes as C
import dataclasses
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


def sweep_sets(base):
    """8 settings: du_bounds of the steering rate and acceleration, and the weights of position / inputs."""
    out = []
    for k in range(8):
        dd = (0.01, 0.02, 0.04, 0.08)[k % 4]
        w = 1.0 if k < 4 else 2.0
        out.append(dataclasses.replace(base, du_bounds=((-12.0 / w, 12.0 / w), (-dd, dd)), q=np.asarray(base.q) * np.array([w, w, 1, 1]),
                                       r=np.asarray(base.r) * w))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--vehicles", type=int, default=8192)
    ap.add_argument("--steps", type=int, default=500)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("params_bench needs a CUDA device")
    from rrt_mpc_b200 import MPCConfig, MPCController, SolverSettings, TrajectoryTracker, params_array
    from rrt_mpc_b200.mpc_controller import params_to_c
    from rrt_mpc_b200.synthetic import make_batch
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)
    N, B = 50, args.batch
    base = dataclasses.replace(MPCConfig(horizon=N).to_parameters(0.8), du_bounds=((-12.0, 12.0), (-0.02, 0.02)))
    st = SolverSettings.early_certified()
    x0, ref, up = make_batch(B, N, 3)
    d_x0, d_ref, d_up = (torch.as_tensor(a).to(dev) for a in (x0, ref, up))
    rows_eq = torch.from_numpy(params_array([base] * B).view(np.uint8).reshape(B, -1)).to(dev)
    out = {"gpu": torch.cuda.get_device_name(dev), "power_limit": gpu_power_limit()}

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record(stream)
        r = fn()
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / 1e3, r

    # (a) shared vs per-problem, all records equal
    ctl = MPCController(base, st, max_batch=8 * B)
    shared = lambda: ctl.solve_batch(d_x0, d_ref, u_prev=d_up)
    perprob = lambda: ctl.solve_batch(d_x0, d_ref, u_prev=d_up, params=rows_eq)
    for _ in range(2):
        shared(); perprob()
    ta, tp = [], []
    for _ in range(3):
        t, rs = timed(shared); ta.append(t)
        t, rp = timed(perprob); tp.append(t)
    same = all(torch.equal(getattr(rs, k), getattr(rp, k)) for k in ("u0", "Xp", "Up", "status", "iters", "info"))
    out["a_bench_batch"] = {"workload": f"{B} problems, horizon {N}, seed 3, steering-rate +-0.02, early_certified",
                            "shared_s": ta, "per_problem_s": tp, "shared_solves_per_s": B / min(ta), "per_problem_solves_per_s": B / min(tp),
                            "per_problem_over_shared_best": min(tp) / min(ta), "outputs_bit_identical": bool(same)}

    # (b) sweep of 8 settings: one launch of 8B problems vs 8 launches after set_params
    sets = sweep_sets(base)
    rows_sw = torch.from_numpy(params_array([p for p in sets for _ in range(B)]).view(np.uint8).reshape(8 * B, -1)).to(dev)
    s_x0, s_ref, s_up = (t.repeat((8,) + (1,) * (t.dim() - 1)) for t in (d_x0, d_ref, d_up))
    h = ctl._handle(8 * B)
    cpar = [params_to_c(p) for p in sets]

    def eight():
        res = []
        for p in cpar:
            assert h.lib.cudampc_set_params(h.ptr, C.byref(p)) == 0
            res.append(ctl.solve_batch(d_x0, d_ref, u_prev=d_up))
        assert h.lib.cudampc_set_params(h.ptr, C.byref(params_to_c(base))) == 0
        return res
    one = lambda: ctl.solve_batch(s_x0, s_ref, u_prev=s_up, params=rows_sw)
    eight(); one()
    te, to = [], []
    for _ in range(3):
        t, re_ = timed(eight); te.append(t)
        t, ro = timed(one); to.append(t)
    same_b = all(torch.equal(torch.cat([getattr(r, k) for r in re_]), getattr(ro, k)) for k in ("u0", "status", "iters"))
    out["b_sweep"] = {"workload": f"8 settings (du_bounds, weights) x {B} problems", "eight_set_params_launches_s": te,
                      "one_per_problem_launch_s": to, "one_over_eight_best": min(to) / min(te), "outputs_bit_identical": bool(same_b),
                      "iters_mean_per_setting": [float(r.iters.double().mean()) for r in re_]}
    del s_x0, s_ref, s_up, rows_sw, ctl
    torch.cuda.empty_cache()

    # (c) config-4 shape with and without all-equal vehicle_params
    V, T = args.vehicles, args.steps
    d = np.load(os.path.join(ROOT, "tests", "golden", "default_scenario.npz"))
    path = np.array(d["path"])
    rng = np.random.default_rng(4)
    noise = rng.normal(size=(V,) + path.shape) * 0.15
    noise[:, 0] = 0.0
    paths = [path + noise[b] for b in range(V)]
    starts = path[0] + rng.normal(size=(V, 2)) * 0.5
    goals = np.full((V, 2), 1e9)
    tr = TrajectoryTracker(MPCConfig(sim_steps=T), None,
                           settings=SolverSettings(eps_abs=1e-6, eps_rel=1e-6, polish_passes=5, polish_retry=2, early_polish=False))
    vp = torch.from_numpy(params_array([MPCConfig().to_parameters(0.8)] * V).view(np.uint8).reshape(V, -1)).to(dev)
    kw = dict(map_resolution=0.8, warm_start=True)
    tr.track_batch(paths[:512], starts[:512], goals[:512], sim_steps=50, **kw)
    tr.track_batch(paths[:512], starts[:512], goals[:512], sim_steps=50, vehicle_params=vp[:512], **kw)
    tc = {"shared_s": [], "per_vehicle_s": []}
    res = {}
    for _ in range(2):
        for name, extra in (("shared_s", {}), ("per_vehicle_s", {"vehicle_params": vp})):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            res[name] = tr.track_batch(paths, starts, goals, **kw, **extra)
            tc[name].append(time.perf_counter() - t0)
    a, b = res["shared_s"], res["per_vehicle_s"]
    same_c = all(np.array_equal(getattr(a, k), getattr(b, k), equal_nan=True) for k in ("states", "controls", "n_steps", "step_iters"))
    out["c_config4"] = {"workload": f"{V} vehicles x {T} steps, horizon 15, eps 1e-6, polish_passes 5, polish_retry 2, warm start",
                        **tc, "vehicle_steps": int(a.n_steps.sum()), "outputs_bit_identical": bool(same_c),
                        "per_vehicle_over_shared_best": min(tc["per_vehicle_s"]) / min(tc["shared_s"])}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
