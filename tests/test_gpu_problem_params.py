"""GPU (B200): per-problem parameters (cudampc_solve_batch_params, cudampc_rollout_batch_params,
cudampc_track_step_batch_params): every problem / vehicle against the reference answers and the certificate of its own
parameter set, the same arithmetic as the shared-parameter kernels, invalid records, and the closed loop."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

from conftest import load_golden, product_params

pytestmark = pytest.mark.gpu
TIGHT = dict(eps_abs=1e-6, eps_rel=1e-6)
INVALID = -100
# the kernel variants a handle selects: horizon 15 (short form), 50 (register form), 100 (two warps), 50 general / pair
VARIANTS = [(15, None), (50, None), (100, None), (50, "general"), (50, "pair")]


def settings(**kw):
    from rrt_mpc_b200 import SolverSettings
    return SolverSettings(**{**dict(polish_passes=5, polish_retry=4, **TIGHT), **kw})


def problems(N, B, seed):
    """Random tracking problems as in test_gpu_parity.test_horizon_edge_cases."""
    rng = np.random.default_rng(seed)
    ref = np.zeros((B, N + 1, 4))
    for b in range(B):
        yaw = 0.4 * (b % 8) + np.cumsum(rng.normal(size=N + 1) * 0.05)
        ref[b, :, 2] = yaw; ref[b, :, 3] = 12.0 + rng.normal(size=N + 1)
        ref[b, :, 0] = 80 + np.cumsum(1.5 * np.cos(yaw)); ref[b, :, 1] = 60 + np.cumsum(1.5 * np.sin(yaw))
    x0 = ref[:, 0] + rng.normal(size=(B, 4)) * [0.5, 0.5, 0.05, 1.0]
    up = rng.uniform(-1, 1, size=(B, 2)) * [3.0, 0.1]
    return x0, ref, up


def param_sets(N):
    """Six parameter sets that differ in wheelbase, weights (one non-diagonal), bounds and slack weights."""
    base = product_params(N)
    m = np.array([[2.0, 0.3, 0.0, 0.1], [0.3, 3.0, 0.2, 0.0], [0.0, 0.2, 0.5, 0.05], [0.1, 0.0, 0.05, 0.2]])
    return [
        base,
        dataclasses.replace(base, wheelbase_px=2.5),
        dataclasses.replace(base, q=m, r=np.array([[0.05, 0.01], [0.01, 0.3]]), q_terminal=2.0 * m),
        dataclasses.replace(base, u_bounds=((-20.0, 20.0), (-0.4, 0.4)), v_bounds=(2.0, 14.0)),
        dataclasses.replace(base, du_bounds=((-4.0, 4.0), (-0.04, 0.05)), wheelbase_px=4.5),
        dataclasses.replace(base, slack_velocity=50.0, slack_input=20.0, slack_rate=10.0, r=np.diag([0.1, 1.0])),
    ]


def to_oracle(p):
    from oracle import mpc_numpy as O
    return O.Params(**{f.name: getattr(p, f.name) for f in dataclasses.fields(O.Params)})


def same(a, b, what, keys=("status", "iters", "u0", "Xp", "Up", "pri_res", "dua_res", "info")):
    for k in keys:
        assert np.array_equal(getattr(a, k), getattr(b, k), equal_nan=True), (what, k)


def set_form(monkeypatch, form):
    if form is None:
        monkeypatch.delenv("CUDAMPC_FORM", raising=False)
    else:
        monkeypatch.setenv("CUDAMPC_FORM", form)


def test_interleaved_reference_answers():
    """n20 of optima.npz (product_params(20)) and nd20 of ref_qp.npz (non-diagonal weights) interleaved in one call."""
    from rrt_mpc_b200 import MPCController
    g, r = load_golden("optima.npz"), load_golden("ref_qp.npz")
    pa = product_params(20)
    pb = dataclasses.replace(pa, q=r["nd20_q"], r=r["nd20_r"], q_terminal=r["nd20_qn"])
    na, nb = len(g["n20_x0"]), len(r["nd20_x0"])
    order = np.argsort(np.r_[np.arange(na) * 2.0, np.arange(nb) * 2.0 + 1.0], kind="stable")      # a b a b ... a a
    cat = lambda k: np.concatenate([g["n20_" + k], r["nd20_" + k]])[order]
    ps = [(pa if i < na else pb) for i in order]
    ctl = MPCController(pa, settings(), max_batch=na + nb)
    launches = ctl.launch_count()
    res = ctl.solve_batch(cat("x0"), cat("ref"), u_prev=cat("up"), params=ps)
    assert ctl.launch_count() == launches + 1
    assert (res.status == 1).all()
    assert np.abs(res.u0 - cat("u0")).max() < 1e-8
    assert np.abs(res.Xp - cat("X")).max() < 1e-6 and np.abs(res.Up - cat("U")).max() < 1e-6


@pytest.mark.parametrize("N,form", VARIANTS)
def test_every_variant_against_the_certificate(N, form, monkeypatch):
    from oracle import mpc_numpy as O
    from rrt_mpc_b200 import MPCController
    set_form(monkeypatch, form)
    B = 24
    x0, ref, up = problems(N, B, seed=N)
    sets = param_sets(N)
    pick = np.random.default_rng(7).integers(0, len(sets), size=B)
    ctl = MPCController(sets[0], settings(), max_batch=B)
    res = ctl.solve_batch(x0, ref, u_prev=up, params=[sets[k] for k in pick])
    assert (res.status == 1).all()
    bar = 1e-6 if N > 64 else 1e-8
    for b in range(B):
        u0, X, U, _ = O.solve_kkt_newton(x0[b], ref[b], up[b], to_oracle(sets[pick[b]]))
        assert np.abs(res.u0[b] - u0).max() < bar, (b, pick[b])
        assert np.abs(res.Xp[b] - X).max() < 1e-6, (b, pick[b])


@pytest.mark.parametrize("N,form", VARIANTS)
def test_same_arithmetic_as_the_shared_parameter_kernels(N, form, monkeypatch):
    """All rows equal to the handle's parameters: bit-identical to the call without params, under early polish, literal OSQP,
    warm start and stateless settings.  A mixed batch: bit-identical to each group solved on a handle of its own."""
    import torch
    from rrt_mpc_b200 import MPCController, params_array
    set_form(monkeypatch, form)
    B = 24
    x0, ref, up = problems(N, B, seed=100 + N)
    base = product_params(N)
    ctl = MPCController(base, settings(), max_batch=B)
    rows = torch.from_numpy(params_array([base] * B).view(np.uint8).reshape(B, -1)).cuda()
    for st in (settings(early_polish=True, check_termination=50), settings(polish_passes=1, polish_retry=0),
               settings(keep_iterate=False, early_polish=True)):
        same(ctl.solve_batch(x0, ref, u_prev=up, settings=st), ctl.solve_batch(x0, ref, u_prev=up, settings=st, params=rows), st)
    warm = settings(warm_start=True)
    ctl.solve_batch(x0, ref, u_prev=up)
    a = ctl.solve_batch(x0 + 0.01, ref, u_prev=up, settings=warm)
    ctl.solve_batch(x0, ref, u_prev=up, params=rows)
    b = ctl.solve_batch(x0 + 0.01, ref, u_prev=up, settings=warm, params=rows)
    same(a, b, "warm start")
    assert a.iters.sum() > 0
    # mixed batch against one handle per parameter set
    sets = param_sets(N)[:3]
    pick = np.arange(B) % 3
    mixed = ctl.solve_batch(x0, ref, u_prev=up, params=[sets[k] for k in pick])
    for k, p in enumerate(sets):
        own = MPCController(p, settings(), max_batch=B).solve_batch(x0[pick == k], ref[pick == k], u_prev=up[pick == k])
        for key in ("status", "iters", "u0", "Xp", "Up", "pri_res", "dua_res", "info"):
            assert np.array_equal(getattr(mixed, key)[pick == k], getattr(own, key)), (k, key)


@pytest.mark.parametrize("N,form", VARIANTS)
def test_invalid_rows_fail_alone(N, form, monkeypatch):
    import torch
    from rrt_mpc_b200 import MPCController, params_array
    set_form(monkeypatch, form)
    B = 16
    x0, ref, up = problems(N, B, seed=200 + N)
    base = product_params(N)
    arr = params_array([base] * B)
    bad = {1: ("q", np.diag([1.0, 1.0, -0.5, 0.1]).reshape(16)), 4: ("slack_input", 0.0), 6: ("dt", np.nan),
           9: ("dt", base.dt * 1.5), 11: ("horizon", N + 1), 13: ("wheelbase_px", 0.0)}
    for i, (k, v) in bad.items():
        arr[k][i] = v
    rows = torch.from_numpy(arr.view(np.uint8).reshape(B, -1)).cuda()
    ok = np.array([i not in bad for i in range(B)])
    ctl = MPCController(base, settings(), max_batch=B)
    ctl.solve_batch(x0, ref, u_prev=up)                                       # every slot holds its problem's iterate
    res = ctl.solve_batch(x0 + 0.02, ref, u_prev=up, params=rows)
    assert (res.status[~ok] == INVALID).all() and (res.iters[~ok] == 0).all()
    for k in ("u0", "Xp", "Up", "pri_res", "dua_res"):
        assert np.isnan(getattr(res, k)[~ok]).all(), k
    alone = MPCController(base, settings(), max_batch=B).solve_batch(x0[ok] + 0.02, ref[ok], u_prev=up[ok], params=[base] * int(ok.sum()))
    for k in ("status", "iters", "u0", "Xp", "Up", "pri_res", "dua_res", "info"):
        assert np.array_equal(getattr(res, k)[ok], getattr(alone, k)), k
    # the invalid rows left their warm-start slots alone: a warm start there finds the iterate of the first call
    warm = settings(warm_start=True)
    hot = ctl.solve_batch(x0 + 0.01, ref, u_prev=up, settings=warm)
    ref_ctl = MPCController(base, settings(), max_batch=B)
    ref_ctl.solve_batch(x0, ref, u_prev=up)
    want = ref_ctl.solve_batch(x0 + 0.01, ref, u_prev=up, settings=warm)
    for k in ("status", "iters", "u0", "Xp", "Up"):
        assert np.array_equal(getattr(hot, k)[~ok], getattr(want, k)[~ok]), k


# ------------------------------------------------------------------------------------------------
# closed loop
# ------------------------------------------------------------------------------------------------
def scenario():
    d = load_golden("default_scenario.npz")
    return d, [tuple(p) for p in d["path"]]


def perturbed(B=48):
    """The vehicles of test_gpu_rollout.test_many_perturbed_vehicles."""
    d, path = scenario()
    rng = np.random.default_rng(4)
    paths, starts = [], []
    for b in range(B):
        pts = np.array(path) + rng.normal(size=(len(path), 2)) * 0.15
        pts[0] = path[0]
        paths.append([tuple(p) for p in pts]); starts.append(pts[0] + rng.normal(size=2) * 0.5)
    return paths, np.array(starts), np.tile(d["goal"], (B, 1))


def fleet(B):
    """Three wheelbases x two du_bounds x two weight sets, assigned in turn."""
    from rrt_mpc_b200 import MPCConfig
    base = MPCConfig().to_parameters(0.8)
    out = []
    for b in range(B):
        L = (3.0, base.wheelbase_px, 4.5)[b % 3]
        du = base.du_bounds if (b // 3) % 2 == 0 else ((-8.0, 8.0), (-0.08, 0.08))
        w = {} if (b // 6) % 2 == 0 else dict(q=np.diag([8.0, 8.0, 1.0, 0.1]), r=np.diag([0.06, 0.5]))
        out.append(dataclasses.replace(base, wheelbase_px=L, du_bounds=du, **w))
    return out


def tracker(T, **kw):
    from rrt_mpc_b200 import MPCConfig, SolverSettings, TrajectoryTracker
    return TrajectoryTracker(MPCConfig(sim_steps=T), None, settings=SolverSettings(**{**dict(polish_passes=3, polish_retry=2, **TIGHT), **kw}))


def same_rollout(a, b, idx=slice(None)):
    for k in ("states", "controls", "n_steps", "goal_reached", "aborted", "relaxed", "step_status", "step_iters"):
        assert np.array_equal(getattr(a, k)[idx], getattr(b, k)[idx], equal_nan=True), k


def test_track_batch_all_equal_vehicle_params_is_the_shared_roll_out():
    from rrt_mpc_b200 import MPCConfig
    T = 80
    tr = tracker(T)
    paths, starts, goals = perturbed()
    vp = [MPCConfig().to_parameters(0.8)] * len(paths)
    for warm in (True, False):
        a = tr.track_batch(paths, starts, goals, map_resolution=0.8, warm_start=warm)
        b = tr.track_batch(paths, starts, goals, map_resolution=0.8, warm_start=warm, vehicle_params=vp)
        same_rollout(a, b)
        assert not b.invalid_params.any() and a.goal_reached.any()


def test_heterogeneous_fleet_matches_the_oracle_per_vehicle():
    from oracle import c_oracle as CO
    from rrt_mpc_b200.control_stage import initial_state
    from rrt_mpc_b200.ref_builder import build_reference
    T = 80
    tr = tracker(T)
    paths, starts, goals = perturbed()
    vp = fleet(len(paths))
    res = tr.track_batch(paths, starts, goals, map_resolution=0.8, warm_start=True, vehicle_params=vp)
    assert (res.n_steps > 0).all() and not res.invalid_params.any()
    for b in range(len(paths)):
        rg = build_reference(paths[b], 15.0, 15, 0.1)
        ora = CO.track(vp[b], rg, initial_state(paths[b], starts[b]), goals[b], T, polish_passes=3, **TIGHT)
        n = int(res.n_steps[b])
        assert n == ora["n_steps"], b
        assert np.abs(res.states[b, :n, :2] - ora["states"][:n, :2]).max() < 1e-3, b


def test_relaxation_retries_each_vehicle_with_its_own_bounds():
    """max_iter = 550 (test_gpu_rollout's relaxation case): every vehicle retries with its own widened du_bounds."""
    from oracle import c_oracle as CO
    from rrt_mpc_b200 import MPCConfig
    from rrt_mpc_b200.control_stage import initial_state
    d, path = scenario()
    base = MPCConfig().to_parameters(0.8)
    vp = [base, dataclasses.replace(base, du_bounds=((-10.0, 10.0), (-0.12, 0.12))), dataclasses.replace(base, wheelbase_px=4.0)]
    tr = tracker(300, polish_passes=1, polish_retry=0, max_iter=550)
    res = tr.track_batch([path] * 3, [d["start"]] * 3, [d["goal"]] * 3, map_resolution=0.8, warm_start=False, vehicle_params=vp)
    s0 = initial_state(path, d["start"])
    assert res.relaxed[0]
    for b, p in enumerate(vp):
        ora = CO.track(p, d["ref_global"], s0, d["goal"], 300, polish_passes=1, scaling=0, z0_projected=1, max_iter=550, **TIGHT)
        n = int(res.n_steps[b])
        assert n == ora["n_steps"], b
        assert bool(res.relaxed[b]) == bool(ora["flags"] & 4) and bool(res.aborted[b]) == bool(ora["flags"] & 2), b
        assert np.array_equal(res.step_status[b, :n], ora["step_status"][:n]), b
        if n:
            assert np.abs(res.states[b, :n] - ora["states"][:n]).max() < 1e-7, b


def test_invalid_vehicle_is_flagged_and_its_neighbours_run():
    from rrt_mpc_b200 import params_array
    T = 40
    tr = tracker(T)
    paths, starts, goals = perturbed(8)
    vp = params_array(fleet(8))
    good = tr.track_batch(paths, starts, goals, map_resolution=0.8, vehicle_params=vp)
    vp["wheelbase_px"][3] = 0.0
    vp["r"][5] = [-1.0, 0.0, 0.0, 1.0]
    res = tr.track_batch(paths, starts, goals, map_resolution=0.8, vehicle_params=vp)
    bad = np.isin(np.arange(8), [3, 5])
    assert np.array_equal(res.invalid_params, bad) and res.aborted[bad].all()
    assert (res.n_steps[bad] == 0).all() and np.isnan(res.states[bad]).all() and (res.step_status[bad] == 0).all()
    same_rollout(good, res, ~bad)
    assert not good.invalid_params.any() and good.n_steps[~bad].min() > 0


def test_session_with_per_vehicle_params_reproduces_track_batch():
    """start_batch(vehicle_params=...) with f_discrete at each vehicle's own (dt, wheelbase) as the plant: bit-identical to
    track_batch(vehicle_params=...), one launch per step.  Vehicle 2's record is invalid."""
    from rrt_mpc_b200 import params_array
    T = 80
    tr = tracker(T)
    paths, starts, goals = perturbed()
    vp = params_array(fleet(len(paths)))
    vp["slack_rate"][2] = 0.0
    for warm in (True, False):
        res = tr.track_batch(paths, starts, goals, map_resolution=0.8, warm_start=warm, vehicle_params=vp)
        sess = tr.start_batch(paths, starts, goals, map_resolution=0.8, warm_start=warm, vehicle_params=vp)
        dtL = np.stack([vp["dt"], vp["wheelbase_px"]], axis=1)
        out = drive(sess, T, lambda x, u, ok: sess.controller.f_discrete_batch(x, u, dt_L=dtL[ok]))
        assert_same_as_track_batch(res, out, sess, T, goals)
        assert np.array_equal(sess.invalid_params.cpu().numpy(), res.invalid_params) and res.invalid_params[2]
        sess.close()


def drive(sess, T, plant):
    """As test_gpu_track_step.drive; the plant also gets the mask of the vehicles that stepped, and every step must be exactly
    one launch (the plant's f_discrete launches on the same handle are outside the count)."""
    B = sess.batch
    x = sess.states0.copy()
    out = dict(states=np.full((B, T, 4), np.nan), controls=np.full((B, T, 2), np.nan),
               step_status=np.zeros((B, T), np.int32), step_iters=np.zeros((B, T), np.int32))
    for t in range(T):
        before = sess.launch_count()
        r = sess.step(x)
        assert sess.launch_count() == before + 1
        out["step_status"][:, t], out["step_iters"][:, t] = r.status, r.iters
        ok = np.isfinite(r.u0).all(axis=1)
        if ok.any():
            x[ok] = plant(x[ok], r.u0[ok], ok)
            out["states"][ok, t], out["controls"][ok, t] = x[ok], r.u0[ok]
        if not sess.active.any():
            break
    return out


def assert_same_as_track_batch(res, out, sess, T, goals):
    """test_gpu_track_step.assert_same_as_track_batch"""
    n = sess.n_steps.cpu().numpy()
    f = {k: getattr(sess, k).cpu().numpy() for k in ("goal_reached", "aborted", "relaxed", "active")}
    assert np.array_equal(n, res.n_steps)
    assert np.array_equal(f["aborted"], res.aborted) and np.array_equal(f["relaxed"], res.relaxed)
    last = n == T
    assert np.array_equal(f["goal_reached"][~last], res.goal_reached[~last])
    assert not f["goal_reached"][last].any()
    for b in np.flatnonzero(last):
        g = np.hypot(*(res.states[b, T - 1, :2] - goals[b])) < 8.0
        assert bool(res.goal_reached[b]) == g
    for k in ("states", "controls"):
        assert np.array_equal(out[k], getattr(res, k), equal_nan=True), k
    for k in ("step_status", "step_iters"):
        assert np.array_equal(out[k], getattr(res, k)), k


def test_solve_batch_params_is_one_launch_and_checks_its_arguments():
    import torch
    from rrt_mpc_b200 import MPCController, _lib, params_array
    N, B = 20, 8
    x0, ref, up = problems(N, B, seed=5)
    base = product_params(N)
    ctl = MPCController(base, settings(), max_batch=B)
    rows = torch.from_numpy(params_array([base] * B).view(np.uint8).reshape(B, -1)).cuda()
    t = lambda a: torch.as_tensor(a).cuda()
    for params in (rows, [base] * B, params_array([base] * B)):
        before = ctl.launch_count()
        r = ctl.solve_batch(t(x0), t(ref), u_prev=t(up), params=params)
        torch.cuda.synchronize()
        assert ctl.launch_count() == before + 1 and (r.status.cpu().numpy() == 1).all()
    with pytest.raises(ValueError):
        ctl.solve_batch(t(x0), t(ref), u_prev=t(up), params=rows[:4])
    lib, h = _lib.load(), ctl._handle(B)
    s = settings().to_c()
    out = [torch.empty(n, dtype=dt, device="cuda") for n, dt in ((2 * B, torch.float64), (4 * (N + 1) * B, torch.float64),
                                                                (2 * N * B, torch.float64), (B, torch.int32), (B, torch.int32))]
    p = lambda x: C.c_void_p(x.data_ptr())
    rc = lib.cudampc_solve_batch_params(h.ptr, B, p(t(x0)), p(t(ref)), None, C.byref(s), None, *map(p, out), None, None, None, None)
    assert rc == -1 and b"NULL" in lib.cudampc_last_error(h.ptr)
