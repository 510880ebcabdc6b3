"""One closed-loop step per call with the plant outside (TrajectoryTracker.start_batch / TrackingSession.step,
cudampc_track_step_batch): bit-identical to track_batch when the plant is f_discrete, the tracker rules of
control_stage.py:126-147 when it is not, and the ABI's argument checks."""
import ctypes as C

import numpy as np
import pytest

from conftest import load_golden

TIGHT = dict(eps_abs=1e-6, eps_rel=1e-6)


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


def drive(sess, T, plant):
    """T calls of sess.step with NumPy states; `plant(x, u0)` moves the vehicles that stepped.  Returns the arrays of a
    BatchTrackingResult (states / controls NaN and status / iters 0 where a vehicle did not step)."""
    B = sess.batch
    x = sess.states0.copy()
    out = dict(states=np.full((B, T, 4), np.nan), controls=np.full((B, T, 2), np.nan),
               step_status=np.zeros((B, T), np.int32), step_iters=np.zeros((B, T), np.int32))
    for t in range(T):
        r = sess.step(x)
        out["step_status"][:, t], out["step_iters"][:, t] = r.status, r.iters
        ok = np.isfinite(r.u0).all(axis=1)
        if ok.any():
            x[ok] = plant(x[ok], r.u0[ok])
            out["states"][ok, t], out["controls"][ok, t] = x[ok], r.u0[ok]
        if not sess.active.any():
            break
    return out, x


def flags_of(sess):
    return {k: getattr(sess, k).cpu().numpy() for k in ("goal_reached", "aborted", "relaxed", "active")}


def assert_same_as_track_batch(res, out, sess, T, goals):
    n = sess.n_steps.cpu().numpy()
    f = flags_of(sess)
    assert np.array_equal(n, res.n_steps)
    assert np.array_equal(f["aborted"], res.aborted) and np.array_equal(f["relaxed"], res.relaxed)
    # the session tests the goal at the start of the next step: a vehicle whose T-th state is at the goal is flagged there
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


@pytest.mark.gpu
@pytest.mark.parametrize("warm", [True, False])
def test_session_with_f_discrete_reproduces_track_batch_bit_for_bit(warm):
    from rrt_mpc_b200 import MPCConfig, SolverSettings, TrajectoryTracker
    d, path = scenario()
    T = 80
    tr = TrajectoryTracker(MPCConfig(sim_steps=T), None, settings=SolverSettings(polish_passes=3, polish_retry=2, **TIGHT))
    paths, starts, goals = perturbed()
    cases = [(paths, starts, goals), ([path], np.array([d["start"]]), np.array([d["goal"]]))]
    for ps, ss, gs in cases:
        res = tr.track_batch(ps, ss, gs, map_resolution=0.8, warm_start=warm)
        sess = tr.start_batch(ps, ss, gs, map_resolution=0.8, warm_start=warm)
        out, _ = drive(sess, T, sess.controller.f_discrete_batch)
        assert_same_as_track_batch(res, out, sess, T, gs)
        assert res.goal_reached.any()
        sess.close()


@pytest.mark.gpu
def test_relaxation_and_abort_match_track_batch():
    """The max_iter = 550 (retry at steps 0, 1, 4, 5, then the goal) and 300 (retry fails, abort at step 0) cases of
    test_gpu_rollout.test_relaxation_branch_is_entered_and_matches_the_oracle, and the abort without the retry."""
    from rrt_mpc_b200 import MPCConfig, SolverSettings, TrajectoryTracker
    d, path = scenario()
    T = 300
    for max_iter, relax in ((550, True), (300, True), (550, False)):
        tr = TrajectoryTracker(MPCConfig(), None, settings=SolverSettings(polish_passes=1, max_iter=max_iter, **TIGHT))
        starts, goals = np.array([d["start"]] * 2), np.array([d["goal"]] * 2)
        res = tr.track_batch([path, path], starts, goals, map_resolution=0.8, warm_start=False, relax_on_failure=relax)
        sess = tr.start_batch([path, path], starts, goals, map_resolution=0.8, warm_start=False, relax_on_failure=relax)
        out, _ = drive(sess, T, sess.controller.f_discrete_batch)
        assert_same_as_track_batch(res, out, sess, T, goals)
        if max_iter == 300 or not relax:
            assert res.aborted.all() and (res.n_steps == 0).all()
            assert (out["step_status"][:, 0] == -2).all() and np.isnan(out["controls"][:, 0]).all()
        else:
            assert res.relaxed.all() and res.goal_reached.all() and (res.n_steps == 63).all()
        sess.close()


def window(ref, path_idx, N):
    w = ref[path_idx:min(path_idx + N + 1, len(ref))]
    if len(w) < N + 1:
        w = np.vstack((w, np.repeat(w[-1:], N + 1 - len(w), axis=0)))
    return w


@pytest.mark.gpu
def test_external_plant_with_model_mismatch_follows_the_tracker_rules():
    """Plant: f_discrete with the wheelbase x 1.15 plus seeded noise on x, y and yaw.  Every step is replayed on the host with
    the rules of control_stage.py:126-147 written out here; u0 is checked against the CPU oracle on the same window, x0 and
    u_prev."""
    import dataclasses
    from oracle import c_oracle as CO, mpc_numpy as O
    from rrt_mpc_b200 import MPCConfig, SolverSettings, TrajectoryTracker, build_reference, f_discrete
    from rrt_mpc_b200.control_stage import initial_state
    B, T, N = 8, 80, 15
    paths, starts, goals = perturbed(B)
    refs = [build_reference(p, 15.0, N, 0.1) for p in paths]
    s0 = np.stack([initial_state(paths[b], starts[b]) for b in range(B)])
    tr = TrajectoryTracker(MPCConfig(sim_steps=T), None, settings=SolverSettings(polish_passes=3, polish_retry=2, **TIGHT))
    sess = tr.start_batch(None, None, goals, map_resolution=0.8, ref_globals=refs, states0=s0, warm_start=True)
    L = sess.controller.params.wheelbase_px * 1.15
    dt = sess.controller.params.dt
    rng = np.random.default_rng(11)
    op = O.Params(horizon=N)
    relaxed_op = dataclasses.replace(op, du_bounds=((op.du_bounds[0][0] - 5.0, op.du_bounds[0][1] + 5.0),
                                                    (op.du_bounds[1][0] - 0.05, op.du_bounds[1][1] + 0.05)))
    x = s0.copy()
    pidx, fl, nst, up = np.zeros(B, int), np.zeros(B, int), np.zeros(B, int), np.zeros((B, 2))
    hist = np.full((B, T, 4), np.nan)
    worst = 0.0
    for t in range(T):
        r = sess.step(x)
        for b in range(B):
            if fl[b] & 3:
                assert r.status[b] == 0 and np.isnan(r.u0[b]).all()
                continue
            if nst[b] > 0:
                if pidx[b] < len(refs[b]) - 2:
                    dx, dy = x[b, 0] - refs[b][pidx[b], 0], x[b, 1] - refs[b][pidx[b], 1]
                    if dx * dx + dy * dy > 25.0:
                        pidx[b] += 1
                if np.hypot(x[b, 0] - goals[b, 0], x[b, 1] - goals[b, 1]) < 8.0:
                    fl[b] |= 1
                    assert r.status[b] == 0 and np.isnan(r.u0[b]).all() and np.isnan(r.Xp[b]).all()
                    continue
            win = window(refs[b], pidx[b], N)
            ora = CO.solve_batch(op, x[b][None], win[None], up[b][None], polish_passes=3, **TIGHT)
            if ora["status"][0] not in (1, 2):
                fl[b] |= 4
                ora = CO.solve_batch(relaxed_op, x[b][None], (win * np.array([1, 1, 1, 0.6]))[None], up[b][None], polish_passes=3, **TIGHT)
            assert r.status[b] in (1, 2) and ora["status"][0] in (1, 2)
            worst = max(worst, float(np.abs(r.u0[b] - ora["u0"][0]).max()))
            up[b] = r.u0[b]
            nst[b] += 1
        assert np.array_equal(sess.path_idx.cpu().numpy(), pidx), t
        got = sess.flags.cpu().numpy()
        assert np.array_equal(got, fl), (t, got, fl)
        ok = np.isfinite(r.u0).all(axis=1)
        for b in np.flatnonzero(ok):
            x[b] = f_discrete(x[b], r.u0[b], dt, L) + rng.normal(size=4) * np.array([0.2, 0.2, 0.005, 0.0])
            hist[b, t] = x[b]
        if not ok.any() and not sess.active.any():
            break
    assert worst < 1e-5, worst
    assert np.array_equal(sess.n_steps.cpu().numpy(), nst) and np.allclose(sess.u_prev.cpu().numpy(), up, rtol=0, atol=0)
    # not vacuous: the plant is not the controller's model, and the rules were exercised
    res = tr.track_batch(None, None, goals, map_resolution=0.8, ref_globals=refs, states0=s0, warm_start=True)
    n = np.minimum(nst, res.n_steps)
    assert max(np.abs(hist[b, :n[b], :2] - res.states[b, :n[b], :2]).max() for b in range(B)) > 1.0
    assert (pidx > 0).any() and (fl & 1).any()
    sess.close()


@pytest.mark.gpu
def test_edge_cases_and_device_tensors():
    import torch
    from rrt_mpc_b200 import MPCConfig, SolverSettings, TrajectoryTracker
    d, path = scenario()
    tr = TrajectoryTracker(MPCConfig(), None, settings=SolverSettings(polish_passes=3, polish_retry=2, **TIGHT))
    # vehicle 0 starts inside its goal radius, 1 is an ordinary vehicle, 2 gets an empty reference (ref_len = 0)
    starts = np.array([d["start"]] * 3)
    goals = np.array([d["start"], d["goal"], d["goal"]])
    sess = tr.start_batch([path] * 3, starts, goals, map_resolution=0.8)
    sess._ref_len[2] = 0
    x = sess.states0.copy()
    r = sess.step(x)                                  # the first step takes no goal test (as K_rollout)
    assert list(r.status[:2]) == [1, 1] and r.status[2] == 0 and r.iters[2] == 0 and np.isnan(r.u0[2]).all()
    assert list(sess.n_steps.cpu().numpy()) == [1, 1, 0] and list(sess.flags.cpu().numpy()) == [0, 0, 2]
    x[:2] = sess.controller.f_discrete_batch(x[:2], r.u0[:2])
    r = sess.step(x)                                  # vehicle 0 is at its goal now; finished and active share the batch
    assert r.status[0] == 0 and np.isnan(r.u0[0]).all() and np.isnan(r.Xp[0]).all() and np.isnan(r.Up[0]).all()
    assert r.status[1] == 1 and np.isfinite(r.Xp[1]).all()
    assert list(sess.goal_reached.cpu().numpy()) == [True, False, False] and list(sess.active.cpu().numpy()) == [False, True, False]
    before = [t.clone() for t in (sess.path_idx, sess.u_prev, sess.n_steps, sess.flags)]
    x[1] = sess.controller.f_discrete_batch(x[1:2], r.u0[1:2])[0]
    # a CUDA tensor: one launch, CUDA tensors back
    xd = torch.as_tensor(x).cuda()
    n0 = sess.launch_count()
    rd = sess.step(xd)
    assert sess.launch_count() == n0 + 1
    assert all(t.is_cuda for t in (rd.u0, rd.Xp, rd.Up, rd.status, rd.iters))
    torch.cuda.synchronize()
    for i in (0, 2):                                  # stopped vehicles: status 0, NaN, tracker state unchanged
        assert int(rd.status[i]) == 0 and int(rd.iters[i]) == 0 and torch.isnan(rd.u0[i]).all()
        for a, b_ in zip(before, (sess.path_idx, sess.u_prev, sess.n_steps, sess.flags)):
            assert torch.equal(a[i], b_[i])
    assert int(rd.status[1]) == 1 and int(sess.n_steps[1]) == 3
    with pytest.raises(ValueError):
        sess.step(xd.float())
    with pytest.raises(ValueError):
        sess.step(xd.cpu())
    with pytest.raises(ValueError):
        sess.step(xd[:2])
    # the ABI's checks with a real handle
    h = sess._h
    lib = h.lib
    ptr = lambda t: C.c_void_p(t.data_ptr())
    st = [ptr(sess._ref), ptr(sess._ref_len)]
    tail = [ptr(sess.path_idx), ptr(sess.u_prev), ptr(sess.n_steps), ptr(sess.flags), ptr(rd.u0), None, None, ptr(rd.status), ptr(rd.iters), None]
    assert lib.cudampc_track_step_batch(h.ptr, 4, *st, sess._stride, ptr(sess._goals), ptr(xd), None, None, *tail) == -1
    assert b"batch out of range" in lib.cudampc_last_error(h.ptr)
    assert lib.cudampc_track_step_batch(h.ptr, 3, *st, 0, ptr(sess._goals), ptr(xd), None, None, *tail) == -1
    assert lib.cudampc_track_step_batch(h.ptr, 3, *st, sess._stride, None, ptr(xd), None, None, *tail) == -1
    assert b"NULL pointer" in lib.cudampc_last_error(h.ptr)
    sess.close()


def test_abi_rejects_a_null_handle_without_touching_the_device():
    from rrt_mpc_b200 import _lib
    lib = _lib.load()
    assert lib.cudampc_track_step_batch(None, 1, *([None] * 2), 1, *([None] * 4), *([None] * 10)) == -1


def test_step_rejects_bad_states_before_any_launch():
    import torch
    from rrt_mpc_b200 import TrackingSession
    sess = object.__new__(TrackingSession)              # no device: the checks come before anything touches one
    sess.batch, sess.horizon, sess.device = 4, 15, torch.device("cuda", 0)
    for bad in (np.zeros((3, 4)), np.zeros((4, 4), np.float32), np.zeros(16), torch.zeros((4, 4), dtype=torch.float64),
                [[0.0] * 4] * 4):
        with pytest.raises(ValueError):
            sess.step(bad)
