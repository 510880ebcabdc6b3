"""GPU (B200): every horizon the library accepts (1..256) through every kernel a horizon dispatches to: the batched solve
against the exact optimum of every problem (tests/certificate.py) and the host emulation of the same source, every override
of the dispatch against the default kernel, the order of a batch and the parameter path (shared / per problem) bit for bit;
the closed loop against the CPU oracle and its one-step twin; K_ref against build_reference.

The horizon picks the kernel of the batched solve, how many problems share an SM (P) and how lanes map onto stages
(cudampc_create): a lane per stage for N <= 31, the two-warp register form for 32..63, one warp in parity form for 64..95,
two warps beyond; CUDAMPC_FORM / CUDAMPC_WPP override the choice.  The closed loop (K_rollout, K_step) runs the short form for N <= 31 and the general form beyond unless
the pair form is forced.  Every problem set mixes make_batch problems at two steering-rate limits with the saturated
problems of test_emulation_horizons."""
import functools
import os
from types import SimpleNamespace as NS

import numpy as np
import pytest

from conftest import load_golden, product_params
from test_emulation_horizons import DUS, SOLVE, by_horizon, certify, horizon_problems, limits_active
from test_gpu_problem_params import param_sets
from test_gpu_track_step import assert_same_as_track_batch, drive, perturbed

pytestmark = pytest.mark.gpu
TIGHT = dict(eps_abs=1e-6, eps_rel=1e-6)
MAX_HORIZON = 256
# every horizon up to 150, every other one beyond (the dispatch does not change from 146 on), and the largest
HORIZONS = list(range(1, 151)) + list(range(151, MAX_HORIZON, 2)) + [MAX_HORIZON]
BOUNDARIES = [1, 31, 32, 63, 64, 70, 71, 95, 96, 145, 146, MAX_HORIZON]
KEYS = ("status", "iters", "u0", "Xp", "Up", "pri_res", "dua_res", "info")

# Against the certificate, by range of horizons, at most 10x the worst error measured on a B200 (1000 W) over the default
# kernel.  A solve that ends polished sits on the KKT point of its active set: POLISHED bars.  A rare problem (at most one
# of a batch of 299..2371, at 14 of the 256 horizons) ends on the eps = 1e-6 ADMM test with every polish rejected; the host
# emulation of the same source ends the same problems the same way (same iteration count, no accepted polish): ADMM bars,
# and a bound on how many.
POLISHED_U0 = {31: 1e-7, 63: 1e-7, 95: 1e-7, 145: 1e-7, MAX_HORIZON: 5e-8}      # measured 2.2e-8, 1.8e-8, 1.6e-8, 1.7e-8, 7.8e-9
POLISHED_X = {31: 1e-7, 63: 2e-7, 95: 1e-7, 145: 5e-7, MAX_HORIZON: 5e-5}       # measured 1.7e-8, 2.5e-8, 1.5e-8, 7.1e-8, 7.5e-6
ADMM_U0, ADMM_X = 3e-6, 2e-4                                                      # measured 4.0e-7, 3.7e-5
MAX_UNPOLISHED = 2                                                                # measured 1
# the six parameter sets of test_gpu_problem_params in one batch (narrower limits, other weights), every problem
MIXED_U0 = {31: 1e-6, 63: 1e-6, 95: 5e-6, 145: 5e-6, MAX_HORIZON: 1e-5}          # measured 2.1e-7, 1.4e-7, 6.3e-7, 7.7e-7, 1.8e-6
MIXED_X = {31: 2e-6, 63: 5e-6, 95: 5e-5, 145: 1e-4, MAX_HORIZON: 1e-4}           # measured 3.6e-7, 7.4e-7, 6.6e-6, 1.7e-5, 1.4e-5
MEASURED = {}           # worst error per (what, range of horizons) of this session: the numbers behind the bars


def within(err, table, N, what):
    key = (what, min(k for k in table if N <= k))
    MEASURED[key] = max(MEASURED.get(key, 0.0), float(err))
    assert err < by_horizon(table, N), (what, N, err)


def check_certificate(N, opt, r, what):
    """u0 and X of every problem against the exact optimum: polished solves at the POLISHED bars, the few others at the
    ADMM bars."""
    pol = r.info[:, 2] > 0
    assert (~pol).sum() <= MAX_UNPOLISHED, (what, N, np.flatnonzero(~pol))
    eu = np.abs(r.u0 - opt["U"][:, :, 0]).max(axis=1)
    ex = np.abs(r.Xp - opt["X"]).max(axis=(1, 2))
    if pol.any():
        within(eu[pol].max(), POLISHED_U0, N, what + " u0")
        within(ex[pol].max(), POLISHED_X, N, what + " X")
    if (~pol).any():
        within(eu[~pol].max(), {MAX_HORIZON: ADMM_U0}, N, what + " u0 unpolished")
        within(ex[~pol].max(), {MAX_HORIZON: ADMM_X}, N, what + " X unpolished")


def same_solves(a, b, what):
    """test_gpu_parity._same_solves for batches of hundreds to thousands of problems: the same status everywhere, the same
    iteration count for 90 % of the problems, and the same result to round-off wherever both ended polished (the KKT point of
    the same active set).  Where one of them did not, the certificate checks each on its own."""
    assert np.array_equal(a.status, b.status), what
    assert (a.iters == b.iters).mean() >= 0.9, (what, (a.iters == b.iters).mean())
    both = (a.info[:, 2] > 0) & (b.info[:, 2] > 0)
    assert np.abs(a.u0 - b.u0)[both].max(initial=0.0) < 1e-8, what
    assert np.abs(a.Xp - b.Xp)[both].max(initial=0.0) < 1e-7 and np.abs(a.Up - b.Up)[both].max(initial=0.0) < 1e-7, what


def settings(**kw):
    from rrt_mpc_b200 import SolverSettings
    return SolverSettings(**{**dict(polish_passes=5, polish_retry=2, early_polish=True, **TIGHT), **kw})


def set_env(monkeypatch, form=None, wpp=None):
    for k, v in (("CUDAMPC_FORM", form), ("CUDAMPC_WPP", wpp)):
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, v)


# ------------------------------------------------------------------------------------------------
# one horizon: two parameter sets, B = 2 * SMs * P + 3 problems each (every resident group solves at least two problems
# back to back), solved by the default kernel and certified once; the tests of the horizon share it
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", params=HORIZONS, ids=lambda N: f"N{N}")
def horizon(request):
    import torch
    from rrt_mpc_b200 import MPCController
    N = request.param
    saved = {k: os.environ.pop(k, None) for k in ("CUDAMPC_FORM", "CUDAMPC_WPP")}
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    sets = []
    try:
        for i, du in enumerate(DUS):
            p = product_params(N, du)
            ctl = MPCController(p, settings())
            B = 2 * sms * ctl.problems_per_sm() + 3
            x0, ref, up = horizon_problems(N, B, seed=10 * N + i)
            res = ctl.solve_batch(x0, ref, u_prev=up)
            A, Bm, c = ctl.linearize_batch(ref)
            opt = certify(p, x0, ref, up, res.Up, A, Bm, device="cuda")
            sets.append(NS(du=du, p=p, ctl=ctl, B=B, x0=x0, ref=ref, up=up, res=res, A=A, Bm=Bm, c=c, opt=opt))
    finally:
        os.environ.update({k: v for k, v in saved.items() if v is not None})
    yield NS(N=N, sets=sets)
    for s in sets:
        s.ctl.close()


def test_default_kernel_against_the_certificate(horizon):
    N = horizon.N
    for s in horizon.sets:
        r = s.res
        assert (r.status == 1).all(), (s.du, np.flatnonzero(r.status != 1))
        pol = r.info[:, 2] > 0
        x0e = np.abs(r.Xp[:, :, 0] - s.x0).max(axis=1)                 # X_0 = x0 is a constraint of the QP, solved with it
        within(x0e[pol].max(initial=0.0), {MAX_HORIZON: 1e-8}, N, "X_0 - x0")             # measured 1.06e-9 (all problems)
        within(x0e.max(), {MAX_HORIZON: 1e-7}, N, "X_0 - x0 unpolished")
        dyn = r.Xp[:, :, 1:] - np.einsum("bkij,bjk->bik", s.A, r.Xp[:, :, :-1]) - np.einsum("bkij,bjk->bik", s.Bm, r.Up) \
            - s.c.transpose(0, 2, 1)
        within(np.abs(dyn).max(), {31: 1e-8, 63: 1e-8, 95: 1e-8, 145: 1e-8, MAX_HORIZON: 1e-6}, N, "dynamics residual")
        first, last = limits_active(s.p, s.up, s.opt)
        assert first.any() and last.any(), (s.du, first.sum(), last.sum())
        check_certificate(N, s.opt, r, "default")


def test_matches_the_host_emulation(horizon):
    """The first problems and the saturated ones against the emulation of the form the horizon dispatches to."""
    import emu_driver as E
    for s in horizon.sets:
        idx = np.r_[np.arange(18), s.B // 3, (2 * s.B) // 3]
        E.set_form(-1)
        e = E.solve(s.p, s.x0[idx], s.ref[idx], s.up[idx], **SOLVE)                   # settings() in the emulation's terms
        dev = NS(**{k: getattr(s.res, k)[idx] for k in ("status", "iters", "u0", "Xp", "Up", "info")})
        same_solves(dev, NS(status=e["status"], iters=e["iters"], u0=e["u0"], Xp=e["Xp"], Up=e["Up"], info=e["info"]), ("emulation", s.du))


def forced(N):
    """(CUDAMPC_FORM, CUDAMPC_WPP) of every override the horizon accepts."""
    out = [("general", None)]
    if N + 1 <= 64:
        out += [("reg", None), ("pair", None)]
    if N + 1 <= 32:
        out += [("short", None)]
    if N >= 96:
        out += [(None, "1")]
    return out


def test_every_override_agrees_with_the_default_kernel(horizon, monkeypatch):
    from rrt_mpc_b200 import MPCController
    N = horizon.N
    for form, wpp in forced(N):
        set_env(monkeypatch, form, wpp)
        for s in horizon.sets:
            ctl = MPCController(s.p, settings(), max_batch=s.B)
            try:
                r = ctl.solve_batch(s.x0, s.ref, u_prev=s.up)
            finally:
                ctl.close()
            same_solves(s.res, r, (f"form={form} wpp={wpp}", s.du))
            check_certificate(N, s.opt, r, f"form={form} wpp={wpp}")


def test_permuted_batch_is_bit_identical(horizon):
    """The same problems in another order land on other groups, after other problems: nothing of a group's previous problem
    may leak into the next one."""
    for s in horizon.sets:
        perm = np.random.default_rng(horizon.N).permutation(s.B)
        r = s.ctl.solve_batch(s.x0[perm], s.ref[perm], u_prev=s.up[perm])
        for k in KEYS:
            assert np.array_equal(getattr(r, k), getattr(s.res, k)[perm], equal_nan=True), (s.du, k)


def test_per_problem_parameter_twin_is_the_same_arithmetic(horizon):
    """Every row equal to the handle's parameters: bit-identical to the shared-parameter kernel (its own P, its own
    shared-memory layout with the Params slot of each group)."""
    import torch
    from rrt_mpc_b200 import params_array
    for s in horizon.sets:
        rows = torch.from_numpy(params_array([s.p] * s.B).view(np.uint8).reshape(s.B, -1)).cuda()
        r = s.ctl.solve_batch(s.x0, s.ref, u_prev=s.up, params=rows)
        for k in KEYS:
            assert np.array_equal(getattr(r, k), getattr(s.res, k), equal_nan=True), (s.du, k)


@pytest.mark.parametrize("N", BOUNDARIES)
def test_mixed_parameter_sets_at_the_dispatch_boundaries(N):
    """A batch of the six parameter sets of test_gpu_problem_params, each problem against the certificate of its own set."""
    import torch
    from rrt_mpc_b200 import MPCController
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    sets = param_sets(N)
    ctl = MPCController(sets[0], settings())
    B = 2 * sms * ctl.problems_per_sm() + 3
    x0, ref, up = horizon_problems(N, B, seed=7 * N)
    pick = np.random.default_rng(N).integers(0, len(sets), size=B)
    r = ctl.solve_batch(x0, ref, u_prev=up, params=[sets[k] for k in pick])
    ctl.close()
    assert (r.status == 1).all(), np.flatnonzero(r.status != 1)
    pol = r.info[:, 2] > 0
    assert (~pol).sum() <= MAX_UNPOLISHED, np.flatnonzero(~pol)
    for k, p in enumerate(sets):
        sel = pick == k
        own = MPCController(p, settings())
        A, Bm, _ = own.linearize_batch(ref[sel])
        own.close()
        opt = certify(p, x0[sel], ref[sel], up[sel], r.Up[sel], A, Bm, device="cuda")
        within(np.abs(r.u0[sel] - opt["U"][:, :, 0]).max(), MIXED_U0, N, "per-problem parameters u0")
        within(np.abs(r.Xp[sel] - opt["X"]).max(), MIXED_X, N, "per-problem parameters X")


# ------------------------------------------------------------------------------------------------
# closed loop
# ------------------------------------------------------------------------------------------------
LOOP = [(31, None), (32, None), (50, None), (63, None), (64, None), (100, None), (256, None), (32, "pair"), (50, "pair"), (63, "pair")]
T = 80                  # the oracle reaches the goal of the default scenario in 64 steps at each of these horizons


def scenario():
    d = load_golden("default_scenario.npz")
    return d, [tuple(p) for p in d["path"]]


@functools.lru_cache(maxsize=None)
def oracle_rollout(N, short):
    """CO.track of the default scenario at horizon N on the reference build_reference makes for N (padded to N + 1 rows), or,
    `short`, on the scenario's 45-row reference as the caller's own ref_global (shorter than N + 1 rows for N >= 45)."""
    from oracle import c_oracle as CO
    from rrt_mpc_b200 import MPCConfig
    from rrt_mpc_b200.control_stage import initial_state
    from rrt_mpc_b200.ref_builder import build_reference
    d, path = scenario()
    rg = d["ref_global"] if short else build_reference(path, 15.0, N, 0.1)
    return CO.track(MPCConfig(horizon=N).to_parameters(0.8), rg, initial_state(path, d["start"]), d["goal"], T, polish_passes=3, **TIGHT)


def tracker(N):
    from rrt_mpc_b200 import MPCConfig, SolverSettings, TrajectoryTracker
    return TrajectoryTracker(MPCConfig(horizon=N, sim_steps=T), None, settings=SolverSettings(polish_passes=3, polish_retry=2, **TIGHT))


def against_oracle(res, ora):
    n = int(res.n_steps[0])
    assert n == ora["n_steps"] and bool(res.goal_reached[0]) and not bool(res.aborted[0]), (n, ora["n_steps"])
    assert np.abs(res.states[0, :n, :2] - ora["states"][:n, :2]).max() < 1e-3
    assert np.abs(res.controls[0, :n] - ora["controls"][:n]).max() < 1e-5


@pytest.mark.parametrize("N,form", LOOP)
def test_closed_loop_at_long_horizons(N, form, monkeypatch):
    """K_rollout against the CPU oracle's closed loop; K_step (TrackingSession, f_discrete as the plant) and the per-vehicle
    twin with every row equal bit-identical to K_rollout.  The window runs past the reference's end: the gather clamps there."""
    from rrt_mpc_b200 import MPCConfig
    from rrt_mpc_b200.control_stage import initial_state
    set_env(monkeypatch, form)
    d, path = scenario()
    tr = tracker(N)
    against_oracle(tr.track_batch([path], [d["start"]], [d["goal"]], map_resolution=0.8, warm_start=False), oracle_rollout(N, False))
    if N in (50, 100) and form is None:                     # the caller's reference, shorter than N + 1 rows
        s0 = initial_state(path, d["start"])[None]
        short = tr.track_batch(None, None, d["goal"][None], map_resolution=0.8, ref_globals=[d["ref_global"]], states0=s0, warm_start=False)
        against_oracle(short, oracle_rollout(N, True))
    paths, starts, goals = perturbed(8)
    paths[0], starts[0] = path, d["start"]
    for warm in (True, False):
        res = tr.track_batch(paths, starts, goals, map_resolution=0.8, warm_start=warm)
        assert res.goal_reached.any()
        sess = tr.start_batch(paths, starts, goals, map_resolution=0.8, warm_start=warm)
        out, _ = drive(sess, T, sess.controller.f_discrete_batch)
        assert_same_as_track_batch(res, out, sess, T, goals)
        sess.close()
        vp = tr.track_batch(paths, starts, goals, map_resolution=0.8, warm_start=warm,
                            vehicle_params=[MPCConfig(horizon=N).to_parameters(0.8)] * len(paths))
        for k in ("states", "controls", "n_steps", "goal_reached", "aborted", "relaxed", "step_status", "step_iters"):
            assert np.array_equal(getattr(vp, k), getattr(res, k), equal_nan=True), (warm, k)


# ------------------------------------------------------------------------------------------------
# K_ref
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [1, 15, 32, 63, 100, 256])
def test_build_reference_batch_against_build_reference(N):
    """Paths shorter and longer than N + 1 samples, one point, zero length, repeated consecutive points."""
    from rrt_mpc_b200 import MPCConfig, MPCController
    from rrt_mpc_b200.ref_builder import build_reference
    from rrt_mpc_b200.synthetic import random_path
    d, path = scenario()
    pts = np.asarray(path, float)
    paths = [pts, pts[:3], random_path(np.random.default_rng(N), 900.0), np.array([[50.0, 40.0]]),
             np.array([[50.0, 40.0]] * 3), np.repeat(pts, 2, axis=0), np.insert(pts, [2, 2, 7], pts[[2, 2, 7]], axis=0)]
    ctl = MPCController(MPCConfig(horizon=N).to_parameters(0.8))
    ref, ref_len = ctl.build_reference_batch(paths, 15.0)
    ref, ref_len = ref.cpu().numpy(), ref_len.cpu().numpy()
    ctl.close()
    for b, pth in enumerate(paths):
        want = build_reference(pth, 15.0, N, 0.1)
        assert ref_len[b] == len(want), (b, ref_len[b], len(want))
        got = ref[b, :len(want)]
        assert np.abs(got[:, :2] - want[:, :2]).max() <= 1e-12 * np.abs(want[:, :2]).max(), b
        assert np.abs(got[:, 2] - want[:, 2]).max() <= 1e-12 * max(1.0, np.abs(want[:, 2]).max()), b
        assert np.abs(got[:, 3] - want[:, 3]).max() <= 1e-12 * 15.0, b
