"""CPU: the host emulation of the solve (tests/emu, the kernels' own headers run lane by lane) at EVERY horizon the library
accepts.  Forms of the ADMM iteration against the general (parity) form, bit for bit, at every horizon they run (1..63); the
general form against the exact optimum of every problem (tests/certificate.py) at every horizon 1..256.

The helpers of this file (problems with limits active at the first and the last stage, the certificate of a batch) are the
ones tests/test_gpu_horizons.py runs the device kernels on."""
import numpy as np
import pytest

import certificate as CT
import emu_driver as E
from conftest import oracle_params

TIGHT = dict(eps_abs=1e-6, eps_rel=1e-6)
SOLVE = dict(polish_passes=5, polish_retry=2, early_polish=1, **TIGHT)
MAX_HORIZON = 256
DUS = (0.15, 0.02)                  # steering-rate limit of the two parameter sets of every horizon
# bars of the emulation (general form, every horizon 1..256), at most 10x the worst measured over each range of horizons.
# The state error and the residual of the dynamics grow with the horizon: positions reach 3000 px at N = 256.
EMU_U0 = 1e-8                       # measured 3.1e-9 (N = 129..192)
EMU_X = {64: 1e-7,                  # measured 1.1e-8
         128: 2e-7,                 # measured 2.4e-8
         192: 5e-6,                 # measured 7.4e-7
         256: 5e-5}                 # measured 7.5e-6
EMU_DYN = {128: 1e-8,               # measured 1.1e-9
           192: 1e-7,               # measured 1.6e-8
           256: 1e-6}               # measured 1.2e-7


def by_horizon(table, N):
    """The bar of the range of horizons N falls in: the smallest key >= N."""
    return table[min(k for k in table if N <= k)]


# ------------------------------------------------------------------------------------------------
# problems
# ------------------------------------------------------------------------------------------------
def saturated(N):
    """Two problems in the style of test_emulation.test_active_limits_everywhere at the product's own limits: the reference
    speeds up to 120 px/s (v_hi = 90) through a hard turn, and u_prev holds the steering at its limit against the turn.  At
    the optimum the rate rows of stage 0 (against u_prev) and the speed row of the last stage are active: the clamped-neighbour
    paths of the first and the last stage.  The start speed (90 px/s at N = 1, 3 px/s less per stage down to 60) lets the
    speed cross v_hi by the last stage at every horizon.  The second problem is the mirror image of the first."""
    v0 = max(60.0, 90.0 - 3.0 * (N - 1))
    yaw = -np.linspace(0.0, 2.5, N + 1)
    ref = np.zeros((N + 1, 4))
    ref[:, 2], ref[:, 3] = yaw, np.linspace(v0, 120.0, N + 1)
    ref[:, 0] = 80.0 + np.concatenate(([0.0], np.cumsum(0.1 * ref[:-1, 3] * np.cos(yaw[:-1]))))
    ref[:, 1] = 60.0 + np.concatenate(([0.0], np.cumsum(0.1 * ref[:-1, 3] * np.sin(yaw[:-1]))))
    x0 = ref[0] + np.array([0.0, 1.0, 0.3, 0.0])
    up = np.array([12.0, 0.6])
    m = np.array([1.0, -1.0, -1.0, 1.0])                       # mirror: y, yaw -> -y, -yaw
    mref = ref * m; mref[:, 1] += 120.0
    mx0 = x0 * m; mx0[1] += 120.0
    return np.stack([x0, mx0]), np.stack([ref, mref]), np.stack([up, up * [1.0, -1.0]])


def horizon_problems(N, n, seed):
    """n - 2 problems of make_batch (x0 noise, u_prev up to the limits) and the two saturated problems, interleaved."""
    from rrt_mpc_b200.synthetic import make_batch
    x0, ref, up = make_batch(n - 2, N, seed=seed)
    sx, sr, su = saturated(N)
    at = [n // 3, (2 * n) // 3]
    for i, j in enumerate(at):
        x0, ref, up = np.insert(x0, j, sx[i], 0), np.insert(ref, j, sr[i], 0), np.insert(up, j, su[i], 0)
    return x0, ref, up


# ------------------------------------------------------------------------------------------------
# certificate
# ------------------------------------------------------------------------------------------------
def certify(p, x0, ref, up, U, A, Bm, device="cpu"):
    """certificate.exact_optimum of every problem, started from the candidate controls U (B,2,N), with the linearisation
    (A, Bm) of the solve under test (linearize_batch / the emulation's hook)."""
    refu = ref.copy()
    refu[:, :, 2] = np.unwrap(ref[:, :, 2], axis=1)
    o = CT.exact_optimum(p, x0, refu, up, U, CT.lin_from_hook(A, Bm), device=device)
    assert o["settled"].all(), np.flatnonzero(~o["settled"])
    return o


def limits_active(p, up, opt):
    """(rate row against u_prev active at stage 0, speed row active at the last stage) per problem, at the exact optimum."""
    U, X = opt["U"], opt["X"]
    rate0 = U[:, :, 0] - up
    lo = np.array([p.du_bounds[0][0], p.du_bounds[1][0]]); hi = np.array([p.du_bounds[0][1], p.du_bounds[1][1]])
    first = ((rate0 < lo - 1e-9) | (rate0 > hi + 1e-9)).any(axis=1)
    v = X[:, 3, -1]
    last = (v > p.v_bounds[1] + 1e-9) | (v < p.v_bounds[0] - 1e-9)
    return first, last


def emu_solve(p, x0, ref, up, form, reverse=0):
    try:
        E.set_form(form)
        return E.solve(p, x0, ref, up, reverse=reverse, **SOLVE)
    finally:
        E.set_form(-1)


# ------------------------------------------------------------------------------------------------
# forms of the iteration: bit-identical to the general form at every horizon they run
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", range(1, 64))
def test_every_form_is_the_general_form_bit_for_bit(N):
    """Short (1, N + 1 <= 32), pair (2), register (3) and register with the state left in the records (7), each with the
    stages of a part visited in order and in reverse, against the general parity form (0): same operands, same order, so every
    output agrees to the last bit, the counters of `info` included."""
    forms = ([1] if N + 1 <= 32 else []) + [2, 3, 7]
    for du in DUS:
        p = oracle_params(N, du)
        x0, ref, up = horizon_problems(N, 5, seed=1000 * N + int(du * 100))
        b = emu_solve(p, x0, ref, up, 0)
        assert (b["status"] == 1).all(), (du, b["status"])
        for form in forms:
            for rev in (0, 1):
                a = emu_solve(p, x0, ref, up, form, rev)
                for k in ("status", "iters", "info", "u0", "Xp", "Up", "pri", "dua"):
                    assert np.array_equal(a[k], b[k]), (du, form, rev, k)


# ------------------------------------------------------------------------------------------------
# the general form against the exact optimum at every horizon
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", range(1, MAX_HORIZON + 1))
def test_general_form_against_the_certificate(N):
    du = DUS[N % 2]                  # both parameter sets, alternating over the horizons
    p = oracle_params(N, du)
    x0, ref, up = horizon_problems(N, 5, seed=N)
    r = emu_solve(p, x0, ref, up, 0)
    assert (r["status"] == 1).all() and (r["info"][:, 2] > 0).all(), (r["status"], r["info"])
    assert np.abs(r["Xp"][:, :, 0] - x0).max() < 1e-9
    A, Bm, c = E.linearize(p, ref)
    res = r["Xp"][:, :, 1:] - np.einsum("bkij,bjk->bik", A, r["Xp"][:, :, :-1]) - np.einsum("bkij,bjk->bik", Bm, r["Up"]) \
        - c.transpose(0, 2, 1)
    assert np.abs(res).max() < by_horizon(EMU_DYN, N)
    o = certify(p, x0, ref, up, r["Up"], A, Bm)
    first, last = limits_active(p, up, o)
    assert first.any() and last.any(), (first, last)
    assert np.abs(r["u0"] - o["U"][:, :, 0]).max() < EMU_U0
    assert np.abs(r["Xp"] - o["X"]).max() < by_horizon(EMU_X, N)
