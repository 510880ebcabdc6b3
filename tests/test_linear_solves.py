"""The linear solves under every ADMM iteration and every polish step, one operation at a time, against an independent
reference in high precision.

Three systems, placed into a problem workspace with the product's own layout (tests/emu/la_systems.h):
  (A) the reduced system of the odd-even solve (mpc_oe.h) on the even stages, random SPD with condition numbers 1e1..1e12;
  (B) the ADMM operator of a real problem at rho in [rho_min, rho_max], solved as an iteration solves it;
  (C) the polish operator (weights {0, 1/delta}, delta = 1e-6) with chosen activity: banded LDL' and twisted sweeps.

Reference: the QP as oracle/mpc_numpy.build_qp states it (no code shared with csrc/), K = P + reg I + A' diag(w) A over
all n = 11N+5 variables, solved with the slack part of the right-hand side zero.  The slack block of K is diagonal, so
the (x,u) part of that solution is the exact solution of the slack-eliminated operator K^ the kernels factorise.
Residuals are formed in np.longdouble.

CPU tier: the sequential statements (tests/emu/emu.cpp).  GPU tier: the lane code of mpc_exec.cuh (tests/emu/la_dev.cu),
against the reference, against the one-lane statements compiled into the same binary (bit for bit), and a write check.
"""
import ctypes
import functools
import os
import shutil
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from conftest import ROOT, load_golden, oracle_params
from emu_driver import lib as emu, pack

LD = np.longdouble
EMU = os.path.join(ROOT, "tests", "emu")
SMEM_OPTIN = 227 * 1024          # shared memory a block can opt in to on sm_100


def _max_horizon():
    """Longest horizon whose workspace plus its GroupShared slot fits 227 KB (one problem per CTA)."""
    gs = emu().emu_group_shared_bytes()
    N = 1
    while 8 * emu().emu_footprint(N + 1) + gs <= SMEM_OPTIN:
        N += 1
    return N


# every horizon to 150 (zero / one step halves, jm = nb and nb + 1, gpad 0 and 2, all fpad / xpad pairs, the 31/32, 63/64
# and 84/85 dispatch boundaries), 200, and the longest that fits
HORIZONS = list(range(1, 151)) + [200, "max"]
RHOS = [1e-6, 1e-4, 1e-2, 0.1, 10.0, 1e3, 1e5, 1e6]     # rho_min, the documented range [1e-4, 1e5], rho_max
CONDS = [1e1, 1e4, 1e8, 1e12]
SIGMA = DELTA = 1e-6
RHO_EQ_FACTOR = 1e3

# ---- bounds: measured by the CPU tier (max over all horizons and cases), at most 10x above it --------------------------
# (A) reduced system, per condition number of the random system: normwise backward error, relative forward error.  The
# explicit pivot inverses are not backward stable on ill-conditioned systems: eta grows with cond (Cholesky would stay near
# eps) and at cond 1e12 the solution has no correct digit.  The ADMM operator (B) does not come near that regime.
ETA_RED = {1e1: 6e-16,           # measured 5.9e-17
           1e4: 2e-14,           # measured 1.6e-15
           1e8: 1.2e-10,         # measured 1.2e-11
           1e12: 8e-9}           # measured 7.7e-10
FWD_RED = {1e1: 8e-15,           # measured 7.5e-16
           1e4: 2e-11,           # measured 1.6e-12
           1e8: 6e-4,            # measured 5.5e-5
           1e12: 1.5e2}          # measured 1.5e1
# (B) ADMM operator, normwise backward error per rho range
ETA_ADMM = {"range": 7e-15,      # rho in [1e-4, 1e5]: measured 6.3e-16 (DESIGN claims 2e-14)
            "ends": 3e-15}       # rho = 1e-6 and 1e6 (rho_eq up to 1e9 against sigma = 1e-6): measured 2.4e-16
FWD_ADMM = {"range": 4e-9,       # relative forward error against the refined reference: measured 4.1e-10 (rho = 1e5)
            "ends": 2.5e-8}      # measured 2.5e-9 (rho = 1e6)
# (C) polish operator (weights 1/delta = 1e6 next to delta = 1e-6)
ETA_POL = 4e-16                  # measured 4.0e-17
FWD_POL = 2.5e-8                 # measured 2.5e-9


def _rho_class(rho):
    return "range" if 1e-4 <= rho <= 1e5 else "ends"


# ---------------------------------------------------------------------------------------------------------------------
# cases
# ---------------------------------------------------------------------------------------------------------------------
def horizon(N):
    return _max_horizon() if N == "max" else N


def _rhs(rng, n, kind):
    """unit-scale, or at the scale of an ADMM right-hand side (|q| up to about 2e3)"""
    return rng.standard_normal(n) if kind == 0 else rng.uniform(-2e3, 2e3, n)


@functools.lru_cache(maxsize=None)
def problem(N):
    """One problem of horizon N: inputs for the harness, the QP as the oracle states it, the (x,u) <-> column map."""
    from oracle import mpc_numpy as O
    from rrt_mpc_b200.synthetic import make_batch
    p = oracle_params(N)
    x0, ref, _ = make_batch(1, N, seed=7000 + N, pool=2)
    P, _, A, l, u, lay = O.build_qp(x0[0], ref[0], None, p)
    xu = np.array([11 * k + j if (k < N or j < 4) else -1 for k in range(N + 1) for j in range(6)])
    real = xu >= 0
    sl = np.setdiff1d(np.arange(lay.n), xu[real])
    par, st = pack(p, sigma=SIGMA, delta=DELTA)
    return dict(N=N, p=p, x0=x0[0], ref=ref[0], P=P.tocsr(), A=A.tocsr(), eq=(l == u), xu=xu, real=real, sl=sl,
                par=par, st=st, lay=lay)


def _csr_ld(M):
    M = M.tocsr()
    return M.data.astype(LD), M.indices, np.repeat(np.arange(M.shape[0]), np.diff(M.indptr)), M.shape[0]


def _mv(Mld, x):
    data, idx, rows, n = Mld
    y = np.zeros(n, LD)
    np.add.at(y, rows, data * x[idx])
    return y


class Operator:
    """K = P + reg I + A' diag(w) A of one problem; the slack-eliminated operator K^ on its 6(N+1) (x,u) unknowns."""

    def __init__(self, pr, reg, w):
        self.pr = pr
        self.reg, self.w = reg, w
        A, P = pr["A"], pr["P"]
        K = (P + reg * sp.identity(P.shape[0]) + A.T @ sp.diags(w) @ A).tocsc()
        xs, sl = pr["xu"][pr["real"]], pr["sl"]
        Kss = K[sl][:, sl]
        assert abs(Kss - sp.diags(Kss.diagonal())).max() == 0.0           # each slack touches only its own rows
        self.kss = Kss.diagonal().astype(LD)
        Kh = K[xs][:, xs] - K[xs][:, sl] @ sp.diags(1.0 / Kss.diagonal()) @ K[sl][:, xs]
        self.norm = max(float(abs(Kh).sum(axis=1).max()), 1.0)            # the dummy rows are identity rows
        self.lu = spla.splu(K)
        self.Pl, self.Al, self.wl = _csr_ld(P), _csr_ld(A), w.astype(LD)
        self.Atl = _csr_ld(A.T)

    def kmul(self, z):
        return _mv(self.Pl, z) + LD(self.reg) * z + _mv(self.Atl, self.wl * _mv(self.Al, z))

    def solve(self, b):
        """reference solution of K^ x = b: K z = [b; 0] in float64, two refinement steps with residuals in longdouble"""
        pr = self.pr
        xs, real = pr["xu"][pr["real"]], pr["real"]
        bf = np.zeros(pr["lay"].n, LD)
        bf[xs] = b[real]
        z = self.lu.solve(bf.astype(float))
        for _ in range(2):
            z = z + self.lu.solve((bf - self.kmul(z.astype(LD))).astype(float))
        x = np.array(b, float)
        x[real] = z[xs]
        return x

    def eta(self, x, b):
        """normwise backward error of x for K^ x = b (slacks eliminated exactly, in longdouble)"""
        pr = self.pr
        xs, sl, real = pr["xu"][pr["real"]], pr["sl"], pr["real"]
        z = np.zeros(pr["lay"].n, LD)
        z[xs] = x[real]
        z[sl] = -self.kmul(z)[sl] / self.kss
        r = np.array(b, LD) - np.array(x, LD)
        r[real] = np.array(b, LD)[real] - self.kmul(z)[xs]
        return float(np.abs(r).max() / (LD(self.norm) * np.abs(np.array(x, LD)).max() + np.abs(np.array(b, LD)).max()))


def fwd(x, xr):
    return float(np.abs(x - xr).max() / np.abs(xr).max())


@functools.lru_cache(maxsize=None)
def admm_cases(N):
    """(rho, b, reference) for every rho and both right-hand-side scales"""
    pr = problem(N)
    rng = np.random.default_rng(100 + N)
    out = []
    for rho in RHOS:
        op = Operator(pr, SIGMA, np.where(pr["eq"], RHO_EQ_FACTOR * rho, rho))
        for kind in (0, 1):
            b = _rhs(rng, 6 * (N + 1), kind)
            out.append((rho, b, op.solve(b), op))
    return out


def act_words(N, rows_active, lay):
    """activity words of mpc_core.h (act()[k]: bit 3g+r soft group g row r, bit 15+r dynamics row r; act()[N+1]: init rows)"""
    a = np.zeros(N + 2, np.int32)
    for i in range(4):
        a[N + 1] |= int(rows_active[lay.r_init(i)]) << i
    for k in range(N + 1):
        rows = [(0, r, lay.r_v(k, r)) for r in range(3)]
        if k < N:
            rows += [(1 + i, r, lay.r_u(k, i, r)) for i in range(2) for r in range(3)]
            rows += [(3 + i, r, lay.r_du(k, i, r)) for i in range(2) for r in range(3)]
            for r in range(4):
                a[k] |= int(rows_active[lay.r_dyn(k, r)]) << (15 + r)
        for g, r, row in rows:
            a[k] |= int(rows_active[row]) << (3 * g + r)
    return a


def golden_active_rows():
    """active set at the certified optimum of the golden n50 problem with the most active slacks: the rows that are tight
    at solve_kkt_newton's solution (equality rows always), so the mask does not come from the code under test"""
    from oracle import mpc_numpy as O
    g = load_golden("optima.npz")
    i = int(np.argmax(g["n50_active_slacks"]))
    p = oracle_params(50, du_delta=0.02)
    _, X, U, _ = O.solve_kkt_newton(g["n50_x0"][i], g["n50_ref"][i], g["n50_up"][i], p)
    P, _, A, l, u, lay = O.build_qp(g["n50_x0"][i], g["n50_ref"][i], g["n50_up"][i], p)
    z = np.zeros(lay.n)
    for k in range(51):
        z[[lay.x(k, j) for j in range(4)]] = X[:, k]
    for k in range(50):
        z[[lay.u(k, j) for j in range(2)]] = U[:, k]
    # slack of a soft group = its distance to [lo, hi]: rows hi/lo read g -/+ s
    g_rows = A @ z
    for k in range(51):
        lo, hi = p.v_bounds
        z[lay.sv(k)] = max(0.0, g_rows[lay.r_v(k, 0)] - hi, lo - g_rows[lay.r_v(k, 1)])
    for k in range(50):
        for i2 in range(2):
            z[lay.su(k, i2)] = max(0.0, g_rows[lay.r_u(k, i2, 0)] - u[lay.r_u(k, i2, 0)], l[lay.r_u(k, i2, 1)] - g_rows[lay.r_u(k, i2, 1)])
            z[lay.sdu(k, i2)] = max(0.0, g_rows[lay.r_du(k, i2, 0)] - u[lay.r_du(k, i2, 0)], l[lay.r_du(k, i2, 1)] - g_rows[lay.r_du(k, i2, 1)])
    Az = A @ z
    tight = (np.abs(Az - l) <= 1e-7 * np.maximum(1.0, np.abs(l))) | (np.abs(Az - u) <= 1e-7 * np.maximum(1.0, np.abs(u)))
    return tight, lay


@functools.lru_cache(maxsize=None)
def polish_cases(N):
    """(activity words, b, reference): all inactive, all active, two random masks (+ the golden active set at N = 50)"""
    pr = problem(N)
    lay, m = pr["lay"], pr["lay"].m
    rng = np.random.default_rng(200 + N)
    masks = [np.zeros(m, bool), np.ones(m, bool), rng.random(m) < 0.5, rng.random(m) < 0.15]
    if N == 50:
        masks.append(golden_active_rows()[0])
    out = []
    for i, act in enumerate(masks):
        op = Operator(pr, DELTA, act * (1.0 / DELTA))
        b = _rhs(rng, 6 * (N + 1), i & 1)
        out.append((act_words(N, act, lay), b, op.solve(b), op))
    return out


@functools.lru_cache(maxsize=None)
def reduced_cases(N):
    """random SPD block-tridiagonal systems K = L L' (L block-bidiagonal) on the J even stages, cond(K) near
    each target (measured 0.19x to 1.5x): (S, F, b, x_ref, K, target)"""
    J = N // 2 + 1
    rng = np.random.default_rng(300 + N)
    out = []
    for cond in CONDS:
        for kind in (0, 1):
            e = np.log10(cond) / 2
            d = 10.0 ** (-e * rng.random(6 * J))
            d[rng.integers(6 * J)] = 1.0
            d[rng.integers(6 * J)] = 10.0 ** -e
            # L = L0 diag(d), L0 unit block-bidiagonal with small off-diagonal blocks (well conditioned at any length)
            Ld = [(np.eye(6) + np.tril(0.1 * rng.standard_normal((6, 6)), -1)) * d[6 * j:6 * j + 6] for j in range(J)]
            Ls = [0.05 * rng.standard_normal((6, 6)) * d[6 * j - 6:6 * j] if j > 0 else None for j in range(J)]
            S = np.zeros((J, 6, 6)); F = np.zeros((J, 6, 6))
            for j in range(J):
                S[j] = Ld[j] @ Ld[j].T + (Ls[j] @ Ls[j].T if j > 0 else 0.0)
                S[j] = 0.5 * (S[j] + S[j].T)
                if j > 0:
                    F[j] = Ls[j] @ Ld[j - 1].T
            K = np.zeros((6 * J, 6 * J))
            for j in range(J):
                K[6 * j:6 * j + 6, 6 * j:6 * j + 6] = S[j]
                if j > 0:
                    K[6 * j:6 * j + 6, 6 * j - 6:6 * j] = F[j]
                    K[6 * j - 6:6 * j, 6 * j:6 * j + 6] = F[j].T
            b = _rhs(rng, 6 * J, kind)
            x = np.linalg.solve(K, b)
            Kl = K.astype(LD)
            for _ in range(2):
                x = x + np.linalg.solve(K, (np.array(b, LD) - Kl @ x.astype(LD)).astype(float))
            out.append((S, F, b, x, K, cond))
    return out


def eta_dense(K, x, b):
    r = np.array(b, LD) - K.astype(LD) @ np.array(x, LD)
    return float(np.abs(r).max() / (LD(np.abs(K).sum(axis=1).max()) * np.abs(np.array(x, LD)).max() + np.abs(np.array(b, LD)).max()))


# ---------------------------------------------------------------------------------------------------------------------
# host runs (the sequential statements)
# ---------------------------------------------------------------------------------------------------------------------
dp = ctypes.POINTER(ctypes.c_double)
ip = ctypes.POINTER(ctypes.c_int)


def _p(a):
    return a.ctypes.data_as(dp)


def host_reduced(N):
    cs = reduced_cases(N)
    J, n = N // 2 + 1, len(cs)
    S = np.ascontiguousarray(np.stack([c[0] for c in cs]))
    F = np.ascontiguousarray(np.stack([c[1] for c in cs]))
    b = np.ascontiguousarray(np.stack([c[2] for c in cs]))
    x = np.zeros((n, 6 * J)); fac = np.zeros((n, emu().emu_oe_doubles(N)))
    emu().emu_la_reduced(N, n, _p(S), _p(F), _p(b), _p(x), _p(fac))
    return x, fac


def _op_inputs(N, mode):
    pr = problem(N)
    cs = admm_cases(N) if mode == 1 else polish_cases(N)
    n = len(cs)
    rho = np.array([c[0] for c in cs]) if mode == 1 else np.zeros(n)
    act = np.ascontiguousarray(np.stack([c[0] for c in cs]).astype(np.int32)) if mode == 2 else np.zeros((n, N + 2), np.int32)
    b = np.ascontiguousarray(np.stack([c[1] for c in cs]))
    x0 = np.ascontiguousarray(np.repeat(pr["x0"][None], n, 0))
    ref = np.ascontiguousarray(np.repeat(pr["ref"][None], n, 0))
    return pr, cs, rho, act, b, x0, ref


def host_operator(N, mode):
    pr, cs, rho, act, b, x0, ref = _op_inputs(N, mode)
    x = np.zeros_like(b)
    emu().emu_la_operator(mode, _p(pr["par"]), _p(pr["st"]), N, len(cs), _p(rho), _p(x0), _p(ref),
                          act.ctypes.data_as(ip), _p(b), _p(x))
    return x


def check_reduced(N, x):
    for (S, F, b, xr, K, cond), xi in zip(reduced_cases(N), x):
        e, f = eta_dense(K, xi, b), fwd(xi, xr)
        assert e <= ETA_RED[cond], (N, cond, e)
        assert f <= FWD_RED[cond], (N, cond, f)


def check_admm(N, x):
    for (rho, b, xr, op), xi in zip(admm_cases(N), x):
        e, f = op.eta(xi, b), fwd(xi, xr)
        assert e <= ETA_ADMM[_rho_class(rho)], (N, rho, e)
        assert f <= FWD_ADMM[_rho_class(rho)], (N, rho, f)


def check_polish(N, x):
    for i, ((act, b, xr, op), xi) in enumerate(zip(polish_cases(N), x)):
        e, f = op.eta(xi, b), fwd(xi, xr)
        assert e <= ETA_POL, (N, i, e)
        assert f <= FWD_POL, (N, i, f)


_ids = [f"N{h}" for h in HORIZONS]


@pytest.mark.parametrize("N", HORIZONS, ids=_ids)
def test_reduced_host(N):
    N = horizon(N)
    x, _ = host_reduced(N)
    check_reduced(N, x)


@pytest.mark.parametrize("N", HORIZONS, ids=_ids)
def test_admm_operator_host(N):
    N = horizon(N)
    check_admm(N, host_operator(N, 1))


@pytest.mark.parametrize("N", HORIZONS, ids=_ids)
def test_polish_operator_host(N):
    N = horizon(N)
    check_polish(N, host_operator(N, 2))


def test_golden_active_set_is_mixed():
    """the golden n50 active set has active and inactive soft rows (otherwise it repeats the all/none masks)"""
    tight, lay = golden_active_rows()
    soft = np.ones(lay.m, bool)
    soft[[lay.r_init(i) for i in range(4)]] = False
    soft[[lay.r_dyn(k, i) for k in range(50) for i in range(4)]] = False
    assert tight[~soft].all()
    assert 0 < tight[soft].sum() < soft.sum()
    # at least one soft limit is crossed (a hi or lo row tight), not only the s >= 0 rows
    hl = [lay.r_v(k, j) for k in range(51) for j in (0, 1)] + [lay.r_du(k, i, j) for k in range(50) for i in range(2) for j in (0, 1)]
    assert tight[hl].any()


def test_writable_sets_are_inside_the_workspace():
    """the write masks the device check uses: the factor and rhs areas only, never a stage record or the header"""
    for N in (1, 2, 3, 50, 151):
        F = emu().emu_footprint(N)
        for mode in (0, 1, 2):
            m = np.zeros(F, np.uint8)
            emu().emu_la_writable(N, mode, m.ctypes.data_as(ctypes.POINTER(ctypes.c_ubyte)))
            assert 0 < m.sum() < F
            hdr = 10 + (N + 3) // 2
            assert not m[:hdr + (N + 1) * 47].any(), (N, mode)


def test_factor_blocks_of_the_two_halves_in_different_bank_groups():
    """mpc_oe.h oe_view: the two chain lanes read block i of gt and of gb at the same step, so gb starts an odd number of
    16-byte columns (mod 8) after gt (gpad = 2 where 18 jm = 0 mod 8); and the factor stays inside oe_doubles(N)"""
    o = np.zeros(6, np.int32)
    for N in range(1, horizon("max") + 1):
        emu().emu_oe_offsets(N, o.ctypes.data_as(ip))
        dinv, sinv, gt, gb, band, nf = (int(v) for v in o)
        J, jm = N // 2 + 1, (N // 2 + 1) // 2
        nb = J - 1 - jm
        assert dinv == band and sinv == dinv + 22 * ((N + 1) // 2) and gt == sinv + 22 * J, N
        assert gt % 2 == 0 and gb % 2 == 0, N                                   # 16-byte aligned blocks
        assert gb - gt in (36 * jm, 36 * jm + 2), N
        if jm >= 1 and nb >= 1:
            assert ((gb - gt) // 2) % 8 != 0, (N, jm, gb - gt)
        assert gb + 36 * nb <= band + nf, N


# ---------------------------------------------------------------------------------------------------------------------
# device runs (the lane code of mpc_exec.cuh, and the one-lane statements in the same binary)
# ---------------------------------------------------------------------------------------------------------------------
DEV_SRC = [os.path.join(EMU, "la_dev.cu"), os.path.join(EMU, "la_systems.h")] + [
    os.path.join(ROOT, "rrt_mpc_b200", "csrc", f) for f in sorted(os.listdir(os.path.join(ROOT, "rrt_mpc_b200", "csrc")))
    if f.endswith((".h", ".cuh"))]


@pytest.fixture(scope="module")
def dev():
    """tests/emu/la_dev.so, built with the product's flags when a source is newer"""
    so = os.path.join(EMU, "la_dev.so")
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in DEV_SRC):
        nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
                        "-shared", "-o", so, DEV_SRC[0]], check=True, cwd=ROOT)
    lib = ctypes.CDLL(so)
    assert lib.la_group_shared_bytes() == emu().emu_group_shared_bytes()
    lib.la_run.argtypes = [ctypes.c_int] * 5 + [ctypes.c_void_p] * 15
    lib.la_run.restype = ctypes.c_int
    return lib


def dev_run(lib, wpp, mode, lanes, N, S=None, Fb=None, b=None, rho=None, x0=None, ref=None, act=None, par=None, st=None):
    import torch
    nsys = b.shape[0]
    P, words = ctypes.c_int(), ctypes.c_int()
    assert lib.la_geometry(wpp, N, ctypes.byref(P), ctypes.byref(words)) >= 1, (wpp, N)
    grid = -(-nsys // P.value)
    cuda = lambda a, dt=torch.float64: None if a is None else torch.as_tensor(np.ascontiguousarray(a)).to("cuda", dt)
    t = dict(rho=cuda(rho), x0=cuda(x0), ref=cuda(ref), act=cuda(act, torch.int32), S=cuda(S), Fb=cuda(Fb), b=cuda(b))
    x = torch.zeros(b.shape, dtype=torch.float64, device="cuda")
    fac = torch.zeros((nsys, emu().emu_oe_doubles(N)), dtype=torch.float64, device="cuda")
    snap = torch.empty(grid * words.value, dtype=torch.float64, device="cuda")
    F = emu().emu_footprint(N)
    m = np.zeros(F, np.uint8)
    emu().emu_la_writable(N, mode, m.ctypes.data_as(ctypes.POINTER(ctypes.c_ubyte)))
    mask = torch.as_tensor(m).cuda()
    changed = torch.zeros(65, dtype=torch.int32, device="cuda")
    if par is None:
        par, st = pack(oracle_params(N), sigma=SIGMA, delta=DELTA)
    vp = lambda a: None if a is None else ctypes.c_void_p(a.data_ptr())
    err = lib.la_run(wpp, mode, lanes, N, nsys, par.ctypes.data, st.ctypes.data, vp(t["rho"]), vp(t["x0"]), vp(t["ref"]),
                     vp(t["act"]), vp(t["S"]), vp(t["Fb"]), vp(t["b"]), vp(x), vp(fac), vp(snap), vp(mask), vp(changed),
                     ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert err == 0, f"la_run: cudaError {err}"
    torch.cuda.synchronize()
    ch = changed.cpu().numpy()
    return x.cpu().numpy(), fac.cpu().numpy(), int(ch[0]), [(int(i) // words.value, int(i) % words.value) for i in ch[1:1 + min(ch[0], 64)]]


def _bits_equal(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.int64), np.ascontiguousarray(b).view(np.int64))


def _agree(x, xh, bound):
    """device and host solutions: both within `bound` of the reference, so within 2 * bound of each other"""
    assert np.abs(x - xh).max() <= 2 * bound * np.abs(xh).max(), float(np.abs(x - xh).max() / np.abs(xh).max())


@pytest.mark.gpu
@pytest.mark.parametrize("wpp", [1, 2])
@pytest.mark.parametrize("N", HORIZONS, ids=_ids)
def test_reduced_device(dev, N, wpp):
    N = horizon(N)
    cs = reduced_cases(N)
    S, F, b = (np.stack([c[i] for c in cs]) for i in range(3))
    x, fac, nch, where = dev_run(dev, wpp, 0, 1, N, S=S, Fb=F, b=b)
    x1, fac1, nch1, where1 = dev_run(dev, wpp, 0, 0, N, S=S, Fb=F, b=b)
    assert nch == 0 and nch1 == 0, ("protected words changed (CTA, word)", where, where1)
    assert _bits_equal(fac, fac1), "oe_factor_lanes: factor differs from the one-lane statements"
    assert _bits_equal(x, x1), "oe_forward_lanes / oe_backward_lanes: solution differs from the one-lane statements"
    check_reduced(N, x)
    xh, _ = host_reduced(N)
    for (S_, F_, b_, xr, K, cond), xd, xhi in zip(cs, x, xh):
        _agree(xd, xhi, FWD_RED[cond])


@pytest.mark.gpu
@pytest.mark.parametrize("wpp", [1, 2])
@pytest.mark.parametrize("N", HORIZONS, ids=_ids)
def test_admm_operator_device(dev, N, wpp):
    N = horizon(N)
    pr, cs, rho, act, b, x0, ref = _op_inputs(N, 1)
    kw = dict(b=b, rho=rho, x0=x0, ref=ref, par=pr["par"], st=pr["st"])
    x, fac, nch, where = dev_run(dev, wpp, 1, 1, N, **kw)
    x1, fac1, nch1, where1 = dev_run(dev, wpp, 1, 0, N, **kw)
    assert nch == 0 and nch1 == 0, ("protected words changed (CTA, word)", where, where1)
    assert _bits_equal(fac, fac1), "GroupExec::oe_factor: factor differs from the one-lane statements"
    assert _bits_equal(x, x1), "ADMM solve: solution differs from the one-lane statements"
    check_admm(N, x)
    xh = host_operator(N, 1)
    for (r, *_), xd, xhi in zip(cs, x, xh):
        _agree(xd, xhi, FWD_ADMM[_rho_class(r)])


@pytest.mark.gpu
@pytest.mark.parametrize("wpp", [1, 2])
@pytest.mark.parametrize("N", HORIZONS, ids=_ids)
def test_polish_operator_device(dev, N, wpp):
    N = horizon(N)
    pr, cs, rho, act, b, x0, ref = _op_inputs(N, 2)
    kw = dict(b=b, act=act, x0=x0, ref=ref, par=pr["par"], st=pr["st"])
    x, _, nch, where = dev_run(dev, wpp, 2, 1, N, **kw)
    x1, _, nch1, where1 = dev_run(dev, wpp, 2, 0, N, **kw)
    assert nch == 0 and nch1 == 0, ("protected words changed (CTA, word)", where, where1)
    assert _bits_equal(x, x1), "factor_twisted_lanes / chain_twisted_lanes: solution differs from the one-lane statements"
    check_polish(N, x)
    _agree(x, host_operator(N, 2), FWD_POL)
