"""Drop-in ``MPCController`` backed by libcudampc.so (hand-written sm_100a CUDA, no CPU path).

Same names, arguments and failure behaviour as /root/reference/src/control/mpc_controller.py:17-145:

* ``MPCParameters``  — same fields and defaults (mpc_controller.py:17-30);
* ``MPCController(params).solve(x0, ref_traj, *, u_init=None, u_prev=None)`` returns
  ``(u0 (2,), Xp (4,N+1), Up (2,N))`` or ``(None, None, None)`` when the solver status is not
  optimal / optimal_inaccurate (mpc_controller.py:137-141); inputs are not mutated; ``u_init`` is
  accepted and ignored exactly as upstream (mpc_controller.py:50-51 computes it and never uses it);
* new: ``solve_batch`` (thousands of independent problems per launch, optionally each with its own
  ``MPCParameters``), ``linearize_batch`` and solver settings as constructor arguments (upstream hard-codes them,
  mpc_controller.py:121-131).
"""
from __future__ import annotations

import ctypes as C
import logging
from dataclasses import dataclass, field
from typing import Optional, Tuple

import numpy as np

from . import _lib

LOG = logging.getLogger(__name__)

STATUS_SOLVED = 1
STATUS_SOLVED_INACCURATE = 2
STATUS_MAX_ITER = -2
_OK = (STATUS_SOLVED, STATUS_SOLVED_INACCURATE)


@dataclass
class MPCParameters:
    wheelbase_px: float
    dt: float
    horizon: int
    q: np.ndarray
    r: np.ndarray
    q_terminal: np.ndarray
    u_bounds: Tuple[Tuple[float, float], Tuple[float, float]]
    v_bounds: Tuple[float, float]
    du_bounds: Tuple[Tuple[float, float], Tuple[float, float]]
    slack_velocity: float = 1e3
    slack_input: float = 5e2
    slack_rate: float = 5e2


@dataclass
class SolverSettings:
    """OSQP-style settings; defaults are what the reference passes (mpc_controller.py:121-131)."""
    eps_abs: float = 1e-3
    eps_rel: float = 1e-3
    max_iter: int = 60000
    polish: bool = True
    polish_passes: int = 1        # 1 = OSQP's single polish; >1 re-identifies the active set (used for 1e-5 parity)
    adaptive_rho: bool = True
    rho: float = 0.1
    alpha: float = 1.6
    sigma: float = 1e-6
    check_termination: int = 25
    adaptive_rho_interval: int = 50
    adaptive_rho_tolerance: float = 5.0
    delta: float = 1e-6
    polish_refine_iter: int = 3
    warm_start: bool = False      # upstream's warm_start=True is a no-op (a new Problem per call)
    keep_iterate: bool = True     # False (with warm_start False): stateless solve, nothing is stored per problem for a later warm start
    polish_retry: int = 0         # rejected polish -> resume ADMM at 10x tighter internal eps, polish again (0 = OSQP)
    early_polish: bool = False    # try the polish as soon as the guessed active set repeats; finish if it certifies a KKT point
    early_polish_start: int = 50

    @classmethod
    def early_certified(cls, eps: float = 1e-6, **kw) -> "SolverSettings":
        """The settings bench.py's headline runs: tolerance `eps`, re-identified active set (5 polish passes), up to 4 resumes after a
        rejected polish, early polish with ONE termination check / polish probe per rho-adaptation interval (check_termination = 50;
        OSQP's 25 costs 15 % of the throughput, DESIGN.md section 8), stateless solves.  Every solve ends on a polished KKT point."""
        base = dict(eps_abs=eps, eps_rel=eps, polish_passes=5, polish_retry=4, early_polish=True, check_termination=50, keep_iterate=False)
        base.update(kw)
        return cls(**base)

    def to_c(self) -> _lib.Settings:
        lib = _lib.load()
        s = _lib.Settings()
        lib.cudampc_default_settings(C.byref(s))
        s.eps_abs, s.eps_rel, s.max_iter = self.eps_abs, self.eps_rel, int(self.max_iter)
        s.polish_passes = int(self.polish_passes) if self.polish else 0
        s.adaptive_rho, s.rho, s.alpha, s.sigma = int(self.adaptive_rho), self.rho, self.alpha, self.sigma
        s.check_termination, s.adaptive_rho_interval = int(self.check_termination), int(self.adaptive_rho_interval)
        s.adaptive_rho_tolerance, s.delta = self.adaptive_rho_tolerance, self.delta
        s.polish_refine_iter = int(self.polish_refine_iter)
        s.warm_start = 1 if self.warm_start else (0 if self.keep_iterate else -1)
        s.polish_retry = int(self.polish_retry)
        s.early_polish, s.early_polish_start = int(self.early_polish), int(self.early_polish_start)
        return s


def params_to_c(p: MPCParameters) -> _lib.Params:
    c = _lib.Params()
    c.wheelbase_px, c.dt, c.horizon = float(p.wheelbase_px), float(p.dt), int(p.horizon)
    c.q[:] = np.asarray(p.q, dtype=float).reshape(16).tolist()
    c.r[:] = np.asarray(p.r, dtype=float).reshape(4).tolist()
    c.q_terminal[:] = np.asarray(p.q_terminal, dtype=float).reshape(16).tolist()
    c.u_bounds[:] = [p.u_bounds[0][0], p.u_bounds[0][1], p.u_bounds[1][0], p.u_bounds[1][1]]
    c.v_bounds[:] = [p.v_bounds[0], p.v_bounds[1]]
    c.du_bounds[:] = [p.du_bounds[0][0], p.du_bounds[0][1], p.du_bounds[1][0], p.du_bounds[1][1]]
    c.slack_velocity, c.slack_input, c.slack_rate = float(p.slack_velocity), float(p.slack_input), float(p.slack_rate)
    return c


def params_array(params) -> np.ndarray:
    """One ``_lib.PARAMS_DTYPE`` record (the layout of ``cudampc_params``) per ``MPCParameters`` of the sequence ``params``.
    The array can be edited field-wise for sweeps (``arr["du_bounds"][:, 3] = ...``) and passed as ``params=`` /
    ``vehicle_params=``."""
    return np.frombuffer(b"".join(bytes(params_to_c(p)) for p in params), dtype=_lib.PARAMS_DTYPE).copy()


def params_rows(params, batch: int, base: MPCParameters):
    """Per-problem parameters checked against a handle created with ``base``: a ``PARAMS_DTYPE`` array of ``batch`` records for
    a sequence of ``MPCParameters`` or such an array, or the CUDA ``uint8`` tensor ``(batch, PARAMS_DTYPE.itemsize)`` as given.
    Raises ``ValueError`` for a wrong shape, or a record whose horizon or dt differs from ``base`` (dt compared exactly); the
    other rules are applied per record on the device (a rejected record gets ``STATUS_INVALID_PARAMS``).  The horizon and dt of
    a tensor's records are checked there too."""
    rec = _lib.PARAMS_DTYPE.itemsize
    if hasattr(params, "is_cuda"):
        import torch
        if tuple(params.shape) != (batch, rec) or params.dtype != torch.uint8 or not params.is_cuda or not params.is_contiguous():
            raise ValueError(f"params: expected a contiguous CUDA uint8 tensor of shape ({batch}, {rec}); "
                             f"got {params.dtype} {tuple(params.shape)} on {params.device}")
        return params
    if isinstance(params, np.ndarray) and params.dtype == _lib.PARAMS_DTYPE:
        arr = np.ascontiguousarray(params)
    elif isinstance(params, np.ndarray):
        raise ValueError(f"params: expected an array of dtype PARAMS_DTYPE or a sequence of MPCParameters; got dtype {params.dtype}")
    else:
        arr = params_array(params)
    if arr.shape != (batch,):
        raise ValueError(f"params: expected {batch} records; got shape {arr.shape}")
    bad = np.flatnonzero((arr["horizon"] != int(base.horizon)) | (arr["dt"] != float(base.dt)))
    if bad.size:
        raise ValueError(f"params: horizon and dt must equal the controller's ({base.horizon}, {base.dt!r}); "
                         f"records {bad[:8].tolist()} differ")
    return arr


def params_to_device(rows, device):
    """``params_rows`` output as the CUDA uint8 tensor the *_params entry points read."""
    import torch
    if hasattr(rows, "is_cuda"):
        if rows.device != device:
            raise ValueError(f"params live on {rows.device}; expected {device}")
        return rows
    return torch.from_numpy(rows.view(np.uint8).reshape(len(rows), _lib.PARAMS_DTYPE.itemsize)).to(device)


@dataclass
class BatchResult:
    u0: object          # (B,2)
    Xp: object          # (B,4,N+1)
    Up: object          # (B,2,N)
    status: object      # (B,) int32, OSQP codes
    iters: object       # (B,) int32
    pri_res: object = None
    dua_res: object = None
    info: object = None  # (B,4) int32: rho updates, factorisations, accepted polish passes, triangular solves

    def __iter__(self):  # (u0, Xp, Up, status, iters) unpacking as in SURVEY §8b
        return iter((self.u0, self.Xp, self.Up, self.status, self.iters))


class _Handle:
    """Owns a cudampc_handle (one per (params, capacity, device))."""

    def __init__(self, params: MPCParameters, max_batch: int, device: int):
        self.lib = _lib.load()
        self.ptr = C.c_void_p()
        cpar = params_to_c(params)
        rc = self.lib.cudampc_create(C.byref(cpar), int(max_batch), int(device), C.byref(self.ptr))
        if rc != 0:
            msg = self.lib.cudampc_last_error(None)
            raise RuntimeError(f"cudampc_create failed (code {rc}): {msg.decode() if msg else ''}")
        self.max_batch, self.device, self.horizon = int(max_batch), int(device), int(params.horizon)

    def close(self):
        if getattr(self, "ptr", None) and self.ptr.value:
            self.lib.cudampc_destroy(self.ptr)
            self.ptr = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _is_torch_cuda(x) -> bool:
    return hasattr(x, "is_cuda") and bool(x.is_cuda)


class MPCController:
    """Quadratic-cost MPC controller with soft bounds and rate limits (batched, GPU)."""

    def __init__(self, params: MPCParameters, settings: Optional[SolverSettings] = None, *, device: int = 0,
                 max_batch: int = 1) -> None:
        self._params = params
        self.settings = settings or SolverSettings()
        self._device = device
        self._capacity = max(1, int(max_batch))
        self._h: Optional[_Handle] = None

    # -- plumbing -------------------------------------------------------------------------------
    def _handle(self, batch: int) -> _Handle:
        if self._h is None or batch > self._h.max_batch:
            if self._h is not None:
                self._h.close()
            self._capacity = max(self._capacity, batch)
            self._h = _Handle(self._params, self._capacity, self._device)
        return self._h

    @property
    def params(self) -> MPCParameters:
        return self._params

    def close(self) -> None:
        if self._h is not None:
            self._h.close()
            self._h = None

    def launch_count(self) -> int:
        return int(self._h.lib.cudampc_launch_count(self._h.ptr)) if self._h else 0

    def problems_per_sm(self) -> int:
        h = self._handle(1)
        return int(h.lib.cudampc_problems_per_sm(h.ptr))

    def rollout_resident(self) -> int:
        """Vehicles the closed-loop kernel keeps in flight on the device."""
        h = self._handle(1)
        return int(h.lib.cudampc_rollout_resident(h.ptr))

    def fp64_peak_tflops(self) -> float:
        h = self._handle(1)
        return float(h.lib.cudampc_fp64_peak_tflops(h.ptr))

    def workspace_doubles(self) -> int:
        h = self._handle(1)
        return int(h.lib.cudampc_workspace_doubles(h.ptr))

    # -- reference signature --------------------------------------------------------------------
    def solve(self, x0, ref_traj, *, u_init=None, u_prev=None):
        N = self._params.horizon
        x0 = np.ascontiguousarray(x0, dtype=float).reshape(1, 4)
        ref = np.ascontiguousarray(np.asarray(ref_traj, dtype=float)[: N + 1]).reshape(1, N + 1, 4)
        up = None if u_prev is None else np.ascontiguousarray(u_prev, dtype=float).reshape(1, 2)
        res = self.solve_batch(x0, ref, u_prev=up)
        status = int(res.status[0])
        if status not in _OK:                      # mpc_controller.py:137-139
            LOG.warning("MPC solve returned status %s", status)
            return None, None, None
        return res.u0[0].copy(), res.Xp[0].copy(), res.Up[0].copy()

    # -- batched entry points -------------------------------------------------------------------
    def solve_batch(self, x0, ref, *, u_prev=None, settings: Optional[SolverSettings] = None, stream=None, params=None) -> BatchResult:
        """``x0 (B,4)``, ``ref (B,N+1,4)``, ``u_prev (B,2)|None`` as NumPy arrays (host path: pinned staging,
        H2D, solve, D2H) or as torch CUDA fp64 tensors (device path: asynchronous on the current stream).

        ``params``: per-problem parameters, problem b solved with its own record (``params_rows``: a sequence of
        ``MPCParameters``, a ``PARAMS_DTYPE`` array or a CUDA uint8 tensor ``(B, 416)``; horizon and dt as this controller's).
        With NumPy inputs the call then stages through device tensors and synchronises.  A record the parameter rules reject
        gets status ``STATUS_INVALID_PARAMS`` and NaN outputs."""
        s = (settings or self.settings).to_c()
        N = self._params.horizon
        if _is_torch_cuda(x0):
            rows = None if params is None else params_rows(params, x0.shape[0], self._params)
            return self._solve_batch_device(x0, ref, u_prev, s, stream, rows)
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        ref = np.ascontiguousarray(ref, dtype=np.float64)
        B = x0.shape[0]
        if x0.shape != (B, 4) or ref.shape != (B, N + 1, 4):
            raise ValueError(f"expected x0 (B,4) and ref (B,{N + 1},4); got {x0.shape} and {ref.shape}")
        up = None
        if u_prev is not None:
            up = np.ascontiguousarray(u_prev, dtype=np.float64)
            if up.shape != (B, 2):
                raise ValueError(f"expected u_prev (B,2); got {up.shape}")
        if params is not None:
            rows = params_rows(params, B, self._params)
            import torch
            dev = torch.device("cuda", self._device)
            t = lambda a: None if a is None else torch.as_tensor(a).to(dev)
            res = self._solve_batch_device(t(x0), t(ref), t(up), s, None, rows)
            torch.cuda.synchronize(dev)
            return BatchResult(*(x.cpu().numpy() for x in (res.u0, res.Xp, res.Up, res.status, res.iters, res.pri_res, res.dua_res, res.info)))
        out = self._host_outputs(B, N)
        if B == 0:
            return out
        h = self._handle(B)
        ptr = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        rc = h.lib.cudampc_solve_batch_host(h.ptr, B, ptr(x0), ptr(ref), ptr(up), C.byref(s), ptr(out.u0), ptr(out.Xp),
                                            ptr(out.Up), ptr(out.status), ptr(out.iters), ptr(out.pri_res),
                                            ptr(out.dua_res), ptr(out.info), None)
        _lib.check(h.lib, h.ptr, rc, "cudampc_solve_batch_host")
        return out

    def _host_outputs(self, B: int, N: int) -> BatchResult:
        """Result arrays of the host path.  With ``pinned_outputs`` they are views of page-locked torch tensors that are
        reused from call to call (so the library copies straight into them, no staging) - copy what you keep."""
        if not getattr(self, "pinned_outputs", False):
            return BatchResult(np.empty((B, 2)), np.empty((B, 4, N + 1)), np.empty((B, 2, N)), np.empty(B, np.int32),
                               np.empty(B, np.int32), np.empty(B), np.empty(B), np.empty((B, 4), np.int32))
        import torch
        cache = self.__dict__.setdefault("_pinned", {})
        if cache.get("B") != B:
            f = lambda *shape: torch.empty(shape, dtype=torch.float64).pin_memory()
            i = lambda *shape: torch.empty(shape, dtype=torch.int32).pin_memory()
            cache.update(B=B, t=(f(B, 2), f(B, 4, N + 1), f(B, 2, N), i(B), i(B), f(B), f(B), i(B, 4)))
        return BatchResult(*(t.numpy() for t in cache["t"]))

    def _solve_batch_device(self, x0, ref, u_prev, s, stream, rows=None) -> BatchResult:
        import torch
        N = self._params.horizon
        B = x0.shape[0]
        for name, t, shape in (("x0", x0, (B, 4)), ("ref", ref, (B, N + 1, 4))) + ((("u_prev", u_prev, (B, 2)),) if u_prev is not None else ()):
            if tuple(t.shape) != shape or t.dtype != torch.float64 or not t.is_contiguous() or not t.is_cuda:
                raise ValueError(f"{name}: expected contiguous CUDA float64 tensor of shape {shape}")
        dev = x0.device
        out = BatchResult(torch.empty((B, 2), dtype=torch.float64, device=dev),
                          torch.empty((B, 4, N + 1), dtype=torch.float64, device=dev),
                          torch.empty((B, 2, N), dtype=torch.float64, device=dev),
                          torch.empty(B, dtype=torch.int32, device=dev), torch.empty(B, dtype=torch.int32, device=dev),
                          torch.empty(B, dtype=torch.float64, device=dev), torch.empty(B, dtype=torch.float64, device=dev),
                          torch.empty((B, 4), dtype=torch.int32, device=dev))
        if B == 0:
            return out
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        if self._h is None:
            self._device = idx
        elif idx != self._h.device:
            raise ValueError(f"tensors live on cuda:{idx} but this controller's handle was created on cuda:{self._h.device}; "
                             "use one MPCController per device")
        h = self._handle(B)
        st = stream if stream is not None else torch.cuda.current_stream(dev).cuda_stream
        p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        if rows is not None:
            d_par = params_to_device(rows, dev)
            rc = h.lib.cudampc_solve_batch_params(h.ptr, B, p(x0), p(ref), p(u_prev), C.byref(s), p(d_par), p(out.u0), p(out.Xp),
                                                  p(out.Up), p(out.status), p(out.iters), p(out.pri_res), p(out.dua_res),
                                                  p(out.info), C.c_void_p(st))
            _lib.check(h.lib, h.ptr, rc, "cudampc_solve_batch_params")
            if stream is not None and d_par is not rows:    # the staged records are freed in the current stream's order
                torch.cuda.synchronize(dev)
            return out
        rc = h.lib.cudampc_solve_batch(h.ptr, B, p(x0), p(ref), p(u_prev), C.byref(s), p(out.u0), p(out.Xp), p(out.Up),
                                       p(out.status), p(out.iters), p(out.pri_res), p(out.dua_res), p(out.info),
                                       C.c_void_p(st))
        _lib.check(h.lib, h.ptr, rc, "cudampc_solve_batch")
        return out

    def build_reference_batch(self, paths, desired_speed: float, *, stride: Optional[int] = None):
        """``build_reference`` (ref_builder.py:10-22) for many polylines on the device.  ``paths``: sequence of ``(n_b, 2)``
        arrays.  Returns ``(ref (B, stride, 4), ref_len (B,))`` as torch CUDA tensors (rows beyond ``ref_len[b]`` are
        unspecified); feed them to ``cudampc_rollout_batch`` / ``TrajectoryTracker.track_batch``."""
        import torch
        N = self._params.horizon
        B = len(paths)
        npts = np.array([len(p) for p in paths], dtype=np.int32)
        if B and npts.min() < 1:
            raise RuntimeError("Planner returned an empty path")          # control_stage.py:71-72
        max_pts = int(npts.max()) if B else 1
        buf = np.zeros((B, max_pts, 2))
        for b, p in enumerate(paths):
            buf[b, :len(p)] = np.asarray(p, dtype=float)
        if stride is None:      # enough rows for the longest polyline: ceil(total / step) + 1, and at least N + 1
            step = max(2.0, 0.8 * desired_speed * self._params.dt)
            seg = np.hypot(*np.diff(buf, axis=1).transpose(2, 0, 1)) * (np.arange(1, max_pts)[None, :] < npts[:, None]) if max_pts > 1 else np.zeros((B, 1))
            stride = int(max(N + 1, np.ceil(seg.sum(axis=1).max() / step) + 2, max_pts))
        dev = torch.device("cuda", self._device)
        d_paths, d_n = torch.as_tensor(buf).to(dev), torch.as_tensor(npts).to(dev)
        ref = torch.empty((B, stride, 4), dtype=torch.float64, device=dev)
        ref_len = torch.empty(B, dtype=torch.int32, device=dev)
        h = self._handle(max(B, 1))
        st = torch.cuda.current_stream(dev).cuda_stream
        rc = h.lib.cudampc_build_reference_batch(h.ptr, B, C.c_void_p(d_paths.data_ptr()), C.c_void_p(d_n.data_ptr()), max_pts,
                                                 C.c_double(desired_speed), C.c_void_p(ref.data_ptr()), C.c_void_p(ref_len.data_ptr()),
                                                 stride, C.c_void_p(st))
        _lib.check(h.lib, h.ptr, rc, "cudampc_build_reference_batch")
        return ref, ref_len

    def f_discrete_batch(self, x, u, dt_L=None):
        """``f_discrete`` (vehicle_model.py:11-21) for ``x (B,4)``, ``u (B,2)`` on the device - the integrator of the closed
        loop, exposed for parity checks.  ``dt_L (B,2)``: per-sample ``(dt, wheelbase_px)``; default: this controller's."""
        import torch
        dev = torch.device("cuda", self._device)
        t = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).to(dev)
        dx, du = t(x).reshape(-1, 4), t(u).reshape(-1, 2)
        B = dx.shape[0]
        if du.shape[0] != B:
            raise ValueError("x and u must have the same leading dimension")
        dd = None if dt_L is None else t(dt_L).reshape(B, 2)
        out = torch.empty((B, 4), dtype=torch.float64, device=dev)
        h = self._handle(max(B, 1))
        st = torch.cuda.current_stream(dev).cuda_stream
        rc = h.lib.cudampc_f_discrete_batch(h.ptr, B, C.c_void_p(dx.data_ptr()), C.c_void_p(du.data_ptr()),
                                            C.c_void_p(dd.data_ptr()) if dd is not None else None, C.c_void_p(out.data_ptr()), C.c_void_p(st))
        _lib.check(h.lib, h.ptr, rc, "cudampc_f_discrete_batch")
        return out.cpu().numpy()

    def linearize_batch(self, ref):
        """(A (B,N,4,4), B (B,N,4,2), c (B,N,4)) as ``solve`` linearises them (mpc_controller.py:59-70,108-109)."""
        import torch
        N = self._params.horizon
        host = not _is_torch_cuda(ref)
        t = torch.as_tensor(np.ascontiguousarray(ref, dtype=np.float64)).cuda(self._device) if host else ref
        B = t.shape[0]
        if tuple(t.shape) != (B, N + 1, 4):
            raise ValueError(f"expected ref (B,{N + 1},4); got {tuple(t.shape)}")
        A = torch.empty((B, N, 4, 4), dtype=torch.float64, device=t.device)
        Bm = torch.empty((B, N, 4, 2), dtype=torch.float64, device=t.device)
        c = torch.empty((B, N, 4), dtype=torch.float64, device=t.device)
        h = self._handle(max(B, 1))
        st = torch.cuda.current_stream(t.device).cuda_stream
        rc = h.lib.cudampc_linearize_batch(h.ptr, B, C.c_void_p(t.data_ptr()), C.c_void_p(A.data_ptr()),
                                           C.c_void_p(Bm.data_ptr()), C.c_void_p(c.data_ptr()), C.c_void_p(st))
        _lib.check(h.lib, h.ptr, rc, "cudampc_linearize_batch")
        if host:
            return A.cpu().numpy(), Bm.cpu().numpy(), c.cpu().numpy()
        return A, Bm, c


__all__ = ["MPCParameters", "SolverSettings", "MPCController", "BatchResult", "params_array"]
