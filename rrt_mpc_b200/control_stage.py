"""Drop-in ``TrajectoryTracker`` (closed-loop MPC tracking) with a batched, device-resident entry point.

Mirror of /root/reference/src/pipeline/control_stage.py:26-157:

* ``TrajectoryTracker(mpc, viz)`` dataclass, ``track(planning, maps, *, map_resolution, visualize, occupancy,
  axis) -> TrackingResult`` and ``_solve_with_relaxation(state, reference, u_prev, base_params)`` keep the
  reference's signatures, constants (v0 = 5.0 :84, advance when farther than 25.0 px^2 :141-145, goal radius
  8.0 px :147) and failure behaviour (RuntimeError for a failed/empty plan :69-72; abort on persistent solver
  failure :108-110);
* new ``track_batch`` runs thousands of vehicles for all steps inside one CUDA launch
  (cudampc_rollout_batch): window gather + tail padding, solve with warm start, relaxation retry,
  ``f_discrete``, ``u_prev`` carry, path-index rule and goal mask all stay on the device;
* new ``start_batch`` returns a ``TrackingSession`` whose ``step(states)`` runs one closed-loop step of every vehicle from
  states measured by a plant the caller owns (cudampc_track_step_batch), the tracker state staying on the device.
"""
from __future__ import annotations

import ctypes as C
import logging
from dataclasses import dataclass, field, replace
from typing import Optional, Sequence, Tuple

import numpy as np

from . import _lib
from .config import params_from_config
from .mpc_controller import MPCController, MPCParameters, SolverSettings, params_to_c
from .ref_builder import build_reference
from .vehicle_model import f_discrete

LOG = logging.getLogger(__name__)


@dataclass
class TrackingResult:
    """Trajectory roll-out information returned by the control stage (artifacts.py:34-38)."""
    states: Sequence[np.ndarray] = field(default_factory=list)


@dataclass
class BatchTrackingResult:
    """Per-vehicle roll-outs; ``states[b, :n_steps[b]]`` is what ``TrackingResult.states`` would hold."""
    states: np.ndarray        # (B, T, 4), NaN after a vehicle stopped
    controls: np.ndarray      # (B, T, 2)
    n_steps: np.ndarray       # (B,) int32
    goal_reached: np.ndarray  # (B,) bool
    aborted: np.ndarray       # (B,) bool   (solver failed even after the relaxation retry)
    step_status: np.ndarray   # (B, T) int32 OSQP codes (0 = not run)
    step_iters: np.ndarray    # (B, T) int32
    relaxed: Optional[np.ndarray] = None   # (B,) bool: the relaxation retry (control_stage.py:45-56) ran at least once
    step_ns: Optional[np.ndarray] = None   # (B, T) int32: wall time of every closed-loop step on the device (ns), if recorded

    def result(self, b: int) -> TrackingResult:
        return TrackingResult(states=[self.states[b, t].copy() for t in range(int(self.n_steps[b]))])

    def save_npz(self, path: str) -> None:
        """Telemetry export (the reference keeps only the post-step states, artifacts.py:34-38): every array of the roll-out."""
        np.savez_compressed(path, states=self.states, controls=self.controls, n_steps=self.n_steps, goal_reached=self.goal_reached,
                            aborted=self.aborted, step_status=self.step_status, step_iters=self.step_iters,
                            relaxed=self.relaxed if self.relaxed is not None else np.zeros(len(self.n_steps), bool))

    @staticmethod
    def load_npz(path: str) -> "BatchTrackingResult":
        d = np.load(path)
        keys = ("states", "controls", "n_steps", "goal_reached", "aborted", "step_status", "step_iters", "relaxed")
        return BatchTrackingResult(**{k: d[k] for k in keys if k in d.files})


def initial_state(path, start) -> np.ndarray:
    """control_stage.py:79-84: heading of the first path segment, v0 = 5.0."""
    if len(path) > 1:
        yaw0 = float(np.arctan2(path[1][1] - path[0][1], path[1][0] - path[0][0]))
    else:
        yaw0 = 0.0
    return np.array([start[0], start[1], yaw0, 5.0], dtype=float)


@dataclass
class TrajectoryTracker:
    """Run MPC closed-loop tracking over the planned path."""

    mpc: object                      # MPCConfig (this package's mirror or the reference's)
    viz: object = None               # VizConfig; only read when visualize=True
    settings: Optional[SolverSettings] = None
    device: int = 0

    # -- reference semantics, one vehicle -----------------------------------------------------------
    def _solve_with_relaxation(self, state, reference, u_prev, base_params: MPCParameters):
        controller = self._controller(base_params)
        u0, Xp, Up = controller.solve(state, reference, u_prev=u_prev)
        if u0 is not None:
            return u0, Xp, Up
        LOG.warning("MPC infeasible; applying rate relaxation and speed reduction")
        relaxed_reference = np.array(reference, dtype=float, copy=True)
        relaxed_reference[:, 3] *= 0.6
        relaxed_params = replace(
            base_params,
            du_bounds=((base_params.du_bounds[0][0] - 5.0, base_params.du_bounds[0][1] + 5.0),
                       (base_params.du_bounds[1][0] - 0.05, base_params.du_bounds[1][1] + 0.05)))
        return self._controller(relaxed_params, key="relaxed").solve(state, relaxed_reference, u_prev=u_prev)

    def _controller(self, params: MPCParameters, key: str = "base") -> MPCController:
        cache = self.__dict__.setdefault("_controllers", {})
        fp = bytes(params_to_c(params))          # field-wise fingerprint (dataclass == is ambiguous on ndarray fields)
        hit = cache.get(key)
        if hit is None or hit[0] != fp:
            hit = (fp, MPCController(params, self.settings, device=self.device))
            cache[key] = hit
        return hit[1]

    def track(self, planning, maps, *, map_resolution: float, visualize: bool = True, occupancy=None, axis=None) -> TrackingResult:
        plan = planning.plan
        if not plan.success:
            raise RuntimeError("Planning stage did not succeed; cannot start control stage")
        if not plan.path:
            raise RuntimeError("Planner returned an empty path")
        base_params = params_from_config(self.mpc, map_resolution)
        horizon, wheelbase_px = base_params.horizon, base_params.wheelbase_px
        path = plan.path
        state = initial_state(path, maps.start)
        u_prev = np.zeros(2)
        ref_global = build_reference(path, self.mpc.v_px_s, horizon, self.mpc.dt)
        LOG.info("Starting MPC tracking (sim_steps=%d, horizon=%d, reference_points=%d)", self.mpc.sim_steps, horizon, len(ref_global))
        plot = _reference_plotter() if (visualize and occupancy is not None) else None
        states: list = []
        path_idx, goal_reached = 0, False
        for step in range(self.mpc.sim_steps):
            window = ref_global[path_idx:min(path_idx + horizon + 1, len(ref_global))]
            if len(window) < horizon + 1:
                window = np.vstack((window, np.repeat(window[-1:], horizon + 1 - len(window), axis=0)))
            u0, Xp, _ = self._solve_with_relaxation(state, window, u_prev, base_params)
            if u0 is None or Xp is None:
                LOG.error("MPC remained infeasible at step %d; aborting tracking", step)
                break
            if plot is not None:
                plot(occupancy, path, Xp, state, step, self.viz, axis, wheelbase_px, u0)
            state = f_discrete(state, u0, self.mpc.dt, wheelbase_px)
            states.append(state.copy())
            u_prev = u0.copy()
            if path_idx < len(ref_global) - 2:
                dx, dy = state[0] - ref_global[path_idx][0], state[1] - ref_global[path_idx][1]
                if dx * dx + dy * dy > 25.0:
                    path_idx += 1
            if np.hypot(state[0] - maps.goal[0], state[1] - maps.goal[1]) < 8.0:
                LOG.info("Reached goal region at step %d", step)
                goal_reached = True
                break
        LOG.info("MPC tracking finished after %d steps (goal_reached=%s)", len(states), goal_reached)
        return TrackingResult(states=states)

    # -- batched, device-resident closed loop ---------------------------------------------------------
    def _references(self, ctl: MPCController, paths, ref_globals, build_on_device: bool):
        """The global references of a batch on ``ctl``'s device: ``(ref (B, stride, 4), ref_len (B,), stride)``."""
        import torch
        N = ctl.params.horizon
        if ref_globals is None and build_on_device:
            # the reference's build_reference (ref_builder.py:10-22) for all paths in one launch (K_ref)
            d_ref, d_len = ctl.build_reference_batch(paths, float(self.mpc.v_px_s))
            return d_ref, d_len, int(d_ref.shape[1])
        if ref_globals is None:
            if any(len(p) < 1 for p in paths):
                raise RuntimeError("Planner returned an empty path")   # control_stage.py:71-72
            ref_globals = [build_reference(p, self.mpc.v_px_s, N, self.mpc.dt) for p in paths]
        B = len(ref_globals)
        if any(len(r) < 1 for r in ref_globals):
            raise RuntimeError("Planner returned an empty path")
        lens = np.array([len(r) for r in ref_globals], dtype=np.int32)
        stride = int(lens.max())
        refg = np.zeros((B, stride, 4))
        for b, r in enumerate(ref_globals):
            refg[b, :len(r)] = r
        dev = torch.device("cuda", self.device)
        return torch.as_tensor(refg).to(dev), torch.as_tensor(lens).to(dev), stride

    def track_batch(self, paths: Sequence, starts, goals, *, map_resolution: float, sim_steps: Optional[int] = None,
                    ref_globals: Optional[Sequence[np.ndarray]] = None, states0=None, warm_start: bool = True,
                    relax_on_failure: bool = True, build_on_device: bool = True, record_step_time: bool = False) -> BatchTrackingResult:
        """Track ``B`` vehicles. ``paths[b]`` is a polyline (as ``PlanResult.path``); ``starts``/``goals`` are
        ``(B,2)``.  Alternatively pass prebuilt ``ref_globals`` (each ``(M_b,4)``) and ``states0 (B,4)``."""
        import torch
        params = params_from_config(self.mpc, map_resolution)
        T = int(self.mpc.sim_steps if sim_steps is None else sim_steps)
        dev = torch.device("cuda", self.device)
        t = lambda a: torch.as_tensor(a).to(dev)
        ctl = self._controller(params, key="rollout")
        d_ref, d_len, stride = self._references(ctl, paths, ref_globals, build_on_device)
        B = int(d_ref.shape[0])
        if states0 is None:
            states0 = np.stack([initial_state(paths[b], starts[b]) for b in range(B)])
        states0 = np.ascontiguousarray(states0, dtype=np.float64).reshape(B, 4)
        goals = np.ascontiguousarray(goals, dtype=np.float64).reshape(B, 2)
        d_s0, d_goal = t(states0), t(goals)
        d_states = torch.empty((B, T, 4), dtype=torch.float64, device=dev)
        d_ctrl = torch.empty((B, T, 2), dtype=torch.float64, device=dev)
        d_n = torch.empty(B, dtype=torch.int32, device=dev)
        d_fl = torch.empty(B, dtype=torch.int32, device=dev)
        d_st = torch.empty((B, T), dtype=torch.int32, device=dev)
        d_it = torch.empty((B, T), dtype=torch.int32, device=dev)
        h = ctl._handle(B)
        s = replace(self.settings or SolverSettings(), warm_start=warm_start).to_c()
        cfg = _lib.RolloutCfg()
        h.lib.cudampc_default_rollout_cfg(C.byref(cfg))
        cfg.sim_steps, cfg.relax_on_failure = T, int(relax_on_failure)
        d_ns = torch.zeros((B, T), dtype=torch.int32, device=dev) if record_step_time else None
        cfg.step_ns_dev = d_ns.data_ptr() if d_ns is not None else None
        p = lambda x: C.c_void_p(x.data_ptr())
        rc = h.lib.cudampc_rollout_batch(h.ptr, B, p(d_ref), p(d_len), stride, p(d_s0), p(d_goal), C.byref(s), C.byref(cfg),
                                         p(d_states), p(d_ctrl), p(d_n), p(d_fl), p(d_st), p(d_it),
                                         C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
        _lib.check(h.lib, h.ptr, rc, "cudampc_rollout_batch")
        torch.cuda.synchronize(dev)
        flags = d_fl.cpu().numpy()
        return BatchTrackingResult(states=d_states.cpu().numpy(), controls=d_ctrl.cpu().numpy(), n_steps=d_n.cpu().numpy(),
                                   goal_reached=(flags & 1).astype(bool), aborted=(flags & 2).astype(bool),
                                   step_status=d_st.cpu().numpy(), step_iters=d_it.cpu().numpy(), relaxed=(flags & 4).astype(bool),
                                   step_ns=d_ns.cpu().numpy() if d_ns is not None else None)

    # -- one closed-loop step per call, the plant outside -----------------------------------------------
    def start_batch(self, paths: Optional[Sequence], starts, goals, *, map_resolution: float,
                    ref_globals: Optional[Sequence[np.ndarray]] = None, states0=None, warm_start: bool = True,
                    relax_on_failure: bool = True, build_on_device: bool = True) -> "TrackingSession":
        """Start tracking ``B`` vehicles whose states come from a plant the caller owns (a simulator, a real vehicle, a model
        with mismatch or noise).  References, starts and goals as ``track_batch``; ``session.step(states)`` then runs one
        closed-loop step of every vehicle in one launch (cudampc_track_step_batch).  ``session.states0`` is the initial state
        of every vehicle (``initial_state`` of its path unless ``states0`` is given), the plant's first input."""
        import torch
        params = params_from_config(self.mpc, map_resolution)
        # the session's own handle: nobody else reuses the warm-start slots of its vehicles between steps
        B = len(ref_globals) if ref_globals is not None else len(paths)
        ctl = MPCController(params, self.settings, device=self.device, max_batch=max(B, 1))
        d_ref, d_len, stride = self._references(ctl, paths, ref_globals, build_on_device)
        if states0 is None:
            states0 = np.stack([initial_state(paths[b], starts[b]) for b in range(B)]) if B else np.zeros((0, 4))
        states0 = np.ascontiguousarray(states0, dtype=np.float64).reshape(B, 4)
        goals = np.ascontiguousarray(goals, dtype=np.float64).reshape(B, 2)
        s = replace(self.settings or SolverSettings(), warm_start=warm_start).to_c()
        cfg = _lib.RolloutCfg()
        _lib.load().cudampc_default_rollout_cfg(C.byref(cfg))
        cfg.relax_on_failure = int(relax_on_failure)
        return TrackingSession(ctl, d_ref, d_len, stride, torch.as_tensor(goals).to(d_ref.device), states0, s, cfg)


@dataclass
class StepResult:
    """What one ``TrackingSession.step`` returns (CUDA tensors for CUDA input, NumPy arrays for NumPy input).  A vehicle that
    did not step (stopped before, at the goal now, or the solve failed) has NaN ``u0``, ``Xp`` and ``Up``; ``status`` is 0
    when no solve ran."""
    u0: object       # (B,2)
    Xp: object       # (B,4,N+1) state-major predicted trajectory
    Up: object       # (B,2,N)
    status: object   # (B,) int32 OSQP codes
    iters: object    # (B,) int32


class TrackingSession:
    """The tracker state of ``B`` vehicles on the device between the steps of an external plant (``TrajectoryTracker.start_batch``).

    ``path_idx``, ``u_prev``, ``n_steps`` and the flag views are CUDA tensors; reading them does not synchronise."""

    def __init__(self, ctl: MPCController, ref, ref_len, stride: int, goals, states0: np.ndarray, settings: _lib.Settings,
                 cfg: _lib.RolloutCfg):
        import torch
        self.controller, self._ref, self._ref_len, self._stride, self._goals = ctl, ref, ref_len, int(stride), goals
        self._settings, self._cfg = settings, cfg
        self.states0 = states0
        self.batch = B = int(ref.shape[0])
        self.horizon = N = ctl.params.horizon
        dev = self.device = ref.device
        self.path_idx = torch.zeros(B, dtype=torch.int32, device=dev)
        self.u_prev = torch.zeros((B, 2), dtype=torch.float64, device=dev)
        self.n_steps = torch.zeros(B, dtype=torch.int32, device=dev)
        self.flags = torch.zeros(B, dtype=torch.int32, device=dev)   # bit0 goal reached, bit1 aborted, bit2 relaxation ran
        self._h = ctl._handle(max(B, 1))

    @property
    def goal_reached(self):
        return (self.flags & 1) != 0

    @property
    def aborted(self):
        return (self.flags & 2) != 0

    @property
    def relaxed(self):
        return (self.flags & 4) != 0

    @property
    def active(self):
        return (self.flags & 3) == 0

    def launch_count(self) -> int:
        return self.controller.launch_count()

    def step(self, states) -> StepResult:
        """One closed-loop step of every vehicle from its measured ``states (B,4)``.  A contiguous CUDA float64 tensor on the
        session's device: asynchronous on the current stream, CUDA tensors out.  A NumPy float64 array: copied in, synchronised,
        NumPy out."""
        import torch
        B, N = self.batch, self.horizon
        host = isinstance(states, np.ndarray)
        if host:
            if states.shape != (B, 4) or states.dtype != np.float64:
                raise ValueError(f"states: expected a float64 array of shape ({B}, 4); got {states.dtype} {states.shape}")
            x = torch.as_tensor(np.ascontiguousarray(states)).to(self.device)
        elif isinstance(states, torch.Tensor):
            if tuple(states.shape) != (B, 4) or states.dtype != torch.float64 or states.device != self.device or not states.is_contiguous():
                raise ValueError(f"states: expected a contiguous float64 tensor of shape ({B}, 4) on {self.device}; "
                                 f"got {states.dtype} {tuple(states.shape)} on {states.device}")
            x = states
        else:
            raise ValueError(f"states: expected a NumPy array or a CUDA tensor; got {type(states).__name__}")
        e = lambda *shape, dt=torch.float64: torch.empty(shape, dtype=dt, device=self.device)
        out = StepResult(e(B, 2), e(B, 4, N + 1), e(B, 2, N), e(B, dt=torch.int32), e(B, dt=torch.int32))
        if B:
            h = self._h
            p = lambda t: C.c_void_p(t.data_ptr())
            rc = h.lib.cudampc_track_step_batch(h.ptr, B, p(self._ref), p(self._ref_len), self._stride, p(self._goals), p(x),
                                                C.byref(self._settings), C.byref(self._cfg), p(self.path_idx), p(self.u_prev),
                                                p(self.n_steps), p(self.flags), p(out.u0), p(out.Xp), p(out.Up), p(out.status),
                                                p(out.iters), C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream))
            _lib.check(h.lib, h.ptr, rc, "cudampc_track_step_batch")
        if host:
            return StepResult(*(t.cpu().numpy() for t in (out.u0, out.Xp, out.Up, out.status, out.iters)))
        return out

    def close(self) -> None:
        self.controller.close()


def _reference_plotter():
    """The reference's own plotting (src/viz, untouched) when this module is dropped into the reference tree."""
    try:  # pragma: no cover - needs matplotlib and the reference package
        from src.viz.vehicle_draw import VehicleParams
        from src.viz.visualization import plot_prediction
    except Exception:
        LOG.info("reference viz modules not importable; tracking without plots")
        return None

    def plot(occupancy, path, Xp, state, step, viz, axis, wheelbase_px, u0):  # pragma: no cover
        plot_prediction(occupancy, path, Xp, state, step, getattr(viz, "prediction_pause", 0.01), ax=axis,
                        vehicle_params=VehicleParams.from_wheelbase(wheelbase_px), control=u0)
    return plot


__all__ = ["TrajectoryTracker", "TrackingResult", "BatchTrackingResult", "TrackingSession", "StepResult", "initial_state"]
