"""rrt_mpc_b200 — B200-native (sm_100a) batched MPC tracking step for RRT-MPC.

Host-side mirror of the reference's operator interface for this path
(``MPCParameters`` / ``MPCController.solve`` / ``TrajectoryTracker.track``) over the C ABI of
``libcudampc.so`` (include/cudampc.h).  Importing the package does not load CUDA; the first solver call
does, and fails loudly if the library or the GPU is missing."""
from .config import MPCConfig, VizConfig
from .control_stage import BatchTrackingResult, StepResult, TrackingResult, TrackingSession, TrajectoryTracker
from .mpc_controller import BatchResult, MPCController, MPCParameters, SolverSettings, params_array
from .ref_builder import build_reference
from .vehicle_model import f_discrete, linearize

__all__ = ["MPCConfig", "VizConfig", "MPCParameters", "SolverSettings", "MPCController", "BatchResult", "params_array",
           "TrajectoryTracker", "TrackingResult", "BatchTrackingResult", "TrackingSession", "StepResult",
           "build_reference", "f_discrete", "linearize"]
