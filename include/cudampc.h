/* cudampc.h — C ABI of libcudampc.so: batched, B200-native (sm_100a) MPC tracking step of RRT-MPC.
 *
 * The reference has no FFI; its operator API for this path is two Python call signatures.  Each entry
 * point below names the reference interface it replaces (paths relative to /root/reference):
 *
 *   cudampc_linearize_batch   <- vehicle_model.linearize as called by MPCController.solve
 *                                (src/control/vehicle_model.py:24-45, src/control/mpc_controller.py:59-70,108-109)
 *   cudampc_solve_batch[_host] <- MPCController.solve(x0, ref_traj, *, u_init, u_prev) -> (u0, X, U) | (None,)*3
 *                                (src/control/mpc_controller.py:39-141)
 *   cudampc_rollout_batch      <- TrajectoryTracker.track closed loop incl. _solve_with_relaxation
 *                                (src/pipeline/control_stage.py:33-56,74-157; vehicle_model.f_discrete :11-21)
 *   cudampc_track_step_batch   <- one step of that loop with the plant left to the caller (control_stage.py:126-147)
 *   cudampc_build_reference_batch <- build_reference(path, desired_speed, horizon, dt) -> (M,4) rows [x,y,yaw,v_ref]
 *                                (src/control/ref_builder.py:10-22, src/common/geometry.py:9-45)
 *   cudampc_params            <- MPCParameters (src/control/mpc_controller.py:17-30; defaults src/config.py:66-92)
 *   cudampc_settings          <- the hard-coded OSQP settings (src/control/mpc_controller.py:121-131) + OSQP defaults
 *
 * Conventions: every function returns 0 on success and a negative CUDAMPC_ERR_* otherwise; nothing throws
 * or aborts; the message of the last failure on a handle is cudampc_last_error(h).  Per-problem outcomes
 * are in status[] (OSQP integer codes).  Plain pointers and sizes only; buffers are caller-owned.
 * "dev" pointers are CUDA device pointers on the handle's device; "host" pointers are host memory
 * (pinned or pageable).  All arrays are C-contiguous fp64 unless stated.  A handle is bound to one device
 * and is not re-entrant; launches are ordered on `stream` (a cudaStream_t passed as void*, NULL = default).
 */
#ifndef CUDAMPC_H_
#define CUDAMPC_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CUDAMPC_VERSION 100 /* 0.1.0 */

enum {
  CUDAMPC_OK = 0,
  CUDAMPC_ERR_INVALID = -1,     /* bad argument (NULL pointer, batch > max_batch, horizon out of range ...) */
  CUDAMPC_ERR_CUDA = -2,        /* a CUDA runtime call failed; see cudampc_last_error */
  CUDAMPC_ERR_UNSUPPORTED = -3, /* e.g. a horizon whose workspace exceeds 227 KB of shared memory */
  CUDAMPC_ERR_NOMEM = -4
};

/* OSQP status codes used in status[] */
enum {
  CUDAMPC_SOLVED = 1,
  CUDAMPC_SOLVED_INACCURATE = 2,
  CUDAMPC_MAX_ITER_REACHED = -2,
  CUDAMPC_UNSOLVED = -10
};

/* Mirror of MPCParameters, field for field (mpc_controller.py:17-30). Matrices row-major. */
typedef struct cudampc_params {
  double wheelbase_px;
  double dt;
  int32_t horizon;
  int32_t _pad;
  double q[16];          /* 4x4 */
  double r[4];           /* 2x2 */
  double q_terminal[16]; /* 4x4 */
  double u_bounds[4];    /* a_lo, a_hi, delta_lo, delta_hi */
  double v_bounds[2];    /* lo, hi */
  double du_bounds[4];   /* da_lo, da_hi, ddelta_lo, ddelta_hi (per step) */
  double slack_velocity;
  double slack_input;
  double slack_rate;
} cudampc_params;

/* Solver settings. cudampc_default_settings() fills the reference's values (eps 1e-3, max_iter 60000,
 * polish on, adaptive rho, rho 0.1, alpha 1.6) and OSQP's defaults for the rest. */
typedef struct cudampc_settings {
  double eps_abs;
  double eps_rel;
  double rho;
  double alpha;
  double sigma;
  double adaptive_rho_tolerance;
  double rho_eq_factor; /* rho multiplier on equality rows (OSQP: 1e3) */
  double rho_min;
  double rho_max;
  double delta;         /* polish regularisation */
  int32_t max_iter;
  int32_t check_termination;
  int32_t adaptive_rho;
  int32_t adaptive_rho_interval; /* fixed iteration interval (upstream 0.6.x uses a wall-clock heuristic) */
  int32_t polish_passes;         /* 0 = no polish, 1 = OSQP's polish, >1 = re-identify the active set up to n times */
  int32_t polish_refine_iter;
  int32_t warm_start;            /* 1: start from the iterate this handle stored for the same slot in the last call;
                                    0: cold start, the final iterate is stored for a later warm start; -1: stateless - cold
                                    start and nothing is stored per problem (the solver's back-ups of the iterate then stay
                                    in a few L2-resident slots, one per resident problem, instead of 12 KB of HBM per problem) */
  int32_t polish_retry;          /* if OSQP's polish is rejected (active set not identified): resume ADMM at a 10x tighter
                                    internal tolerance and polish again, up to this many times (0 = OSQP behaviour) */
  int32_t early_polish;          /* 1: also try the polish at termination checks whose guessed active set repeated; a polish that
                                    ends on a KKT point of a settled active set finishes the solve early (0 = OSQP behaviour) */
  int32_t early_polish_start;    /* first iteration for such a try (default 50) */
} cudampc_settings;

/* Closed-loop constants of TrajectoryTracker.track (control_stage.py:84,141-150) */
typedef struct cudampc_rollout_cfg {
  int32_t sim_steps;        /* MPCConfig.sim_steps (config.py:70) */
  int32_t relax_on_failure; /* 1: retry a failed solve once with v_ref*0.6 and widened du_bounds (control_stage.py:45-56) */
  double advance_dist2;     /* 25.0 px^2 : path index advances when the new state is farther than this from ref[path_idx] */
  double goal_radius;       /* 8.0 px */
  double relax_v_scale;     /* 0.6 */
  double relax_da;          /* 5.0 */
  double relax_ddelta;      /* 0.05 */
  int32_t* step_ns_dev;     /* optional device array (B, sim_steps) int32: wall time of every closed-loop step of every vehicle
                               in nanoseconds (%globaltimer around window gather + solve (+ retry) + f_discrete + path-index
                               rule + goal test), 0 for steps not run; NULL = not recorded.  What "p99 per-step latency" is measured from. */
} cudampc_rollout_cfg;

typedef struct cudampc_handle cudampc_handle;

int cudampc_version(void);
void cudampc_default_settings(cudampc_settings* s);
void cudampc_default_rollout_cfg(cudampc_rollout_cfg* c);

/* Create a solver for up to max_batch problems of params->horizon stages on CUDA device `device`.
 * Allocates the per-slot HBM workspace (warm-start iterate + polish back-up). */
int cudampc_create(const cudampc_params* params, int max_batch, int device, cudampc_handle** out);
int cudampc_destroy(cudampc_handle* h);
const char* cudampc_last_error(const cudampc_handle* h); /* h may be NULL: message of the last failed create */

/* Replace the parameters (same horizon) — used by the relaxation fallback and by callers that sweep limits. */
int cudampc_set_params(cudampc_handle* h, const cudampc_params* params);

/* (A_k, B_k, c_k), k = 0..N-1, exactly as MPCController.solve linearises them: stage k at the unwrapped
 * reference row max(k-1,0) with ulin = 0.   ref_dev (B,N+1,4) -> A_dev (B,N,4,4), B_dev (B,N,4,2), c_dev (B,N,4). */
int cudampc_linearize_batch(cudampc_handle* h, int batch, const double* ref_dev, double* A_dev, double* B_dev,
                            double* c_dev, void* stream);

/* x_{k+1} = f_discrete(x_k, u_k) (vehicle_model.py:11-21), the integrator of the closed loop, as a parity hook.
 *   x (B,4), u (B,2) -> out (B,4); dt_L (B,2) per-sample (dt, wheelbase_px) or NULL = the handle's parameters. */
int cudampc_f_discrete_batch(cudampc_handle* h, int batch, const double* x_dev, const double* u_dev, const double* dt_L_dev,
                             double* out_dev, void* stream);

/* Solve `batch` independent tracking QPs.  Device pointers.
 *   in : x0 (B,4); ref (B,N+1,4) time-major [x,y,yaw,v]; u_prev (B,2) or NULL (= 0)
 *   out: u0 (B,2); Xp (B,4,N+1) state-major; Up (B,2,N); status (B) int32; iters (B) int32;
 *        pri_res, dua_res (B) or NULL; info (B,4) int32 or NULL = {rho updates, factorisations, accepted polish
 *        passes, triangular solves}.  Problems whose status is not SOLVED/SOLVED_INACCURATE still return their
 *        last iterate; the Python wrapper maps them to (None, None, None) as mpc_controller.py:137-139 does. */
int cudampc_solve_batch(cudampc_handle* h, int batch, const double* x0_dev, const double* ref_dev,
                        const double* u_prev_dev, const cudampc_settings* settings, double* u0_dev, double* Xp_dev,
                        double* Up_dev, int32_t* status_dev, int32_t* iters_dev, double* pri_res_dev,
                        double* dua_res_dev, int32_t* info_dev, void* stream);

/* Same call with HOST buffers: stages inputs through pinned memory, copies H2D, solves, copies D2H and
 * synchronises the stream before returning (what MPCController.solve_batch uses for NumPy arrays). */
int cudampc_solve_batch_host(cudampc_handle* h, int batch, const double* x0, const double* ref, const double* u_prev,
                             const cudampc_settings* settings, double* u0, double* Xp, double* Up, int32_t* status,
                             int32_t* iters, double* pri_res, double* dua_res, int32_t* info, void* stream);

/* build_reference for `batch` polylines (the input producer of the tracker, SURVEY.md 8f row 3).  Device pointers.
 *   in : paths (B, max_pts, 2) with n_pts[b] valid points each; desired_speed = MPCConfig.v_px_s; dt and horizon from params
 *   out: ref (B, ref_stride, 4) rows [x, y, unwrapped yaw, v_ref]; ref_len[b] = rows written, >= horizon+1 (tail padded),
 *        0 for an empty polyline (n_pts[b] < 1);
 *        a path that would need more than ref_stride rows is truncated to ref_stride (ref_len[b] == ref_stride). */
int cudampc_build_reference_batch(cudampc_handle* h, int batch, const double* paths_dev, const int32_t* n_pts_dev, int max_pts,
                                  double desired_speed, double* ref_dev, int32_t* ref_len_dev, int ref_stride, void* stream);

/* Closed-loop tracking of `batch` vehicles for cfg->sim_steps steps without host round trips
 * (TrajectoryTracker.track semantics per vehicle: window gather with tail padding, solve (+relaxation),
 * f_discrete, u_prev carry, path-index rule, goal mask).  Device pointers.
 *   in : ref_global (B, ref_stride, 4) with ref_len[b] valid rows each (build_reference pads to N+1; a vehicle with
 *        ref_len[b] < 1 takes no step and is flagged aborted, where control_stage.py:71-72 raises for an empty path);
 *        state0 (B,4); goal (B,2)
 *   out: states (B, sim_steps, 4) post-step states (rows after a vehicle stops are NaN);
 *        controls (B, sim_steps, 2) or NULL; n_steps (B) int32 = len(TrackingResult.states);
 *        flags (B) int32: bit0 goal reached, bit1 aborted on solver failure, bit2 the relaxation retry ran at least once;
 *        step_status (B, sim_steps) int32 or NULL; step_iters (B, sim_steps) int32 or NULL. */
int cudampc_rollout_batch(cudampc_handle* h, int batch, const double* ref_global_dev, const int32_t* ref_len_dev,
                          int ref_stride, const double* state0_dev, const double* goal_dev,
                          const cudampc_settings* settings, const cudampc_rollout_cfg* cfg, double* states_dev,
                          double* controls_dev, int32_t* n_steps_dev, int32_t* flags_dev, int32_t* step_status_dev,
                          int32_t* step_iters_dev, void* stream);

/* One closed-loop step of `batch` vehicles whose states come from a plant the caller owns (a simulator, a real vehicle, a
 * model with mismatch or noise): the per-step half of cudampc_rollout_batch, one kernel launch per call.  Device pointers.
 *   in : ref_global (B, ref_stride, 4) with ref_len[b] valid rows each, goal (B,2) as for cudampc_rollout_batch;
 *        state (B,4) the measured state of every vehicle;
 *        cfg: relax_on_failure, advance_dist2, goal_radius and relax_* are read (NULL = defaults); sim_steps and step_ns_dev
 *        are not read.
 *   in/out, the tracker state: path_idx (B) int32, u_prev (B,2), n_steps (B) int32, flags (B) int32 (the bits of
 *        cudampc_rollout_batch).  The caller owns these arrays and zeroes them before the first step of a roll-out.
 *   out: u0 (B,2); Xp (B,4,N+1) and Up (B,2,N) as cudampc_solve_batch, or NULL (not returned); status (B), iters (B) int32.
 * Per vehicle: ref_len[b] < 1 sets flags = 2 (aborted) and solves nothing.  A stopped vehicle (flags bit 0 or 1) gets status 0,
 * iters 0 and NaN u0 / Xp / Up, and its tracker state does not change.  From its second step on, the path-index rule and the
 * goal test run on the measured state first (as cudampc_rollout_batch runs them after each step); a vehicle at the goal
 * sets bit 0 and stops there.  Otherwise the window at path_idx is solved from the measured state and u_prev (+ the
 * relaxation retry, bit 2).  On success u0 is carried into u_prev and n_steps grows by one; on failure bit 1 is set and
 * u0 / Xp / Up are NaN (status and iters are those of the failed solve).  With f_discrete as the plant the steps reproduce
 * cudampc_rollout_batch.
 * Warm start (settings->warm_start = 1) uses the iterate the handle stored in slot b, the slot cudampc_solve_batch and
 * cudampc_rollout_batch use for problem b: another call on the same handle between two steps changes the next step's
 * starting point (and iteration count), not the optimum it converges to. */
int cudampc_track_step_batch(cudampc_handle* h, int batch, const double* ref_global_dev, const int32_t* ref_len_dev,
                             int ref_stride, const double* goal_dev, const double* state_dev,
                             const cudampc_settings* settings, const cudampc_rollout_cfg* cfg,
                             int32_t* path_idx_dev, double* u_prev_dev, int32_t* n_steps_dev, int32_t* flags_dev,
                             double* u0_dev, double* Xp_dev, double* Up_dev, int32_t* status_dev, int32_t* iters_dev,
                             void* stream);

/* Introspection used by bench.py / tests: shared-memory doubles per problem, problems resident per SM,
 * number of kernel launches issued by this handle so far. */
int cudampc_workspace_doubles(const cudampc_handle* h);
int cudampc_problems_per_sm(const cudampc_handle* h);
int cudampc_rollout_resident(const cudampc_handle* h);   /* vehicles K_rollout keeps in flight on the device (SMs x resident one-warp CTAs) */
int64_t cudampc_launch_count(const cudampc_handle* h);

/* Measured fp64 FMA throughput of the handle's device (TFLOP/s, ~50 ms of independent DFMA chains): the
 * roofline denominator bench.py reports against (MEASURED_PEAKS.json holds no fp64 figure). < 0 on failure. */
double cudampc_fp64_peak_tflops(cudampc_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* CUDAMPC_H_ */
