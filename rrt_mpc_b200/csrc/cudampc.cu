// cudampc.cu — libcudampc.so: CUDA kernels (sm_100a) + C ABI (include/cudampc.h).
//
// A group of warps (one warp up to horizon ~80, two beyond) owns one tracking problem; the whole problem (ADMM
// iterate, linearisation, banded LDL' factor, right-hand side) lives in shared memory for the entire solve
// (DESIGN.md §3).  Stage-parallel phases run with lanes striding over the N+1 stages; the banded factorisation /
// triangular sweeps are the sequential chain (twisted: two lanes, one per half of the horizon).  One CTA per SM
// holds as many groups as shared memory allows; groups are independent of each other and fetch problems from a
// global counter, so a launch is persistent: grid = SMs regardless of the batch size.
//
// There is no CPU fallback: every entry point fails with CUDAMPC_ERR_CUDA if the device is unusable.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <new>

#include "../../include/cudampc.h"
#include "mpc_kernels.cuh"

using namespace mpc;

// ------------------------------------------------------------------------------------------------
// K_lin: batched linearisation hook (parity at 1e-12 against vehicle_model.linearize)
// ------------------------------------------------------------------------------------------------
__global__ void mpc_linearize_kernel(Params p, int batch, const double* ref, double* A, double* Bm, double* c) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int N = p.N;
  double* uy = smem + (size_t)wid * (N + 1);
  for (int b = blockIdx.x * wpb + wid; b < batch; b += gridDim.x * wpb) {
    RefWin rw{ref + (size_t)4 * (N + 1) * b, 0, N + 1, 1.0};
    if (lane == 0) unwrap_window(rw, N + 1, uy);
    __syncwarp();
    for (int k = lane; k < N; k += 32) {
      int kl = k > 0 ? k - 1 : 0;
      const double* r = rw.row(kl);
      double lin[7];
      linearize_point(p, r[0], r[1], uy[kl], r[3], lin);
      double* a = A + ((size_t)b * N + k) * 16;
      double* bm = Bm + ((size_t)b * N + k) * 8;
      double* cc = c + ((size_t)b * N + k) * 4;
#pragma unroll
      for (int i = 0; i < 16; ++i) a[i] = 0.0;
#pragma unroll
      for (int i = 0; i < 8; ++i) bm[i] = 0.0;
      a[0] = a[5] = a[10] = a[15] = 1.0;
      a[2] = lin[0]; a[3] = lin[1]; a[6] = lin[2]; a[7] = lin[3];
      bm[5] = lin[4]; bm[6] = p.dt;
      cc[0] = lin[5]; cc[1] = lin[6]; cc[2] = 0.0; cc[3] = 0.0;
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------
// K_f: batched f_discrete hook (parity at 1e-12 against vehicle_model.f_discrete, vehicle_model.py:11-21); the very
// function the closed loop integrates with.  dt_L: optional per-sample (dt, wheelbase_px) pairs, else the handle's.
// ------------------------------------------------------------------------------------------------
__global__ void mpc_f_discrete_kernel(double dt0, double L0, int batch, const double* x, const double* u, const double* dt_L, double* out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  const double dt = dt_L ? dt_L[2 * (size_t)b] : dt0;
  const double L = dt_L ? dt_L[2 * (size_t)b + 1] : L0;
  double o[4];
  f_discrete_vals(dt, L, x + 4 * (size_t)b, u + 2 * (size_t)b, o);
#pragma unroll
  for (int i = 0; i < 4; ++i) out[4 * (size_t)b + i] = o[i];
}

// ------------------------------------------------------------------------------------------------
// K_ref: batched build_reference (src/control/ref_builder.py:10-22 + src/common/geometry.py:9-45), one thread per path:
// arc-length resampling at step = max(2, 0.8 v dt) (np.arange + np.isclose end rule, np.interp two-pointer walk),
// heading of successive differences with np.unwrap (first heading = atan2(0,0) = 0), curvature slow-down,
// tail padding to horizon+1 rows.  Products/sums are written with explicit _rn intrinsics so that no fma contraction
// changes the rounding of np.interp's  slope*(x - xp[j]) + fp[j].
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double interp_np(double x, double x0, double x1, double f0, double f1) {
  if (x == x0) return f0;
  const double slope = __ddiv_rn(__dsub_rn(f1, f0), __dsub_rn(x1, x0));
  return __dadd_rn(__dmul_rn(slope, __dsub_rn(x, x0)), f0);
}
__global__ void mpc_build_reference_kernel(int batch, const double* paths, const int* n_pts, int max_pts, double v, double dt, int N,
                                           double* ref, int* ref_len, int stride) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  const double PI = 3.141592653589793;
  const double* P = paths + (size_t)2 * max_pts * b;
  double* R = ref + (size_t)4 * stride * b;
  const int n = n_pts[b];
  if (n < 1) { ref_len[b] = 0; return; }                   // empty polyline: no reference (the tracker flags such a vehicle as aborted)
  const double step = fmax(2.0, 0.8 * v * dt);
  // total arc length (sequential cumsum, as np.cumsum)
  double total = 0.0;
  for (int i = 1; i < n; ++i) total = __dadd_rn(total, hypot(P[2 * i] - P[2 * i - 2], P[2 * i + 1] - P[2 * i - 1]));
  int M = 0;
  if (n < 2 || total < 1e-9) {
    M = n < stride ? n : stride;
    for (int i = 0; i < M; ++i) { R[4 * i] = P[2 * i]; R[4 * i + 1] = P[2 * i + 1]; }
  } else {
    int na = (int)ceil(total / step);                      // len(np.arange(0, total, step))
    const double last = __dmul_rn((double)(na - 1), step);
    const bool close = fabs(last - total) <= 1e-8 + 1e-5 * fabs(total);   // np.isclose(samples[-1], total)
    M = close ? na : na + 1;
    if (M > stride) M = stride;
    int j = 0;                                             // current segment [s0, s1]
    double s0 = 0.0, s1 = hypot(P[2] - P[0], P[3] - P[1]);
    for (int i = 0; i < M; ++i) {
      const double x = (i < na) ? __dmul_rn((double)i, step) : total;
      while (j + 1 < n - 1 && x >= s1) {                   // np.interp: xp[j] <= x < xp[j+1]
        ++j; s0 = s1;
        s1 = __dadd_rn(s1, hypot(P[2 * j + 2] - P[2 * j], P[2 * j + 3] - P[2 * j + 1]));
      }
      if (x >= s1) { R[4 * i] = P[2 * (n - 1)]; R[4 * i + 1] = P[2 * (n - 1) + 1]; }       // x == xp[-1]
      else { R[4 * i] = interp_np(x, s0, s1, P[2 * j], P[2 * j + 2]); R[4 * i + 1] = interp_np(x, s0, s1, P[2 * j + 1], P[2 * j + 3]); }
    }
  }
  // heading (first difference is the zero vector), np.unwrap, slow-down
  double prev_raw = 0.0, cum = 0.0, prev_un = 0.0;
  for (int i = 0; i < M; ++i) {
    const double dx = i ? R[4 * i] - R[4 * i - 4] : 0.0, dy = i ? R[4 * i + 1] - R[4 * i - 3] : 0.0;
    const double raw = atan2(dy, dx);
    if (i) {
      const double dd = raw - prev_raw;
      double ddmod = np_mod(dd + PI, 2.0 * PI) - PI;
      if (ddmod == -PI && dd > 0.0) ddmod = PI;
      double corr = ddmod - dd;
      if (fabs(dd) < PI) corr = 0.0;
      cum += corr;
    }
    const double un = raw + cum;
    double hd = i ? fabs(un - prev_un) : 0.0;
    hd = fmin(hd, PI - hd);
    R[4 * i + 2] = un;
    R[4 * i + 3] = v * (0.6 + 0.4 * (1.0 / (1.0 + 4.0 * hd)));
    prev_raw = raw; prev_un = un;
  }
  int len = M;
  for (; len < N + 1 && len < stride; ++len)
    for (int c = 0; c < 4; ++c) R[4 * len + c] = R[4 * (M - 1) + c];
  ref_len[b] = len;
}

// ------------------------------------------------------------------------------------------------
// fp64 pipe peak (roofline denominator measured on the device the solver runs on)
// ------------------------------------------------------------------------------------------------
__global__ void fp64_peak_kernel(double* out, int iters, double a, double b) {
  double acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = threadIdx.x * 1e-3 + i;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = fma(acc[i], a, b);
  }
  double sum = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) sum += acc[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = sum;
}

// ------------------------------------------------------------------------------------------------
// Handle + C ABI
// ------------------------------------------------------------------------------------------------
struct cudampc_handle {
  int device, max_batch, N;
  Params p;
  double *warm, *scratch, *work, *fsave;   // fsave: the ADMM factor of every resident group while a polish uses its place
  int* counter;
  // staging for the host-pointer entry point
  double *h_in, *h_out, *d_in, *d_out;
  size_t in_doubles, out_doubles;
  int sms, smem_bytes, roll_per_sm;   // K_rollout: one-warp CTAs of smem_bytes each, roll_per_sm resident per SM
  int grp_P, grp_wpp, grp_smem;        // K_solve: one CTA per SM with grp_P groups of grp_wpp warps
  int variant;                         // SolveVariant
  // per-problem-parameter kernels (the *_params entry points), configured on first use: a Params slot per group / CTA on top of
  // the shared-parameter layout, so at most as many groups and resident CTAs as above (the allocations are sized for those)
  bool pp_ready;
  int pp_P, pp_smem, pp_roll_per_sm, pp_roll_smem;
  int form;                            // form of the ADMM phases (mpc_solve.h FORM_*): K_solve one-warp groups, K_rollout
  unsigned long long* tags;            // dev builds (MPC_TIMING): per-tag cycle counters
  long long launches;
  char err[512];
};

static char g_create_err[512] = "";

// launchers of the kernel instantiations (mpc_kernels_tu.cu, one translation unit each)
cudaError_t solve_set_smem_0(int), solve_set_smem_1(int), solve_set_smem_2(int), solve_set_smem_3(int), solve_set_smem_4(int), solve_set_smem_5(int);
void solve_launch_0(int, int, int, cudaStream_t, const Params&, const Settings&, const BatchArgs&, int, int);
void solve_launch_1(int, int, int, cudaStream_t, const Params&, const Settings&, const BatchArgs&, int, int);
void solve_launch_2(int, int, int, cudaStream_t, const Params&, const Settings&, const BatchArgs&, int, int);
void solve_launch_3(int, int, int, cudaStream_t, const Params&, const Settings&, const BatchArgs&, int, int);
void solve_launch_4(int, int, int, cudaStream_t, const Params&, const Settings&, const BatchArgs&, int, int);
void solve_launch_5(int, int, int, cudaStream_t, const Params&, const Settings&, const BatchArgs&, int, int);
int solve_reg_max_threads_4();
cudaError_t rollout_set_smem_short(int), rollout_set_smem_general(int), rollout_set_smem_pair(int);
cudaError_t rollout_occupancy_short(int, int*), rollout_occupancy_general(int, int*), rollout_occupancy_pair(int, int*);
void rollout_launch_short(int, int, cudaStream_t, const Params&, const Settings&, const cudampc_rollout_cfg&, const RolloutArgs&);
void rollout_launch_general(int, int, cudaStream_t, const Params&, const Settings&, const cudampc_rollout_cfg&, const RolloutArgs&);
void rollout_launch_pair(int, int, cudaStream_t, const Params&, const Settings&, const cudampc_rollout_cfg&, const RolloutArgs&);
cudaError_t step_set_smem_short(int), step_set_smem_general(int), step_set_smem_pair(int);
void step_launch_short(int, int, cudaStream_t, const Params&, const Settings&, const cudampc_rollout_cfg&, const StepArgs&);
void step_launch_general(int, int, cudaStream_t, const Params&, const Settings&, const cudampc_rollout_cfg&, const StepArgs&);
void step_launch_pair(int, int, cudaStream_t, const Params&, const Settings&, const cudampc_rollout_cfg&, const StepArgs&);
// the per-problem-parameter instantiations (mpc_kernels_tu.cu 9..17)
cudaError_t solve_set_smem_pp0(int), solve_set_smem_pp1(int), solve_set_smem_pp2(int), solve_set_smem_pp3(int), solve_set_smem_pp4(int), solve_set_smem_pp5(int);
void solve_launch_pp0(int, int, int, cudaStream_t, const Params&, const Settings&, const BatchArgs&, int, int);
void solve_launch_pp1(int, int, int, cudaStream_t, const Params&, const Settings&, const BatchArgs&, int, int);
void solve_launch_pp2(int, int, int, cudaStream_t, const Params&, const Settings&, const BatchArgs&, int, int);
void solve_launch_pp3(int, int, int, cudaStream_t, const Params&, const Settings&, const BatchArgs&, int, int);
void solve_launch_pp4(int, int, int, cudaStream_t, const Params&, const Settings&, const BatchArgs&, int, int);
void solve_launch_pp5(int, int, int, cudaStream_t, const Params&, const Settings&, const BatchArgs&, int, int);
cudaError_t rollout_set_smem_pp_short(int), rollout_set_smem_pp_general(int), rollout_set_smem_pp_pair(int);
cudaError_t rollout_occupancy_pp_short(int, int*), rollout_occupancy_pp_general(int, int*), rollout_occupancy_pp_pair(int, int*);
void rollout_launch_pp_short(int, int, cudaStream_t, const Params&, const Settings&, const cudampc_rollout_cfg&, const RolloutArgs&);
void rollout_launch_pp_general(int, int, cudaStream_t, const Params&, const Settings&, const cudampc_rollout_cfg&, const RolloutArgs&);
void rollout_launch_pp_pair(int, int, cudaStream_t, const Params&, const Settings&, const cudampc_rollout_cfg&, const RolloutArgs&);
cudaError_t step_set_smem_pp_short(int), step_set_smem_pp_general(int), step_set_smem_pp_pair(int);
void step_launch_pp_short(int, int, cudaStream_t, const Params&, const Settings&, const cudampc_rollout_cfg&, const StepArgs&);
void step_launch_pp_general(int, int, cudaStream_t, const Params&, const Settings&, const cudampc_rollout_cfg&, const StepArgs&);
void step_launch_pp_pair(int, int, cudaStream_t, const Params&, const Settings&, const cudampc_rollout_cfg&, const StepArgs&);

typedef void (*SolveLaunchFn)(int, int, int, cudaStream_t, const Params&, const Settings&, const BatchArgs&, int, int);
static cudaError_t (*const k_solve_set_smem[2][6])(int) = {
  {solve_set_smem_0, solve_set_smem_1, solve_set_smem_2, solve_set_smem_3, solve_set_smem_4, solve_set_smem_5},
  {solve_set_smem_pp0, solve_set_smem_pp1, solve_set_smem_pp2, solve_set_smem_pp3, solve_set_smem_pp4, solve_set_smem_pp5}};
static const SolveLaunchFn k_solve_launch[2][6] = {
  {solve_launch_0, solve_launch_1, solve_launch_2, solve_launch_3, solve_launch_4, solve_launch_5},
  {solve_launch_pp0, solve_launch_pp1, solve_launch_pp2, solve_launch_pp3, solve_launch_pp4, solve_launch_pp5}};
cudaError_t solve_set_smem(int v, int bytes, bool pp) { return k_solve_set_smem[pp][v < 5 ? v : 5](bytes); }
void solve_launch(int v, int grid, int threads, int smem, cudaStream_t st, const Params& p, const Settings& s, const BatchArgs& a, int P, int F, bool pp) {
  k_solve_launch[pp][v < 5 ? v : 5](grid, threads, smem, st, p, s, a, P, F);
}
cudaError_t rollout_set_smem(int f, int bytes, bool pp) {
  if (pp) return f == FORM_SHORT ? rollout_set_smem_pp_short(bytes) : f == FORM_PAIR ? rollout_set_smem_pp_pair(bytes) : rollout_set_smem_pp_general(bytes);
  return f == FORM_SHORT ? rollout_set_smem_short(bytes) : f == FORM_PAIR ? rollout_set_smem_pair(bytes) : rollout_set_smem_general(bytes);
}
cudaError_t rollout_occupancy(int f, int bytes, int* n, bool pp) {
  if (pp) return f == FORM_SHORT ? rollout_occupancy_pp_short(bytes, n) : f == FORM_PAIR ? rollout_occupancy_pp_pair(bytes, n) : rollout_occupancy_pp_general(bytes, n);
  return f == FORM_SHORT ? rollout_occupancy_short(bytes, n) : f == FORM_PAIR ? rollout_occupancy_pair(bytes, n) : rollout_occupancy_general(bytes, n);
}
void rollout_launch(int f, int grid, int smem, cudaStream_t st, const Params& p, const Settings& s, const cudampc_rollout_cfg& cfg, const RolloutArgs& a, bool pp) {
  if (pp) {
    if (f == FORM_SHORT) rollout_launch_pp_short(grid, smem, st, p, s, cfg, a);
    else if (f == FORM_PAIR) rollout_launch_pp_pair(grid, smem, st, p, s, cfg, a);
    else rollout_launch_pp_general(grid, smem, st, p, s, cfg, a);
  } else if (f == FORM_SHORT) rollout_launch_short(grid, smem, st, p, s, cfg, a);
  else if (f == FORM_PAIR) rollout_launch_pair(grid, smem, st, p, s, cfg, a);
  else rollout_launch_general(grid, smem, st, p, s, cfg, a);
}
cudaError_t step_set_smem(int f, int bytes, bool pp) {
  if (pp) return f == FORM_SHORT ? step_set_smem_pp_short(bytes) : f == FORM_PAIR ? step_set_smem_pp_pair(bytes) : step_set_smem_pp_general(bytes);
  return f == FORM_SHORT ? step_set_smem_short(bytes) : f == FORM_PAIR ? step_set_smem_pair(bytes) : step_set_smem_general(bytes);
}
void step_launch(int f, int grid, int smem, cudaStream_t st, const Params& p, const Settings& s, const cudampc_rollout_cfg& cfg, const StepArgs& a, bool pp) {
  if (pp) {
    if (f == FORM_SHORT) step_launch_pp_short(grid, smem, st, p, s, cfg, a);
    else if (f == FORM_PAIR) step_launch_pp_pair(grid, smem, st, p, s, cfg, a);
    else step_launch_pp_general(grid, smem, st, p, s, cfg, a);
  } else if (f == FORM_SHORT) step_launch_short(grid, smem, st, p, s, cfg, a);
  else if (f == FORM_PAIR) step_launch_pair(grid, smem, st, p, s, cfg, a);
  else step_launch_general(grid, smem, st, p, s, cfg, a);
}

// Every entry point runs on the handle's device and leaves the caller's current device as it found it.
struct DeviceGuard {
  int prev = -1; bool switched = false; cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int dev) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != dev) { err = cudaSetDevice(dev); switched = (err == cudaSuccess); }
  }
  ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};
#define ON_DEVICE(h) DeviceGuard guard_((h)->device); CU(h, guard_.err)

static int fail(cudampc_handle* h, int code, const char* fmt, const char* detail) {
  char* dst = h ? h->err : g_create_err;
  snprintf(dst, 512, fmt, detail ? detail : "");
  return code;
}
#define CU(h, call)                                                                         \
  do {                                                                                      \
    cudaError_t e_ = (call);                                                                \
    if (e_ != cudaSuccess) {                                                                \
      char buf_[400];                                                                       \
      snprintf(buf_, sizeof buf_, "%s -> %s", #call, cudaGetErrorString(e_));              \
      return fail(h, CUDAMPC_ERR_CUDA, "CUDA failure: %s", buf_);                          \
    }                                                                                       \
  } while (0)

static int convert_params(const cudampc_params* in, Params* p, cudampc_handle* h) {
  if (!in) return fail(h, CUDAMPC_ERR_INVALID, "%s", "params is NULL");
  static const char* const why[] = {"", "horizon must be in [1, 256]", "dt and wheelbase_px must be > 0",
                                    "q must be positive semidefinite and non-zero", "q_terminal must be positive semidefinite and non-zero",
                                    "r must be positive semidefinite and non-zero", "slack weights must be > 0"};
  const int rc = params_from_c(in, p);
  return rc == PARAMS_OK ? CUDAMPC_OK : fail(h, CUDAMPC_ERR_INVALID, "%s", why[rc]);
}

static int convert_settings(const cudampc_settings* in, Settings* s, cudampc_handle* h) {
  cudampc_settings d;
  if (!in) { cudampc_default_settings(&d); in = &d; }
  if (!(in->eps_abs >= 0.0) || !(in->eps_rel >= 0.0) || !(in->rho > 0.0) || !(in->alpha > 0.0 && in->alpha < 2.0) ||
      !(in->sigma > 0.0) || in->max_iter < 1 || !(in->delta > 0.0))
    return fail(h, CUDAMPC_ERR_INVALID, "%s", "settings out of range");
  if (!(in->rho_min > 0.0) || !(in->rho_max >= in->rho_min) || !(in->rho_eq_factor > 0.0) || !(in->adaptive_rho_tolerance >= 1.0) ||
      in->check_termination < 0 || in->adaptive_rho_interval < 0 || in->polish_passes < 0 || in->polish_refine_iter < 0)
    return fail(h, CUDAMPC_ERR_INVALID, "%s", "settings out of range (rho_min > 0, rho_max >= rho_min, rho_eq_factor > 0, adaptive_rho_tolerance >= 1, intervals >= 0)");
  s->eps_abs = in->eps_abs; s->eps_rel = in->eps_rel; s->rho0 = in->rho; s->alpha = in->alpha; s->sigma = in->sigma;
  s->adaptive_rho_tolerance = in->adaptive_rho_tolerance; s->rho_eq_factor = in->rho_eq_factor;
  s->rho_min = in->rho_min; s->rho_max = in->rho_max; s->delta = in->delta;
  s->max_iter = in->max_iter; s->check_termination = in->check_termination; s->adaptive_rho = in->adaptive_rho;
  // OSQP's adaptive_rho_interval = 0 means "automatic" (wall-clock based upstream, hence non-deterministic); its documented
  // fixed fallback is a multiple of check_termination.  Map 0 to 2 * check_termination (= this library's default of 50).
  s->adaptive_rho_interval = in->adaptive_rho_interval > 0 ? in->adaptive_rho_interval : 2 * (in->check_termination > 0 ? in->check_termination : 25);
  s->polish_passes = in->polish_passes;
  s->polish_refine_iter = in->polish_refine_iter; s->warm_start = in->warm_start > 0 ? 1 : 0;   /* < 0: stateless, see solve_batch */
  s->polish_retry = in->polish_retry < 0 ? 0 : in->polish_retry;
  s->early_polish = in->early_polish; s->early_polish_start = in->early_polish_start;
  return CUDAMPC_OK;
}

// Launch configuration of the per-problem-parameter kernels (first *_params call on a handle; the caller holds the device).
// K_solve: the handle's variant with one Params slot per group after the GroupShared array; K_rollout / K_step: the handle's form
// with the slot after the workspace.  Both at most the shared-parameter counts, which the handle's allocations are sized for.
static int pp_configure(cudampc_handle* h) {
  if (h->pp_ready) return CUDAMPC_OK;
  int optin = 0;
  CU(h, cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
  const int F = footprint(h->N), per = F * (int)sizeof(double) + (int)sizeof(GroupShared) + (int)sizeof(Params);
  int P = (optin - 64) / per;
  if (P > h->grp_P) P = h->grp_P;
  if (P < 1) return fail(h, CUDAMPC_ERR_UNSUPPORTED, "%s", "horizon too long for per-problem parameters in 227 KB of shared memory");
  const int smem = P * per + 16;
  CU(h, solve_set_smem(h->variant, smem, true));
  const int rsmem = h->smem_bytes + (int)sizeof(Params);
  int occ = 0;
  CU(h, rollout_set_smem(h->form, rsmem, true));
  CU(h, step_set_smem(h->form, rsmem, true));
  CU(h, rollout_occupancy(h->form, rsmem, &occ, true));
  if (occ < 1) return fail(h, CUDAMPC_ERR_UNSUPPORTED, "%s", "horizon too long for per-vehicle parameters in 227 KB of shared memory");
  h->pp_P = P; h->pp_smem = smem;
  h->pp_roll_per_sm = occ < h->roll_per_sm ? occ : h->roll_per_sm; h->pp_roll_smem = rsmem;
  h->pp_ready = true;
  return CUDAMPC_OK;
}

extern "C" {

int cudampc_version(void) { return CUDAMPC_VERSION; }

void cudampc_default_settings(cudampc_settings* s) {
  if (!s) return;
  memset(s, 0, sizeof *s);
  s->eps_abs = 1e-3; s->eps_rel = 1e-3; s->rho = 0.1; s->alpha = 1.6;       /* mpc_controller.py:121-131 */
  s->sigma = 1e-6; s->adaptive_rho_tolerance = 5.0; s->rho_eq_factor = 1e3; s->rho_min = 1e-6; s->rho_max = 1e6;
  s->delta = 1e-6; s->max_iter = 60000; s->check_termination = 25; s->adaptive_rho = 1; s->adaptive_rho_interval = 50;
  s->polish_passes = 1; s->polish_refine_iter = 3; s->warm_start = 0; s->polish_retry = 0;
  s->early_polish = 0; s->early_polish_start = 50;
}

void cudampc_default_rollout_cfg(cudampc_rollout_cfg* c) {
  if (!c) return;
  memset(c, 0, sizeof *c);
  c->sim_steps = 300; c->relax_on_failure = 1; c->advance_dist2 = 25.0; c->goal_radius = 8.0;
  c->relax_v_scale = 0.6; c->relax_da = 5.0; c->relax_ddelta = 0.05;
}

const char* cudampc_last_error(const cudampc_handle* h) { return h ? h->err : g_create_err; }

int cudampc_create(const cudampc_params* params, int max_batch, int device, cudampc_handle** out) {
  if (!out) return fail(nullptr, CUDAMPC_ERR_INVALID, "%s", "out is NULL");
  *out = nullptr;
  if (max_batch < 1) return fail(nullptr, CUDAMPC_ERR_INVALID, "%s", "max_batch must be >= 1");
  Params p;
  int rc = convert_params(params, &p, nullptr);
  if (rc) return rc;
  int ndev = 0;
  CU(nullptr, cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(nullptr, CUDAMPC_ERR_INVALID, "%s", "device index out of range");
  DeviceGuard guard_(device);
  CU(nullptr, guard_.err);
  cudampc_handle* h = new (std::nothrow) cudampc_handle();
  if (!h) return fail(nullptr, CUDAMPC_ERR_NOMEM, "%s", "host allocation failed");
  memset(h, 0, sizeof *h);
  h->device = device; h->max_batch = max_batch; h->N = p.N; h->p = p;
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) { delete h; return fail(nullptr, CUDAMPC_ERR_CUDA, "CUDA failure: %s", cudaGetErrorString(e)); }
  h->sms = prop.multiProcessorCount;
  const int F = footprint(p.N);
  h->smem_bytes = F * (int)sizeof(double);
  const int optin = (int)prop.sharedMemPerBlockOptin;
  if (h->smem_bytes + (int)sizeof(GroupShared) > optin) { delete h; return fail(nullptr, CUDAMPC_ERR_UNSUPPORTED, "%s", "horizon too long for one problem per 227 KB of shared memory"); }
  // K_rollout: one-warp CTAs.  Form of the ADMM phases (mpc_solve.h): a lane per stage for N+1 <= 32 (short), a lane per
  // pair of stages for N+1 <= 64 (pair), one parity of stages at a time beyond (general).
  h->form = p.N + 1 <= 32 ? FORM_SHORT : FORM_GENERAL;      // the pair form (N+1 <= 64) is opt-in: measured slower (profiles/README.md)
  if (const char* fe = getenv("CUDAMPC_FORM")) {                                                          // tuning knob
    if (!strcmp(fe, "general")) h->form = FORM_GENERAL;
    else if (!strcmp(fe, "pair") && p.N + 1 <= 64) h->form = FORM_PAIR;
    else if (!strcmp(fe, "short") && p.N + 1 <= 32) h->form = FORM_SHORT;
  }
  e = rollout_set_smem(h->form, h->smem_bytes);
  if (e == cudaSuccess) e = step_set_smem(h->form, h->smem_bytes);     // K_step: K_rollout's form and workspace
  int occ = 0;
  if (e == cudaSuccess) e = rollout_occupancy(h->form, h->smem_bytes, &occ);
  if (e != cudaSuccess || occ < 1) { delete h; return fail(nullptr, CUDAMPC_ERR_CUDA, "CUDA failure: %s", cudaGetErrorString(e)); }
  h->roll_per_sm = occ;
  // K_solve: one CTA per SM with P independent groups.  P <= 8: with more resident warps the 255-register budget of the
  // driver would have to shrink.  Two warps per group pay off only when few problems fit (long horizons: the SM is
  // latency-bound there); at P >= 3 the extra barriers cost more than the second warp saves (measured again in round 2:
  // branch item-form-experiment).
  {
    // K_solve: horizons with 32 < N+1 <= 64 run the two-warp register form (mpc_reg.h; 279 k / 369 k solves/s against 268 k / 364 k for
    // the one-warp parity form at horizon 50); CUDAMPC_FORM=reg selects it for short horizons too, general / pair / short override it
    int solve_form = (p.N + 1 > 32 && p.N + 1 <= 64) ? FORM_REG : h->form;
    if (const char* fe = getenv("CUDAMPC_FORM")) {
      if (!strcmp(fe, "reg") && p.N + 1 <= 64) solve_form = FORM_REG;
      else if (!strcmp(fe, "general") || !strcmp(fe, "pair") || !strcmp(fe, "short")) solve_form = h->form;
    }
    int P = (optin - 64) / (F * (int)sizeof(double) + (int)sizeof(GroupShared));
    if (P > 8) P = 8;
    if (const char* pe = getenv("CUDAMPC_P")) { int v = atoi(pe); if (v >= 1 && v < P) P = v; }   // tuning knobs
    h->grp_P = P;
    h->grp_wpp = (P <= 2 && p.N + 1 > 32) ? 2 : 1;
    if (const char* we = getenv("CUDAMPC_WPP")) { int v = atoi(we); if (v == 1 || (v == 2 && P <= 2)) h->grp_wpp = v; }
    h->variant = h->grp_wpp == 2 ? SOLVE_W2 : (h->form == FORM_SHORT ? SOLVE_W1_SHORT : h->form == FORM_PAIR ? SOLVE_W1_PAIR : SOLVE_W1);
    // register form (mpc_reg.h): two warps per problem, as many problems as the kernel was compiled for (256 threads: 255
    // registers; more: 168 registers)
    if (solve_form == FORM_REG && p.N + 1 <= 32) { if (P > 8) { P = 8; h->grp_P = 8; } h->grp_wpp = 1; h->variant = SOLVE_W1_REG; }      // a lane per stage, one warp
    else if (solve_form == FORM_REG) { const int pm = solve_reg_max_threads_4() / 64; if (P > pm) { P = pm; h->grp_P = pm; } h->grp_wpp = 2; h->variant = SOLVE_W2_REG; }
    h->grp_smem = P * (F * (int)sizeof(double) + (int)sizeof(GroupShared)) + 16;
    e = solve_set_smem(h->variant, h->grp_smem);
    if (e != cudaSuccess) { delete h; return fail(nullptr, CUDAMPC_ERR_CUDA, "CUDA failure: %s", cudaGetErrorString(e)); }
  }
  // warm / scratch: one slot per problem of the largest batch, then one per resident group (stateless solves)
  const size_t ws = (size_t)warm_size(p.N) * ((size_t)max_batch + (size_t)h->sms * h->grp_P) * sizeof(double);
  const size_t wk = (size_t)(16 + 4 * (p.N + 1) + 2 * p.N) * max_batch * sizeof(double);
  h->in_doubles = (size_t)max_batch * (4 + 4 * (p.N + 1) + 2);
  h->out_doubles = (size_t)max_batch * (2 + 4 * (p.N + 1) + 2 * p.N + 2 + 4);   // + pri, dua, (status, iters, info[4] as int32 in 3 doubles.. rounded to 4)
  e = cudaMalloc(&h->warm, ws);
  if (e == cudaSuccess) e = cudaMalloc(&h->scratch, ws);
  {
    int slots = h->sms * h->grp_P; if (h->sms * h->roll_per_sm > slots) slots = h->sms * h->roll_per_sm;
    if (e == cudaSuccess) e = cudaMalloc(&h->fsave, (size_t)slots * oe_doubles(p.N) * sizeof(double));
  }
  if (e == cudaSuccess) e = cudaMalloc(&h->work, wk);
  if (e == cudaSuccess) e = cudaMalloc(&h->counter, sizeof(int));
#ifdef MPC_TIMING
  if (e == cudaSuccess) e = cudaMalloc(&h->tags, sizeof(unsigned long long) * 32);
  if (e == cudaSuccess) e = cudaMemset(h->tags, 0, sizeof(unsigned long long) * 32);
#endif
  if (e == cudaSuccess) e = cudaMemset(h->warm, 0, ws);
  if (e != cudaSuccess) {
    snprintf(g_create_err, sizeof g_create_err, "CUDA failure: allocation -> %s", cudaGetErrorString(e));
    cudampc_destroy(h);
    return CUDAMPC_ERR_CUDA;
  }
  *out = h;
  return CUDAMPC_OK;
}

int cudampc_destroy(cudampc_handle* h) {
  if (!h) return CUDAMPC_OK;
  DeviceGuard guard_(h->device);
  cudaFree(h->warm); cudaFree(h->scratch); cudaFree(h->fsave); cudaFree(h->work); cudaFree(h->counter); cudaFree(h->tags);
  cudaFree(h->d_in); cudaFree(h->d_out);
  if (h->h_in) cudaFreeHost(h->h_in);
  if (h->h_out) cudaFreeHost(h->h_out);
  delete h;
  return CUDAMPC_OK;
}

int cudampc_set_params(cudampc_handle* h, const cudampc_params* params) {
  if (!h) return CUDAMPC_ERR_INVALID;
  Params p;
  int rc = convert_params(params, &p, h);
  if (rc) return rc;
  if (p.N != h->N) return fail(h, CUDAMPC_ERR_INVALID, "%s", "horizon cannot change on an existing handle");
  h->p = p;
  return CUDAMPC_OK;
}

double cudampc_fp64_peak_tflops(cudampc_handle* h) {
  if (!h) return -1.0;
  DeviceGuard guard_(h->device);
  if (guard_.err != cudaSuccess) return -1.0;
  const int blocks = h->sms * 8, threads = 256, iters = 20000;
  double* out = nullptr;
  if (cudaMalloc(&out, sizeof(double) * blocks * threads) != cudaSuccess) return -1.0;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  float best = 1e30f;
  for (int r = 0; r < 6; ++r) {
    cudaEventRecord(e0);
    fp64_peak_kernel<<<blocks, threads>>>(out, iters, 0.999999, 1e-6);
    cudaEventRecord(e1);
    if (cudaEventSynchronize(e1) != cudaSuccess) { best = -1.f; break; }
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    if (r > 0 && ms < best) best = ms;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
  if (best <= 0.f) return -1.0;
  return 2.0 * 8 * (double)iters * blocks * threads / (best * 1e-3) / 1e12;
}

int cudampc_workspace_doubles(const cudampc_handle* h) { return h ? footprint(h->N) : 0; }
int cudampc_problems_per_sm(const cudampc_handle* h) { return h ? h->grp_P : 0; }
int cudampc_rollout_resident(const cudampc_handle* h) { return h ? h->sms * h->roll_per_sm : 0; }
int64_t cudampc_launch_count(const cudampc_handle* h) { return h ? h->launches : 0; }

int cudampc_linearize_batch(cudampc_handle* h, int batch, const double* ref_dev, double* A_dev, double* B_dev,
                            double* c_dev, void* stream) {
  if (!h) return CUDAMPC_ERR_INVALID;
  if (batch < 0 || !ref_dev || !A_dev || !B_dev || !c_dev) return fail(h, CUDAMPC_ERR_INVALID, "%s", "linearize_batch: NULL pointer or negative batch");
  if (batch == 0) return CUDAMPC_OK;
  ON_DEVICE(h);
  const int wpb = 4;
  int grid = (batch + wpb - 1) / wpb;
  if (grid > h->sms * 8) grid = h->sms * 8;
  size_t sm = (size_t)wpb * (h->N + 1) * sizeof(double);
  mpc_linearize_kernel<<<grid, 32 * wpb, sm, (cudaStream_t)stream>>>(h->p, batch, ref_dev, A_dev, B_dev, c_dev);
  h->launches++;
  CU(h, cudaGetLastError());
  return CUDAMPC_OK;
}

int cudampc_f_discrete_batch(cudampc_handle* h, int batch, const double* x_dev, const double* u_dev, const double* dt_L_dev,
                             double* out_dev, void* stream) {
  if (!h) return CUDAMPC_ERR_INVALID;
  if (batch < 0 || !x_dev || !u_dev || !out_dev) return fail(h, CUDAMPC_ERR_INVALID, "%s", "f_discrete_batch: NULL pointer or negative batch");
  if (batch == 0) return CUDAMPC_OK;
  ON_DEVICE(h);
  mpc_f_discrete_kernel<<<(batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->p.dt, h->p.L, batch, x_dev, u_dev, dt_L_dev, out_dev);
  h->launches++;
  CU(h, cudaGetLastError());
  return CUDAMPC_OK;
}

// cudampc_solve_batch (params_dev NULL) and cudampc_solve_batch_params
static int solve_batch_impl(cudampc_handle* h, int batch, const double* x0_dev, const double* ref_dev,
                            const double* u_prev_dev, const cudampc_settings* settings, const cudampc_params* params_dev,
                            double* u0_dev, double* Xp_dev, double* Up_dev, int32_t* status_dev, int32_t* iters_dev,
                            double* pri_res_dev, double* dua_res_dev, int32_t* info_dev, void* stream, const char* name) {
  if (!h) return CUDAMPC_ERR_INVALID;
  if (batch < 0 || batch > h->max_batch) return fail(h, CUDAMPC_ERR_INVALID, "%s: batch out of range for this handle", name);
  if (!x0_dev || !ref_dev || !u0_dev || !Xp_dev || !Up_dev || !status_dev || !iters_dev)
    return fail(h, CUDAMPC_ERR_INVALID, "%s: NULL pointer", name);
  Settings s;
  int rc = convert_settings(settings, &s, h);
  if (rc) return rc;
  if (batch == 0) return CUDAMPC_OK;
  ON_DEVICE(h);
  const bool pp = params_dev != nullptr;
  if (pp && (rc = pp_configure(h))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  CU(h, cudaMemsetAsync(h->counter, 0, sizeof(int), st));
  BatchArgs a;
  a.x0 = x0_dev; a.ref = ref_dev; a.u_prev = u_prev_dev; a.warm = h->warm; a.scratch = h->scratch; a.fsave = getenv("CUDAMPC_NO_FSAVE") ? nullptr : h->fsave;
  a.group_state = settings && settings->warm_start < 0 ? 1 : 0;
  a.group_slot0 = h->max_batch;
  a.u0 = u0_dev; a.Xp = Xp_dev; a.Up = Up_dev; a.status = status_dev; a.iters = iters_dev;
  a.pri = pri_res_dev; a.dua = dua_res_dev; a.info = info_dev; a.counter = h->counter; a.batch = batch; a.tags = h->tags;
  a.params = params_dev;
  const int P = pp ? h->pp_P : h->grp_P;
  int grid = (batch + P - 1) / P;
  if (grid > h->sms) grid = h->sms;
  const int threads = 32 * h->grp_wpp * P;
  solve_launch(h->variant, grid, threads, pp ? h->pp_smem : h->grp_smem, st, h->p, s, a, P, footprint(h->N), pp);
  h->launches++;
  CU(h, cudaGetLastError());
  return CUDAMPC_OK;
}

int cudampc_solve_batch(cudampc_handle* h, int batch, const double* x0_dev, const double* ref_dev,
                        const double* u_prev_dev, const cudampc_settings* settings, double* u0_dev, double* Xp_dev,
                        double* Up_dev, int32_t* status_dev, int32_t* iters_dev, double* pri_res_dev,
                        double* dua_res_dev, int32_t* info_dev, void* stream) {
  return solve_batch_impl(h, batch, x0_dev, ref_dev, u_prev_dev, settings, nullptr, u0_dev, Xp_dev, Up_dev, status_dev, iters_dev,
                          pri_res_dev, dua_res_dev, info_dev, stream, "solve_batch");
}

int cudampc_solve_batch_params(cudampc_handle* h, int batch, const double* x0_dev, const double* ref_dev,
                               const double* u_prev_dev, const cudampc_settings* settings, const cudampc_params* params_dev,
                               double* u0_dev, double* Xp_dev, double* Up_dev, int32_t* status_dev, int32_t* iters_dev,
                               double* pri_res_dev, double* dua_res_dev, int32_t* info_dev, void* stream) {
  if (h && !params_dev) return fail(h, CUDAMPC_ERR_INVALID, "%s", "solve_batch_params: NULL pointer");
  return solve_batch_impl(h, batch, x0_dev, ref_dev, u_prev_dev, settings, params_dev, u0_dev, Xp_dev, Up_dev, status_dev, iters_dev,
                          pri_res_dev, dua_res_dev, info_dev, stream, "solve_batch_params");
}

static bool is_pinned(const void* p) {
  if (!p) return true;
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeHost;
}

int cudampc_solve_batch_host(cudampc_handle* h, int batch, const double* x0, const double* ref, const double* u_prev,
                             const cudampc_settings* settings, double* u0, double* Xp, double* Up, int32_t* status,
                             int32_t* iters, double* pri_res, double* dua_res, int32_t* info, void* stream) {
  if (!h) return CUDAMPC_ERR_INVALID;
  if (batch < 0 || batch > h->max_batch) return fail(h, CUDAMPC_ERR_INVALID, "%s", "solve_batch_host: batch out of range for this handle");
  if (!x0 || !ref || !u0 || !Xp || !Up || !status || !iters) return fail(h, CUDAMPC_ERR_INVALID, "%s", "solve_batch_host: NULL pointer");
  if (batch == 0) return CUDAMPC_OK;
  ON_DEVICE(h);
  cudaStream_t st = (cudaStream_t)stream;
  const int N = h->N;
  const size_t B = (size_t)batch;
  if (!h->d_in) {          // device staging of the host path: allocated on first use (a device-only caller never pays for it)
    CU(h, cudaMalloc(&h->d_in, h->in_doubles * sizeof(double)));
    CU(h, cudaMalloc(&h->d_out, h->out_doubles * sizeof(double)));
  }
  const size_t n_x0 = 4 * B, n_ref = 4 * (size_t)(N + 1) * B, n_up = 2 * B;
  const size_t n_u0 = 2 * B, n_xp = 4 * (size_t)(N + 1) * B, n_upo = 2 * (size_t)N * B;
  double* d_x0 = h->d_in; double* d_ref = d_x0 + n_x0; double* d_up = d_ref + n_ref;
  double* d_u0 = h->d_out; double* d_xp = d_u0 + n_u0; double* d_upo = d_xp + n_xp;
  double* d_pri = d_upo + n_upo; double* d_dua = d_pri + B;
  int32_t* d_int = reinterpret_cast<int32_t*>(d_dua + B);   // status[B], iters[B], info[4B]
  // page-locked caller buffers (cudaHostAlloc / cudaHostRegister / torch pin_memory) are copied directly;
  // pageable ones go through the handle's pinned staging area
  const bool in_pinned = is_pinned(x0) && is_pinned(ref) && is_pinned(u_prev);
  if (in_pinned) {
    CU(h, cudaMemcpyAsync(d_x0, x0, n_x0 * sizeof(double), cudaMemcpyHostToDevice, st));
    CU(h, cudaMemcpyAsync(d_ref, ref, n_ref * sizeof(double), cudaMemcpyHostToDevice, st));
    if (u_prev) CU(h, cudaMemcpyAsync(d_up, u_prev, n_up * sizeof(double), cudaMemcpyHostToDevice, st));
    else CU(h, cudaMemsetAsync(d_up, 0, n_up * sizeof(double), st));
  } else {
    if (!h->h_in) CU(h, cudaMallocHost(&h->h_in, h->in_doubles * sizeof(double)));       // pinned staging for pageable callers
    memcpy(h->h_in, x0, n_x0 * sizeof(double));
    memcpy(h->h_in + n_x0, ref, n_ref * sizeof(double));
    if (u_prev) memcpy(h->h_in + n_x0 + n_ref, u_prev, n_up * sizeof(double));
    else memset(h->h_in + n_x0 + n_ref, 0, n_up * sizeof(double));
    CU(h, cudaMemcpyAsync(h->d_in, h->h_in, (n_x0 + n_ref + n_up) * sizeof(double), cudaMemcpyHostToDevice, st));
  }
  int rc = cudampc_solve_batch(h, batch, d_x0, d_ref, d_up, settings, d_u0, d_xp, d_upo, d_int, d_int + B, d_pri, d_dua,
                               d_int + 2 * B, stream);
  if (rc) return rc;
  const bool out_pinned = is_pinned(u0) && is_pinned(Xp) && is_pinned(Up) && is_pinned(status) && is_pinned(iters) &&
                          is_pinned(pri_res) && is_pinned(dua_res) && is_pinned(info);
  if (out_pinned) {
    CU(h, cudaMemcpyAsync(u0, d_u0, n_u0 * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(h, cudaMemcpyAsync(Xp, d_xp, n_xp * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(h, cudaMemcpyAsync(Up, d_upo, n_upo * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (pri_res) CU(h, cudaMemcpyAsync(pri_res, d_pri, B * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (dua_res) CU(h, cudaMemcpyAsync(dua_res, d_dua, B * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(h, cudaMemcpyAsync(status, d_int, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU(h, cudaMemcpyAsync(iters, d_int + B, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (info) CU(h, cudaMemcpyAsync(info, d_int + 2 * B, 4 * B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU(h, cudaStreamSynchronize(st));
    return CUDAMPC_OK;
  }
  if (!h->h_out) CU(h, cudaMallocHost(&h->h_out, h->out_doubles * sizeof(double)));
  const size_t n_out = n_u0 + n_xp + n_upo + 2 * B + 3 * B;   // 6 int32 per problem = 3 doubles
  CU(h, cudaMemcpyAsync(h->h_out, h->d_out, n_out * sizeof(double), cudaMemcpyDeviceToHost, st));
  CU(h, cudaStreamSynchronize(st));
  memcpy(u0, h->h_out, n_u0 * sizeof(double));
  memcpy(Xp, h->h_out + n_u0, n_xp * sizeof(double));
  memcpy(Up, h->h_out + n_u0 + n_xp, n_upo * sizeof(double));
  const double* hp = h->h_out + n_u0 + n_xp + n_upo;
  if (pri_res) memcpy(pri_res, hp, B * sizeof(double));
  if (dua_res) memcpy(dua_res, hp + B, B * sizeof(double));
  const int32_t* hi = reinterpret_cast<const int32_t*>(hp + 2 * B);
  memcpy(status, hi, B * sizeof(int32_t));
  memcpy(iters, hi + B, B * sizeof(int32_t));
  if (info) memcpy(info, hi + 2 * B, 4 * B * sizeof(int32_t));
  return CUDAMPC_OK;
}

int cudampc_build_reference_batch(cudampc_handle* h, int batch, const double* paths_dev, const int32_t* n_pts_dev, int max_pts,
                                  double desired_speed, double* ref_dev, int32_t* ref_len_dev, int ref_stride, void* stream) {
  if (!h) return CUDAMPC_ERR_INVALID;
  if (batch < 0 || !paths_dev || !n_pts_dev || !ref_dev || !ref_len_dev || max_pts < 1 || ref_stride < h->N + 1 || !(desired_speed > 0.0))
    return fail(h, CUDAMPC_ERR_INVALID, "%s", "build_reference_batch: NULL pointer, max_pts < 1, ref_stride < horizon+1 or speed <= 0");
  if (batch == 0) return CUDAMPC_OK;
  ON_DEVICE(h);
  mpc_build_reference_kernel<<<(batch + 63) / 64, 64, 0, (cudaStream_t)stream>>>(batch, paths_dev, n_pts_dev, max_pts, desired_speed, h->p.dt,
                                                                                 h->N, ref_dev, ref_len_dev, ref_stride);
  h->launches++;
  CU(h, cudaGetLastError());
  return CUDAMPC_OK;
}

// cudampc_rollout_batch (params_dev NULL) and cudampc_rollout_batch_params
static int rollout_batch_impl(cudampc_handle* h, int batch, const double* ref_global_dev, const int32_t* ref_len_dev,
                              int ref_stride, const double* state0_dev, const double* goal_dev,
                              const cudampc_settings* settings, const cudampc_rollout_cfg* cfg, const cudampc_params* params_dev,
                              double* states_dev, double* controls_dev, int32_t* n_steps_dev, int32_t* flags_dev,
                              int32_t* step_status_dev, int32_t* step_iters_dev, void* stream, const char* name) {
  if (!h) return CUDAMPC_ERR_INVALID;
  if (batch < 0 || batch > h->max_batch) return fail(h, CUDAMPC_ERR_INVALID, "%s: batch out of range for this handle", name);
  if (!ref_global_dev || !ref_len_dev || !state0_dev || !goal_dev || !states_dev || !n_steps_dev || !flags_dev || ref_stride < 1)
    return fail(h, CUDAMPC_ERR_INVALID, "%s: NULL pointer or bad stride", name);
  cudampc_rollout_cfg c;
  if (cfg) c = *cfg; else cudampc_default_rollout_cfg(&c);
  if (c.sim_steps < 1) return fail(h, CUDAMPC_ERR_INVALID, "%s: sim_steps must be >= 1", name);
  Settings s;
  int rc = convert_settings(settings, &s, h);
  if (rc) return rc;
  if (batch == 0) return CUDAMPC_OK;
  ON_DEVICE(h);
  const bool pp = params_dev != nullptr;
  if (pp && (rc = pp_configure(h))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  CU(h, cudaMemsetAsync(h->counter, 0, sizeof(int), st));
  RolloutArgs a;
  a.ref_global = ref_global_dev; a.ref_len = ref_len_dev; a.ref_stride = ref_stride; a.state0 = state0_dev; a.goal = goal_dev;
  a.warm = h->warm; a.scratch = h->scratch; a.fsave = getenv("CUDAMPC_NO_FSAVE") ? nullptr : h->fsave; a.work = h->work;
  a.states = states_dev; a.controls = controls_dev; a.n_steps = n_steps_dev; a.flags = flags_dev;
  a.step_status = step_status_dev; a.step_iters = step_iters_dev; a.counter = h->counter; a.batch = batch; a.params = params_dev;
  {
    int grid = h->sms * (pp ? h->pp_roll_per_sm : h->roll_per_sm);
    if (grid > batch) grid = batch;
    rollout_launch(h->form, grid, pp ? h->pp_roll_smem : h->smem_bytes, st, h->p, s, c, a, pp);
  }
  h->launches++;
  CU(h, cudaGetLastError());
  return CUDAMPC_OK;
}

int cudampc_rollout_batch(cudampc_handle* h, int batch, const double* ref_global_dev, const int32_t* ref_len_dev,
                          int ref_stride, const double* state0_dev, const double* goal_dev,
                          const cudampc_settings* settings, const cudampc_rollout_cfg* cfg, double* states_dev,
                          double* controls_dev, int32_t* n_steps_dev, int32_t* flags_dev, int32_t* step_status_dev,
                          int32_t* step_iters_dev, void* stream) {
  return rollout_batch_impl(h, batch, ref_global_dev, ref_len_dev, ref_stride, state0_dev, goal_dev, settings, cfg, nullptr, states_dev,
                            controls_dev, n_steps_dev, flags_dev, step_status_dev, step_iters_dev, stream, "rollout_batch");
}

int cudampc_rollout_batch_params(cudampc_handle* h, int batch, const double* ref_global_dev, const int32_t* ref_len_dev,
                                 int ref_stride, const double* state0_dev, const double* goal_dev,
                                 const cudampc_settings* settings, const cudampc_rollout_cfg* cfg,
                                 const cudampc_params* params_dev, double* states_dev, double* controls_dev,
                                 int32_t* n_steps_dev, int32_t* flags_dev, int32_t* step_status_dev, int32_t* step_iters_dev,
                                 void* stream) {
  if (h && !params_dev) return fail(h, CUDAMPC_ERR_INVALID, "%s", "rollout_batch_params: NULL pointer or bad stride");
  return rollout_batch_impl(h, batch, ref_global_dev, ref_len_dev, ref_stride, state0_dev, goal_dev, settings, cfg, params_dev, states_dev,
                            controls_dev, n_steps_dev, flags_dev, step_status_dev, step_iters_dev, stream, "rollout_batch_params");
}

// cudampc_track_step_batch (params_dev NULL) and cudampc_track_step_batch_params
static int track_step_impl(cudampc_handle* h, int batch, const double* ref_global_dev, const int32_t* ref_len_dev,
                           int ref_stride, const double* goal_dev, const double* state_dev,
                           const cudampc_settings* settings, const cudampc_rollout_cfg* cfg, const cudampc_params* params_dev,
                           int32_t* path_idx_dev, double* u_prev_dev, int32_t* n_steps_dev, int32_t* flags_dev,
                           double* u0_dev, double* Xp_dev, double* Up_dev, int32_t* status_dev, int32_t* iters_dev,
                           void* stream, const char* name) {
  if (!h) return CUDAMPC_ERR_INVALID;
  if (batch < 0 || batch > h->max_batch) return fail(h, CUDAMPC_ERR_INVALID, "%s: batch out of range for this handle", name);
  if (!ref_global_dev || !ref_len_dev || !goal_dev || !state_dev || !path_idx_dev || !u_prev_dev || !n_steps_dev || !flags_dev ||
      !u0_dev || !status_dev || !iters_dev || ref_stride < 1)
    return fail(h, CUDAMPC_ERR_INVALID, "%s: NULL pointer or bad stride", name);
  cudampc_rollout_cfg c;
  if (cfg) c = *cfg; else cudampc_default_rollout_cfg(&c);
  Settings s;
  int rc = convert_settings(settings, &s, h);
  if (rc) return rc;
  if (batch == 0) return CUDAMPC_OK;
  ON_DEVICE(h);
  const bool pp = params_dev != nullptr;
  if (pp && (rc = pp_configure(h))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  CU(h, cudaMemsetAsync(h->counter, 0, sizeof(int), st));
  StepArgs a;
  a.ref_global = ref_global_dev; a.ref_len = ref_len_dev; a.ref_stride = ref_stride; a.goal = goal_dev; a.state = state_dev;
  a.warm = h->warm; a.scratch = h->scratch; a.fsave = getenv("CUDAMPC_NO_FSAVE") ? nullptr : h->fsave; a.work = h->work;
  a.path_idx = path_idx_dev; a.u_prev = u_prev_dev; a.n_steps = n_steps_dev; a.flags = flags_dev;
  a.u0 = u0_dev; a.Xp = Xp_dev; a.Up = Up_dev; a.status = status_dev; a.iters = iters_dev; a.counter = h->counter; a.batch = batch;
  a.params = params_dev;
  int grid = h->sms * (pp ? h->pp_roll_per_sm : h->roll_per_sm);
  if (grid > batch) grid = batch;
  step_launch(h->form, grid, pp ? h->pp_roll_smem : h->smem_bytes, st, h->p, s, c, a, pp);
  h->launches++;
  CU(h, cudaGetLastError());
  return CUDAMPC_OK;
}

int cudampc_track_step_batch(cudampc_handle* h, int batch, const double* ref_global_dev, const int32_t* ref_len_dev,
                             int ref_stride, const double* goal_dev, const double* state_dev,
                             const cudampc_settings* settings, const cudampc_rollout_cfg* cfg,
                             int32_t* path_idx_dev, double* u_prev_dev, int32_t* n_steps_dev, int32_t* flags_dev,
                             double* u0_dev, double* Xp_dev, double* Up_dev, int32_t* status_dev, int32_t* iters_dev,
                             void* stream) {
  return track_step_impl(h, batch, ref_global_dev, ref_len_dev, ref_stride, goal_dev, state_dev, settings, cfg, nullptr, path_idx_dev,
                         u_prev_dev, n_steps_dev, flags_dev, u0_dev, Xp_dev, Up_dev, status_dev, iters_dev, stream, "track_step_batch");
}

int cudampc_track_step_batch_params(cudampc_handle* h, int batch, const double* ref_global_dev, const int32_t* ref_len_dev,
                                    int ref_stride, const double* goal_dev, const double* state_dev,
                                    const cudampc_settings* settings, const cudampc_rollout_cfg* cfg,
                                    const cudampc_params* params_dev, int32_t* path_idx_dev, double* u_prev_dev,
                                    int32_t* n_steps_dev, int32_t* flags_dev, double* u0_dev, double* Xp_dev, double* Up_dev,
                                    int32_t* status_dev, int32_t* iters_dev, void* stream) {
  if (h && !params_dev) return fail(h, CUDAMPC_ERR_INVALID, "%s", "track_step_batch_params: NULL pointer or bad stride");
  return track_step_impl(h, batch, ref_global_dev, ref_len_dev, ref_stride, goal_dev, state_dev, settings, cfg, params_dev, path_idx_dev,
                         u_prev_dev, n_steps_dev, flags_dev, u0_dev, Xp_dev, Up_dev, status_dev, iters_dev, stream, "track_step_batch_params");
}

// dev tool (tools/tag_times.py, libraries built with -DMPC_TIMING): cycles between the driver's tags, summed over a launch
int cudampc_debug_tag_cycles(cudampc_handle* h, unsigned long long* out32, int reset) {
  if (!h || !h->tags) return CUDAMPC_ERR_INVALID;
  if (cudaMemcpy(out32, h->tags, sizeof(unsigned long long) * 32, cudaMemcpyDeviceToHost) != cudaSuccess) return CUDAMPC_ERR_CUDA;
  if (reset && cudaMemset(h->tags, 0, sizeof(unsigned long long) * 32) != cudaSuccess) return CUDAMPC_ERR_CUDA;
  return CUDAMPC_OK;
}

}  // extern "C"
