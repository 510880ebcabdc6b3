// mpc_kernels.cuh — the heavy kernels of libcudampc.so (K_solve, K_rollout, K_step) as templates, and the launch interface of
// their instantiations.  Every instantiation lives in its own translation unit (mpc_kernels_tu.cu compiled with
// -DMPC_TU=n) so that the library builds in parallel; cudampc.cu (C ABI + the small kernels) only sees the launchers.
#pragma once
#include <cuda_runtime.h>
#include "../../include/cudampc.h"
#include "mpc_exec.cuh"
#include "mpc_params.h"

using namespace mpc;

struct BatchArgs {
  const double* x0; const double* ref; const double* u_prev;
  double* warm; double* scratch; double* fsave;     // fsave: oe_doubles(N) per resident group (grid x P), or null
  double* u0; double* Xp; double* Up; int* status; int* iters; double* pri; double* dua; int* info;
  int* counter;
  int batch;
  int group_state;             // 1: stateless solve - the iterate back-ups (warm, scratch) use the resident group's slot, not the problem's
  int group_slot0;             // first of the per-group slots (behind the per-problem ones)
  unsigned long long* tags;    // dev builds only (MPC_TIMING)
  const cudampc_params* params;  // per-problem kernels (PP): batch records, problem order
};

// ------------------------------------------------------------------------------------------------
// Per-problem parameters (the PP instantiations).  Each problem / vehicle b reads its own record params[b]: one lane runs the
// rules of mpc_params.h on it into the group's Params slot in shared memory, and the group syncs before reading the slot.  A
// record the rules reject, or whose horizon or dt differs from the launch's (the workspace layout and the time grid of the
// register-form block are the launch's), leaves slot->N = 0.  Such a problem is not solved.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void load_params(const cudampc_params* rows, int b, const Params& launch, Params* slot) {
  const cudampc_params* in = rows + b;
  if (params_from_c(in, slot) != PARAMS_OK || in->horizon != launch.N || !(in->dt == launch.dt)) slot->N = 0;
}
// Outputs of a problem whose record is invalid: status CUDAMPC_INVALID_PARAMS, iters 0, NaN u0 / Xp / Up / pri / dua, info 0.
// The warm-start slot is not touched.
template <class Exec>
__device__ __forceinline__ void invalid_problem(Exec& ex, const ProblemIO& io, int N) {
  const double nan_ = __longlong_as_double(0x7ff8000000000000LL);
  ex.stages(4 * (N + 1), [&](int i) { io.Xp[i] = nan_; });
  ex.stages(2 * N, [&](int i) { io.Up[i] = nan_; });
  ex.single([&]() {
    io.u0[0] = nan_; io.u0[1] = nan_; *io.status = CUDAMPC_INVALID_PARAMS; *io.iters = 0;
    if (io.pri_res) *io.pri_res = nan_;
    if (io.dua_res) *io.dua_res = nan_;
    if (io.info) for (int i = 0; i < 4; ++i) io.info[i] = 0;
  });
}

// ------------------------------------------------------------------------------------------------
// K_solve: batched MPCController.solve.  The CTA holds P problems, each owned by a group of WPP warps (GroupExec).
// <256,1>: P <= 8 one-warp groups, 255 registers; <128,2>: P <= 2 two-warp groups for long horizons.
// PP: per-problem parameters; the P Params slots follow the GroupShared array.
// ------------------------------------------------------------------------------------------------
template <int MAXT, int WPP, int FORM, bool PP>
__global__ void __launch_bounds__(MAXT, 1) mpc_solve_kernel(Params p, Settings s, BatchArgs a, int P, int F) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int N = p.N;
  GroupShared* sh = reinterpret_cast<GroupShared*>(smem + (size_t)P * F) + warp / WPP;
  int fpad, xpad; layout_pads(N, fpad, xpad);
  View w{smem + (size_t)(warp / WPP) * F, N, fpad, xpad};
  GroupExec<WPP> ex{lane, warp, sh};
#ifdef MPC_TIMING
  ex.tags = a.tags;
#endif
  const int ws = warm_size(N);
  for (int b = ex.fetch(a.counter); b < a.batch; b = ex.fetch(a.counter)) {
    ProblemIO io;
    io.x0 = a.x0 + 4 * (size_t)b;
    io.ref = RefWin{a.ref + (size_t)4 * (N + 1) * b, 0, N + 1, 1.0};
    io.u_prev = a.u_prev ? a.u_prev + 2 * (size_t)b : nullptr;
    const size_t slot = a.group_state ? (size_t)a.group_slot0 + (size_t)blockIdx.x * P + warp / WPP : (size_t)b;
    io.warm = a.warm + (size_t)ws * slot;
    io.scratch = a.scratch + (size_t)ws * slot;
    io.fsave = a.fsave ? a.fsave + (size_t)oe_doubles(N) * ((size_t)blockIdx.x * P + warp / WPP) : nullptr;
    io.u0 = a.u0 + 2 * (size_t)b;
    io.Xp = a.Xp + (size_t)4 * (N + 1) * b;
    io.Up = a.Up + (size_t)2 * N * b;
    io.status = a.status + b; io.iters = a.iters + b;
    io.pri_res = a.pri ? a.pri + b : nullptr; io.dua_res = a.dua ? a.dua + b : nullptr;
    io.info = a.info ? a.info + 4 * (size_t)b : nullptr;
    if constexpr (PP) {
      Params* pb = reinterpret_cast<Params*>(reinterpret_cast<GroupShared*>(smem + (size_t)P * F) + P) + warp / WPP;
      if (ex.gl() == 0) load_params(a.params, b, p, pb);
      ex.group_sync();
      if (pb->N == 0) invalid_problem(ex, io, N);
      else solve_problem<FORM>(ex, w, *pb, s, io);
    } else {
      solve_problem<FORM>(ex, w, p, s, io);
    }
    ex.group_sync();
  }
}

// ------------------------------------------------------------------------------------------------
// K_solve, register form (mpc_reg.h, mpc_drv.h): two warps per problem; the iteration blocks are inlined HERE, at the top
// level of the kernel, and everything else of the driver runs in three inlined pieces that keep their state in shared memory
// (the after-block piece also runs once per polish pass, without a block before it).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ ProblemIO batch_io(const BatchArgs& a, int b, int N, int group) {
  const int ws = warm_size(N);
  ProblemIO io;
  io.x0 = a.x0 + 4 * (size_t)b;
  io.ref = RefWin{a.ref + (size_t)4 * (N + 1) * b, 0, N + 1, 1.0};
  io.u_prev = a.u_prev ? a.u_prev + 2 * (size_t)b : nullptr;
  const size_t slot = a.group_state ? (size_t)a.group_slot0 + (size_t)group : (size_t)b;
  io.warm = a.warm + (size_t)ws * slot;
  io.scratch = a.scratch + (size_t)ws * slot;
  io.fsave = a.fsave ? a.fsave + (size_t)oe_doubles(N) * group : nullptr;
  io.u0 = a.u0 + 2 * (size_t)b;
  io.Xp = a.Xp + (size_t)4 * (N + 1) * b;
  io.Up = a.Up + (size_t)2 * N * b;
  io.status = a.status + b; io.iters = a.iters + b;
  io.pri_res = a.pri ? a.pri + b : nullptr; io.dua_res = a.dua ? a.dua + b : nullptr;
  io.info = a.info ? a.info + 4 * (size_t)b : nullptr;
  return io;
}
struct RegCtx { const Params* p; const Settings* s; const BatchArgs* a; double* base; GroupShared* sh; int N, fpad, xpad, lane, warp, group; };
template <int WPP>
__device__ __forceinline__ GroupExec<WPP> reg_exec(const RegCtx& c) {
  GroupExec<WPP> ex{c.lane, c.warp, c.sh};
#ifdef MPC_TIMING
  ex.tags = c.a->tags;
#endif
  return ex;
}
template <int WPP>
__device__ __forceinline__ void reg_drv_begin(RegCtx c, int b) {
  const View w{c.base, c.N, c.fpad, c.xpad};
  GroupExec<WPP> ex = reg_exec<WPP>(c);
  const ProblemIO io = batch_io(*c.a, b, c.N, c.group);
  Drv d;
  drv_begin(ex, w, *c.p, *c.s, io, d);
  drv_prepare(ex, w, *c.p, *c.s, d);
  if (ex.gl() == 0) c.sh->drv = d;
  ex.group_sync();
}
template <int WPP>
__device__ __forceinline__ void reg_drv_after(RegCtx c, int b) {
  const View w{c.base, c.N, c.fpad, c.xpad};
  GroupExec<WPP> ex = reg_exec<WPP>(c);
  const ProblemIO io = batch_io(*c.a, b, c.N, c.group);
  Drv d = c.sh->drv;
  ex.group_sync();                          // every lane has its copy before lane 0 writes the new one
  drv_after(ex, w, *c.p, *c.s, io, d);
  if (!d.finished && d.phase == PH_ADMM) drv_prepare(ex, w, *c.p, *c.s, d);
  if (ex.gl() == 0) c.sh->drv = d;
  ex.group_sync();
}
template <int WPP>
__device__ __forceinline__ void reg_drv_finish(RegCtx c, int b) {
  const View w{c.base, c.N, c.fpad, c.xpad};
  GroupExec<WPP> ex = reg_exec<WPP>(c);
  const ProblemIO io = batch_io(*c.a, b, c.N, c.group);
  const Drv d = c.sh->drv;
  drv_finish(ex, w, io, d);
  ex.group_sync();
}
template <int MAXT, int STATE, int WPP, bool PP>
__global__ void __launch_bounds__(MAXT, 1) mpc_solve_reg_kernel(const __grid_constant__ Params p, const __grid_constant__ Settings s,
                                                                const __grid_constant__ BatchArgs a, int P, int F) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int N = p.N;
  GroupShared* sh = reinterpret_cast<GroupShared*>(smem + (size_t)P * F) + warp / WPP;
  int fpad, xpad; layout_pads(N, fpad, xpad);
  double* base = smem + (size_t)(warp / WPP) * F;
  GroupExec<WPP> ex{lane, warp, sh};
  const int ev = ex.chain_warp() ? 1 : 0, bar_id = 1 + ex.grp();
#ifdef MPC_TIMING
  unsigned long long* tg = a.tags;
#else
  unsigned long long* tg = nullptr;
#endif
  for (int b = ex.fetch(a.counter); b < a.batch; b = ex.fetch(a.counter)) {
    const int group = (int)blockIdx.x * P + warp / WPP;
    const Params* pc = &p;
    if constexpr (PP) {     // the pieces read the problem's slot; the iteration block keeps the launch's dt
      Params* pb = reinterpret_cast<Params*>(reinterpret_cast<GroupShared*>(smem + (size_t)P * F) + P) + warp / WPP;
      if (ex.gl() == 0) load_params(a.params, b, p, pb);
      ex.group_sync();
      if (pb->N == 0) { invalid_problem(ex, batch_io(a, b, N, group), N); continue; }
      pc = pb;
    }
    // The pieces of the driver are inlined; none of their values is alive across a block (Drv lives in shared memory
    // between them).
    const RegCtx c{pc, &s, &a, base, sh, N, fpad, xpad, lane, warp, group};
    reg_drv_begin<WPP>(c, b);
    while (!*(volatile int*)&sh->drv.finished) {
      if (*(volatile int*)&sh->drv.phase == PH_ADMM) {       // else a polish pass ran its solves: its residuals are next
        const int nb = *(volatile int*)&sh->drv.nb;
        reg_block_run<STATE, WPP>(base, N, fpad, xpad, p.dt, &sh->drv.ic, nb, lane, ev, bar_id, tg);
      }
      reg_drv_after<WPP>(c, b);
    }
    reg_drv_finish<WPP>(c, b);
  }
}

__device__ __forceinline__ void f_discrete_vals(double dt, double L, const double* x, const double* u, double* out) {
  // vehicle_model.py:11-21 (beta = 0.0 is added to the yaw there)
  const double yaw = x[2], v = x[3];
  out[0] = x[0] + dt * v * cos(yaw + 0.0);
  out[1] = x[1] + dt * v * sin(yaw + 0.0);
  out[2] = yaw + dt * (v / L) * tan(u[1]);
  out[3] = v + dt * u[0];
}

// ------------------------------------------------------------------------------------------------
// K_rollout: TrajectoryTracker.track for a batch of vehicles, all steps on the device
// ------------------------------------------------------------------------------------------------
struct RolloutArgs {
  const double* ref_global; const int* ref_len; int ref_stride;
  const double* state0; const double* goal;
  double* warm; double* scratch; double* fsave; double* work;   // fsave: oe_doubles(N) per CTA, or null; work: per vehicle 16 doubles (state, u_prev, u0 out) + Xp/Up scratch
  double* states; double* controls; int* n_steps; int* flags; int* step_status; int* step_iters;
  int* counter; int batch;
  const cudampc_params* params;  // per-vehicle kernels (PP): batch records, vehicle order
};

__device__ __forceinline__ void f_discrete_dev(const Params& p, const double* x, const double* u, double* out) {
  f_discrete_vals(p.dt, p.L, x, u, out);
}

// The pieces of one closed-loop step that K_rollout and K_step share (control_stage.py:126-147).
// (a) The solve of the step (_solve_with_relaxation, control_stage.py:45-56,126-129): window at path_idx with tail padding,
// warm start from the problem's slot once the vehicle has stepped, one cold retry with v_ref * relax_v_scale and widened
// du_bounds on failure (sets flags bit 2).  io carries everything but the window.  Returns the final status.
// PP: p is the vehicle's Params slot in shared memory; the retry widens the slot's own du_bounds and restores them afterwards
// (a copy of the slot would take 416 bytes of local memory in every lane).
template <int FORM, bool PP, class Exec>
__device__ __forceinline__ int track_solve(Exec& ex, const View& w, const Params& p, const Settings& s, const cudampc_rollout_cfg& cfg,
                                           ProblemIO io, const double* refg, int path_idx, int len, bool stepped, int& flags) {
  io.ref = RefWin{refg, path_idx, len, 1.0};
  Settings ss = s;
  ss.warm_start = (s.warm_start && stepped) ? 1 : 0;
  solve_problem<FORM>(ex, w, p, ss, io);
  ex.group_sync();
  int status = *io.status;
  if (status != STATUS_SOLVED && status != STATUS_SOLVED_INACCURATE && cfg.relax_on_failure) {
    io.ref.vscale = cfg.relax_v_scale;
    ss.warm_start = 0;
    if constexpr (PP) {
      Params& pr = const_cast<Params&>(p);
      const double lo0 = pr.du_lo[0], hi0 = pr.du_hi[0], lo1 = pr.du_lo[1], hi1 = pr.du_hi[1];
      ex.single([&]() {
        pr.du_lo[0] -= cfg.relax_da; pr.du_hi[0] += cfg.relax_da;
        pr.du_lo[1] -= cfg.relax_ddelta; pr.du_hi[1] += cfg.relax_ddelta;
      });
      solve_problem<FORM>(ex, w, pr, ss, io);
      ex.group_sync();
      ex.single([&]() { pr.du_lo[0] = lo0; pr.du_hi[0] = hi0; pr.du_lo[1] = lo1; pr.du_hi[1] = hi1; });
    } else {
      Params pr = p;
      pr.du_lo[0] -= cfg.relax_da; pr.du_hi[0] += cfg.relax_da;
      pr.du_lo[1] -= cfg.relax_ddelta; pr.du_hi[1] += cfg.relax_ddelta;
      solve_problem<FORM>(ex, w, pr, ss, io);
      ex.group_sync();
    }
    status = *io.status;
    flags |= 4;
  }
  return status;
}

// (b) The path-index rule (control_stage.py:138-141: advance when x is farther than sqrt(advance_dist2) from ref[path_idx])
// followed by the goal test (:142: within goal_radius of the goal).  Returns whether x is at the goal.
__device__ __forceinline__ bool track_advance(const cudampc_rollout_cfg& cfg, const double* refg, int len, const double* goal,
                                              const double* x, int& path_idx) {
  if (path_idx < len - 2) {
    double dx = x[0] - refg[4 * (size_t)path_idx], dy = x[1] - refg[4 * (size_t)path_idx + 1];
    if (dx * dx + dy * dy > cfg.advance_dist2) path_idx += 1;
  }
  return hypot(x[0] - goal[0], x[1] - goal[1]) < cfg.goal_radius;
}

// A vehicle that takes no step: NaN states / controls, zero step status / iters, n_steps 0
template <class Exec>
__device__ __forceinline__ void stopped_vehicle(Exec& ex, const cudampc_rollout_cfg& cfg, const RolloutArgs& a, int b, int flags) {
  const double nan_ = __longlong_as_double(0x7ff8000000000000LL);
  const int T0 = cfg.sim_steps;
  ex.stages(T0 * 4, [&](int i) { a.states[(size_t)T0 * b * 4 + i] = nan_; });
  if (a.controls) ex.stages(T0 * 2, [&](int i) { a.controls[(size_t)T0 * b * 2 + i] = nan_; });
  if (a.step_status) ex.stages(T0, [&](int i) { a.step_status[(size_t)T0 * b + i] = 0; });
  if (a.step_iters) ex.stages(T0, [&](int i) { a.step_iters[(size_t)T0 * b + i] = 0; });
  ex.single([&]() { a.n_steps[b] = 0; a.flags[b] = flags; });
}

// One vehicle, all steps (TrajectoryTracker.track loop body, control_stage.py:100-150), generic in the execution policy
template <int FORM, bool PP, class Exec>
__device__ __forceinline__ void rollout_vehicle(Exec& ex, const View& w, const Params& p, const Settings& s,
                                                const cudampc_rollout_cfg& cfg, const RolloutArgs& a, int b) {
  const int N = p.N;
  const int ws = warm_size(N);
  const int wk = 16 + 4 * (N + 1) + 2 * N;   // per-vehicle global scratch
  const double nan_ = __longlong_as_double(0x7ff8000000000000LL);
  double* wkb = a.work + (size_t)wk * b;     // [0..3] state, [4..5] u_prev, [6..7] u0, [10..11] status/iters (int), 16.. Xp, Up
  const double* refg = a.ref_global + (size_t)4 * a.ref_stride * b;
  const int len = a.ref_len[b];
  if (len < 1) {                                           // control_stage.py:71-72 raises for an empty path; per vehicle: aborted, no steps
    stopped_vehicle(ex, cfg, a, b, 2);
    return;
  }
  ex.single([&]() {
    for (int i = 0; i < 4; ++i) wkb[i] = a.state0[4 * (size_t)b + i];
    wkb[4] = 0.0; wkb[5] = 0.0;
  });
  int path_idx = 0, flags = 0, nst = 0;
  for (int step = 0; step < cfg.sim_steps; ++step) {
    unsigned long long t_step = 0;
    if (cfg.step_ns_dev) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_step));
    int* st_out = a.step_status ? a.step_status + (size_t)cfg.sim_steps * b + step : reinterpret_cast<int*>(wkb + 10);
    int* it_out = a.step_iters ? a.step_iters + (size_t)cfg.sim_steps * b + step : reinterpret_cast<int*>(wkb + 10) + 1;
    ProblemIO io;
    io.x0 = wkb; io.u_prev = wkb + 4;
    io.warm = a.warm + (size_t)ws * b; io.scratch = a.scratch + (size_t)ws * b;
    io.fsave = a.fsave ? a.fsave + (size_t)oe_doubles(N) * blockIdx.x : nullptr;
    io.u0 = wkb + 6; io.Xp = wkb + 16; io.Up = wkb + 16 + 4 * (N + 1);
    io.status = st_out; io.iters = it_out; io.pri_res = nullptr; io.dua_res = nullptr; io.info = nullptr;
    const int status = track_solve<FORM, PP>(ex, w, p, s, cfg, io, refg, path_idx, len, step > 0, flags);
    if (status != STATUS_SOLVED && status != STATUS_SOLVED_INACCURATE) { flags |= 2; break; }
    // integrate, carry u_prev, path index rule, goal test (control_stage.py:127-150)
    double xn[4];
    f_discrete_dev(p, wkb, wkb + 6, xn);
    const double u0a = wkb[6], u0d = wkb[7];
    ex.group_sync();
    ex.single([&]() {
      for (int i = 0; i < 4; ++i) { wkb[i] = xn[i]; a.states[((size_t)cfg.sim_steps * b + step) * 4 + i] = xn[i]; }
      wkb[4] = u0a; wkb[5] = u0d;
      if (a.controls) { a.controls[((size_t)cfg.sim_steps * b + step) * 2] = u0a; a.controls[((size_t)cfg.sim_steps * b + step) * 2 + 1] = u0d; }
    });
    nst = step + 1;
    const bool at_goal = track_advance(cfg, refg, len, a.goal + 2 * (size_t)b, xn, path_idx);
    if (cfg.step_ns_dev) {
      unsigned long long t_end;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_end));
      ex.single([&]() { cfg.step_ns_dev[(size_t)cfg.sim_steps * b + step] = (int)(t_end - t_step); });
    }
    if (at_goal) { flags |= 1; break; }
  }
  // rows after the vehicle stopped
  const int T = cfg.sim_steps, skip = nst + ((flags & 2) ? 1 : 0);
  ex.stages(T * 4, [&](int i) { if (i >= nst * 4) a.states[(size_t)T * b * 4 + i] = nan_; });
  if (a.controls) ex.stages(T * 2, [&](int i) { if (i >= nst * 2) a.controls[(size_t)T * b * 2 + i] = nan_; });
  if (a.step_status) ex.stages(T, [&](int i) { if (i >= skip) a.step_status[(size_t)T * b + i] = 0; });
  if (a.step_iters) ex.stages(T, [&](int i) { if (i >= skip) a.step_iters[(size_t)T * b + i] = 0; });
  ex.single([&]() { a.n_steps[b] = nst; a.flags[b] = flags; });
}

// PP: per-vehicle parameters, the Params slot follows the workspace.  A vehicle with an invalid record takes no step and is
// flagged aborted (bit 1) with invalid parameters (bit 3).
template <int FORM, bool PP>
__global__ void __launch_bounds__(32) mpc_rollout_kernel(Params p, Settings s, cudampc_rollout_cfg cfg, RolloutArgs a) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31;
  int fpad, xpad; layout_pads(p.N, fpad, xpad);
  View w{smem, p.N, fpad, xpad};
  GroupExec<1> ex{lane, 0, nullptr};
  for (int b = ex.fetch(a.counter); b < a.batch; b = ex.fetch(a.counter)) {
    if constexpr (PP) {
      Params* pb = reinterpret_cast<Params*>(smem + footprint(p.N));
      if (lane == 0) load_params(a.params, b, p, pb);
      __syncwarp();
      if (pb->N == 0) stopped_vehicle(ex, cfg, a, b, 2 | 8);
      else rollout_vehicle<FORM, true>(ex, w, *pb, s, cfg, a, b);
    } else {
      rollout_vehicle<FORM, false>(ex, w, p, s, cfg, a, b);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K_step: one closed-loop step of TrajectoryTracker.track for a batch of vehicles whose state comes from an external plant.
// The tracker state (path_idx, u_prev, n_steps, flags) lives in caller-owned device arrays between calls; the step runs the
// pieces of K_rollout (track_solve, track_advance), so with f_discrete as the plant it reproduces K_rollout's roll-out.
// ------------------------------------------------------------------------------------------------
struct StepArgs {
  const double* ref_global; const int* ref_len; int ref_stride;
  const double* goal; const double* state;
  double* warm; double* scratch; double* fsave; double* work;   // as RolloutArgs; work: Xp/Up scratch when the caller passes none
  int* path_idx; double* u_prev; int* n_steps; int* flags;
  double* u0; double* Xp; double* Up; int* status; int* iters;
  int* counter; int batch;
  const cudampc_params* params;  // per-vehicle kernels (PP): batch records, vehicle order
};

// bad (PP only): the vehicle's record is invalid; it is flagged aborted (bit 1) with invalid parameters (bit 3) and solves nothing
template <int FORM, bool PP, class Exec>
__device__ __forceinline__ void step_vehicle(Exec& ex, const View& w, const Params& p, const Settings& s,
                                             const cudampc_rollout_cfg& cfg, const StepArgs& a, int b, bool bad) {
  const int N = p.N;
  const int ws = warm_size(N);
  const int wk = 16 + 4 * (N + 1) + 2 * N;
  const double nan_ = __longlong_as_double(0x7ff8000000000000LL);
  // the solve reads state and u_prev from, and writes u0 to, the vehicle's work row as K_rollout does (the pointers of the
  // solve then share one base, which keeps this kernel within K_rollout's registers)
  double* wkb = a.work + (size_t)wk * b;
  const double* refg = a.ref_global + (size_t)4 * a.ref_stride * b;
  const int len = a.ref_len[b];
  const int stepped = a.n_steps[b] > 0;
  int flags = a.flags[b], path_idx = a.path_idx[b];
  if constexpr (PP) {
    if (len < 1) flags = bad ? 2 | 8 : 2;
    else if (bad) flags |= 2 | 8;
    else if (!(flags & 3) && stepped && track_advance(cfg, refg, len, a.goal + 2 * (size_t)b, a.state + 4 * (size_t)b, path_idx)) flags |= 1;
  } else {
    if (len < 1) flags = 2;                                // empty path: aborted, no solve (as K_rollout)
    else if (!(flags & 3) && stepped && track_advance(cfg, refg, len, a.goal + 2 * (size_t)b, a.state + 4 * (size_t)b, path_idx)) flags |= 1;
  }
  double* Xp = a.Xp ? a.Xp + (size_t)4 * (N + 1) * b : wkb + 16;
  double* Up = a.Up ? a.Up + (size_t)2 * N * b : wkb + 16 + 4 * (N + 1);
  if (!(flags & 3)) {
    ex.single([&]() {
      for (int i = 0; i < 4; ++i) wkb[i] = a.state[4 * (size_t)b + i];
      wkb[4] = a.u_prev[2 * (size_t)b]; wkb[5] = a.u_prev[2 * (size_t)b + 1];
    });
    ProblemIO io;
    io.x0 = wkb; io.u_prev = wkb + 4;
    io.warm = a.warm + (size_t)ws * b; io.scratch = a.scratch + (size_t)ws * b;
    io.fsave = a.fsave ? a.fsave + (size_t)oe_doubles(N) * blockIdx.x : nullptr;
    io.u0 = wkb + 6; io.Xp = Xp; io.Up = Up;
    io.status = a.status + b; io.iters = a.iters + b; io.pri_res = nullptr; io.dua_res = nullptr; io.info = nullptr;
    const int status = track_solve<FORM, PP>(ex, w, p, s, cfg, io, refg, path_idx, len, stepped, flags);
    if (status == STATUS_SOLVED || status == STATUS_SOLVED_INACCURATE) {
      ex.single([&]() {
        a.u0[2 * (size_t)b] = wkb[6]; a.u0[2 * (size_t)b + 1] = wkb[7];
        a.u_prev[2 * (size_t)b] = wkb[6]; a.u_prev[2 * (size_t)b + 1] = wkb[7];
        a.n_steps[b] += 1; a.path_idx[b] = path_idx; a.flags[b] = flags;
      });
      return;
    }
    flags |= 2;                                            // the reference returns (None, None, None): NaN outputs
  } else {
    ex.single([&]() { a.status[b] = 0; a.iters[b] = 0; });
  }
  // stopped or failed: NaN u0 / Xp / Up, tracker state as it was (flags and the path index of a goal test updated)
  ex.stages(4 * (N + 1), [&](int i) { Xp[i] = nan_; });
  ex.stages(2 * N, [&](int i) { Up[i] = nan_; });
  ex.single([&]() { a.u0[2 * (size_t)b] = nan_; a.u0[2 * (size_t)b + 1] = nan_; a.path_idx[b] = path_idx; a.flags[b] = flags; });
}

// PP: as K_rollout; an invalid vehicle's slot gets the launch's horizon (the sizes of its NaN outputs), and bad = true stops it
template <int FORM, bool PP>
__global__ void __launch_bounds__(32) mpc_track_step_kernel(Params p, Settings s, cudampc_rollout_cfg cfg, StepArgs a) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31;
  int fpad, xpad; layout_pads(p.N, fpad, xpad);
  View w{smem, p.N, fpad, xpad};
  GroupExec<1> ex{lane, 0, nullptr};
  for (int b = ex.fetch(a.counter); b < a.batch; b = ex.fetch(a.counter)) {
    if constexpr (PP) {
      Params* pb = reinterpret_cast<Params*>(smem + footprint(p.N));
      int bad = 0;
      if (lane == 0) {
        load_params(a.params, b, p, pb);
        bad = pb->N == 0;
        if (bad) pb->N = p.N;
      }
      bad = __shfl_sync(0xffffffffu, bad, 0);
      step_vehicle<FORM, true>(ex, w, *pb, s, cfg, a, b, bad != 0);
    } else {
      step_vehicle<FORM, false>(ex, w, p, s, cfg, a, b, false);
    }
  }
}


// ------------------------------------------------------------------------------------------------
// Instantiations and their launchers
// ------------------------------------------------------------------------------------------------
// K_solve: one warp per problem with the short (N+1 <= 32), pair (N+1 <= 64) or general form of the phases, two warps per
// problem (general form, long horizons); K_rollout and K_step: one warp per vehicle, any of the three forms (mpc_solve.h FORM_*),
// both in the rollout's translation unit of that form.
enum SolveVariant { SOLVE_W1_SHORT = 0, SOLVE_W1 = 1, SOLVE_W2 = 2, SOLVE_W1_PAIR = 3, SOLVE_W2_REG = 4, SOLVE_W1_REG = 5 };
// pp: the per-problem-parameter instantiation of the same variant / form
cudaError_t solve_set_smem(int variant, int bytes, bool pp = false);
void solve_launch(int variant, int grid, int threads, int smem, cudaStream_t st, const Params& p, const Settings& s, const BatchArgs& a, int P, int F, bool pp = false);
cudaError_t rollout_set_smem(int form, int bytes, bool pp = false);
cudaError_t rollout_occupancy(int form, int bytes, int* blocks_per_sm, bool pp = false);
void rollout_launch(int form, int grid, int smem, cudaStream_t st, const Params& p, const Settings& s, const cudampc_rollout_cfg& cfg, const RolloutArgs& a, bool pp = false);
cudaError_t step_set_smem(int form, int bytes, bool pp = false);
void step_launch(int form, int grid, int smem, cudaStream_t st, const Params& p, const Settings& s, const cudampc_rollout_cfg& cfg, const StepArgs& a, bool pp = false);
