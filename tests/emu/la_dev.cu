// la_dev.cu — TEST INFRASTRUCTURE (tests/test_linear_solves.py): the linear solves of the kernels, one operation at a time, on
// the device.  Each group of WPP warps places one system into its workspace (tests/emu/la_systems.h), runs the product's
// lane code (mpc_exec.cuh: oe_factor_lanes, oe_forward_lanes / oe_backward_lanes, factor_twisted_lanes / chain_twisted_lanes
// through GroupExec) or the one-lane statements on lane 0 of the group, and returns the solution and the factor area.
// P groups share a CTA as in the product, so chain_warp() and the named barriers 1 + grp() of several groups are exercised.
//
// Write check: every word of shared memory (all groups' workspaces, the GroupShared slots) is first filled with a marked NaN
// (its index in the payload), then the inputs are placed and the image is saved to global memory.  After the run every word
// that the mode may not write (la::writable, the same for every group) must be bit-identical to its saved value.
// Never linked into libcudampc.so.
#include <cuda_runtime.h>
#include "la_systems.h"
#include "../../rrt_mpc_b200/csrc/mpc_exec.cuh"

using namespace mpc;

namespace {

struct LaArgs {
  int mode, lanes, N, nsys, P, F, words;
  Params p; Settings s;
  const double* rho;           // [nsys]                        (B)
  const double* x0;            // [nsys][4]                     (B, C)
  const double* ref;           // [nsys][N+1][4]                (B, C)
  const int* act;              // [nsys][N+2]                   (C)
  const double* S;             // [nsys][J][36]                 (A)
  const double* Fb;            // [nsys][J][36]                 (A)
  const double* b;             // [nsys][J][6] (A) or [nsys][N+1][6]
  double* x;                   // same shape as b
  double* fac;                 // [nsys][oe_doubles(N)]         (A, B)
  double* snap;                // [grid][words]: the shared-memory image before the run
  const unsigned char* wmask;  // [F]: 1 = a group may change this word of its workspace
  int* changed;                // [0]: protected words that changed, [1..64]: the first of them (CTA * words + word)
};

constexpr int MAX_CHANGED = 64;

__device__ __forceinline__ double canary(int i) { return __longlong_as_double(0x7ff4dead00000000LL | (long long)i); }

template <int WPP>
__global__ void __launch_bounds__(256, 1) la_kernel(const __grid_constant__ LaArgs a) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = warp / WPP, N = a.N;
  const int sys = blockIdx.x * a.P + g;
  const bool on = sys < a.nsys;                  // uniform over the group: its barriers are all or nothing
  GroupShared* sh = reinterpret_cast<GroupShared*>(smem + (size_t)a.P * a.F) + g;
  GroupExec<WPP> ex{lane, warp, sh};
  const View w = la::view(smem + (size_t)g * a.F, N);
  const Params& p = a.p;
  const Settings& s = a.s;
  for (int i = threadIdx.x; i < a.words; i += blockDim.x) smem[i] = canary(i);
  __syncthreads();

  const int J = oe_neven(N), nx = a.mode == la::MODE_RED ? 6 * J : 6 * (N + 1);
  const double* b = a.b + (size_t)nx * sys;
  if (on) {
    if (a.mode == la::MODE_RED) {
      const double* S = a.S + (size_t)36 * J * sys;
      const double* F = a.Fb + (size_t)36 * J * sys;
      ex.stages(J, [&](int j) { la::red_place(w, S, F, b, j); });
    } else {
      const double* ref = a.ref + (size_t)4 * (N + 1) * sys;
      ex.single([&]() { la::prob_head(w, a.x0 + 4 * (size_t)sys, ref, a.mode == la::MODE_POLISH ? a.act + (size_t)(N + 2) * sys : nullptr); });
      ex.stages(N + 1, [&](int k) { la::prob_stage(w, p, ref, k); });
    }
  }
  __syncthreads();
  double* snap = a.snap + (size_t)a.words * blockIdx.x;
  for (int i = threadIdx.x; i < a.words; i += blockDim.x) snap[i] = smem[i];
  __syncthreads();

  if (on) {
    const OEView oe = oe_view(w);
    if (a.mode == la::MODE_RED) {
      if (a.lanes) {
        if (ex.chain_warp()) oe_factor_lanes(lane, w, oe);
        ex.group_sync();
        ex.oe_forward(w, oe);
        ex.stages_par(N + 1, 0, [&](int k) { oe_diag_stage(w, oe, k); });
        ex.oe_backward(w, oe);
      } else {
        ex.single([&]() { la::red_solve_seq(w); });
      }
    } else if (a.mode == la::MODE_ADMM) {
      const double rho = a.rho[sys];
      if (a.lanes) {
        const IterConst c = iter_const(w, p, s, rho);
        ex.oe_factor(w, p, admm_mode(rho, s), oe);
        ex.stages(N + 1, [&](int k) { la::admm_place(w, oe, b, k); });
        ex.stages_par(N + 1, 0, [&](int k) { oe_even_fixup(w, p, c, k); });
        ex.oe_forward(w, oe);
        ex.stages_par(N + 1, 0, [&](int k) { oe_diag_stage(w, oe, k); });
        ex.oe_backward(w, oe);
        ex.stages_par(N + 1, 1, [&](int k) { oe_expand_odd(w, p, c, oe, k); });
      } else {
        ex.single([&]() { la::admm_seq(w, p, s, rho, b); });
      }
    } else {
      if (a.lanes) {
        const Mode m = polish_mode(s);
        ex.stages(N + 1, [&](int k) { assemble_stage(w, p, m, k); });
        ex.factor(w);
        ex.stages(N + 1, [&](int k) { la::pol_place(w, b, k); });
        ex.solve(w);
      } else {
        ex.single([&]() { la::pol_seq(w, p, s, b); });
      }
    }
  }
  __syncthreads();

  const int gw = a.P * a.F;                      // words behind the workspaces: the GroupShared slots (never written here)
  for (int i = threadIdx.x; i < a.words; i += blockDim.x) {
    const bool may = i < gw && a.wmask[i % a.F];
    if (!may && __double_as_longlong(smem[i]) != __double_as_longlong(snap[i])) {
      const int n = atomicAdd(a.changed, 1);
      if (n < MAX_CHANGED) a.changed[1 + n] = blockIdx.x * a.words + i;
    }
  }
  if (on) {
    double* x = a.x + (size_t)nx * sys;
    if (a.mode == la::MODE_RED) ex.stages(J, [&](int j) { la::red_read(w, x, j); });
    else if (a.mode == la::MODE_ADMM) ex.stages(N + 1, [&](int k) { la::admm_read(w, x, k); });
    else ex.stages(N + 1, [&](int k) { la::pol_read(w, x, k); });
    if (a.mode != la::MODE_POLISH) {
      const int nf = oe_doubles(N);
      double* fac = a.fac + (size_t)nf * sys;
      const double* src = w.base + band_offset(N);
      ex.stages(nf, [&](int t) { fac[t] = src[t]; });
    }
  }
}

constexpr int SMEM_MAX = 227 * 1024;

}  // namespace

extern "C" {

int la_group_shared_bytes() { return (int)sizeof(GroupShared); }

// groups per CTA and shared-memory words per CTA for horizon N with WPP warps per group: up to 8 one-warp or 4 two-warp
// groups, as many as fit 227 KB.  Returns 0 if not even one group fits.
int la_geometry(int wpp, int N, int* P, int* words) {
  const int F = footprint(N);
  const int per = F * 8 + (int)sizeof(GroupShared);
  int q = wpp == 2 ? 4 : 8;
  while (q > 0 && q * per > SMEM_MAX) --q;
  *P = q;
  *words = (q * per + 7) / 8;
  return q;
}

// One launch on `stream` over nsys systems (device pointers from torch tensors; par / set are host arrays, la::unpack).
// Returns a cudaError_t value (0 = launched).
int la_run(int wpp, int mode, int lanes, int N, int nsys, const double* par, const double* set, const double* rho,
           const double* x0, const double* ref, const int* act, const double* S, const double* Fb, const double* b,
           double* x, double* fac, double* snap, const unsigned char* wmask, int* changed, void* stream) {
  LaArgs a;
  a.mode = mode; a.lanes = lanes; a.N = N; a.nsys = nsys; a.F = footprint(N);
  la::unpack(par, set, N, a.p, a.s);
  a.rho = rho; a.x0 = x0; a.ref = ref; a.act = act; a.S = S; a.Fb = Fb; a.b = b; a.x = x; a.fac = fac;
  a.snap = snap; a.wmask = wmask; a.changed = changed;
  if (la_geometry(wpp, N, &a.P, &a.words) == 0) return (int)cudaErrorInvalidValue;
  const int grid = (nsys + a.P - 1) / a.P, threads = 32 * wpp * a.P, bytes = a.words * 8;
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e;
  if (wpp == 2) {
    e = cudaFuncSetAttribute(la_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return (int)e;
    la_kernel<2><<<grid, threads, bytes, st>>>(a);
  } else {
    e = cudaFuncSetAttribute(la_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return (int)e;
    la_kernel<1><<<grid, threads, bytes, st>>>(a);
  }
  return (int)cudaGetLastError();
}

}
