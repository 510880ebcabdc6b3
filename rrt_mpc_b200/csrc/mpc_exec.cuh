// mpc_exec.cuh — CUDA execution policy for the per-problem driver (mpc_solve.h): how stage-parallel
// phases, reductions and the sequential chain operations map onto the warps that own a problem.
#pragma once
#include <cuda_runtime.h>
#include "mpc_solve.h"

namespace mpc {

// One lane sweeps one half of one problem: `bottom` selects the half, `partner` is the lane that holds the other
// half of the same problem.  Called by ALL 32 lanes of the warp (inactive lanes only take part in the shuffles).
// PIPE selects the sweep variant of mpc_core.h: 0 plain, 1 two register sets, 2 rolling refill.
template <int PIPE>
__device__ __forceinline__ void chain_twisted_lanes(bool active, bool bottom, int partner, const View& w) {
  double a[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0}, o[6], xm[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  const HalfView h = bottom ? w.bottom() : w.top();
  if (active) half_forward<PIPE>(h, a);
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 6; ++j) o[j] = __shfl_sync(0xffffffffu, a[5 - j], partner);      // partner's border accumulators, index-reversed
  if (active && !bottom) {
#pragma unroll
    for (int j = 0; j < 6; ++j) a[j] += o[j];
    middle_solve(w, a, xm);
  }
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 6; ++j) o[j] = __shfl_sync(0xffffffffu, xm[5 - j], partner);     // bottom lanes receive the reversed middle solution
  if (active) half_backward<PIPE>(h, bottom ? o : xm);
  __syncwarp();
}
// twisted factorisation of local stages [i0, i1) of both halves by two lanes; `last` also forms the middle block
__device__ __forceinline__ void factor_twisted_lanes(int lane, const View& w, int i0, int i1, bool last) {
  const HalfView h = lane == 1 ? w.bottom() : w.top();
  if (lane < 2) factor_half(h, i0, i1);            // ONE instruction stream for both halves (two branches would serialise them)
  __syncwarp();
  if (last && lane == 0) factor_middle(w);
  __syncwarp();
}

// ------------------------------------------------------------------------------------------------
// Sweeps of the odd-even block solve (mpc_oe.h), one lane per ROW of a half: lanes 0..5 the top half, 6..11 the bottom
// half, one instruction stream.  Called by all 32 lanes of the chain warp (lanes >= 12 only keep the warp converged).
// Per step and lane: 3 x LDS.128 (block row, requested one step ahead) + 6 fmas + one 64-bit store of its element of the
// new vector, __syncwarp, 3 x LDS.128 to read the whole vector back.  The loop is branch-free: both halves run the trip
// count of the longer one, a half that is done keeps computing on in-bounds words of the workspace and stores nothing
// (predicated), so the warp never diverges inside the dependent chain.  Shared-memory accesses are explicit PTX on 32-bit
// shared addresses (through generic pointers every access pays an address-space conversion), two register sets, unrolled
// by two.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void lds_row(unsigned a, double* r) {
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(r[0]), "=d"(r[1]) : "r"(a));
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2+16];" : "=d"(r[2]), "=d"(r[3]) : "r"(a));
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2+32];" : "=d"(r[4]), "=d"(r[5]) : "r"(a));
}
__device__ __forceinline__ void lds_col(unsigned a, double* r) {       // six doubles 48 bytes apart (a block column)
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(r[0]) : "r"(a));
  asm volatile("ld.shared.f64 %0, [%1+48];" : "=d"(r[1]) : "r"(a));
  asm volatile("ld.shared.f64 %0, [%1+96];" : "=d"(r[2]) : "r"(a));
  asm volatile("ld.shared.f64 %0, [%1+144];" : "=d"(r[3]) : "r"(a));
  asm volatile("ld.shared.f64 %0, [%1+192];" : "=d"(r[4]) : "r"(a));
  asm volatile("ld.shared.f64 %0, [%1+240];" : "=d"(r[5]) : "r"(a));
}
__device__ __forceinline__ double lds_f64(unsigned a) { double v; asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts_f64_if(bool p, unsigned a, double v) {
  asm volatile("{ .reg .pred q; setp.ne.u32 q, %0, 0; @q st.shared.f64 [%1], %2; }" ::"r"((unsigned)p), "r"(a), "d"(v) : "memory");
}
// The twelve row lanes run the sweep inside ONE divergent region (the other twenty lanes of the warp wait at its end), with
// warp barriers and shuffles over the twelve-lane mask.  With all 32 lanes executing the loads (the idle ones on duplicate
// addresses, to keep the warp converged) every 128-bit load cost the shared-memory pipe 4-5 wavefronts instead of 2: with
// five chain warps per SM that saturated the pipe - 108 cycles per step alone, 170 with five warps sweeping
// (tools/microbench/oe_bench.cu).  The loop is branch-free between the two halves: both run the trip count of the longer
// one, a half that is done keeps computing on in-bounds words of the workspace and stores nothing (predicated).
#define MPC_ROW_LANES 0x00000fffu
__device__ __forceinline__ void oe_forward_lanes(int lane, const View& w, const OEView& oe) {
  if (lane < 12) {
    const bool bottom = lane >= 6;
    const int r = bottom ? lane - 6 : lane;
    const OEHalf h = oe_half(w, oe, bottom);
    const int cnt = h.cnt, cmax = oe.jm > oe.nb ? oe.jm : oe.nb;     // uniform trip count
    const int xs = h.xstep * 8;                                      // bytes between consecutive local rows (+-48)
    const unsigned xlast = smem_u32(h.xlast) + 8 * r;
    unsigned xrow = smem_u32(h.x0) + xs;                             // row of local stage i (i = 1)
    unsigned gp = smem_u32(h.g0) + 48 * r;                           // row r of the block of step i
    double a[6], gA[6], gB[6], nbA, nbB, y;
    lds_row(smem_u32(h.x0), a);                                      // y_0 = b'_0
    double ymid = lds_f64(xlast);                                    // the half's term for the middle if it has no step
    lds_row(gp, gA); nbA = lds_f64(cnt == 1 ? xlast : xrow + 8 * r);
    for (int i = 1; i <= cmax; i += 2) {
      lds_row(gp + 288, gB); nbB = lds_f64(i + 1 == cnt ? xlast : xrow + xs + 8 * r);          // step i+1
      y = oe_row_dot(gA, nbA, a);
      ymid = (i == cnt) ? y : ymid;
      sts_f64_if(i < cnt, xrow + 8 * r, y);
      __syncwarp(MPC_ROW_LANES);
      lds_row(xrow, a);
      if (i + 1 > cmax) break;
      lds_row(gp + 576, gA); nbA = lds_f64(i + 2 == cnt ? xlast : xrow + 2 * xs + 8 * r);      // step i+2
      y = oe_row_dot(gB, nbB, a);
      ymid = (i + 1 == cnt) ? y : ymid;
      sts_f64_if(i + 1 < cnt, xrow + xs + 8 * r, y);
      __syncwarp(MPC_ROW_LANES);
      lds_row(xrow + xs, a);
      gp += 576; xrow += 2 * xs;
    }
    // middle stage: x_m = S'_m^-1 (top term + bottom term); lanes r and r + 6 hold element r of the two terms
    const double yo = __shfl_sync(MPC_ROW_LANES, ymid, bottom ? lane - 6 : lane + 6);
    double* mrow = w.nx(2 * oe.jm);
    if (lane < 6) mrow[r] = ymid + yo;
    __syncwarp(MPC_ROW_LANES);
    double xm = 0.0;
    if (lane < 6) {
      double s[6];
      row_load(mrow, s);
      xm = oe_sym_row(oe.sinv + OE_SYM * oe.jm, r, s);
    }
    __syncwarp(MPC_ROW_LANES);
    if (lane < 6) mrow[r] = xm;
  }
  __syncwarp();
}
__device__ __forceinline__ void oe_backward_lanes(int lane, const View& w, const OEView& oe) {
  if (lane < 12) {
    const bool bottom = lane >= 6;
    const int c = bottom ? lane - 6 : lane;
    const OEHalf h = oe_half(w, oe, bottom);
    const int cmax = oe.jm > oe.nb ? oe.jm : oe.nb;
    const int xs = h.xstep * 8;
    int i = h.cnt - 1;                                               // local stage of this half at the current step (< 0: done)
    unsigned xrow = smem_u32(h.x0) + xs * i;                         // row of local stage i
    unsigned gp = smem_u32(h.g0) + 288 * i + 8 * c;                  // column c of the block of step i+1
    double a[6], gA[6], gB[6], zA, zB;
    lds_row(smem_u32(w.nx(2 * oe.jm)), a);                           // x_m
    lds_col(gp, gA); zA = lds_f64(xrow + 8 * c);
    for (int s = 0; s < cmax; s += 2, i -= 2) {
      lds_col(gp - 288, gB); zB = lds_f64(xrow - xs + 8 * c);        // local stage i-1
      sts_f64_if(i >= 0, xrow + 8 * c, oe_row_dot(gA, zA, a));
      __syncwarp(MPC_ROW_LANES);
      lds_row(xrow, a);
      if (s + 1 >= cmax) break;
      lds_col(gp - 576, gA); zA = lds_f64(xrow - 2 * xs + 8 * c);    // local stage i-2
      sts_f64_if(i - 1 >= 0, xrow - xs + 8 * c, oe_row_dot(gB, zB, a));
      __syncwarp(MPC_ROW_LANES);
      lds_row(xrow - xs, a);
      gp -= 576; xrow -= 2 * xs;
    }
  }
  __syncwarp();
}

// Sequential half of the ADMM factorisation (mpc_oe.h oe_factor_half) in the same row lanes: at step i, lane r of a half
// forms row r of G_{i+1} = F_{i+1} S'_i^-1 and row r of the update G_{i+1} F_{i+1}' of S'_{i+1} (no lane needs another lane's
// row of G).  Every lane of the half inverts the 6x6 pivot itself with spd6_inverse, and every entry is formed by the
// statements of oe_factor_half, so the factor is bit-identical to the one-lane version.  The two halves can differ by one
// step: a warp barrier covers the lanes whose half has step i.  The middle stage (oe_factor_middle) stays on one lane.
__device__ __forceinline__ void oe_factor_lanes(int lane, const View& w, const OEView& oe) {
  if (lane < 12) {
    const bool bottom = lane >= 6;
    const int r = bottom ? lane - 6 : lane;
    const OEHalf h = oe_half(w, oe, bottom);
    double u[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};                   // row r of the middle's update U (entries c <= r)
#pragma unroll 1
    for (int i = 0; i < h.cnt; ++i) {
      const unsigned mask = (i < oe.jm ? 0x3fu : 0u) | (i < oe.nb ? 0xfc0u : 0u);
      double* sp = h.s0 + h.sstep * i;
      double S[6][6], sv[OE_SYM];
      sym_load(sp, sv);
      sym_expand(sv, S);
      spd6_inverse(S, sv);
      sym_expand(sv, S);                                           // S = S'_i^-1 (full)
      double* g = h.g0 + OE_G * i;                                 // block of step i+1
      double F[OE_G], Fr[6], G[6];
      blk_load(g, F);
      row_load(g + 6 * r, Fr);
      __syncwarp(mask);                                            // S'_i and F read by the whole half before they are overwritten
      if (r == 0) {
#pragma unroll
        for (int t = 0; t < OE_SYM; ++t) sp[t] = sv[t];
      }
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        double acc = Fr[0] * S[0][c];
#pragma unroll
        for (int t = 1; t < 6; ++t) acc = fma(Fr[t], S[t][c], acc);
        G[c] = acc;
      }
      row_store(g + 6 * r, G);
      double* sn = h.s0 + h.sstep * (i + 1) + MPC_SP(r, 0);         // row r of S'_{i+1}
      const bool last = (i + 1 == h.cnt);
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        if (c > r) break;
        double acc = G[0] * F[6 * c];
#pragma unroll
        for (int t = 1; t < 6; ++t) acc = fma(G[t], F[6 * c + t], acc);
        if (last) u[c] = acc; else sn[c] -= acc;
      }
      __syncwarp(mask);                                            // S'_{i+1} complete
    }
    // middle stage: S'_m = S_m - U_top - U_bot (row r by lane r), then inverted by lane 0
    double uo[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) uo[c] = __shfl_sync(MPC_ROW_LANES, u[c], bottom ? lane : lane + 6);
    double* sm = oe.sinv + OE_SYM * oe.jm;
    if (!bottom) {
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        if (c > r) break;
        sm[MPC_SP(r, c)] -= u[c] + uo[c];
      }
    }
    __syncwarp(MPC_ROW_LANES);
    if (lane == 0) {
      double S[6][6], sv[OE_SYM];
      sym_load(sm, sv);
      sym_expand(sv, S);
      spd6_inverse(S, sv);
#pragma unroll
      for (int t = 0; t < OE_SYM; ++t) sm[t] = sv[t];
    }
  }
  __syncwarp();
}

__device__ __forceinline__ int next_problem_warp(int* counter, int lane) {
  int p = 0;
  if (lane == 0) p = atomicAdd(counter, 1);
  return __shfl_sync(0xffffffffu, p, 0);
}

// ------------------------------------------------------------------------------------------------
// Group execution policy: a group of WPP warps owns one problem and runs it independently of every other group in
// the CTA (no CTA-wide rendezvous).  Stage-parallel phases stride over the 32*WPP lanes of the group; the twisted
// sweeps / factorisation run in two lanes of ONE warp of the group, chosen so that the chain warps of the resident
// groups spread over the four SM sub-partitions (warp w issues on sub-partition w % 4).
// ------------------------------------------------------------------------------------------------
struct GroupShared {
  int next;
  int anyv[2];
  double red[2][8];
  Drv drv;            // register form: the driver's state between its pieces (mpc_drv.h); drv.ic is read inside the blocks
};

// Register form (mpc_reg.h): a block of nb iterations of one problem by its two warps.  Meant to be inlined at the TOP LEVEL
// of the kernel (mpc_kernels.cuh: mpc_solve_reg_kernel), where nothing else is alive: there the stage record, the
// temporaries of the fused pass and the sweeps fit the 255 registers without a spill (250 used).  Inlined into the driver,
// or as a real call (callee-saved registers of the ABI), ptxas parks part of the record in local memory, which with 227 KB
// of shared memory carved out of the L1 is slow.  `ev`: this warp owns the even stages and runs the sweeps.
// WPP = 2: two warps per problem (lane j of the even / odd warp owns stage 2j / 2j+1, 64-thread named barriers);
// WPP = 1: horizons with N + 1 <= 32, one warp per problem, lane k owns stage k (parity = parity of the lane, warp barriers).
template <int STATE, int WPP>
__device__ __forceinline__ void reg_block_run(double* base, int N, int fpad, int xpad, double dt, const IterConst* csm, int nb,
                                           int lane, int ev_warp, int bar_id, unsigned long long* tags) {
#ifdef MPC_TIMING     // dev builds: cycles of the parts of an iteration as the even warp's lane 0 sees them (tags 20..26)
  long long tq = clock64(), tacc[7] = {0, 0, 0, 0, 0, 0, 0};
#define MPC_BTAG(n) do { const long long now_ = clock64(); tacc[(n) - 20] += now_ - tq; tq = now_; } while (0)
#else
#define MPC_BTAG(n) do { } while (0)
#endif
  const View w{base, N, fpad, xpad};
  const OEView oe = oe_view(w);
  const volatile IterConst& c = *csm;          // read where used (see mpc_pair.h: pair_stage)
  Params p;
  p.dt = dt; p.N = N;
  const int k = WPP == 2 ? 2 * lane + (ev_warp ? 0 : 1) : lane;
  const bool ev = WPP == 2 ? ev_warp != 0 : !(lane & 1);          // this lane owns an even stage
  const bool sweeper = WPP == 2 ? ev_warp != 0 : true;              // this warp runs the sweeps (its lanes 0..11)
  const bool on = k <= N;
  // every word defined here: a register that is read without a definition on some path (the lanes beyond the horizon) is
  // live from the kernel's entry, i.e. across the driver's code as well
  StageRegs R;
  StageTmp T;
#pragma unroll
  for (int j = 0; j < SR; ++j) R.r[j] = 0.0;
#pragma unroll
  for (int j = 0; j < 6; ++j) { T.xt[j] = 0.0; T.xn[j] = 0.0; T.b[j] = 0.0; }
#pragma unroll
  for (int j = 0; j < 5; ++j) T.G[j] = 0.0;
  T.ua = 0.0; T.ud = 0.0;
  if (on) reg_load<STATE>(w, k, R);
  // One loop for both warp roles: the update and the right-hand side are ONE copy of code shared by the two warps (two
  // loops - one per role - measured slower with early polish: the iteration loop competes for the 32 KB instruction cache
  // with the polish code other resident problems run).
#define MPC_BAR() do { if (WPP == 2) asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory"); else __syncwarp(); } while (0)
#pragma unroll 1
  for (int i = 0; i < nb; ++i) {
    MPC_BTAG(26);
    if (sweeper) {
      oe_forward_lanes(lane, w, oe);
      MPC_BTAG(20);
      if (ev && on) oe_diag_stage(w, oe, k);
      __syncwarp();
      MPC_BTAG(21);
      oe_backward_lanes(lane, w, oe);
      MPC_BTAG(22);
    }
    MPC_BAR();                                        // B_a: x~ of the even stages
    if (!ev && on) reg_expand(w, p, c, oe, k, R, T);
    MPC_BAR();                                        // B_b: x~ of the odd stages
    MPC_BTAG(23);
    if (ev && on) reg_gather_even(w, k, T);
    if (on) reg_update<STATE>(w, p, c, k, R, T);
    MPC_BAR();                                        // B_c: (d, G) of every stage
    MPC_BTAG(24);
    if (on) reg_rhs<STATE>(w, p, c, oe, k, R, T);
    MPC_BAR();                                        // B_d: t_o
    MPC_BTAG(25);
    if (ev && on) reg_fixup(w, p, c, k, T);
    if (sweeper) __syncwarp();
  }
#ifdef MPC_TIMING
  if (sweeper && lane == 0 && tags) for (int q = 0; q < 7; ++q) atomicAdd(&tags[20 + q], (unsigned long long)tacc[q]);
#endif
  MPC_BAR();
  if (on) reg_store<STATE>(w, k, R);
  MPC_BAR();
}

template <int WPP>
struct GroupExec {
  int lane, warp;     // warp index within the CTA
  GroupShared* sh;    // this group's slot
  __device__ __forceinline__ int grp() const { return warp / WPP; }
  __device__ __forceinline__ int sub() const { return warp % WPP; }
  __device__ __forceinline__ int gl() const { return sub() * 32 + lane; }
  // groups 0,1,2,3,4,5 (warps 2g, 2g+1) -> chain warps 0,2,5,7,8,10 -> sub-partitions 0,2,1,3,0,2
  __device__ __forceinline__ bool chain_warp() const { return WPP == 1 || sub() == ((grp() >> 1) & 1); }
  __device__ __forceinline__ void group_sync() const {
    if (WPP == 1) __syncwarp();
    else asm volatile("bar.sync %0, %1;" ::"r"(1 + grp()), "r"(32 * WPP) : "memory");
  }
#ifdef MPC_TIMING     // dev builds only (tools/tag_times.py): cycles between consecutive tags, summed per tag over the launch
  long long t_last = 0; int t_cur = 0; unsigned long long* tags = nullptr;
  __device__ __forceinline__ void tag(int n) {
    const long long now = clock64();
    if (gl() == 0 && t_last && tags) atomicAdd(&tags[t_cur], (unsigned long long)(now - t_last));
    t_last = now; t_cur = n;
  }
#else
  __device__ __forceinline__ void tag(int) {}
#endif
  template <class Fn> __device__ __forceinline__ void stages(int n, Fn f) {
    for (int k = gl(); k < n; k += 32 * WPP) f(k);
    group_sync();
  }
  // stages of one parity (par = 1: odd, 0: even), lanes over them
  template <class Fn> __device__ __forceinline__ void stages_par(int n, int par, Fn f) {
    for (int k = 2 * gl() + par; k < n; k += 64 * WPP) f(k);
    group_sync();
  }
  template <class Fn> __device__ __forceinline__ void single(Fn f) {
    if (gl() == 0) f();
    group_sync();
  }
  template <class Fn> __device__ __forceinline__ void reduce_max(int n, double* r, int nr, Fn f) {
    for (int i = 0; i < nr; ++i) r[i] = 0.0;
    for (int k = gl(); k < n; k += 32 * WPP) f(k, r);
    for (int i = 0; i < nr; ++i) {
      double v = r[i];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
      r[i] = v;
    }
    if (WPP > 1) {
      if (lane == 0) for (int i = 0; i < nr; ++i) sh->red[sub()][i] = r[i];
      group_sync();
      for (int i = 0; i < nr; ++i) r[i] = fmax(sh->red[0][i], sh->red[1][i]);
    }
    group_sync();
  }
  template <class Fn> __device__ __forceinline__ int any(int n, Fn f) {
    int a = 0;
    for (int k = gl(); k < n; k += 32 * WPP) a |= f(k);
    a = __any_sync(0xffffffffu, a);
    if (WPP > 1) {
      if (lane == 0) sh->anyv[sub()] = a;
      group_sync();
      a = sh->anyv[0] | sh->anyv[1];
    }
    group_sync();
    return a;
  }
  __device__ __forceinline__ int fetch(int* counter) {
    if (WPP == 1) return next_problem_warp(counter, lane);
    if (gl() == 0) sh->next = atomicAdd(counter, 1);
    group_sync();
    const int b = sh->next;
    group_sync();
    return b;
  }
  // callers reach solve()/factor() right after a phase's group_sync, so the right-hand side / band is visible
  __device__ __forceinline__ void solve(const View& w) {           // polish / refinement solves: compact code
    if (chain_warp()) chain_twisted_lanes<0>(lane < 2, lane == 1, lane ^ 1, w);
    group_sync();
  }
  // ---- odd-even block solve of the ADMM iterations (mpc_oe.h): stage-parallel parts with lanes over stages, the two
  // halves of the reduced system in lanes 0 (top) and 1 (bottom) of the group's chain warp, one instruction stream
  __device__ __forceinline__ void oe_factor(const View& w, const Params& p, const Mode& m, const OEView& oe) {
    stages_par(w.N + 1, 1, [&](int k) { oe_factor_odd(w, p, m, oe, k); });
    stages_par(w.N + 1, 0, [&](int k) { oe_factor_even(w, p, m, oe, k); });
    if (chain_warp()) oe_factor_lanes(lane, w, oe);
    group_sync();
  }
  __device__ __forceinline__ void oe_forward(const View& w, const OEView& oe) {
    if (chain_warp()) oe_forward_lanes(lane, w, oe);
    group_sync();
  }
  __device__ __forceinline__ void oe_backward(const View& w, const OEView& oe) {
    if (chain_warp()) oe_backward_lanes(lane, w, oe);
    group_sync();
  }
  // ---- pair form of an iteration (mpc_pair.h): one lane per pair of stages, neighbours exchanged through shuffles.
  // One warp per problem only (N + 1 <= 64).
  __device__ __forceinline__ void pair_pass(const View& w, const Params& p, const IterConst& c, const OEView& oe) {
    const unsigned full = 0xffffffffu;
    const bool on = lane < pair_lanes(w.N);
    PairCtx cx;        // every word defined on every path (a register read without a definition is live from the kernel's entry)
#pragma unroll
    for (int j = 0; j < 6; ++j) { cx.xe[j] = 0.0; cx.xo[j] = 0.0; cx.xn[j] = 0.0; cx.be[j] = 0.0; cx.bo[j] = 0.0; cx.t[j] = 0.0; }
#pragma unroll
    for (int j = 0; j < 4; ++j) { cx.de[j] = 0.0; cx.dd[j] = 0.0; }
#pragma unroll
    for (int j = 0; j < 5; ++j) { cx.Ge[j] = 0.0; cx.Go[j] = 0.0; }
    if (on) pair_expand(w, p, c, oe, lane, cx);
    double ua = __shfl_up_sync(full, cx.xo[4], 1), ud = __shfl_up_sync(full, cx.xo[5], 1);
    if (lane == 0) { ua = 0.0; ud = 0.0; }
    if (on) pair_update(w, p, c, lane, cx, ua, ud);
    double dprev[4], rnext[2], tprev[6];
#pragma unroll
    for (int r = 0; r < 4; ++r) dprev[r] = __shfl_up_sync(full, cx.dd[r], 1);
#pragma unroll
    for (int i = 0; i < 2; ++i) rnext[i] = __shfl_down_sync(full, cx.Ge[3 + i], 1);
    if (on) pair_rhs(w, p, c, oe, lane, cx, dprev, rnext);
#pragma unroll
    for (int j = 0; j < 6; ++j) tprev[j] = __shfl_up_sync(full, cx.t[j], 1);
    if (on) pair_fixup(w, p, c, lane, cx, tprev);
    group_sync();
  }
  // ---- register form of the iterations (mpc_reg.h): two warps per problem, the chain warp owns the even stages and runs
  // the sweeps, the other warp the odd stages; lane j <-> stage 2j (+1).  nb iterations, then the records are written back.
  __device__ __forceinline__ void admm_block(const View& w, const Params& p, const IterConst& c, const OEView&, int nb) {
    // generic path (state in the records); the product kernels are mpc_solve_reg_kernel<.., WPP>
    if (gl() == 0) sh->drv.ic = c;
    group_sync();
#ifdef MPC_TIMING
    unsigned long long* tg = tags;
#else
    unsigned long long* tg = nullptr;
#endif
    reg_block_run<0, WPP>(w.base, w.N, w.fpad, w.xpad, p.dt, &sh->drv.ic, nb, lane, chain_warp() ? 1 : 0, 1 + grp(), tg);
  }
  __device__ __forceinline__ void factor(const View& w) {
    if (chain_warp()) factor_twisted_lanes(lane, w, 0, max(half_top(w.N), half_bot(w.N)), true);
    group_sync();
  }
};

}  // namespace mpc
