// mpc_reg.h — the "register" form of the ADMM iterations: every stage is owned by ONE lane that keeps the stage's state
// (x/u, slacks, merged row states, dynamics duals, s-tilde: 35 doubles of mpc_core.h's stage record) in REGISTERS for a whole
// block of iterations (up to the next termination check / rho adaptation).  Two warps per problem: one owns the even
// stages (and runs the sweeps over them), the other the odd stages; for N + 1 <= 32 also one warp with a lane per stage.
//
// Why: with the records in shared memory an iteration moved 1,811 wavefronts (~200 KB) per problem through the shared-memory
// pipe (ncu: 53 % of its peak over the whole launch, 84 % in steady state): the phases re-read and re-write every record four
// times per iteration.  Here shared memory only carries what crosses lanes, one 6-double row each:
//
//   sweeps (even warp)                                x~_e -> row nx(e)
//   B_a  T1  odd : x~_o = t_o - D_o^-1 (E_o x~_{o-1} + E_{o+1}' x~_{o+1})            -> row nx(o)
//   B_b  T2  all : A1 (relaxation, row states, duals) + the stage's own part of A2  -> row mb(k) = (d_k[4], G_k[3], G_k[4])
//   B_c  T3  all : b_k from mb(k-1), mb(k+1);   odd: t_o = D_o^-1 b_o                  -> row nx(o)
//   B_d  T4  even: b'_e = b_e - E_e t_{e-1} - E_{e+1}' t_{e+1}                        -> row nx(e), next sweeps
//
// (B_x: barrier of the two warps).  The arithmetic - operands and order of every sum - is that of the general parity form
// (admm_update_stage_oe / admm_rhs_stage_oe) through pair_stage / pair_assemble of mpc_pair.h, so the iterates are the same
// to the last bit.  Between blocks the records are written back: termination checks, rho adaptation, polish and the first
// right-hand side after a (re)factorisation run on the records exactly as in the other forms.
// Rows: mb(k) is the s-tilde slot of the record (s-tilde lives in registers inside a block).  Horizons with N + 1 <= 64.
// STATE = 0 keeps the same two-warp schedule with the state left in the records (no mailbox: the neighbours' values are read
// from their records): one fused read-modify-write of every record per iteration instead of four parity passes.
#pragma once

namespace mpc {

struct StageRegs {
  double r[SR];        // the stage record, same layout as in shared memory; only the state (R_XU .. R_YE) and s-tilde (R_ST)
                       // live here - the constants (R_LIN, R_Q) are read from the record where they are used
};
// what a lane carries from one part of an iteration to the next
struct StageTmp {
  double xt[6], xn[6]; // x~ of the stage and of stage k+1 (T1 -> T2)
  double ua, ud;       // x~ inputs of stage k-1           (T1 -> T2)
  double G[5];         // group sums                        (T2 -> T3)
  double b[6];         // even stages: b_k                  (T3 -> T4)
};

// An address in the problem's shared-memory window, as the register form keeps it for a whole block of iterations.  The
// device holds a 32-bit shared-state-space address (one register; an access through p() compiles to ld.shared / st.shared
// on it with the word's offset as an immediate), the host emulation a plain pointer: both run the same statements.
#ifdef __CUDACC__
// A value formed once per block and kept in a register: with every register taken, ptxas would otherwise re-derive it
// (from N, k, the lane) at each use in the iterations - rematerialisation, the integer work these values are there to remove.
__device__ __forceinline__ unsigned opaque_u32(unsigned v) { asm volatile("mov.b32 %0, %0;" : "+r"(v)); return v; }
#endif
struct SAddr {
#ifdef __CUDA_ARCH__
  unsigned a;
  __device__ __forceinline__ static SAddr of(const double* q) { return SAddr{opaque_u32((unsigned)__cvta_generic_to_shared(q))}; }
  __device__ __forceinline__ double* p() const { return static_cast<double*>(__cvta_shared_to_generic(a)); }
#else
  double* a;
  MPC_HD static SAddr of(double* q) { return SAddr{q}; }
  MPC_HD double* p() const { return a; }
#endif
};
// Everything the stage of a lane reads or writes in an iteration, computed once at the entry of a block, so that the
// iterations spend no integer instructions on record and row offsets.  Neighbours are clamped as the branch-free phases
// need them: stage 0 reads its own record / row in place of stage -1's (the value is dropped by a select), the last stage
// its own record in place of stage N+1's and the row of zeros in place of row N+1.
struct StageAddr {
  SAddr hdr;          // the problem's header
  SAddr rec, rp, rn;  // records of stages k, max(k-1, 0), min(k+1, N)
  SAddr x, xp, xn;    // rows nx(k), nx(max(k-1, 0)), nx(k+1) (k = N: the row of zeros)
  SAddr di;           // odd k: D_k^-1; even k: S'^-1 of its reduced stage (the diagonal step)
};
MPC_HD StageAddr stage_addr(const View& w, const OEView& oe, int k) {
  const int N = w.N, kp = k >= 1 ? k - 1 : 0, kn = k + 1 <= N ? k + 1 : N;
  StageAddr a;
  a.hdr = SAddr::of(w.hdr());
  a.rec = SAddr::of(w.rec(k)); a.rp = SAddr::of(w.rec(kp)); a.rn = SAddr::of(w.rec(kn));
  a.x = SAddr::of(w.nx(k)); a.xp = SAddr::of(w.nx(kp)); a.xn = SAddr::of(k + 1 <= N ? w.nx(k + 1) : w.nx_zero());
  a.di = SAddr::of(((k & 1) ? oe.dinv : oe.sinv) + OE_SYM * (k >> 1));
  return a;
}

MPC_HD double* reg_mb(SAddr rec) { return rec.p() + R_ST; }          // 6 doubles (R_ST[5] + pad)

// STATE = 1: the ADMM state of the stage lives in R.r for the block; STATE = 2: only the row states and slacks (v, s,
// s-tilde: 25 of the 35 doubles) do, x / u and the dynamics duals stay in the record; STATE = 0: everything stays in the record
template <int STATE>
MPC_HD void reg_load(SAddr rec, StageRegs& R) {
  const double* rc = rec.p();
  if (STATE) {
#pragma unroll
  for (int j = (STATE == 2 ? R_S : 0); j < (STATE == 2 ? R_YE : R_LIN); ++j) R.r[j] = rc[j];
#pragma unroll
  for (int j = 0; j < 5; ++j) R.r[R_ST + j] = rc[R_ST + j];
  }
}
// state + s-tilde back to the record, t_o back to its row (the constants never change)
template <int STATE>
MPC_HD void reg_store(SAddr rec, const StageRegs& R) {
  double* rc = rec.p();
  if (STATE) {
#pragma unroll
  for (int j = (STATE == 2 ? R_S : 0); j < (STATE == 2 ? R_YE : R_LIN); ++j) rc[j] = R.r[j];
#pragma unroll
  for (int j = 0; j < 5; ++j) rc[R_ST + j] = R.r[R_ST + j];
  }
}

// T1, odd k: x~ of the stage from the even neighbours' rows
template <class C>
MPC_HD void reg_expand(const StageAddr& a, const Params& p, const C& c, int k, const StageRegs& R, StageTmp& T) {
  const int N = p.N;
  const double re = c.rho_eq, kap = c.kap;
  double xp[6], di[OE_SYM], v[6], y[6], u[6];
  row_load(a.xp.p(), xp);
#pragma unroll
  for (int j = 0; j < 6; ++j) T.xn[j] = 0.0;
  cross_mul(a.rp.p() + R_LIN, p.dt, re, kap, k < N, xp, v);
  // no branch for the last stage: the row of zeros stands in for row N+1 and the terminal record's lin is zero, so the term is an exact +-0
  row_load(a.xn.p(), T.xn);
  cross_mul_t(a.rec.p() + R_LIN, p.dt, re, kap, k + 1 < N, T.xn, y);
#pragma unroll
  for (int j = 0; j < 6; ++j) v[j] += y[j];
  sym_load(a.di.p(), di);
  symv6(di, v, u);
  double t[6];
  row_load(a.x.p(), t);                    // t_o, published in this row by the last right-hand side
#pragma unroll
  for (int j = 0; j < 6; ++j) T.xt[j] = t[j] - u[j];
  T.ua = k < N ? xp[4] : 0.0; T.ud = k < N ? xp[5] : 0.0;
  row_store(a.x.p(), T.xt);
}
// T2 inputs of an even stage: its own row from the sweeps, the odd neighbours' rows from T1
MPC_HD void reg_gather_even(const StageAddr& a, int N, int k, StageTmp& T) {
  row_load(a.x.p(), T.xt);
  row_load(a.xn.p(), T.xn);                // beyond the horizon: the row of zeros
  const double* xp = a.xp.p();             // branch-free: clamped index + select
  const double ua = xp[4], ud = xp[5];
  const bool ib = k > 0 && k < N;
  T.ua = ib ? ua : 0.0; T.ud = ib ? ud : 0.0;
}
// T2: A1 + own part of A2 on the registers, publish (d, G[3], G[4])
template <int STATE, class C>
MPC_HD void reg_update(const StageAddr& a, const Params& p, const C& c, int k, StageRegs& R, StageTmp& T) {
  double* st = STATE ? R.r : a.rec.p();
  double* sx = STATE == 1 ? R.r : a.rec.p();
  pair_stage(st, st, sx, sx, a.rec.p(), a.hdr.p(), p, c, p.N, k, T.xt, T.xn, T.ua, T.ud, T.G);
  if (STATE) {                     // the record's state slots are stale inside a block: publish what the neighbours need
    double d[4];
    stage_d(sx, a.rec.p(), c, k < p.N, d);
    double* mb = reg_mb(a.rec);
#pragma unroll
    for (int r = 0; r < 4; ++r) mb[r] = d[r];
    mb[4] = T.G[3]; mb[5] = T.G[4];
  }
}
// T3: right-hand side of the stage; odd: t_o and its two products for the even neighbours
template <int STATE, class C>
MPC_HD void reg_rhs(const StageAddr& a, const Params& p, const C& c, int k, StageRegs& R, StageTmp& T) {
  const int N = p.N;
  const double re = c.rho_eq, kap = c.kap;
  // branch-free: the neighbours' values through clamped indices, then selects (stage 0: the initial-state rows)
  double dp[4], rn[2];
  {
    const double* h = a.hdr.p();
    double di_[4], dm[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) di_[r] = re * h[H_X0 + r] - h[H_YI + r];
    if (STATE) {
      const double* mp = reg_mb(a.rp);
#pragma unroll
      for (int r = 0; r < 4; ++r) dm[r] = mp[r];
      const double* mn = reg_mb(a.rn);
      rn[0] = mn[4]; rn[1] = mn[5];
    } else {
      stage_d(a.rp.p(), a.rp.p(), c, true, dm);
      const double* rnx = a.rn.p();                     // G[3], G[4] of stage k+1 from its row states (admm_rhs_vals)
      const double rho = c.rho;
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const double v0 = rnx[R_V + 3 * (3 + i)], v1 = rnx[R_V + 3 * (3 + i) + 1];
        const double z0 = dmin2(v0, c.hi[3 + i]), z1 = dmax2(v1, c.lo[3 + i]);
        rn[i] = rho * (z0 + (z0 - v0)) + rho * (z1 + (z1 - v1));
      }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) dp[r] = k >= 1 ? dm[r] : di_[r];
  }
  double val[6], d[4], base[6];
  const double* sx = STATE == 1 ? R.r : a.rec.p();
  stage_d(sx, a.rec.p(), c, k < N, d);              // functions of the state: nothing but G is carried over B_c
  stage_base(sx, a.rec.p(), c, k < N, base);
  pair_assemble(a.rec.p() + R_LIN, p, N, k, dp, d, T.G, rn, base, val);
  if (k & 1) {
    double di[OE_SYM];
    sym_load(a.di.p(), di);
    double t[6];
    symv6(di, val, t);
    row_store(a.x.p(), t);                              // for the even neighbours' fixup and the next expand
  } else {
#pragma unroll
    for (int j = 0; j < 6; ++j) T.b[j] = val[j];
  }
}
// T4, even k: b'_k = b_k - E_k t_{k-1} - E_{k+1}' t_{k+1} -> row nx(k)
template <class C>
MPC_HD void reg_fixup(const StageAddr& a, const Params& p, const C& c, int k, StageTmp& T) {
  const int N = p.N;
  const double re = c.rho_eq, kap = c.kap;
  // branch-free: stage 0 reads a clamped row and drops the term with a select; beyond the last stage the row of zeros and the
  // terminal record's zero lin give an exact +-0
  double t[6], y[6], t2[6], y2[6];
  row_load(a.xp.p(), t);
  row_load(a.xn.p(), t2);
  cross_mul(a.rp.p() + R_LIN, p.dt, re, kap, k < N, t, y);
  cross_mul_t(a.rec.p() + R_LIN, p.dt, re, kap, k + 1 < N, t2, y2);
#pragma unroll
  for (int j = 0; j < 6; ++j) T.b[j] -= (k >= 1) ? y[j] : 0.0;
#pragma unroll
  for (int j = 0; j < 6; ++j) T.b[j] -= y2[j];
  row_store(a.x.p(), T.b);
}

// a block of nb iterations, stage after stage (host emulation; `reverse`: stages of every part in the other order)
template <int STATE>
MPC_HD void reg_block_seq(const View& w, const Params& p, const IterConst& c, const OEView& oe, int nb, StageRegs* R, StageTmp* T, bool reverse) {
  const int NS = w.N + 1;
  auto each = [&](int par, auto f) {          // par: 0 even stages, 1 odd stages, 2 all
    for (int i = 0; i < NS; ++i) { const int k = reverse ? NS - 1 - i : i; if (par == 2 || (k & 1) == par) f(k, stage_addr(w, oe, k)); }
  };
  each(2, [&](int k, const StageAddr& a) { reg_load<STATE>(a.rec, R[k]); });
  for (int it = 0; it < nb; ++it) {
    oe_forward_seq(w);
    each(0, [&](int k, const StageAddr& a) { if (k != 2 * oe.jm) oe_diag(a.di.p(), a.x.p()); });
    oe_backward_seq(w);
    each(1, [&](int k, const StageAddr& a) { reg_expand(a, p, c, k, R[k], T[k]); });
    each(0, [&](int k, const StageAddr& a) { reg_gather_even(a, w.N, k, T[k]); });
    each(2, [&](int k, const StageAddr& a) { reg_update<STATE>(a, p, c, k, R[k], T[k]); });
    each(2, [&](int k, const StageAddr& a) { reg_rhs<STATE>(a, p, c, k, R[k], T[k]); });
    each(0, [&](int k, const StageAddr& a) { reg_fixup(a, p, c, k, T[k]); });
  }
  each(2, [&](int k, const StageAddr& a) { reg_store<STATE>(a.rec, R[k]); });
}

}  // namespace mpc
