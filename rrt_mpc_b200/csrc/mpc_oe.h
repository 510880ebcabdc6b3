// mpc_oe.h — the linear solve of every ADMM iteration: odd-even block elimination + twisted block-bidiagonal sweeps.
//
// The slack-eliminated ADMM matrix  M = P + sigma I + A' rho A  is block tridiagonal over the N+1 stages (6x6 blocks:
// D_k on the diagonal, E_k = M[stage k][stage k-1] below it; mpc_core.h stage_diag / stage_cross).  The banded LDL' of
// mpc_core.h walks the stages one after the other in two lanes; that chain of 2 x 25 dependent stage steps was 2/3 of an
// ADMM iteration at horizon 50.  Here the chain is cut to 2 x 12 steps of one dense 6x6 matrix-vector product each, and
// everything else runs with LANES OVER STAGES:
//
//   1. one level of cyclic reduction: the odd stages are eliminated first (they only couple to their two even
//      neighbours).  D_o^-1 is stored explicitly (symmetric, 21 numbers), so  t_o = D_o^-1 b_o  and later
//      x_o = t_o - D_o^-1 (E_o x_{o-1} + E_{o+1}' x_{o+1})  are stage-parallel, fused into the ADMM phases that produce b
//      and consume x (no extra pass over the stages);
//   2. the reduced system on the even stages j = 0..J-1 (diagonal S_j, sub-diagonal F_j, all dense 6x6) is factorised as a
//      BLOCK LDL' with explicit pivot inverses:  G_j = F_j S'_{j-1}^-1,  S'_j = S_j - G_j F_j'.  A solve is then
//         forward   y_j = b'_j - G_j y_{j-1}        (sequential, one dense 6x6 mat-vec per step, no in-stage pivot chain)
//         diagonal  z_j = S'_j^-1 y_j               (stage-parallel)
//         backward  x_j = z_j - G_{j+1}' x_{j+1}    (sequential, same blocks)
//      twisted as before: the top half runs j = 0 -> middle in one lane, the bottom half j = J-1 -> middle in another lane
//      of the same instruction stream, the middle stage collects both.
//
// Accuracy: block elimination with explicit inverses of the SPD pivot blocks; measured backward error <= 2e-14 relative
// for rho in [1e-4, 1e5] (Cholesky: 4e-16) - far inside what ADMM needs, and the termination test uses true residuals.
// It is NOT used for the polish (weights 1/delta = 1e6 next to delta = 1e-6: explicit inverses lose four digits there);
// the polish keeps the banded LDL' of mpc_core.h.
#pragma once

namespace mpc {

enum { OE_SYM = 22, OE_G = 36 };                          // packed symmetric 6x6 (21 + pad), dense 6x6
MPC_HD int oe_nodd(int N) { return (N + 1) / 2; }         // odd stages 1, 3, .. <= N
MPC_HD int oe_neven(int N) { return N / 2 + 1; }          // even stages 0, 2, .. <= N  (index j = stage / 2)
MPC_HD int oe_mid(int N) { return oe_neven(N) / 2; }      // middle even index: top half j < jm, bottom half j > jm
#define MPC_SP(r, c) ((r) * ((r) + 1) / 2 + (c))          /* packed lower triangle, c <= r */

struct OEView {
  double* dinv;    // D_o^-1 of odd stage o at dinv + OE_SYM * (o >> 1)
  double* sinv;    // S'_j^-1 (before the factorisation: S_j) of even index j at sinv + OE_SYM * j
  double* gt;      // top half:    block of local step i = 1..jm        at gt + OE_G * (i - 1)   (couples j = i with j - 1)
  double* gb;      // bottom half: block of local step i = 1..J-1-jm    at gb + OE_G * (i - 1)   (couples j = J-1-i with j + 1)
  int J, jm, nb;   // even stages, middle index, bottom steps
};
MPC_HD OEView oe_view(const View& w) {
  OEView o;
  const int N = w.N;
  o.J = oe_neven(N); o.jm = oe_mid(N); o.nb = o.J - 1 - o.jm;
  o.dinv = w.base + band_offset(N);
  o.sinv = o.dinv + OE_SYM * oe_nodd(N);
  o.gt = o.sinv + OE_SYM * o.J;
  const int gpad = ((18 * o.jm) & 7) ? 0 : 2;             // the two chain lanes read gt / gb at the same step: keep them in different 16-byte bank groups
  o.gb = o.gt + OE_G * o.jm + gpad;
  return o;
}

// doubles of the factor (dinv, sinv, gt, pad, gb) behind band_offset(N): what a polish overwrites and a resume needs back
MPC_HD int oe_doubles(int N) { return OE_SYM * (oe_nodd(N) + oe_neven(N)) + OE_G * (oe_neven(N) - 1) + 2; }
// element i of the factor area <-> a per-group slot in global memory (lanes stride over i: coalesced)
MPC_HD void oe_save_word(const View& w, int i, double* g) { g[i] = (w.base + band_offset(w.N))[i]; }
MPC_HD void oe_restore_word(const View& w, int i, const double* g) {
  (w.base + band_offset(w.N))[i] = g[i];
  if (i < BXS) w.nx_zero()[i] = 0.0;                      // the row of zeros the bottom half reads (the polish used the rows)
}

// ------------------------------------------------------------------------------------------------
// 6x6 helpers
// ------------------------------------------------------------------------------------------------
// inverse of an SPD matrix given by its lower triangle S[r][c], c <= r (destroyed) -> packed lower triangle (21 + pad)
MPC_HD void spd6_inverse(double (*S)[6], double* out) {
  double L[6][6], Li[6][6], dinv[6];
#pragma unroll
  for (int jp = 0; jp < 6; ++jp) {
    dinv[jp] = 1.0 / S[jp][jp];
#pragma unroll
    for (int j = jp + 1; j < 6; ++j) {
      const double l = S[j][jp] * dinv[jp];
      L[j][jp] = l;
#pragma unroll
      for (int j2 = jp + 1; j2 <= j; ++j2) S[j][j2] = fma(-l, S[j2][jp], S[j][j2]);   // S[j2][jp] still unscaled
    }
  }
#pragma unroll
  for (int c = 0; c < 5; ++c)
#pragma unroll
    for (int j = c + 1; j < 6; ++j) {
      double v = -L[j][c];
#pragma unroll
      for (int t = c + 1; t < j; ++t) v = fma(-L[j][t], Li[t][c], v);
      Li[j][c] = v;
    }
#pragma unroll
  for (int r = 0; r < 6; ++r)
#pragma unroll
    for (int c = 0; c <= r; ++c) {
      double acc = 0.0;
#pragma unroll
      for (int t = r; t < 6; ++t) {
        const double a = (t == r) ? dinv[t] : Li[t][r] * dinv[t];
        acc = (t == c) ? acc + a : fma(a, Li[t][c], acc);
      }
      out[MPC_SP(r, c)] = acc;
    }
  out[21] = 0.0;
}
// 22 doubles (16-byte aligned) -> registers
MPC_HD void sym_load(const double* a, double* r) {
  const D2* __restrict__ pa = reinterpret_cast<const D2*>(a);
#pragma unroll
  for (int i = 0; i < 11; ++i) { D2 u = pa[i]; r[2 * i] = u.x; r[2 * i + 1] = u.y; }
}
MPC_HD void row_load(const double* a, double* r) {
  const D2* __restrict__ pa = reinterpret_cast<const D2*>(a);
#pragma unroll
  for (int i = 0; i < 3; ++i) { D2 u = pa[i]; r[2 * i] = u.x; r[2 * i + 1] = u.y; }
}
MPC_HD void row_store(double* a, const double* r) {
  D2* pa = reinterpret_cast<D2*>(a);
#pragma unroll
  for (int i = 0; i < 3; ++i) { D2 u; u.x = r[2 * i]; u.y = r[2 * i + 1]; pa[i] = u; }
}
MPC_HD void blk_load(const double* a, double* r) {
  const D2* __restrict__ pa = reinterpret_cast<const D2*>(a);
#pragma unroll
  for (int i = 0; i < 18; ++i) { D2 u = pa[i]; r[2 * i] = u.x; r[2 * i + 1] = u.y; }
}
// y = A x, A symmetric packed (in registers)
MPC_HD void symv6(const double* a, const double* x, double* y) {
#pragma unroll
  for (int r = 0; r < 6; ++r) y[r] = a[MPC_SP(r, 0)] * x[0];
#pragma unroll
  for (int c = 1; c < 6; ++c)
#pragma unroll
    for (int r = 0; r < 6; ++r) y[r] = fma(r >= c ? a[MPC_SP(r, c)] : a[MPC_SP(c, r)], x[c], y[r]);
}

// E_k = M[stage k rows][stage k-1 cols] of the ADMM matrix (stage_cross with uniform weights): rows 0..3 are -rho_eq times
// the dynamics rows of stage k-1 (lin = that stage's a02 a03 a12 a13 b21), rows 4,5 the rate coupling -kappa (kappa = 2 rho)
// when stage k has inputs.     y = E_k v      and      y = E_k' v
MPC_HD void cross_mul(const double* lin, double dt, double re, double kap, bool has_u, const double* v, double* y) {
  y[0] = -re * (v[0] + lin[0] * v[2] + lin[1] * v[3]);
  y[1] = -re * (v[1] + lin[2] * v[2] + lin[3] * v[3]);
  y[2] = -re * (v[2] + lin[4] * v[5]);
  y[3] = -re * (v[3] + dt * v[4]);
  y[4] = has_u ? -kap * v[4] : 0.0;
  y[5] = has_u ? -kap * v[5] : 0.0;
}
MPC_HD void cross_mul_t(const double* lin, double dt, double re, double kap, bool has_u, const double* v, double* y) {
  y[0] = -re * v[0];
  y[1] = -re * v[1];
  y[2] = -re * (lin[0] * v[0] + lin[2] * v[1] + v[2]);
  y[3] = -re * (lin[1] * v[0] + lin[3] * v[1] + v[3]);
  y[4] = -re * (dt * v[3]) - (has_u ? kap * v[4] : 0.0);
  y[5] = -re * (lin[4] * v[2]) - (has_u ? kap * v[5] : 0.0);
}

// ------------------------------------------------------------------------------------------------
// Factorisation (ADMM mode only)
// ------------------------------------------------------------------------------------------------
// odd stage o: D_o^-1
MPC_HD void oe_factor_odd(const View& w, const Params& p, const Mode& m, const OEView& oe, int k) {
  double D[6][6];
  stage_diag(w, p, m, k, D);
  spd6_inverse(D, oe.dinv + OE_SYM * (k >> 1));
}
// even stage e = 2j:  S_j = D_e - E_e D_{e-1}^-1 E_e' - E_{e+1}' D_{e+1}^-1 E_{e+1}   -> sinv slot j (inverted later)
//                     F_j = M'[j][j-1] = -E_e D_{e-1}^-1 E_{e-1}                      -> the block that couples j and j-1
MPC_HD void oe_factor_even(const View& w, const Params& p, const Mode& m, const OEView& oe, int k) {
  const int N = w.N, j = k >> 1;
  const double re = m.rho_eq, kap = 2.0 * m.rho;
  double S[6][6];
  stage_diag(w, p, m, k, S);
  if (k >= 1) {
    double di[OE_SYM];
    sym_load(oe.dinv + OE_SYM * ((k - 1) >> 1), di);
    const double* lin1 = w.rec(k - 1) + R_LIN;               // E_k is built from the dynamics of stage k-1
    double T[6][6];                                          // T = E_k D^-1   (column c of D^-1 = its row c)
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      double col[6], y[6];
#pragma unroll
      for (int r = 0; r < 6; ++r) col[r] = r >= c ? di[MPC_SP(r, c)] : di[MPC_SP(c, r)];
      cross_mul(lin1, p.dt, re, kap, k < N, col, y);
#pragma unroll
      for (int r = 0; r < 6; ++r) T[r][c] = y[r];
    }
#pragma unroll
    for (int r = 0; r < 6; ++r) {                            // (T E_k')[r][:] = E_k T[r][:]'
      double y[6];
      cross_mul(lin1, p.dt, re, kap, k < N, T[r], y);
#pragma unroll
      for (int c = 0; c <= r; ++c) S[r][c] -= y[c];
    }
    if (k >= 2) {
      const double* lin2 = w.rec(k - 2) + R_LIN;             // E_{k-1}: dynamics of stage k-2; stage k-1 < N always has inputs
      double F[OE_G];
#pragma unroll
      for (int r = 0; r < 6; ++r) {                          // F[r][:] = -(T E_{k-1})[r][:] = -E_{k-1}' T[r][:]'
        double y[6];
        cross_mul_t(lin2, p.dt, re, kap, true, T[r], y);
#pragma unroll
        for (int c = 0; c < 6; ++c) F[6 * r + c] = -y[c];
      }
      if (j <= oe.jm) {
        double* g = oe.gt + OE_G * (j - 1);
#pragma unroll
        for (int i = 0; i < OE_G; ++i) g[i] = F[i];
      } else {                                               // bottom half: the block couples local i = J-j (index j-1) with i-1 (index j): F'
        double* g = oe.gb + OE_G * (oe.J - j - 1);
#pragma unroll
        for (int r = 0; r < 6; ++r)
#pragma unroll
          for (int c = 0; c < 6; ++c) g[6 * c + r] = F[6 * r + c];
      }
    }
  }
  if (k + 1 <= N) {
    double di[OE_SYM];
    sym_load(oe.dinv + OE_SYM * ((k + 1) >> 1), di);
    const double* lin0 = w.rec(k) + R_LIN;                   // E_{k+1}: dynamics of stage k
    const bool hu = k + 1 < N;
    double T[6][6];                                          // T = D^-1 E_{k+1}: column c = D^-1 (E_{k+1} e_c); row r of T' = ...
#pragma unroll
    for (int c = 0; c < 6; ++c) {                            // W[:, c] = E_{k+1}' D^-1[:, c]   =>  W = E' D^-1,  S -= W E
      double col[6], y[6];
#pragma unroll
      for (int r = 0; r < 6; ++r) col[r] = r >= c ? di[MPC_SP(r, c)] : di[MPC_SP(c, r)];
      cross_mul_t(lin0, p.dt, re, kap, hu, col, y);
#pragma unroll
      for (int r = 0; r < 6; ++r) T[r][c] = y[r];
    }
#pragma unroll
    for (int r = 0; r < 6; ++r) {                            // (W E)[r][:] = E' W[r][:]'
      double y[6];
      cross_mul_t(lin0, p.dt, re, kap, hu, T[r], y);
#pragma unroll
      for (int c = 0; c <= r; ++c) S[r][c] -= y[c];
    }
  }
  double* sp = oe.sinv + OE_SYM * j;
#pragma unroll
  for (int r = 0; r < 6; ++r)
#pragma unroll
    for (int c = 0; c <= r; ++c) sp[MPC_SP(r, c)] = S[r][c];
  sp[21] = 0.0;
  if (k == 0) {                                              // the row of zeros the bottom half reads at the middle step
    double* z = w.nx_zero();
#pragma unroll
    for (int i = 0; i < BXS; ++i) z[i] = 0.0;
  }
}

// one half of the reduced system as a chain lane sees it: local stage i = 0..cnt-1 (cnt = the steps towards the middle)
struct OEHalf {
  double* s0; int sstep;       // S' / S'^-1 slot of local stage i: s0 + sstep * i
  double* g0;                  // block of local step i = 1..cnt: g0 + OE_G * (i - 1)
  double* x0; int xstep;       // rhs / solution row of local stage i: x0 + xstep * i
  double* xlast;               // row read at the middle step (the middle's own row for the top half, zeros for the bottom)
  int cnt;
};
MPC_HD OEHalf oe_half(const View& w, const OEView& oe, bool bottom) {
  OEHalf h;
  if (!bottom) { h.s0 = oe.sinv; h.sstep = OE_SYM; h.g0 = oe.gt; h.x0 = w.nx(0); h.xstep = BXS; h.xlast = w.nx(2 * oe.jm); h.cnt = oe.jm; }
  else {
    h.s0 = oe.sinv + OE_SYM * (oe.J - 1); h.sstep = -OE_SYM; h.g0 = oe.gb;
    h.x0 = w.nx(2 * (oe.J - 1)); h.xstep = -BXS; h.xlast = w.nx_zero(); h.cnt = oe.nb;
  }
  return h;
}
MPC_HD void sym_expand(const double* a, double (*A)[6]) {
#pragma unroll
  for (int r = 0; r < 6; ++r)
#pragma unroll
    for (int c = 0; c < 6; ++c) A[r][c] = r >= c ? a[MPC_SP(r, c)] : a[MPC_SP(c, r)];
}
// Sequential block LDL' of one half: for i = 0..cnt-1: S'_i^-1; G_{i+1} = F_{i+1} S'_i^-1; S'_{i+1} -= G_{i+1} F_{i+1}'.
// The last update belongs to the middle stage: it is returned in U (packed lower triangle), not applied.
// Sequential statement (host emulation); the kernel runs mpc_exec.cuh oe_factor_lanes, the same statements with one lane per row.
MPC_HD void oe_factor_half(const OEHalf& h, double* U) {
#pragma unroll
  for (int i = 0; i < 21; ++i) U[i] = 0.0;
  for (int i = 0; i < h.cnt; ++i) {
    double* sp = h.s0 + h.sstep * i;
    double S[6][6], sv[OE_SYM];
    sym_load(sp, sv);
    sym_expand(sv, S);
    spd6_inverse(S, sv);
#pragma unroll
    for (int t = 0; t < OE_SYM; ++t) sp[t] = sv[t];
    sym_expand(sv, S);                                        // S = S'_i^-1 (full)
    double* g = h.g0 + OE_G * i;                              // block of step i+1
    double F[OE_G], G[OE_G];
    blk_load(g, F);
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        double acc = F[6 * r] * S[0][c];
#pragma unroll
        for (int t = 1; t < 6; ++t) acc = fma(F[6 * r + t], S[t][c], acc);
        G[6 * r + c] = acc;
      }
#pragma unroll
    for (int t = 0; t < OE_G; ++t) g[t] = G[t];
    double* sn = h.s0 + h.sstep * (i + 1);
    const bool last = (i + 1 == h.cnt);
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
      for (int c = 0; c <= r; ++c) {
        double acc = G[6 * r] * F[6 * c];
#pragma unroll
        for (int t = 1; t < 6; ++t) acc = fma(G[6 * r + t], F[6 * c + t], acc);
        if (last) U[MPC_SP(r, c)] = acc; else sn[MPC_SP(r, c)] -= acc;
      }
  }
}
// middle stage: S'_m = S_m - U_top - U_bot, inverted in place
MPC_HD void oe_factor_middle(const OEView& oe, const double* Ut, const double* Ub) {
  double* sp = oe.sinv + OE_SYM * oe.jm;
  double S[6][6], sv[OE_SYM];
  sym_load(sp, sv);
#pragma unroll
  for (int t = 0; t < 21; ++t) sv[t] -= Ut[t] + Ub[t];
  sym_expand(sv, S);
  spd6_inverse(S, sv);
#pragma unroll
  for (int t = 0; t < OE_SYM; ++t) sp[t] = sv[t];
}

// ------------------------------------------------------------------------------------------------
// Solve: sequential sweeps of one half (one lane each), the stage-parallel diagonal step
// ------------------------------------------------------------------------------------------------
// Row kernels of the sweeps.  The CUDA policy gives every ROW of a half its own lane (6 + 6 lanes of the chain warp): a
// step is then six fmas per lane instead of 36, the block row comes with three 128-bit loads instead of 18, and the new
// vector is exchanged through the row it is stored to anyway.  The products are summed as a fixed tree (three independent
// pairs) so that the dependent latency of a step is two fmas and two adds; host emulation and kernel use the same tree.
//   forward   y[r] = nb[r] - sum_c G[r][c] a[c]        g = row r of the block
//   backward  x[c] = z[c]  - sum_r G[r][c] a[r]        g = column c of the block
MPC_HD double oe_row_dot(const double* g, double nb, const double* a) {
  const double p0 = fma(-g[1], a[1], fma(-g[0], a[0], nb));
  const double p1 = fma(-g[3], a[3], -(g[2] * a[2]));
  const double p2 = fma(-g[5], a[5], -(g[4] * a[4]));
  return (p0 + p1) + p2;
}
// row r of a packed symmetric matrix times x (same tree)
MPC_HD double oe_sym_row(const double* sp, int r, const double* x) {
  double g[6];
#pragma unroll
  for (int c = 0; c < 6; ++c) g[c] = -sp[r >= c ? MPC_SP(r, c) : MPC_SP(c, r)];
  return oe_row_dot(g, 0.0, x);
}
// Sequential statement of the sweeps of one half (host emulation; the kernel runs mpc_exec.cuh: oe_forward_lanes /
// oe_backward_lanes, the same row kernels with one lane per row).
//   forward: y_0 = b'_0, y_i = b'_i - G_i y_{i-1}; stores y_1 .. y_{cnt-1}; returns in a[] the half's term for the middle stage
MPC_HD void oe_forward_half(const OEHalf& h, double* a) {
  if (h.cnt == 0) { for (int r = 0; r < 6; ++r) a[r] = h.xlast[r]; return; }
  for (int r = 0; r < 6; ++r) a[r] = h.x0[r];
  for (int i = 1; i <= h.cnt; ++i) {
    const double* g = h.g0 + OE_G * (i - 1);
    double* row = (i == h.cnt) ? h.xlast : h.x0 + h.xstep * i;
    double y[6];
    for (int r = 0; r < 6; ++r) y[r] = oe_row_dot(g + 6 * r, row[r], a);
    for (int r = 0; r < 6; ++r) { a[r] = y[r]; if (i < h.cnt) row[r] = y[r]; }
  }
}
//   backward from the middle solution xm: x_i = z_i - G_{i+1}' x_{i+1}, i = cnt-1 .. 0 (z_i in place, overwritten by x_i)
MPC_HD void oe_backward_half(const OEHalf& h, const double* xm) {
  double a[6];
  for (int r = 0; r < 6; ++r) a[r] = xm[r];
  for (int i = h.cnt - 1; i >= 0; --i) {
    const double* g = h.g0 + OE_G * i;
    double* row = h.x0 + h.xstep * i;
    double x[6];
    for (int c = 0; c < 6; ++c) {
      const double col[6] = {g[c], g[6 + c], g[12 + c], g[18 + c], g[24 + c], g[30 + c]};
      x[c] = oe_row_dot(col, row[c], a);
    }
    for (int c = 0; c < 6; ++c) { a[c] = x[c]; row[c] = x[c]; }
  }
}
// middle stage: x_m = S'_m^-1 (top term + bottom term)
MPC_HD void oe_middle(const OEView& oe, const double* at, const double* ab, double* xm) {
  double y[6];
  for (int r = 0; r < 6; ++r) y[r] = at[r] + ab[r];
  for (int r = 0; r < 6; ++r) xm[r] = oe_sym_row(oe.sinv + OE_SYM * oe.jm, r, y);
}
// diagonal step of even stage k != middle: z = S'^-1 y, in place
MPC_HD void oe_diag_stage(const View& w, const OEView& oe, int k) {
  const int j = k >> 1;
  if (j == oe.jm) return;
  double sv[OE_SYM], y[6], z[6];
  sym_load(oe.sinv + OE_SYM * j, sv);
  row_load(w.nx(k), y);
  symv6(sv, y, z);
  row_store(w.nx(k), z);
}

// whole factorisation / solve, sequential (host emulation; the CUDA policy runs the same pieces with lanes over stages)
MPC_HD void oe_factor_seq(const View& w, const Params& p, const Mode& m) {
  const OEView oe = oe_view(w);
  for (int k = 1; k <= w.N; k += 2) oe_factor_odd(w, p, m, oe, k);
  for (int k = 0; k <= w.N; k += 2) oe_factor_even(w, p, m, oe, k);
  double Ut[21], Ub[21];
  oe_factor_half(oe_half(w, oe, false), Ut);
  oe_factor_half(oe_half(w, oe, true), Ub);
  oe_factor_middle(oe, Ut, Ub);
}
MPC_HD void oe_forward_seq(const View& w) {
  const OEView oe = oe_view(w);
  double at[6], ab[6], xm[6];
  oe_forward_half(oe_half(w, oe, false), at);
  oe_forward_half(oe_half(w, oe, true), ab);
  oe_middle(oe, at, ab, xm);
  row_store(w.nx(2 * oe.jm), xm);
}
MPC_HD void oe_backward_seq(const View& w) {
  const OEView oe = oe_view(w);
  double xm[6];
  row_load(w.nx(2 * oe.jm), xm);
  oe_backward_half(oe_half(w, oe, false), xm);
  oe_backward_half(oe_half(w, oe, true), xm);
}

}  // namespace mpc
