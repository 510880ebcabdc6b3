// la_systems.h — TEST INFRASTRUCTURE: places one linear system into the workspace of one problem with the product's own
// layout (View with layout_pads, oe_view, w.nx, bx_set / bx_get) and reads the result back.  Included by tests/emu/emu.cpp
// (host, the sequential statements) and tests/emu/la_dev.cu (device, the lane code of mpc_exec.cuh), so the layout logic of
// the linear-algebra tests exists once.  Never linked into libcudampc.so.
//
// Three systems (tests/test_linear_solves.py):
//   (A) the reduced system of the odd-even solve on the J = oe_neven(N) even stages: SPD blocks S_j and couplings
//       F_j = M'[j][j-1], written where oe_factor_even leaves them (bottom-half blocks transposed), rhs on the even rows;
//   (B) the ADMM operator of a real problem (admm_mode), solved as an ADMM iteration does: odd rows scaled by D_o^-1,
//       even fix-up, sweeps of the reduced system, odd expansion;
//   (C) the polish operator (polish_mode, activity bits in w.act()): banded LDL' and the twisted sweeps.
#pragma once
#include "../../rrt_mpc_b200/csrc/mpc_solve.h"

namespace la {
using namespace mpc;

enum { MODE_RED = 0, MODE_ADMM = 1, MODE_POLISH = 2 };

MPC_HD View view(double* base, int N) {
  int fpad, xpad;
  layout_pads(N, fpad, xpad);
  return View{base, N, fpad, xpad};
}

// params/settings as flat double arrays (tests/emu_driver.py pack)
//  par: L, dt, (Q+Q')[16], (R+R')[4], (QN+QN')[16], u_lo[2], u_hi[2], v_lo, v_hi, du_lo[2], du_hi[2], w_v, w_u, w_du   (51)
//  set: eps_abs, eps_rel, rho0, alpha, sigma, adaptive_rho_tolerance, rho_eq_factor, rho_min, rho_max, delta, max_iter,
//       check_termination, adaptive_rho, adaptive_rho_interval, polish_passes, polish_refine_iter, warm_start, polish_retry,
//       early_polish, early_polish_start (20)
MPC_HD void unpack(const double* par, const double* set, int N, Params& p, Settings& s) {
  int i = 0;
  p.L = par[i++]; p.dt = par[i++];
  for (int a = 0; a < 4; ++a) for (int b = 0; b < 4; ++b) p.pq[a][b] = par[i++];      // already symmetrised: Q + Q'
  for (int a = 0; a < 2; ++a) for (int b = 0; b < 2; ++b) p.pr[a][b] = par[i++];
  for (int a = 0; a < 4; ++a) for (int b = 0; b < 4; ++b) p.pqn[a][b] = par[i++];
  for (int j = 0; j < 2; ++j) p.u_lo[j] = par[i++];
  for (int j = 0; j < 2; ++j) p.u_hi[j] = par[i++];
  p.v_lo = par[i++]; p.v_hi = par[i++];
  for (int j = 0; j < 2; ++j) p.du_lo[j] = par[i++];
  for (int j = 0; j < 2; ++j) p.du_hi[j] = par[i++];
  p.w_v = par[i++]; p.w_u = par[i++]; p.w_du = par[i++];
  p.N = N;
  i = 0;
  s.eps_abs = set[i++]; s.eps_rel = set[i++]; s.rho0 = set[i++]; s.alpha = set[i++]; s.sigma = set[i++];
  s.adaptive_rho_tolerance = set[i++]; s.rho_eq_factor = set[i++]; s.rho_min = set[i++]; s.rho_max = set[i++];
  s.delta = set[i++];
  s.max_iter = (int)set[i++]; s.check_termination = (int)set[i++]; s.adaptive_rho = (int)set[i++];
  s.adaptive_rho_interval = (int)set[i++]; s.polish_passes = (int)set[i++]; s.polish_refine_iter = (int)set[i++];
  s.warm_start = (int)set[i++]; s.polish_retry = (int)set[i++]; s.early_polish = (int)set[i++]; s.early_polish_start = (int)set[i++];
}

// ---- (A) reduced system: S, F are [J][6][6] row-major (F_0 unused), b and the solution [J][6] ------------------------------
MPC_HD void red_place(const View& w, const double* S, const double* F, const double* b, int j) {
  const OEView oe = oe_view(w);
  double* sp = oe.sinv + OE_SYM * j;
  for (int r = 0; r < 6; ++r)
    for (int c = 0; c <= r; ++c) sp[MPC_SP(r, c)] = S[36 * j + 6 * r + c];
  sp[21] = 0.0;
  if (j >= 1) {                                              // as oe_factor_even stores F_j
    const double* f = F + 36 * j;
    if (j <= oe.jm) { double* g = oe.gt + OE_G * (j - 1); for (int i = 0; i < OE_G; ++i) g[i] = f[i]; }
    else {
      double* g = oe.gb + OE_G * (oe.J - j - 1);
      for (int r = 0; r < 6; ++r) for (int c = 0; c < 6; ++c) g[6 * c + r] = f[6 * r + c];
    }
  }
  for (int r = 0; r < 6; ++r) w.nx(2 * j)[r] = b[6 * j + r];
  if (j == 0) for (int r = 0; r < BXS; ++r) w.nx_zero()[r] = 0.0;
}
MPC_HD void red_read(const View& w, double* x, int j) {
  for (int r = 0; r < 6; ++r) x[6 * j + r] = w.nx(2 * j)[r];
}
// the one-lane statements
MPC_HD void red_solve_seq(const View& w) {
  const OEView oe = oe_view(w);
  double Ut[21], Ub[21];
  oe_factor_half(oe_half(w, oe, false), Ut);
  oe_factor_half(oe_half(w, oe, true), Ub);
  oe_factor_middle(oe, Ut, Ub);
  oe_forward_seq(w);
  for (int k = 0; k <= w.N; k += 2) oe_diag_stage(w, oe, k);
  oe_backward_seq(w);
}

// ---- problem setup of (B) and (C): x0 [4], reference window [N+1][4], activity words [N+2] ---------------------------------
MPC_HD void prob_head(const View& w, const double* x0, const double* ref, const int* act) {
  double* h = w.hdr();
  for (int i = 0; i < 4; ++i) h[H_X0 + i] = x0[i];
  for (int i = 0; i < 2; ++i) h[H_UPREV + i] = 0.0;
  for (int i = 0; i < w.N + 2; ++i) w.act()[i] = act ? act[i] : 0;
  unwrap_window(RefWin{ref, 0, w.N + 1, 1.0}, w.N + 1, w.scratch());
}
MPC_HD void prob_stage(const View& w, const Params& p, const double* ref, int k) {
  setup_stage(w, p, k, RefWin{ref, 0, w.N + 1, 1.0}, w.scratch());
}

// ---- (B) ADMM operator: b and the solution [N+1][6] over the (x,u) unknowns ------------------------------------------------
// rhs of stage k as the ADMM right-hand side phase leaves it: odd rows t_o = D_o^-1 b_o, even rows b_e (fixed up next)
MPC_HD void admm_place(const View& w, const OEView& oe, const double* b, int k) {
  double v[6];
  for (int j = 0; j < 6; ++j) v[j] = b[6 * k + j];
  if (k & 1) {
    double di[OE_SYM], t[6];
    sym_load(oe.dinv + OE_SYM * (k >> 1), di);
    symv6(di, v, t);
    row_store(w.nx(k), t);
  } else {
    row_store(w.nx(k), v);
  }
}
MPC_HD void admm_read(const View& w, double* x, int k) {
  for (int j = 0; j < 6; ++j) x[6 * k + j] = w.nx(k)[j];
}
MPC_HD void admm_seq(const View& w, const Params& p, const Settings& s, double rho, const double* b) {
  const OEView oe = oe_view(w);
  const IterConst c = iter_const(w, p, s, rho);
  oe_factor_seq(w, p, admm_mode(rho, s));
  for (int k = 0; k <= w.N; ++k) admm_place(w, oe, b, k);
  for (int k = 0; k <= w.N; k += 2) oe_even_fixup(w, p, c, k);
  oe_forward_seq(w);
  for (int k = 0; k <= w.N; k += 2) oe_diag_stage(w, oe, k);
  oe_backward_seq(w);
  for (int k = 1; k <= w.N; k += 2) oe_expand_odd(w, p, c, oe, k);
}

// ---- (C) polish operator: b and the solution [N+1][6] ------------------------------------------------------------------------
MPC_HD void pol_place(const View& w, const double* b, int k) {
  for (int j = 0; j < 6; ++j) w.bx_set(k, j, b[6 * k + j]);
}
MPC_HD void pol_read(const View& w, double* x, int k) {
  for (int j = 0; j < 6; ++j) x[6 * k + j] = w.bx_get(k, j);
}
MPC_HD void pol_seq(const View& w, const Params& p, const Settings& s, const double* b) {
  const Mode m = polish_mode(s);
  for (int k = 0; k <= w.N; ++k) assemble_stage(w, p, m, k);
  factor_band(w);
  for (int k = 0; k <= w.N; ++k) pol_place(w, b, k);
  chain_solve(w);
}

// ---- words of a problem's workspace that a mode may change once its inputs are placed (1 = may change) ------------------
MPC_HD void mark(const View& w, unsigned char* m, const double* p, int n) {
  for (int i = 0; i < n; ++i) m[(p - w.base) + i] = 1;
}
MPC_HD void writable(const View& w, int mode, unsigned char* m) {
  const int N = w.N;
  const OEView oe = oe_view(w);
  for (int i = 0; i < footprint(N); ++i) m[i] = 0;
  if (mode == MODE_RED || mode == MODE_ADMM) {
    if (mode == MODE_ADMM) mark(w, m, oe.dinv, OE_SYM * oe_nodd(N));
    mark(w, m, oe.sinv, OE_SYM * oe.J);
    mark(w, m, oe.gt, OE_G * oe.jm);
    mark(w, m, oe.gb, OE_G * oe.nb);
    for (int k = 0; k <= N; ++k)
      if (mode == MODE_ADMM || !(k & 1)) mark(w, m, w.nx(k), BXS);
    if (mode == MODE_ADMM) mark(w, m, w.nx_zero(), BXS);
  } else {
    const HalfView T = w.top(), B = w.bottom();
    mark(w, m, T.blk(0), BLK * T.H);
    mark(w, m, B.blk(0), BLK * B.H);
    mark(w, m, w.mid(), 22);
    mark(w, m, T.bx(0), BXS * T.H);
    mark(w, m, B.bx(0), BXS * B.H);
  }
}

}  // namespace la
