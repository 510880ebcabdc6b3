// Lane-emulation harness (TEST INFRASTRUCTURE, host only): runs the very same per-problem driver that
// the CUDA kernel runs (rrt_mpc_b200/csrc/mpc_solve.h) with a sequential execution policy, so that the
// index logic can be debugged and hazard-checked (forward vs reverse stage order must agree bit for
// bit) in a container without a GPU.  Never linked into libcudampc.so and never used by the product.
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "../../rrt_mpc_b200/csrc/mpc_solve.h"
#include "la_systems.h"

using namespace mpc;

static int g_reg_state = 1;   // register form: 1 = stage state in per-stage copies (registers), 0 = left in the records

struct EmuExec {
  int reverse;
  void tag(int) {}
  template <class F> void stages(int n, F f) {
    if (!reverse) for (int k = 0; k < n; ++k) f(k);
    else for (int k = n - 1; k >= 0; --k) f(k);
  }
  template <class F> void single(F f) { f(); }
  template <class F> void reduce_max(int n, double* r, int nr, F f) {
    for (int i = 0; i < nr; ++i) r[i] = 0.0;
    stages(n, [&](int k) { f(k, r); });
  }
  template <class F> int any(int n, F f) {
    int a = 0;
    stages(n, [&](int k) { a |= f(k); });
    return a;
  }
  template <class F> void stages_par(int n, int par, F f) {
    if (!reverse) for (int k = par; k < n; k += 2) f(k);
    else for (int k = ((n - 1 - par) / 2) * 2 + par; k >= 0; k -= 2) f(k);
  }
  void factor(const View& w) { factor_band(w); }
  void solve(const View& w) { chain_solve(w); }
  // odd-even block solve of the ADMM iterations: the same pieces the CUDA policy runs with lanes over stages / two chain lanes
  void oe_factor(const View& w, const Params& p, const Mode& m, const OEView& oe) {
    stages_par(w.N + 1, 1, [&](int k) { oe_factor_odd(w, p, m, oe, k); });
    stages_par(w.N + 1, 0, [&](int k) { oe_factor_even(w, p, m, oe, k); });
    double Ut[21], Ub[21];
    if (!reverse) { oe_factor_half(oe_half(w, oe, false), Ut); oe_factor_half(oe_half(w, oe, true), Ub); }
    else { oe_factor_half(oe_half(w, oe, true), Ub); oe_factor_half(oe_half(w, oe, false), Ut); }
    oe_factor_middle(oe, Ut, Ub);
  }
  // pair form of an iteration: the parts of mpc_pair.h lane after lane (in either order), neighbours' values from their contexts
  void pair_pass(const View& w, const Params& p, const IterConst& c, const OEView& oe) {
    std::vector<PairCtx> cx(pair_lanes(w.N));
    pair_pass_seq(w, p, c, oe, cx.data(), reverse != 0);
  }
  // register form: a block of iterations on per-stage copies of the records
  void admm_block(const View& w, const Params& p, const IterConst& c, const OEView& oe, int nb) {
    std::vector<StageRegs> R(w.N + 1);
    std::vector<StageTmp> T(w.N + 1);
    if (g_reg_state) reg_block_seq<1>(w, p, c, oe, nb, R.data(), T.data(), reverse != 0);
    else reg_block_seq<0>(w, p, c, oe, nb, R.data(), T.data(), reverse != 0);
  }
  void oe_forward(const View& w, const OEView&) { oe_forward_seq(w); }
  void oe_backward(const View& w, const OEView&) { oe_backward_seq(w); }
};

extern "C" {

int emu_footprint(int N) { return footprint(N); }
int emu_warm_size(int N) { return warm_size(N); }

static void unpack(const double* par, const double* set, int N, Params& p, Settings& s) { la::unpack(par, set, N, p, s); }

static int g_fsave = 1;       // keep the ADMM factor in a side buffer over a polish (0: refactorise on resume)
void emu_set_fsave(int f) { g_fsave = f; }
static int g_form = -1;      // -1: what the library picks (short form for N+1 <= 32, register form for N+1 <= 64), else FORM_* of mpc_solve.h
void emu_set_form(int f) { g_form = f & 3; g_reg_state = (f & 4) ? 0 : 1; if (f < 0) { g_form = -1; g_reg_state = 1; } }

int emu_solve_batch(const double* par, const double* set, int N, int B, int reverse,
                    const double* x0, const double* ref, const double* u_prev, double* warm,
                    double* u0, double* Xp, double* Up, int* status, int* iters, double* pri, double* dua, int* info) {
  Params p; Settings s; unpack(par, set, N, p, s);
  std::vector<double> ws(footprint(N)), scratch(warm_size(N)), warm_local(warm_size(N)), fsave(oe_doubles(N));
  for (int b = 0; b < B; ++b) {
    std::fill(ws.begin(), ws.end(), 0.0);
    View w{ws.data(), N, 4, 2};   // arbitrary non-zero (even: 16-byte aligned) pads: the layout must work with any
    ProblemIO io;
    io.x0 = x0 + 4 * b; io.ref = RefWin{ref + (size_t)4 * (N + 1) * b, 0, N + 1, 1.0}; io.u_prev = u_prev ? u_prev + 2 * b : nullptr;
    io.warm = warm ? warm + (size_t)warm_size(N) * b : warm_local.data();
    io.scratch = scratch.data();
    io.fsave = g_fsave ? fsave.data() : nullptr;
    io.u0 = u0 + 2 * b; io.Xp = Xp + (size_t)4 * (N + 1) * b; io.Up = Up + (size_t)2 * N * b;
    io.status = status + b; io.iters = iters + b; io.pri_res = pri + b; io.dua_res = dua + b; io.info = info + 4 * b;
    Settings sb = s;
    if (!warm) sb.warm_start = 0;
    EmuExec ex{reverse};
    const int form = g_form >= 0 ? g_form : (N + 1 <= 32 ? FORM_SHORT : (N + 1 <= 64 ? FORM_REG : FORM_GENERAL));
    if (form == FORM_SHORT && N + 1 <= 32) solve_problem<FORM_SHORT>(ex, w, p, sb, io);
    else if (form == FORM_PAIR && N + 1 <= 64) solve_problem<FORM_PAIR>(ex, w, p, sb, io);
    else if (form == FORM_REG && N + 1 <= 64) solve_problem<FORM_REG>(ex, w, p, sb, io);
    else solve_problem<FORM_GENERAL>(ex, w, p, sb, io);
  }
  return 0;
}

// linearisation hook: A (B,N,4,4), Bm (B,N,4,2), c (B,N,4) exactly as the solve path computes them
int emu_linearize_batch(const double* par, const double* set, int N, int B, const double* ref, double* A, double* Bm, double* c) {
  Params p; Settings s; unpack(par, set, N, p, s);
  std::vector<double> uy(N + 1);
  for (int b = 0; b < B; ++b) {
    const double* r = ref + (size_t)4 * (N + 1) * b;
    unwrap_yaw(r + 2, 4, N + 1, uy.data(), 1);
    for (int k = 0; k < N; ++k) {
      int kl = k > 0 ? k - 1 : 0;
      double lin[7];
      linearize_point(p, r[4 * kl], r[4 * kl + 1], uy[kl], r[4 * kl + 3], lin);
      double* a = A + ((size_t)b * N + k) * 16; double* bm = Bm + ((size_t)b * N + k) * 8; double* cc = c + ((size_t)b * N + k) * 4;
      for (int i = 0; i < 16; ++i) a[i] = 0.0;
      for (int i = 0; i < 8; ++i) bm[i] = 0.0;
      a[0] = a[5] = a[10] = a[15] = 1.0;
      a[2] = lin[0]; a[3] = lin[1]; a[6] = lin[2]; a[7] = lin[3];
      bm[2 * 2 + 1] = lin[4]; bm[3 * 2 + 0] = p.dt;
      cc[0] = lin[5]; cc[1] = lin[6]; cc[2] = 0.0; cc[3] = 0.0;
    }
  }
  return 0;
}

// ---- linear solves one at a time (tests/test_linear_solves.py, la_systems.h), the sequential statements ------------------
int emu_oe_doubles(int N) { return oe_doubles(N); }
// bytes of mpc_exec.cuh GroupShared (a CUDA header): same members, same order
int emu_group_shared_bytes() {
  struct GS { int next; int anyv[2]; double red[2][8]; Drv drv; };
  return (int)sizeof(GS);
}

// offsets (doubles from the workspace base) of the odd-even factor: dinv, sinv, gt, gb, and band_offset, oe_doubles
int emu_oe_offsets(int N, int* o) {
  std::vector<double> ws(footprint(N));
  const View w = la::view(ws.data(), N);
  const OEView oe = oe_view(w);
  o[0] = (int)(oe.dinv - w.base); o[1] = (int)(oe.sinv - w.base); o[2] = (int)(oe.gt - w.base); o[3] = (int)(oe.gb - w.base);
  o[4] = band_offset(N); o[5] = oe_doubles(N);
  return 0;
}

// words of a problem's workspace (footprint(N)) that `mode` may change once its inputs are placed
int emu_la_writable(int N, int mode, unsigned char* m) {
  std::vector<double> ws(footprint(N));
  la::writable(la::view(ws.data(), N), mode, m);
  return 0;
}

// (A) reduced systems: S, F [nsys][J][36], b, x [nsys][J][6], fac [nsys][oe_doubles(N)] (the factor area afterwards)
int emu_la_reduced(int N, int nsys, const double* S, const double* F, const double* b, double* x, double* fac) {
  const int J = oe_neven(N), nf = oe_doubles(N);
  std::vector<double> ws(footprint(N));
  for (int i = 0; i < nsys; ++i) {
    std::fill(ws.begin(), ws.end(), 0.0);
    const View w = la::view(ws.data(), N);
    for (int j = 0; j < J; ++j) la::red_place(w, S + (size_t)36 * J * i, F + (size_t)36 * J * i, b + (size_t)6 * J * i, j);
    la::red_solve_seq(w);
    for (int j = 0; j < J; ++j) la::red_read(w, x + (size_t)6 * J * i, j);
    for (int t = 0; t < nf; ++t) fac[(size_t)nf * i + t] = (w.base + band_offset(N))[t];
  }
  return 0;
}

// (B) mode 1, ADMM operator at rho[i];  (C) mode 2, polish operator with activity words act [nsys][N+2].
// x0 [nsys][4], ref [nsys][N+1][4], b, x [nsys][N+1][6]
int emu_la_operator(int mode, const double* par, const double* set, int N, int nsys, const double* rho, const double* x0,
                    const double* ref, const int* act, const double* b, double* x) {
  Params p; Settings s; unpack(par, set, N, p, s);
  std::vector<double> ws(footprint(N));
  const size_t nb = (size_t)6 * (N + 1);
  for (int i = 0; i < nsys; ++i) {
    std::fill(ws.begin(), ws.end(), 0.0);
    const View w = la::view(ws.data(), N);
    la::prob_head(w, x0 + 4 * i, ref + (size_t)4 * (N + 1) * i, mode == la::MODE_POLISH ? act + (size_t)(N + 2) * i : nullptr);
    for (int k = 0; k <= N; ++k) la::prob_stage(w, p, ref + (size_t)4 * (N + 1) * i, k);
    if (mode == la::MODE_ADMM) {
      la::admm_seq(w, p, s, rho[i], b + nb * i);
      for (int k = 0; k <= N; ++k) la::admm_read(w, x + nb * i, k);
    } else {
      la::pol_seq(w, p, s, b + nb * i);
      for (int k = 0; k <= N; ++k) la::pol_read(w, x + nb * i, k);
    }
  }
  return 0;
}
}
