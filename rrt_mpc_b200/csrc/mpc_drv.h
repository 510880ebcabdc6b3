// mpc_drv.h — the per-problem driver of mpc_solve.h as a resumable state machine, for the register form (mpc_reg.h).
//
// The register form keeps every stage record in registers across a block of ADMM iterations.  That only works if the
// iteration block is compiled at the TOP LEVEL of the kernel with nothing else alive: inlined into solve_problem the
// driver's own state (settings, residuals, counters, pointers) is alive across the block and competes for the 255 registers,
// and as a real function call the ABI's register conventions do (ptxas then parks part of the record in local memory -
// measured: 120k instead of 260k solves/s).  So the driver is cut at the block boundary into pieces that keep ALL their state
// in one struct (Drv):
//
//   drv_begin    load + linearise, initial iterate
//   drv_prepare  (re)factorise if needed, first right-hand side after a factorisation, length of the next block
//   [block of d.nb iterations: Exec::admm_block / the kernel's inline loop]
//   drv_after    termination check, early / final polish, rho adaptation            (-> d.finished)
//                after a block (d.phase = PH_ADMM), or after the solves of one polish pass (PH_POLISH: no block runs
//                before it); both reach the one residual check of the piece
//   drv_finish   outputs
//
// The kernel (mpc_kernels.cuh: mpc_solve_reg_kernel) inlines the pieces through wrappers that load Drv from shared memory and
// store it back, so that no value of a piece is alive in the block; the host emulation (and solve_problem<FORM_REG>) runs
// them back to back on a local Drv.  The logic is that of solve_problem
// statement by statement (tests/test_emulation.py holds the two bit-identical, early polish and retries included).
#pragma once
#include "mpc_solve.h"

namespace mpc {

struct Drv {
  double rho, pri, dua, se_abs, se_rel;      // se_*: effective tolerances (tightened by polish_retry)
  Residuals res;
  int status, it, retries, n_rho, n_fac, n_solve, n_pol, nb;
  int finished, need_restore, need_factor, need_rhs;
  int phase;                                 // PH_ADMM: a block of iterations ran; PH_POLISH: polish pass `pass` ran its solves
  int last, check, adapt, converged;         // the event being handled (the check that started a polish)
  int pass, acc;                             // polish: current pass, passes accepted
  double pp, dd;                             // polish: residuals of the last accepted pair
  IterConst ic;
};
enum { PH_ADMM = 0, PH_POLISH = 1 };

template <class Exec>
MPC_HD void drv_begin(Exec& ex, const View& w, const Params& p, const Settings& s, const ProblemIO& io, Drv& d) {
  const int N = w.N, NS = N + 1;
  ex.tag(0);
  ex.single([&]() {
    double* h = w.hdr();
    for (int i = 0; i < 4; ++i) h[H_X0 + i] = io.x0[i];
    for (int i = 0; i < 2; ++i) h[H_UPREV + i] = io.u_prev ? io.u_prev[i] : 0.0;
    for (int i = 0; i < N + 2; ++i) w.act()[i] = 0;
    unwrap_window(io.ref, NS, w.scratch());
  });
  ex.stages(NS, [&](int k) { setup_stage(w, p, k, io.ref, w.scratch()); });
  d.rho = s.rho0;
  const double rho_slot = (s.warm_start && io.warm) ? io.warm[30 * NS + 4] : 0.0;      // see solve_problem: rho word = valid marker
  if (rho_slot >= s.rho_min && rho_slot <= s.rho_max) {
    ex.stages(NS, [&](int k) { load_stage(w, k, io.warm); });
    ex.single([&]() { for (int r = 0; r < 4; ++r) w.hdr()[H_YI + r] = io.warm[30 * NS + r]; });
    d.rho = rho_slot;
  } else {
    ex.stages(NS, [&](int k) { cold_start_stage(w, p, k); });
  }
  d.ic = iter_const(w, p, s, d.rho);
  d.status = STATUS_UNSOLVED; d.it = 0;
  d.res.pri = d.res.dua = 1e300; d.res.eps_p = d.res.eps_d = 0.0; d.res.sp = d.res.sd = 0.0; d.res.nz = d.res.nq = 0.0;
  d.pri = d.dua = 1e300;
  d.se_abs = s.eps_abs; d.se_rel = s.eps_rel;
  d.retries = s.polish_retry;
  d.n_rho = d.n_fac = d.n_solve = d.n_pol = 0; d.nb = 0;
  d.finished = 0; d.need_restore = 0; d.need_factor = 1; d.need_rhs = 1;
  d.phase = PH_ADMM;
  d.last = d.check = d.adapt = d.converged = 0; d.pass = d.acc = 0; d.pp = d.dd = 0.0;
}

template <class Exec>
MPC_HD void drv_prepare(Exec& ex, const View& w, const Params& p, const Settings& s, Drv& d) {
  const int NS = w.N + 1;
  const OEView oe = oe_view(w);
  if (d.need_factor) {
    const Mode mode = admm_mode(d.rho, s);
    ex.tag(5); ex.oe_factor(w, p, mode, oe); ++d.n_fac;
    d.ic = iter_const(w, p, s, d.rho);
    d.need_factor = 0;
    d.need_rhs = 1;
  }
  if (d.need_rhs) {                        // the first right-hand side after a (re)factorisation: the general parity passes
    ex.tag(6);
    const IterConst ic = d.ic;
#pragma unroll 1
    for (int par = 1; par >= 0; --par) ex.stages_par(NS, par, [&](int k) { admm_rhs_stage_oe(w, p, ic, oe, k); });
    d.need_rhs = 0;
  }
  // iterations up to the next event: termination check, rho adaptation, iteration limit
  int nb = s.max_iter - d.it;
  if (s.check_termination > 0) { const int n = s.check_termination - d.it % s.check_termination; if (n < nb) nb = n; }
  if (s.adaptive_rho && s.adaptive_rho_interval > 0) { const int n = s.adaptive_rho_interval - d.it % s.adaptive_rho_interval; if (n < nb) nb = n; }
  d.nb = nb < 1 ? 1 : nb;
  ex.tag(2);
}

// after a block of d.nb iterations (d.phase == PH_ADMM): what solve_problem's after_update does after the update of iteration
// d.it; after the solves of polish pass d.pass (d.phase == PH_POLISH): that pass's residuals and decision.  The polish loop
// of solve_problem is cut into one piece per pass, so that the termination check and the polish's own check run through ONE
// copy of compute_residuals (ymode from the phase): the check is about 1.4 k instructions, and the code other resident
// problems run between their iteration blocks competes with the iteration loop for the instruction cache.
template <class Exec>
MPC_HD void drv_after(Exec& ex, const View& w, const Params& p, const Settings& s, const ProblemIO& io, Drv& d) {
  const int NS = w.N + 1;
  const bool can_polish = s.polish_passes > 0 && io.warm && io.scratch;
  const bool polishing = d.phase == PH_POLISH;
  if (!polishing) {
    d.it += d.nb; d.n_solve += d.nb;
    d.last = d.it >= s.max_iter;
    d.check = d.last || ((s.check_termination > 0) && (d.it % s.check_termination == 0));
    d.adapt = !d.last && s.adaptive_rho && (s.adaptive_rho_interval > 0) && (d.it % s.adaptive_rho_interval == 0);
    if (!(d.check || d.adapt)) return;
  }
  Settings se = s; se.eps_abs = d.se_abs; se.eps_rel = d.se_rel;
  const IterConst ic = d.ic;
  ex.tag(polishing ? 12 : 3);
  const Residuals rr = compute_residuals(ex, w, p, se, ic, polishing ? 1 : 0);
  bool run_pass = false, polish_end = false, settled = false;
  int rejected = 0;
  if (!polishing) {
    d.res = rr;
    d.pri = rr.pri; d.dua = rr.dua;
    if (d.check) {
      const bool last = d.last;
      const bool converged = rr.pri <= rr.eps_p && rr.dua <= rr.eps_d;
      if (converged && d.status == STATUS_UNSOLVED) d.status = STATUS_SOLVED;
      if (last && d.status == STATUS_UNSOLVED) {
        const double ep10 = 10.0 * s.eps_abs + 10.0 * s.eps_rel * rr.nz, ed10 = 10.0 * s.eps_abs + 10.0 * s.eps_rel * rr.nq;
        d.status = (rr.pri <= ep10 && rr.dua <= ed10) ? STATUS_SOLVED_INACCURATE : STATUS_MAX_ITER;
      }
      bool attempt = converged || (last && d.status == STATUS_SOLVED);
      if (!attempt && !last && s.early_polish && can_polish) {
        ex.tag(15);
        const int changed = ex.any(NS, [&](int k) { return activity_probe_stage(w, p, k); });
        attempt = (!changed || s.early_polish >= 2) && d.it >= s.early_polish_start;
      }
      if (attempt || last) {
        ex.tag(8);
        if (io.warm) {                                                   // save the ADMM iterate
          ex.stages(NS, [&](int k) { save_stage(w, k, io.warm); });
          const double rho = d.rho;
          ex.single([&]() {
            for (int r = 0; r < 4; ++r) io.warm[30 * NS + r] = w.hdr()[H_YI + r];
            io.warm[30 * NS + 4] = (rr.pri < 1e300 && rr.dua < 1e300) ? rho : 0.0;
          });
        }
        if (attempt && can_polish) {
          if (io.fsave && !last && !(converged && d.retries <= 0)) ex.stages(oe_doubles(w.N), [&](int i) { oe_save_word(w, i, io.fsave); });
          // ---- polish (solve_problem: polish lambda), pass 0 ----
          d.converged = converged;
          d.pass = 0; d.acc = 0;
          d.pp = rr.pri; d.dd = rr.dua;
          run_pass = true;
        } else {
          d.finished = 1;
        }
      }
    }
  } else {                                                               // decision of polish pass d.pass
    const int pass = d.pass;
    const double pp = d.pp, dd = d.dd, nz = d.res.nz, nq = d.res.nq;
    bool ok;
    if (pass == 0) ok = (rr.pri < pp && rr.dua < dd) || (rr.pri < pp && dd < 1e-10) || (rr.dua < dd && pp < 1e-10);
    else ok = rr.pri <= dmax(10.0 * pp, 1e-9 * dmax(1.0, nz)) && rr.dua <= dmax(10.0 * dd, 1e-9 * dmax(1.0, nq));
    if (ok) {
      d.pp = rr.pri; d.dd = rr.dua; d.acc = pass + 1;
      d.pass = pass + 1;
      if (d.pass < s.polish_passes) run_pass = true; else polish_end = true;
    } else {
      rejected = pass == 0 ? 1 : 2;
      polish_end = true;
    }
  }
  if (run_pass) {                                                        // polish pass d.pass up to its residuals
    const int pass = d.pass;
    ex.tag(9);
    if (pass > 0) {
      ex.stages(NS, [&](int k) { save_stage(w, k, io.scratch); });
      ex.single([&]() { for (int r = 0; r < 4; ++r) io.scratch[30 * NS + r] = w.hdr()[H_YI + r]; });
    }
    const double rho = d.rho;
    const int changed = ex.any(NS, [&](int k) { return polish_activity_stage(w, p, rho, pass == 0, k); });
    if (pass > 0 && !changed) {
      settled = true;
      polish_end = true;
    } else {
      const Mode pm = polish_mode(s);
      const PolConst pc = pol_const(w, p, s);
      ex.stages(NS, [&](int k) { polish_zero_stage(w, k); });
      ex.stages(NS, [&](int k) { assemble_stage(w, p, pm, k); });
      ex.tag(10); ex.factor(w); ++d.n_fac;
      ex.tag(11);
      for (int step = 0; step <= s.polish_refine_iter; ++step) {
        ex.stages(NS, [&](int k) { polish_rhs_fast(w, p, pc, k); });
        ex.solve(w); ++d.n_solve;
        ex.stages(NS, [&](int k) { polish_dual_fast(w, p, pc, k); });
        ex.stages(NS, [&](int k) { polish_primal_stage(w, k); });
      }
      ex.tag(12);
      d.phase = PH_POLISH;                                               // next: this pass's residuals (no ADMM block)
      return;
    }
  }
  if (polish_end) {
    d.phase = PH_ADMM;
    if (rejected == 2) {
      ex.stages(NS, [&](int k) { load_stage(w, k, io.scratch); });
      ex.single([&]() { for (int r = 0; r < 4; ++r) w.hdr()[H_YI + r] = io.scratch[30 * NS + r]; });
    }
    const int acc = d.acc;
    const double pp = d.pp, dd = d.dd;
    if (acc > 0) { d.pri = pp; d.dua = dd; }
    d.n_pol = acc;
    const bool clean = acc > 0 && (settled || s.polish_passes == 1) && pp <= 1e-9 * dmax(1.0, d.res.nz) && dd <= 1e-9 * dmax(1.0, d.res.nq);
    // ---- decision ----
    const bool converged = d.converged;
    if (clean) { d.status = STATUS_SOLVED; d.finished = 1; }
    else if (d.last || (converged && d.retries <= 0)) {
      d.finished = 1;
      if (d.n_pol == 0) d.need_restore = 1;
    } else {
      if (converged) { --d.retries; d.se_abs *= 0.1; d.se_rel *= 0.1; }
      d.n_pol = 0;                                                      // resume ADMM from the saved iterate
      ex.tag(13);
      ex.stages(NS, [&](int k) { load_stage(w, k, io.warm); });
      ex.single([&]() { for (int r = 0; r < 4; ++r) w.hdr()[H_YI + r] = io.warm[30 * NS + r]; });
      if (io.fsave) { ex.stages(oe_doubles(w.N), [&](int i) { oe_restore_word(w, i, io.fsave); }); d.need_rhs = 1; }
      else d.need_factor = 1;
    }
  }
  if (d.adapt && !d.finished) {
    const Residuals res = d.res;
    double rho_new = d.rho * sqrt(res.sp / (res.sd + 1e-10));
    rho_new = fmin(fmax(rho_new, s.rho_min), s.rho_max);
    if (rho_new > d.rho * s.adaptive_rho_tolerance || rho_new < d.rho / s.adaptive_rho_tolerance) {
      const double rho_old = d.rho;
      ex.stages(NS, [&](int k) { rescale_v_stage(w, p, rho_old, rho_new, k); });
      d.rho = rho_new; ++d.n_rho;
      d.need_factor = 1;
    }
  }
}

template <class Exec>
MPC_HD void drv_finish(Exec& ex, const View& w, const ProblemIO& io, const Drv& d) {
  const int N = w.N, NS = N + 1;
  ex.tag(7);
  if (d.need_restore) {
    ex.stages(NS, [&](int k) { load_stage(w, k, io.warm); });
    ex.single([&]() { for (int r = 0; r < 4; ++r) w.hdr()[H_YI + r] = io.warm[30 * NS + r]; });
  }
  ex.stages(NS, [&](int k) {
    const double* rc = w.rec(k);
    for (int j = 0; j < 4; ++j) io.Xp[j * NS + k] = rc[R_XU + j];
    if (k < N) { io.Up[k] = rc[R_XU + 4]; io.Up[N + k] = rc[R_XU + 5]; }
    if (k == 0) {
      io.u0[0] = rc[R_XU + 4]; io.u0[1] = rc[R_XU + 5];
      *io.status = d.status; *io.iters = d.it;
      if (io.pri_res) *io.pri_res = d.pri;
      if (io.dua_res) *io.dua_res = d.dua;
      if (io.info) { io.info[0] = d.n_rho; io.info[1] = d.n_fac; io.info[2] = d.n_pol; io.info[3] = d.n_solve; }
    }
  });
}

// the register form, pieces back to back on a local Drv (host emulation; the CUDA kernel: mpc_kernels.cuh mpc_solve_reg_kernel)
template <class Exec>
MPC_HD void solve_problem_reg(Exec& ex, const View& w, const Params& p, const Settings& s, const ProblemIO& io) {
  Drv d;
  drv_begin(ex, w, p, s, io, d);
  const OEView oe = oe_view(w);
  while (!d.finished) {
    if (d.phase == PH_ADMM) {
      drv_prepare(ex, w, p, s, d);
      ex.admm_block(w, p, d.ic, oe, d.nb);
    }
    drv_after(ex, w, p, s, io, d);
  }
  drv_finish(ex, w, io, d);
}

}  // namespace mpc
