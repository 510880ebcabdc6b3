// mpc_params.h — the one statement of the parameter rules: cudampc_params -> Params and its checks.  The C ABI runs it on the
// host for the handle's parameters (cudampc_create, cudampc_set_params); the per-problem kernels run it on the device for every
// row of a params array.
#pragma once
#include "../../include/cudampc.h"
#include "mpc_core.h"

namespace mpc {

// Why params_from_c rejected a record (0: accepted)
enum { PARAMS_OK = 0, PARAMS_BAD_HORIZON, PARAMS_BAD_DT_L, PARAMS_BAD_Q, PARAMS_BAD_QN, PARAMS_BAD_R, PARAMS_BAD_SLACK };

// Smallest eigenvalue of the symmetric n x n matrix W (n <= 4), cyclic Jacobi.  cp.quad_form (mpc_controller.py:74-75,112)
// accepts any PSD matrix; the library accepts exactly those (relative tolerance 1e-12) and rejects indefinite ones.
MPC_HD double min_eig_sym(const double* Win, int n, double* scale) {
  double a[4][4];
  double mx = 0.0;
  for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) { a[i][j] = Win[i * n + j]; if (fabs(a[i][j]) > mx) mx = fabs(a[i][j]); }
  *scale = mx;
  for (int sweep = 0; sweep < 50; ++sweep) {
    double off = 0.0;
    for (int i = 0; i < n; ++i) for (int j = 0; j < i; ++j) off += a[i][j] * a[i][j];
    if (off <= 1e-30 * mx * mx) break;
    for (int p = 0; p < n; ++p)
      for (int q = p + 1; q < n; ++q) {
        if (a[p][q] == 0.0) continue;
        const double th = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
        const double t = (th >= 0 ? 1.0 : -1.0) / (fabs(th) + sqrt(th * th + 1.0)), c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
        for (int k = 0; k < n; ++k) { const double x = a[k][p], y = a[k][q]; a[k][p] = c * x - sn * y; a[k][q] = sn * x + c * y; }
        for (int k = 0; k < n; ++k) { const double x = a[p][k], y = a[q][k]; a[p][k] = c * x - sn * y; a[q][k] = sn * x + c * y; }
      }
  }
  double mn = a[0][0];
  for (int i = 1; i < n; ++i) if (a[i][i] < mn) mn = a[i][i];
  return mn;
}

MPC_HD bool psd_nonzero(const double* W, int n) {
  double sc;
  const double e = min_eig_sym(W, n, &sc);
  return sc > 0.0 && e >= -1e-12 * sc && isfinite(e);
}

// Fills p from in; returns PARAMS_OK or the first rule the record breaks (p is then partly written).
MPC_HD int params_from_c(const cudampc_params* in, Params* p) {
  if (in->horizon < 1 || in->horizon > 256) return PARAMS_BAD_HORIZON;
  if (!(in->dt > 0.0) || !(in->wheelbase_px > 0.0)) return PARAMS_BAD_DT_L;
  p->L = in->wheelbase_px; p->dt = in->dt; p->N = in->horizon;
  // quad_form(e, W) = e'We = 1/2 e'(W + W')e: the P block of the QP is the symmetric matrix W + W'
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) { p->pq[i][j] = in->q[4 * i + j] + in->q[4 * j + i]; p->pqn[i][j] = in->q_terminal[4 * i + j] + in->q_terminal[4 * j + i]; }
  for (int i = 0; i < 2; ++i)
    for (int j = 0; j < 2; ++j) p->pr[i][j] = in->r[2 * i + j] + in->r[2 * j + i];
  if (!psd_nonzero(&p->pq[0][0], 4)) return PARAMS_BAD_Q;
  if (!psd_nonzero(&p->pqn[0][0], 4)) return PARAMS_BAD_QN;
  if (!psd_nonzero(&p->pr[0][0], 2)) return PARAMS_BAD_R;
  p->u_lo[0] = in->u_bounds[0]; p->u_hi[0] = in->u_bounds[1]; p->u_lo[1] = in->u_bounds[2]; p->u_hi[1] = in->u_bounds[3];
  p->v_lo = in->v_bounds[0]; p->v_hi = in->v_bounds[1];
  p->du_lo[0] = in->du_bounds[0]; p->du_hi[0] = in->du_bounds[1]; p->du_lo[1] = in->du_bounds[2]; p->du_hi[1] = in->du_bounds[3];
  p->w_v = in->slack_velocity; p->w_u = in->slack_input; p->w_du = in->slack_rate;
  if (!(p->w_v > 0.0) || !(p->w_u > 0.0) || !(p->w_du > 0.0)) return PARAMS_BAD_SLACK;
  return PARAMS_OK;
}

}  // namespace mpc
