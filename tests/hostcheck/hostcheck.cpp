// CPU harness around dvi_ekf_b200/csrc/eskf_math.cuh (TEST INFRASTRUCTURE).
// Compiles the exact host/device math header with g++ and replays, sequentially,
// what one CTA does for one filter: the scalar role followed by the eight
// covariance lanes (column pass, then row pass).  Lets the not-gpu test suite
// check the device arithmetic against the oracle without a GPU.
#include "../../dvi_ekf_b200/csrc/eskf_cov3.cuh"
#include <string.h>

using namespace eskf;

static void load_nominal(Nominal& s, const double* x, const double* u, const double* Ro) {
  memcpy(s.p, x + 0, 24); memcpy(s.v, x + 3, 24); memcpy(s.q, x + 6, 32);
  memcpy(s.dofs, x + 10, 48); memcpy(s.notch, x + 16, 24); memcpy(s.pc, x + 19, 24); memcpy(s.qc, x + 22, 32);
  memcpy(s.om_old, u, 24); memcpy(s.acc_old, u + 3, 24); memcpy(s.R_old, Ro, 72);
}
static void store_nominal(const Nominal& s, double* x, double* u, double* Ro) {
  memcpy(x + 0, s.p, 24); memcpy(x + 3, s.v, 24); memcpy(x + 6, s.q, 32);
  memcpy(x + 10, s.dofs, 48); memcpy(x + 16, s.notch, 24); memcpy(x + 19, s.pc, 24); memcpy(x + 22, s.qc, 32);
  memcpy(u, s.om_old, 24); memcpy(u + 3, s.acc_old, 24); memcpy(Ro, s.R_old, 72);
}

extern "C" {

// model = {L, angle, frozen_mask, flags}
void hc_propagate(const double* model, double* x, double* P, double* u, double* Ro, double dt, const double* om_acc,
                  const double* qd, const double* sig_om, double* fx_out) {
  Model m{model[0], sin(model[1]), cos(model[1]), (int)model[2], (int)model[3]};
  Nominal s; load_nominal(s, x, u, Ro);
  ProbeKin pk; ProbeTrig t;
  probe_eval(m, s.dofs, s.notch, pk, t);
  double R_WB[9]; quat_to_rot(s.q, R_WB);
  double fx[FX_STRIDE];
  const bool imu_q = (qd[3] != 0.0) || (qd[4] != 0.0) || (qd[5] != 0.0);
  propagate_scalar(m, s, pk, t, R_WB, dt, om_acc, om_acc + 3, sig_om, imu_q, fx);
  constexpr int RS = 25;
  double Ps[24 * RS];
  for (int i = 0; i < 24; ++i) for (int j = 0; j < 24; ++j) Ps[i * RS + j] = P[i * 24 + j];
  for (int g = 0; g < 8; ++g) fx_apply3<RS, 1>(Ps + 3 * g, fx);          // T = Fx P   (columns)
  for (int g = 0; g < 8; ++g) {                                            // P' = T Fx^T (rows) + Fi Q Fi^T
    fx_apply3<1, RS>(Ps + 3 * g * RS, fx);
    add_process_noise3<1, RS>(Ps + 3 * g * RS, 3 * g, fx, qd, imu_q);
  }
  for (int i = 0; i < 24; ++i) for (int j = 0; j < 24; ++j) P[i * 24 + j] = Ps[i * RS + j];
  store_nominal(s, x, u, Ro);
  if (fx_out) memcpy(fx_out, fx, sizeof(double) * FX_SIZE);
}

// returns 1 if the update was applied, 0 if skipped (singular S)
int hc_update(const double* model, double* x, double* P, const double* u, const double* Ro, const double* cam /*pos3 quat4*/,
              double notch, const double* rd, double* K_out) {
  Model m{model[0], sin(model[1]), cos(model[1]), (int)model[2], (int)model[3]};
  Nominal s; double uu[6], RR[9]; memcpy(uu, u, 48); memcpy(RR, Ro, 72);
  load_nominal(s, x, uu, RR);
  constexpr int RS = 25;
  double Ps[24 * RS];
  for (int i = 0; i < 24; ++i) for (int j = 0; j < 24; ++j) Ps[i * RS + j] = P[i * 24 + j];
  double up[UP_SIZE];
  double S[49];
  for (int a = 0; a < 7; ++a) for (int b = 0; b < 7; ++b) S[7 * a + b] = Ps[ESKF_HSET(a) * RS + ESKF_HSET(b)] + (a == b ? rd[a] : 0.0);
  bool ok = inv7(S, up + UP_SINV);
  ok = update_residual(s, cam, cam + 3, notch, up + UP_RES) && ok;
  if (!ok) return 0;
  for (int g = 0; g < 8; ++g) gain_rows3<RS>(Ps, 3 * g, up);
  inject_error(m, s, up + UP_DELTA);
  for (int g = 0; g < 8; ++g) joseph_apply3<RS, 1>(Ps + 3 * g, up);
  for (int g = 0; g < 8; ++g) joseph_rows_finish3<RS>(Ps + 3 * g * RS, 3 * g, up, rd);
  for (int i = 0; i < 24; ++i) for (int j = 0; j < 24; ++j) P[i * 24 + j] = Ps[i * RS + j];
  store_nominal(s, x, uu, RR);
  if (K_out)
    for (int r = 0; r < 24; ++r) for (int mm = 0; mm < 7; ++mm)
      K_out[7 * r + mm] = (ESKF_HSET(mm) == r) ? up[UP_KD + mm] : up[UP_KZ + 7 * r + mm];
  return 1;
}

// The same step through the building blocks of the warp-specialised kernel (eskf_kernel3.cuh): split scalar
// roles, Jacobian row groups on strided views, register tile: T = Fx X stored, transposition, X <- Fx X, process noise.
void hc_propagate3(const double* model, double* x, double* P, double* u, double* Ro, double dt, const double* om_acc,
                   const double* qd, const double* sig_om, double* fx_out) {
  Model m{model[0], sin(model[1]), cos(model[1]), (int)model[2], (int)model[3]};
  Nominal s; load_nominal(s, x, u, Ro);
  ProbeKin pk; ProbeTrig t;
  probe_eval(m, s.dofs, s.notch, pk, t);  // kinematics at the pre-step (dofs, notch)
  double R_WB[9]; quat_to_rot(s.q, R_WB);
  const bool imu_q = (qd[3] != 0.0) || (qd[4] != 0.0) || (qd[5] != 0.0);
  // CAMERA role (pre-step v, R_WB, probe kinematics, notch')
  cam_nominal_step(s.pc, s.qc, s.v, R_WB, dt, s.om_old, om_acc, pk.p, pk.R, pk.z6, s.notch[1]);
  // JACOB role
  alignas(16) double fx3[FX3_SIZE];
  for (int i = 0; i < FX3_SIZE; ++i) fx3[i] = 0.0;
  const PKView<1> pkv{reinterpret_cast<double*>(&pk)};
  const TRView<1> trv{reinterpret_cast<double*>(&t)};
  if (dofs_notch_step(m, s.dofs, s.notch, dt)) probe_update_v(m, s.dofs, s.notch, pkv, trv);
  jac_rows_h2(m, s.notch[1], pkv, trv, dt, s.om_old, sig_om, fx3);
  jac_rows_h1(m, s.dofs, pkv, trv, s.R_old, dt, s.om_old, sig_om, fx3);
  if (imu_q) jac_rows_noise(pkv, s.R_old, dt, fx3);
  jac_rows_ab(s.R_old, dt, s.om_old, s.acc_old, fx3);  // (IMU role)
  // IMU role
  double Rn[9];
  imu_nominal_step(s.p, s.v, s.q, R_WB, dt, s.om_old, s.acc_old, om_acc, om_acc + 3, Rn);
  for (int i = 0; i < 9; ++i) s.R_old[i] = Rn[i];
  for (int i = 0; i < 3; ++i) { s.om_old[i] = om_acc[i]; s.acc_old[i] = om_acc[3 + i]; }
  // COVARIANCE role: eight lanes, tile of three columns each
  const d2* f2 = reinterpret_cast<const d2*>(fx3);
  static double X[8][24][3];
  double T[24][24];
  for (int g = 0; g < 8; ++g) {
    for (int i = 0; i < 24; ++i) for (int v = 0; v < 3; ++v) X[g][i][v] = P[i * 24 + 3 * g + v];
    fx3_apply_store<1, 24>(X[g], f2, &T[0][0] + 3 * g);  // all 24 rows are exchanged (eskf_cov3.cuh)
  }
  auto qdf = [&](int j) { return qd[j]; };
  for (int g = 0; g < 8; ++g) {
    for (int k = 0; k < 24; ++k) for (int v = 0; v < 3; ++v) X[g][k][v] = T[3 * g + v][k];
    fx3_apply_inplace<1>(X[g], f2);
    double qdv[3];
    fx3_noise_diag(g, qdf, qdv);
    fx3_process_noise<1>(X[g], g, f2, qdv, qdf, imu_q);
    for (int j = 0; j < 24; ++j) for (int v = 0; v < 3; ++v) P[(3 * g + v) * 24 + j] = X[g][j][v];
  }
  store_nominal(s, x, u, Ro);
  if (fx_out) memcpy(fx_out, fx3, sizeof(double) * FX3_SIZE);
}

// Pass 2 of the covariance propagation both ways for one filter: reload + fx3_apply_inplace (out_a) and the streaming
// pass fx3_apply_stream (out_b), from the same transposition buffer T[24][24] and fx3 record.  Both [8][24][3].
void hc_pass2_both(const double* T, const double* fx3, double* out_a, double* out_b) {
  alignas(16) double rec[FX3_SIZE];
  alignas(16) double Tb[24 * 24];
  memcpy(rec, fx3, sizeof(rec));
  memcpy(Tb, T, sizeof(Tb));
  const d2* f2 = reinterpret_cast<const d2*>(rec);
  for (int g = 0; g < 8; ++g) {
    double Xa[24][3], Xb[24][3];
    fx3_load_transposed<24>(Xa, Tb + 3 * g * 24);
    fx3_apply_inplace<1>(Xa, f2);
    for (int i = 0; i < 24; ++i) for (int v = 0; v < 3; ++v) Xb[i][v] = -7.0;  // write-only operand: must be overwritten
    fx3_apply_stream<1, 24>(Xb, f2, Tb + 3 * g * 24);
    memcpy(out_a + g * 72, Xa, sizeof(Xa));
    memcpy(out_b + g * 72, Xb, sizeof(Xb));
  }
}

// Filter.update through the register-tile building blocks of eskf_kernel3.cuh: the eight lanes of a filter
// replayed phase by phase around the u3 exchange record (warp-level synchronisation points = loop boundaries).
int hc_update3(const double* model, double* x, double* P, const double* u, const double* Ro, const double* cam /*pos3 quat4*/,
               double notch, const double* rd, double* K_out) {
  Model m{model[0], sin(model[1]), cos(model[1]), (int)model[2], (int)model[3]};
  Nominal s; double uu[6], RR[9]; memcpy(uu, u, 48); memcpy(RR, Ro, 72);
  load_nominal(s, x, uu, RR);
  static double X[8][24][3];
  for (int g = 0; g < 8; ++g)
    for (int i = 0; i < 24; ++i) for (int v = 0; v < 3; ++v) X[g][i][v] = P[(3 * g + v) * 24 + i];  // rows used as columns
  alignas(16) double rec[U3_SIZE];
  for (int g = 0; g < 8; ++g) upd3_publish_S<1>(X[g], g, rd, rec);
  double S[49], Si[49];
#if ESKF_OPT_UPD  // the tile's view of S comes from the H P record (inv7_group3): S^T(j, i) = H P(j, h_i) + [i == j] R_i
  for (int i = 0; i < 7; ++i) for (int j = 0; j < 7; ++j) rec[U3_S + 7 * j + i] = rec[U3_HP + 24 * j + ESKF_HSET(i)] + ((i == j) ? rd[i] : 0.0);
#endif
  for (int i = 0; i < 7; ++i) for (int j = 0; j < 7; ++j) S[7 * i + j] = rec[U3_S + 7 * j + i];  // the record holds S^T (eskf_cov3.cuh)
  bool ok = inv7(S, Si);
  for (int j = 0; j < 49; ++j) rec[U3_SINV + j] = Si[j];
  double res[7];
  ok = update_residual(s, cam, cam + 3, notch, res) && ok;
  if (!ok) return 0;
  double K[8][3][7], delta[24];
  for (int g = 0; g < 8; ++g) {
    double dl[3];
    upd3_gain<1>(g, rec, res, K[g], dl);
    for (int v = 0; v < 3; ++v) delta[3 * g + v] = dl[v];
  }
  inject_error(m, s, delta);
  for (int g = 0; g < 8; ++g) upd3_w_pass<1>(X[g], g, rec);
  for (int g = 0; g < 8; ++g) upd3_finish<1, 1, 1>(X[g], g, rec, rd, delta + 6, delta + 21);
  for (int g = 0; g < 8; ++g)
    for (int i = 0; i < 24; ++i) for (int v = 0; v < 3; ++v) P[(3 * g + v) * 24 + i] = X[g][i][v];
  store_nominal(s, x, uu, RR);
  if (K_out)
    for (int g = 0; g < 8; ++g) for (int v = 0; v < 3; ++v) for (int mm = 0; mm < 7; ++mm) K_out[7 * (3 * g + v) + mm] = K[g][v][mm];
  return 1;
}

// CTA mapping of stacked trajectories (stacked_grid / stacked_cta, what eskf_launch3.cu and eskf_kernel3 run) for every
// batch size N = 1 .. n_traj * fpt - filter_id0 of one geometry: one row {N, grid, block, f0, nf, traj, tl} per block, traj =
// the trajectory the kernel derives from the CTA's first global filter id, tl = the decoded one counted from the batch's
// first trajectory.  Returns the number of rows (-1: cap too small).
int64_t hc_stacked_sweep(int F, int64_t fpt, int64_t n_traj, int64_t filter_id0, int64_t* rows, int64_t cap) {
  int64_t r = 0;
  for (int64_t N = 1; filter_id0 + N <= n_traj * fpt; ++N) {
    const int64_t grid = stacked_grid(N, fpt, F);
    for (int64_t b = 0; b < grid; ++b) {
      if (r >= cap) return -1;
      int64_t f0, tl;
      int nf;
      stacked_cta(b, N, fpt, F, f0, nf, tl);
      int64_t* o = rows + 7 * r++;
      o[0] = N, o[1] = grid, o[2] = b, o[3] = f0, o[4] = nf, o[5] = (filter_id0 + f0) / fpt, o[6] = tl;
    }
  }
  return r;
}

}  // extern "C"
