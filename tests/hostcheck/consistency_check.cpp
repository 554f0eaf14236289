// CPU harness for the filter-consistency arithmetic of the device (TEST INFRASTRUCTURE): the replay of hostcheck.cpp plus
// the NIS of the register-tile update (upd3_nis, eskf_cov3.cuh) and the NEES of the estimated DOFs (nees_dofs,
// eskf_math.cuh).  Built by tests/test_consistency_host.py.
#include "hostcheck.cpp"

extern "C" {

// NIS of the update hc_update3 would apply: the same record up to the gain, then upd3_nis on it.  Nothing is modified;
// NaN if the update would be skipped.
double hc_nis3(const double* x, const double* P, const double* u, const double* Ro, const double* cam /*pos3 quat4*/,
               double notch, const double* rd) {
  Nominal s; double xx[NX], uu[6], RR[9]; memcpy(xx, x, sizeof(xx)); memcpy(uu, u, 48); memcpy(RR, Ro, 72);
  load_nominal(s, xx, uu, RR);
  static double X[8][24][3];
  for (int g = 0; g < 8; ++g)
    for (int i = 0; i < 24; ++i) for (int v = 0; v < 3; ++v) X[g][i][v] = P[(3 * g + v) * 24 + i];
  alignas(16) double rec[U3_SIZE];
  for (int g = 0; g < 8; ++g) upd3_publish_S<1>(X[g], g, rd, rec);
  double S[49], Si[49];
#if ESKF_OPT_UPD
  for (int i = 0; i < 7; ++i) for (int j = 0; j < 7; ++j) rec[U3_S + 7 * j + i] = rec[U3_HP + 24 * j + ESKF_HSET(i)] + ((i == j) ? rd[i] : 0.0);
#endif
  for (int i = 0; i < 7; ++i) for (int j = 0; j < 7; ++j) S[7 * i + j] = rec[U3_S + 7 * j + i];
  bool ok = inv7(S, Si);
  for (int j = 0; j < 49; ++j) rec[U3_SINV + j] = Si[j];
  double res[7];
  ok = update_residual(s, cam, cam + 3, notch, res) && ok;
  if (!ok) return NAN;
  double K[3][7], dl[3];
  for (int g = 0; g < 8; ++g) upd3_gain<1>(g, rec, res, K, dl);
  return upd3_nis<1>(rec, res);
}

// NEES of the estimated DOFs (nees_dofs) of n blocks B [n][36], errors eps [n][6] and masks [n]
void hc_nees(const double* B, const double* eps, const int32_t* mask, int64_t n, double* out) {
  for (int64_t i = 0; i < n; ++i) out[i] = nees_dofs(B + 36 * i, eps + 6 * i, mask[i]);
}

}  // extern "C"
