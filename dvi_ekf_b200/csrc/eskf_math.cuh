// Per-filter scalar math of the VI-ESKF hot path (FP64), written as
// straight-line host/device functions so that the very same arithmetic can be
// exercised on the CPU by tests/hostcheck (no GPU needed) and by the sm_100a
// kernels in eskf_kernels.cu.
//
// Reference behaviour restated here (paths relative to the reference repo):
//   Quaternion ops ............ dvi_ekf/tools/Quaternion.py:56-224
//   State / ErrorState ........ dvi_ekf/filter/state.py:11-129
//   f_predict ................. dvi_ekf/kinematics/equations.py:44-50,72-100
//   probe forward kinematics .. dvi_ekf/models/Probe.py:147-167,289-306,431-480
//   error Jacobians ........... dvi_ekf/filter/Filter.py:249-342,
//                               dvi_ekf/kinematics/symbols.py:134-200
//   update .................... dvi_ekf/filter/Filter.py:351-395
// The CasADi-generated Jacobians are re-emitted as closed forms; DESIGN.md
// derives them and tests/ checks them against the oracle's generic DH chain
// and against sympy autodiff of the literal symbolic expressions.
#pragma once

#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define ESKF_HD __host__ __device__ __forceinline__
#else
#define ESKF_HD inline
#endif

namespace eskf {

// ---- sizes and layouts ---------------------------------------------------
constexpr int NX = 26;  // nominal state: p v q(xyzw) dofs notch(3) p_cam q_cam(xyzw)
constexpr int NE = 24;  // error state:  dp dv dth ddofs(6) dnotch(3) dpc dthc
constexpr int NM = 7;   // measurement:  cam pos, cam theta, notch
constexpr int NQ = 13;  // process noise: n_a n_om n_dofs(6) n_notch_acc

// measurement rows of H (Filter.py:83-85): H[0:6,18:24] = I, H[6,15] = 1
#define ESKF_HSET(m) ((m) < 6 ? 18 + (m) : 15)

// model flags
constexpr int FLAG_ZERO_FROZEN = 1;  // quirk Q7 (HEAD): Filter.py:243-245 zeroes frozen DOFs

// Per-step Jacobian blocks handed from the scalar role to the covariance role
// ("fx record", doubles):
constexpr int FX_DT = 0;
constexpr int FX_A = 1;    // 3x3  Fx[3:6,6:9]   = -dt R_old [acc_old]x
constexpr int FX_B = 10;   // 3x3  Fx[6:9,6:9]   = rot(Om_old)^T
constexpr int FX_C1 = 19;  // 3x3  Fx[18:21,6:9] = -dt R_old [w]x
constexpr int FX_C2 = 28;  // 3x6  Fx[18:21,9:15]
constexpr int FX_D = 46;   // 3x4  Fx[21:24,{9,10,11,15}]
constexpr int FX_E = 58;   // 3x3  Fx[21:24,19:22]
constexpr int FX_NP = 67;  // 3x3  Fi[18:21,3:6] = dt R_old [p]x     (only used when Q[3:6] != 0)
constexpr int FX_NT = 76;  // 3x3  Fi[21:24,3:6] = -dt R_p^T
constexpr int FX_SIZE = 85;
constexpr int FX_STRIDE = 86;  // doubles per filter per buffer

// Per-filter constant parameters kept next to P ("par record", doubles)
constexpr int PAR_QD = 0;     // 13: diag(Q)
constexpr int PAR_RD = 13;    // 7:  diag(R)
constexpr int PAR_SIGOM = 20; // 3:  gyro noise std used inside the Jacobians (quirk Q6)
constexpr int PAR_SIZE = 23;
constexpr int PAR_STRIDE = 24;

// Update scratch ("upd record", doubles)
constexpr int UP_SINV = 0;   // 49
constexpr int UP_RES = 49;   // 7
constexpr int UP_DELTA = 56; // 24
constexpr int UP_KZ = 80;    // 24x7: K with K[h_m][m] zeroed
constexpr int UP_KD = 248;   // 7:  K[h_m][m]
constexpr int UP_CD = 255;   // 24: diag(I - K H)
constexpr int UP_OK = 279;   // 1:  0 => update skipped (LinAlgError branch, Filter.py:358-361)
constexpr int UP_SIZE = 280;

struct Model {
  double L;       // scope length        (config.yaml model.length)
  double sa, ca;  // sin / cos of the camera angle (model.angle)
  int frozen_mask;  // bit i set => DOF i frozen (simulation.frozen_dofs)
  int flags;
};

// What the scalar role carries in registers for one filter
struct Nominal {
  double p[3], v[3], q[4], dofs[6], notch[3], pc[3], qc[4];
  double om_old[3], acc_old[3];
  double R_old[9];  // rot(q) as of the end of the last propagate (quirk Q8)
};

// Cached probe kinematics at the current (dofs, notch)
struct ProbeKin {
  double p[3];
  double R[9];
  double z6[3];
};

// ---- tiny linear algebra ---------------------------------------------------
ESKF_HD void cross3(const double* a, const double* b, double* c) {
  c[0] = a[1] * b[2] - a[2] * b[1];
  c[1] = a[2] * b[0] - a[0] * b[2];
  c[2] = a[0] * b[1] - a[1] * b[0];
}
ESKF_HD double dot3(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
// y = M x (row-major 3x3)
ESKF_HD void mv3(const double* M, const double* x, double* y) {
  y[0] = M[0] * x[0] + M[1] * x[1] + M[2] * x[2];
  y[1] = M[3] * x[0] + M[4] * x[1] + M[5] * x[2];
  y[2] = M[6] * x[0] + M[7] * x[1] + M[8] * x[2];
}
// y = M^T x
ESKF_HD void mtv3(const double* M, const double* x, double* y) {
  y[0] = M[0] * x[0] + M[3] * x[1] + M[6] * x[2];
  y[1] = M[1] * x[0] + M[4] * x[1] + M[7] * x[2];
  y[2] = M[2] * x[0] + M[5] * x[1] + M[8] * x[2];
}
// C = M [w]x   (row-major):  column j of [w]x is  w x e_j ... written out
ESKF_HD void mul_skew(const double* M, const double* w, double* C) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double a = M[3 * i], b = M[3 * i + 1], c = M[3 * i + 2];
    C[3 * i + 0] = b * w[2] - c * w[1];
    C[3 * i + 1] = c * w[0] - a * w[2];
    C[3 * i + 2] = a * w[1] - b * w[0];
  }
}

// ---- quaternions (xyzw) ------------------------------------------------------
// Quaternion.rot -> Rotation.from_quat(q).as_matrix() for an already unit q
// (scipy's extra re-normalisation of a unit quaternion is a <=1 ulp effect and
// is skipped; tolerance budget is 1e-9).
ESKF_HD void quat_to_rot(const double* q, double* R) {
  const double x = q[0], y = q[1], z = q[2], w = q[3];
  const double x2 = x * x, y2 = y * y, z2 = z * z, w2 = w * w;
  const double xy = x * y, zw = z * w, xz = x * z, yw = y * w, yz = y * z, xw = x * w;
  R[0] = x2 - y2 - z2 + w2;
  R[1] = 2.0 * (xy - zw);
  R[2] = 2.0 * (xz + yw);
  R[3] = 2.0 * (xy + zw);
  R[4] = -x2 + y2 - z2 + w2;
  R[5] = 2.0 * (yz - xw);
  R[6] = 2.0 * (xz - yw);
  R[7] = 2.0 * (yz + xw);
  R[8] = -x2 - y2 + z2 + w2;
}

// Quaternion.normalise (Quaternion.py:195-206): divide by the norm, force w >= 0.
ESKF_HD void quat_normalise(double* q) {
  const double d = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  // q / d as q * (1 / d): one division instead of four (<= 1 ulp from the reference's quotient, far
  // inside the 1e-9 budget); the sign flip is exact and folded into the factor
  const double r = ((q[3] < 0.0) ? -1.0 : 1.0) / d;
  q[0] = q[0] * r;
  q[1] = q[1] * r;
  q[2] = q[2] * r;
  q[3] = q[3] * r;
}

// Quaternion(val=M, do_normalise=True): scipy-1.10.1 Rotation.from_matrix
// (Markley's method on the RAW, generally non-orthonormal matrix -- quirk Q1)
// followed by normalisation and the w >= 0 convention.
ESKF_HD void quat_from_matrix(const double* M, double* q) {
  const double d0 = M[0], d1 = M[4], d2 = M[8];
  const double tr = d0 + d1 + d2;
  int choice = 0;
  double best = d0;
  if (d1 > best) { best = d1; choice = 1; }
  if (d2 > best) { best = d2; choice = 2; }
  if (tr > best) { choice = 3; }
  if (choice == 3) {
    q[0] = M[7] - M[5];
    q[1] = M[2] - M[6];
    q[2] = M[3] - M[1];
    q[3] = 1.0 + tr;
  } else if (choice == 0) {  // i=0 j=1 k=2
    q[0] = 1.0 - tr + 2.0 * d0;
    q[1] = M[3] + M[1];
    q[2] = M[6] + M[2];
    q[3] = M[7] - M[5];
  } else if (choice == 1) {  // i=1 j=2 k=0
    q[1] = 1.0 - tr + 2.0 * d1;
    q[2] = M[7] + M[5];
    q[0] = M[1] + M[3];
    q[3] = M[2] - M[6];
  } else {  // i=2 j=0 k=1
    q[2] = 1.0 - tr + 2.0 * d2;
    q[0] = M[2] + M[6];
    q[1] = M[5] + M[7];
    q[3] = M[3] - M[1];
  }
  quat_normalise(q);
}

// Quaternion.__mul__ (Quaternion.py:170-183): Hamilton product, re-normalised, w >= 0.
ESKF_HD void quat_mul(const double* a, const double* b, double* r) {
  const double w = a[3] * b[3] - (a[0] * b[0] + a[1] * b[1] + a[2] * b[2]);
  double c[3];
  cross3(a, b, c);
  r[0] = a[3] * b[0] + b[3] * a[0] + c[0];
  r[1] = a[3] * b[1] + b[3] * a[1] + c[1];
  r[2] = a[3] * b[2] + b[3] * a[2] + c[2];
  r[3] = w;
  quat_normalise(r);
}

// Quaternion.about_axis (Quaternion.py:208-224)
ESKF_HD void quat_about_axis(double angle, const double* axis, double* q) {
  const double qlen = sqrt(axis[0] * axis[0] + axis[1] * axis[1] + axis[2] * axis[2]);
  double s, c;
  sincos(0.5 * angle, &s, &c);
  double f = 1.0;
  if (qlen > 4.0 * 2.220446049250313e-16) f = s / qlen;
  q[0] = axis[0] * f;
  q[1] = axis[1] * f;
  q[2] = axis[2] * f;
  q[3] = c;
  quat_normalise(q);
}

// ---- probe kinematics -----------------------------------------------------------
// Closed form of the 8-joint DH chain (Probe.py:147-167) with q8 = 0:
//   triad  e_a(t) = (s1 s2 st - c1 ct,  s1 ct + c1 s2 st,  c2 st)
//          e_b(t) = (s1 s2 ct + c1 st,  c1 s2 ct - s1 st,  c2 ct)
//          z6     = (-s1 c2, -c1 c2, s2)                (notch joint axis)
//   p = (L - q4) z6 + q5 e_a(q3) + q6 e_b(q3)
//   R = [ -e_a(d) | sa z6 + ca e_b(d) | ca z6 - sa e_b(d) ],  d = q3 - q7
//   v = acc = 0, om = z6 q7', alp = z6 q7''
struct ProbeTrig {
  double s1, c1, s2, c2, s3, c3, sd, cd;
  double ea3[3], eb3[3], ead[3], ebd[3];
  double a1, a2, a3, ad;  // the angles the sines / cosines above belong to (probe_update)
};

// products of the cached sines / cosines: triads, joint axis, p and R
ESKF_HD void probe_assemble(const Model& m, const double* dofs, ProbeKin& k, ProbeTrig& t) {
  const double s1s2 = t.s1 * t.s2, c1s2 = t.c1 * t.s2;
  t.ea3[0] = s1s2 * t.s3 - t.c1 * t.c3;
  t.ea3[1] = t.s1 * t.c3 + c1s2 * t.s3;
  t.ea3[2] = t.c2 * t.s3;
  t.eb3[0] = s1s2 * t.c3 + t.c1 * t.s3;
  t.eb3[1] = c1s2 * t.c3 - t.s1 * t.s3;
  t.eb3[2] = t.c2 * t.c3;
  t.ead[0] = s1s2 * t.sd - t.c1 * t.cd;
  t.ead[1] = t.s1 * t.cd + c1s2 * t.sd;
  t.ead[2] = t.c2 * t.sd;
  t.ebd[0] = s1s2 * t.cd + t.c1 * t.sd;
  t.ebd[1] = c1s2 * t.cd - t.s1 * t.sd;
  t.ebd[2] = t.c2 * t.cd;
  k.z6[0] = -t.s1 * t.c2;
  k.z6[1] = -t.c1 * t.c2;
  k.z6[2] = t.s2;
  const double lq = m.L - dofs[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    k.p[i] = lq * k.z6[i] + dofs[4] * t.ea3[i] + dofs[5] * t.eb3[i];
    k.R[3 * i + 0] = -t.ead[i];
    k.R[3 * i + 1] = m.sa * k.z6[i] + m.ca * t.ebd[i];
    k.R[3 * i + 2] = m.ca * k.z6[i] - m.sa * t.ebd[i];
  }
}

ESKF_HD void probe_eval(const Model& m, const double* dofs, const double* notch, ProbeKin& k, ProbeTrig& t) {
  t.a1 = dofs[0];
  t.a2 = dofs[1];
  t.a3 = dofs[2];
  t.ad = dofs[2] - notch[0];
  sincos(t.a1, &t.s1, &t.c1);
  sincos(t.a2, &t.s2, &t.c2);
  sincos(t.a3, &t.s3, &t.c3);
  sincos(t.ad, &t.sd, &t.cd);
  probe_assemble(m, dofs, k, t);
}

// probe_eval for a (pk, t) that is valid for earlier (dofs, notch): only the sines / cosines whose angle
// changed are evaluated again -- same inputs, same results as a full probe_eval.  Between camera updates
// only the notch angle moves (equations.py:87), i.e. one sincos per step instead of four.
ESKF_HD void probe_update(const Model& m, const double* dofs, const double* notch, ProbeKin& k, ProbeTrig& t) {
  const double ad = dofs[2] - notch[0];
  if (dofs[0] != t.a1) {
    t.a1 = dofs[0];
    sincos(t.a1, &t.s1, &t.c1);
  }
  if (dofs[1] != t.a2) {
    t.a2 = dofs[1];
    sincos(t.a2, &t.s2, &t.c2);
  }
  if (dofs[2] != t.a3) {
    t.a3 = dofs[2];
    sincos(t.a3, &t.s3, &t.c3);
  }
  if (ad != t.ad) {
    t.ad = ad;
    sincos(t.ad, &t.sd, &t.cd);
  }
  probe_assemble(m, dofs, k, t);
}

// dofs / notch part of f_predict (equations.py:87; Filter.py:243-245).  Returns true when the probe
// kinematics have to be re-evaluated (their inputs changed).
ESKF_HD bool dofs_notch_step(const Model& m, double* dofs, double* notch, double dt) {
  bool changed = false;
  const double n0 = notch[0] + dt * notch[1];
  const double n1 = notch[1] + dt * notch[2];
  changed = (n0 != notch[0]);
  notch[0] = n0;
  notch[1] = n1;
  if (m.flags & FLAG_ZERO_FROZEN) {
#pragma unroll
    for (int i = 0; i < 6; ++i)
      if ((m.frozen_mask >> i) & 1) {
        changed = changed || (dofs[i] != 0.0);
        dofs[i] = 0.0;
      }
  }
  return changed;
}

// ---- propagate: nominal state + Jacobian blocks -------------------------------------
// One Filter.propagate (Filter.py:219-230) minus the covariance product.
//   s        in: pre-step state and buffers; out: post-step state and buffers
//   pk, t    in: probe kinematics at the pre-step (dofs, notch); out: at the post-step ones
//   R_WB     rot(q) of the pre-step quaternion (== s.R_old unless an update intervened)
//   fx       out: Jacobian blocks (FX_* layout)
ESKF_HD void propagate_scalar(const Model& m, Nominal& s, ProbeKin& pk, ProbeTrig& t, const double* R_WB, double dt,
                              const double* om, const double* acc, const double* sig_om, bool want_noise_jac,
                              double* fx) {
  // ---- f_predict (equations.py:44-50,72-100) with the pre-step state ----
  double om_avg[3], dth[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    om_avg[i] = (s.om_old[i] + om[i]) / 2.0;
    dth[i] = dt * om_avg[i];
  }
  double Rn[9], RS[9];
  mul_skew(R_WB, dth, RS);
#pragma unroll
  for (int i = 0; i < 9; ++i) Rn[i] = R_WB[i] + RS[i];
  double a0[3], a1[3], acc_avg[3];
  mv3(R_WB, s.acc_old, a0);
  mv3(Rn, acc, a1);
  const double hdt2 = dt * dt / 2.0;
#pragma unroll
  for (int i = 0; i < 3; ++i) acc_avg[i] = (a0[i] + a1[i]) / 2.0;

  // camera position: p_C + dt v + dt R_WB (v_p + om_avg x p_p), v_p = 0
  double oxp[3], Roxp[3];
  cross3(om_avg, pk.p, oxp);
  mv3(R_WB, oxp, Roxp);
  // camera rotation: R_WC + R_WC [dt R_p^T (om_old + om_p)]x, om_p = z6 * notch_d
  double omt[3], om_c[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) omt[i] = s.om_old[i] + pk.z6[i] * s.notch[1];
  mtv3(pk.R, omt, om_c);
#pragma unroll
  for (int i = 0; i < 3; ++i) om_c[i] = dt * om_c[i];
  double Rc[9], RcS[9];
  quat_to_rot(s.qc, Rc);
  mul_skew(Rc, om_c, RcS);
#pragma unroll
  for (int i = 0; i < 9; ++i) Rc[i] = Rc[i] + RcS[i];

#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double vi = s.v[i];
    s.pc[i] = s.pc[i] + dt * vi + dt * Roxp[i];
    s.p[i] = s.p[i] + dt * vi + hdt2 * acc_avg[i];
    s.v[i] = vi + dt * acc_avg[i];
  }
  const bool probe_changed = dofs_notch_step(m, s.dofs, s.notch, dt);
  // State.from_array (state.py:62-74): Markley quaternions of the first-order matrices
  quat_from_matrix(Rn, s.q);
  quat_from_matrix(Rc, s.qc);

  // ---- error Jacobians (Filter.py:249-342) with the buffered R_old / om_old / acc_old
  //      and the POST-predict dofs / notch ----
  if (probe_changed) probe_update(m, s.dofs, s.notch, pk, t);  // (pk, t) persist: same inputs, same kinematics
  const double* Ro = s.R_old;
  fx[FX_DT] = dt;
  {  // A = (-R_old [acc_old]x) dt
    double T[9];
    mul_skew(Ro, s.acc_old, T);
#pragma unroll
    for (int i = 0; i < 9; ++i) fx[FX_A + i] = -T[i] * dt;
  }
  {  // B = rot(normalise(quat(w=1, v=dt/2 om_old)))^T   (Filter.py:132-134,255)
    double qo[4] = {0.5 * dt * s.om_old[0], 0.5 * dt * s.om_old[1], 0.5 * dt * s.om_old[2], 1.0};
    quat_normalise(qo);
    double Rb[9];
    quat_to_rot(qo, Rb);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) fx[FX_B + 3 * i + j] = Rb[3 * j + i];
  }
  double wt[3];  // om_tr = om_old - sigma_om (noise symbols evaluated at sigma, quirk Q6)
#pragma unroll
  for (int i = 0; i < 3; ++i) wt[i] = s.om_old[i] - sig_om[i];
  {  // C1 = -dt R_old [w]x,  w = p + om_tr x p   (v_tr = p_tr, quirk Q2)
    double w[3], T[9];
    cross3(wt, pk.p, w);
#pragma unroll
    for (int i = 0; i < 3; ++i) w[i] = pk.p[i] + w[i];
    mul_skew(Ro, w, T);
#pragma unroll
    for (int i = 0; i < 9; ++i) fx[FX_C1 + i] = -dt * T[i];
  }
  {  // C2 = dt R_old (I + [om_tr]x) dp/dq(1..6)
    double Mw[9], S[9];
    mul_skew(Ro, wt, S);
#pragma unroll
    for (int i = 0; i < 9; ++i) Mw[i] = dt * (Ro[i] + S[i]);
    const double lq = m.L - s.dofs[3];
    const double dz2[3] = {t.s1 * t.s2, t.c1 * t.s2, t.c2};  // d z6 / d q2
    const double k2 = s.dofs[4] * t.s3 + s.dofs[5] * t.c3;
    double col[6][3];
    col[0][0] = pk.p[1];
    col[0][1] = -pk.p[0];
    col[0][2] = 0.0;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      col[1][i] = lq * dz2[i] - k2 * pk.z6[i];
      col[2][i] = s.dofs[4] * t.eb3[i] - s.dofs[5] * t.ea3[i];
      col[3][i] = -pk.z6[i];
      col[4][i] = t.ea3[i];
      col[5][i] = t.eb3[i];
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      double y[3];
      mv3(Mw, col[k], y);
      fx[FX_C2 + 0 * 6 + k] = y[0];
      fx[FX_C2 + 1 * 6 + k] = y[1];
      fx[FX_C2 + 2 * 6 + k] = y[2];
    }
  }
  {  // D = dt d/dq{1,2,3,7} [ R(q)^T om_tr ]   (R^T om_p is constant: no contribution)
    const double al = dot3(t.ead, wt), be = dot3(t.ebd, wt), ze = dot3(pk.z6, wt);
    const double al1 = t.ead[1] * wt[0] - t.ead[0] * wt[1];
    const double be1 = t.ebd[1] * wt[0] - t.ebd[0] * wt[1];
    const double ze1 = pk.z6[1] * wt[0] - pk.z6[0] * wt[1];
    const double al2 = -t.sd * ze, be2 = -t.cd * ze, ze2 = t.sd * al + t.cd * be;
    // rows: (-alpha, sa zeta + ca beta, ca zeta - sa beta)
    fx[FX_D + 0] = dt * (-al1);
    fx[FX_D + 4] = dt * (m.sa * ze1 + m.ca * be1);
    fx[FX_D + 8] = dt * (m.ca * ze1 - m.sa * be1);
    fx[FX_D + 1] = dt * (-al2);
    fx[FX_D + 5] = dt * (m.sa * ze2 + m.ca * be2);
    fx[FX_D + 9] = dt * (m.ca * ze2 - m.sa * be2);
    // d/dq3: alpha' = beta, beta' = -alpha, zeta' = 0 ; d/dq7 = - d/dq3
    fx[FX_D + 2] = dt * (-be);
    fx[FX_D + 6] = dt * (-m.ca * al);
    fx[FX_D + 10] = dt * (m.sa * al);
    fx[FX_D + 3] = -fx[FX_D + 2];
    fx[FX_D + 7] = -fx[FX_D + 6];
    fx[FX_D + 11] = -fx[FX_D + 10];
  }
  {  // E = I - dt/2 [a + b]x,  a = R_p^T (om_tr + om_p), b = R_p^T (om_old + om_p)
    double ua[3], ub[3], a[3], b[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const double omp = pk.z6[i] * s.notch[1];
      ua[i] = wt[i] + omp;
      ub[i] = s.om_old[i] + omp;
    }
    mtv3(pk.R, ua, a);
    mtv3(pk.R, ub, b);
    const double h = 0.5 * dt;
    const double e0 = h * (a[0] + b[0]), e1 = h * (a[1] + b[1]), e2 = h * (a[2] + b[2]);
    fx[FX_E + 0] = 1.0;
    fx[FX_E + 1] = e2;
    fx[FX_E + 2] = -e1;
    fx[FX_E + 3] = -e2;
    fx[FX_E + 4] = 1.0;
    fx[FX_E + 5] = e0;
    fx[FX_E + 6] = e1;
    fx[FX_E + 7] = -e0;
    fx[FX_E + 8] = 1.0;
  }
  if (want_noise_jac) {  // rows 18:24 of Fi (only matter when Q[3:6] != 0)
    double T[9];
    mul_skew(Ro, pk.p, T);
#pragma unroll
    for (int i = 0; i < 9; ++i) fx[FX_NP + i] = dt * T[i];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) fx[FX_NT + 3 * i + j] = -dt * pk.R[3 * j + i];
  }

  // ---- buffers (Filter.py:224-227) ----
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    s.om_old[i] = om[i];
    s.acc_old[i] = acc[i];
  }
  quat_to_rot(s.q, s.R_old);
}

// ---- covariance propagation:  y = Fx x  applied in place to three 24-vectors ----
// Element i of vector v lives at x[v * VS + i * ES].  Column pass of P:
// ES = row stride, VS = 1; row pass: ES = 1, VS = row stride.
template <int ES, int VS>
ESKF_HD void fx_apply3(double* x, const double* fx) {
  const double dt = fx[FX_DT];
  double xv[3][3], xt[3][3], xd[3][6], xn[3][3], xpc[3][3], xtc[3][3];
#pragma unroll
  for (int v = 0; v < 3; ++v) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      xv[v][i] = x[v * VS + (3 + i) * ES];
      xt[v][i] = x[v * VS + (6 + i) * ES];
      xn[v][i] = x[v * VS + (15 + i) * ES];
      xpc[v][i] = x[v * VS + (18 + i) * ES];
      xtc[v][i] = x[v * VS + (21 + i) * ES];
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) xd[v][i] = x[v * VS + (9 + i) * ES];
  }
  // rows 18:21 (camera position error)
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    double y[3];
#pragma unroll
    for (int v = 0; v < 3; ++v) y[v] = dt * xv[v][i];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double c = fx[FX_C1 + 3 * i + k];
#pragma unroll
      for (int v = 0; v < 3; ++v) y[v] += c * xt[v][k];
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const double c = fx[FX_C2 + 6 * i + k];
#pragma unroll
      for (int v = 0; v < 3; ++v) y[v] += c * xd[v][k];
    }
    // mis-aligned identity block (quirk Q3): Fx[18+i, 16+i] = 1
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      y[v] += (i == 0) ? xn[v][1] : (i == 1) ? xn[v][2] : xpc[v][0];
      x[v * VS + (18 + i) * ES] = y[v];
    }
  }
  // rows 21:24 (camera orientation error)
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    double y[3];
#pragma unroll
    for (int v = 0; v < 3; ++v) y[v] = (i == 0) ? 0.0 : xtc[v][i];  // Fx[22,22] = Fx[23,23] = 1
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double c = fx[FX_D + 4 * i + k];
#pragma unroll
      for (int v = 0; v < 3; ++v) y[v] += c * xd[v][k];
    }
    {
      const double c = fx[FX_D + 4 * i + 3];
#pragma unroll
      for (int v = 0; v < 3; ++v) y[v] += c * xn[v][0];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double c = fx[FX_E + 3 * i + k];
#pragma unroll
      for (int v = 0; v < 3; ++v) y[v] += c * ((k == 0) ? xpc[v][1] : (k == 1) ? xpc[v][2] : xtc[v][0]);
    }
#pragma unroll
    for (int v = 0; v < 3; ++v) x[v * VS + (21 + i) * ES] = y[v];
  }
  // rows 0:3  p += dt v
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) x[v * VS + i * ES] = x[v * VS + i * ES] + dt * xv[v][i];
  // rows 3:6  v += A theta ; rows 6:9 theta = B theta
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    double yv[3], yt[3];
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      yv[v] = xv[v][i];
      yt[v] = 0.0;
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double a = fx[FX_A + 3 * i + k], b = fx[FX_B + 3 * i + k];
#pragma unroll
      for (int v = 0; v < 3; ++v) {
        yv[v] += a * xt[v][k];
        yt[v] += b * xt[v][k];
      }
    }
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      x[v * VS + (3 + i) * ES] = yv[v];
      x[v * VS + (6 + i) * ES] = yt[v];
    }
  }
  // rows 15:17 notch chain
#pragma unroll
  for (int v = 0; v < 3; ++v) {
    x[v * VS + 15 * ES] = xn[v][0] + dt * xn[v][1];
    x[v * VS + 16 * ES] = xn[v][1] + dt * xn[v][2];
  }
}

// Fi Q Fi^T for rows r0..r0+2 of P (row pass epilogue; Filter.py:349).
// With Q[3:6] == 0 (the reference's normal flow, quirk Q5) this is a diagonal add.
template <int ES, int VS>
ESKF_HD void add_process_noise3(double* x, int r0, const double* fx, const double* qd, bool imu_q) {
#pragma unroll
  for (int v = 0; v < 3; ++v) {
    const int r = r0 + v;
    double add = 0.0;
    if (r >= 3 && r < 15) add = qd[r - 3];  // Fi[3:15,0:12] = I
    if (r == 17) add = qd[12];               // Fi[17,12] = 1
    if (add != 0.0) x[v * VS + r * ES] += add;
  }
  if (imu_q && (r0 == 6 || r0 == 18 || r0 == 21)) {
    // n_om drives theta (I), p_C (Np) and theta_C (Nt): L Q_om L^T on rows/cols {6:9,18:21,21:24}
    // the diagonal part of the theta rows was added above.
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      double Lr[3];
#pragma unroll
      for (int k = 0; k < 3; ++k)
        Lr[k] = (r0 == 6) ? ((k == v) ? 1.0 : 0.0) : (r0 == 18) ? fx[FX_NP + 3 * v + k] : fx[FX_NT + 3 * v + k];
#pragma unroll
      for (int cb = 0; cb < 3; ++cb) {
        const int c0 = (cb == 0) ? 6 : (cb == 1) ? 18 : 21;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          if (r0 == 6 && cb == 0) continue;  // already added (diagonal of Q_om)
          double acc = 0.0;
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            const double Lc = (cb == 0) ? ((k == j) ? 1.0 : 0.0) : (cb == 1) ? fx[FX_NP + 3 * j + k] : fx[FX_NT + 3 * j + k];
            acc += Lr[k] * qd[3 + k] * Lc;
          }
          x[v * VS + (c0 + j) * ES] += acc;
        }
      }
    }
  }
}

// ---- update: scalar part ---------------------------------------------------------------
// 7x7 inverse by LU with partial pivoting (np.linalg.inv -> LAPACK gesv, Filter.py:357).
// Fully unrolled so everything stays in registers.  Returns false if a pivot is exactly
// zero or the result is not finite (the reference's LinAlgError branch).
ESKF_HD bool inv7(const double* S, double* Sinv) {
  double a[7][7], b[7][7];
#pragma unroll
  for (int i = 0; i < 7; ++i)
#pragma unroll
    for (int j = 0; j < 7; ++j) {
      a[i][j] = S[7 * i + j];
      b[i][j] = (i == j) ? 1.0 : 0.0;
    }
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    // pivot search: first maximum of |a[i][k]|, i >= k (idamax)
    int piv = k;
    double best = fabs(a[k][k]);
#pragma unroll
    for (int i = k + 1; i < 7; ++i) {
      const double v = fabs(a[i][k]);
      if (v > best) {
        best = v;
        piv = i;
      }
    }
    ok = ok && (best != 0.0);
#pragma unroll
    for (int i = k + 1; i < 7; ++i) {
      if (piv == i) {
#pragma unroll
        for (int j = 0; j < 7; ++j) {
          double tmp = a[k][j];
          a[k][j] = a[i][j];
          a[i][j] = tmp;
          tmp = b[k][j];
          b[k][j] = b[i][j];
          b[i][j] = tmp;
        }
      }
    }
    const double rp = 1.0 / a[k][k];
#pragma unroll
    for (int i = k + 1; i < 7; ++i) {
      const double l = a[i][k] * rp;
#pragma unroll
      for (int j = k + 1; j < 7; ++j) a[i][j] -= l * a[k][j];
#pragma unroll
      for (int j = 0; j < 7; ++j) b[i][j] -= l * b[k][j];
    }
  }
  // back substitution U X = B
#pragma unroll
  for (int i = 6; i >= 0; --i) {
    const double rd = 1.0 / a[i][i];
#pragma unroll
    for (int j = 0; j < 7; ++j) {
      double v = b[i][j];
#pragma unroll
      for (int k = i + 1; k < 7; ++k) v -= a[i][k] * b[k][j];
      b[i][j] = v * rd;
    }
  }
  double chk = 0.0;
#pragma unroll
  for (int i = 0; i < 7; ++i)
#pragma unroll
    for (int j = 0; j < 7; ++j) {
      Sinv[7 * i + j] = b[i][j];
      chk += b[i][j] * 0.0;  // NaN / inf detector
    }
  return ok && (chk == 0.0);
}

// Residual of Filter.update (Filter.py:363-375).  cam_q is the RAW file quaternion (xyzw).
ESKF_HD bool update_residual(const Nominal& s, const double* cam_pos, const double* cam_q, double ang_notch,
                             double* res) {
  double sn, cn;
  sincos(0.5 * ang_notch, &sn, &cn);
  const double nq[4] = {0.0, 0.0, sn, cn};  // Rotation.from_euler("xyz", [0, 0, ang]).as_quat()
  double qm[4], qmc[4], e[4];
  quat_mul(nq, cam_q, qm);
  qmc[0] = -qm[0];
  qmc[1] = -qm[1];
  qmc[2] = -qm[2];
  qmc[3] = qm[3];
  quat_mul(qmc, s.qc, e);
  const double nv = sqrt(e[0] * e[0] + e[1] * e[1] + e[2] * e[2]);
  const double ang = asin(nv);  // quirk Q9: asin|v|, not 2 acos w
  // axis = 0 iff math.isclose(angle, 0) (rel_tol 1e-9, abs_tol 0) <=> angle == 0
  const double f = (ang == 0.0) ? 0.0 : ang / nv;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    res[i] = cam_pos[i] - s.pc[i];
    res[3 + i] = f * e[i];
  }
  res[6] = ang_notch - s.notch[0];
  return nv <= 1.0;  // math.asin raises for |v| > 1
}

// state (+) error state  (state.py:46-60,105-129) incl. the dqc axis slip (quirk Q4)
ESKF_HD void inject_error(const Model& m, Nominal& s, const double* d) {
  const double* th = d + 6;
  const double* thc = d + 21;
  const double nth = sqrt(th[0] * th[0] + th[1] * th[1] + th[2] * th[2]);
  const double nthc = sqrt(thc[0] * thc[0] + thc[1] * thc[1] + thc[2] * thc[2]);
  double dq[4], dqc[4], qn[4];
  quat_about_axis(nth, th, dq);
  quat_about_axis(nthc, th, dqc);  // axis = theta (IMU), not theta_c: state.py:124
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    s.p[i] += d[i];
    s.v[i] += d[3 + i];
    s.notch[i] += d[15 + i];
    s.pc[i] += d[18 + i];
  }
#pragma unroll
  for (int i = 0; i < 6; ++i)
    if (!((m.frozen_mask >> i) & 1)) s.dofs[i] += d[9 + i];  // Filter.py:377-379
  quat_mul(s.q, dq, qn);
#pragma unroll
  for (int i = 0; i < 4; ++i) s.q[i] = qn[i];
  quat_mul(s.qc, dqc, qn);
#pragma unroll
  for (int i = 0; i < 4; ++i) s.qc[i] = qn[i];
}

// ---- update: covariance part ---------------------------------------------------------------
// Gain rows r0..r0+2:  K = (P H^T) inv(S);  delta = K res;  bookkeeping for Joseph.
// P is addressed as P[i * RS + j].
template <int RS>
ESKF_HD void gain_rows3(const double* P, int r0, double* up) {
#pragma unroll
  for (int v = 0; v < 3; ++v) {
    const int r = r0 + v;
    double ph[7], k[7];
#pragma unroll
    for (int j = 0; j < 7; ++j) ph[j] = P[r * RS + ESKF_HSET(j)];
    double dl = 0.0;
#pragma unroll
    for (int mm = 0; mm < 7; ++mm) {
      double acc = 0.0;
#pragma unroll
      for (int j = 0; j < 7; ++j) acc += ph[j] * up[UP_SINV + 7 * j + mm];
      k[mm] = acc;
      dl += acc * up[UP_RES + mm];
    }
    up[UP_DELTA + r] = dl;
    double cd = 1.0;
#pragma unroll
    for (int mm = 0; mm < 7; ++mm) {
      const bool diag = (ESKF_HSET(mm) == r);
      up[UP_KZ + 7 * r + mm] = diag ? 0.0 : k[mm];
      if (diag) {
        up[UP_KD + mm] = k[mm];
        cd = 1.0 - k[mm];  // (I - K H)[r][r]
      }
    }
    up[UP_CD + r] = cd;
  }
}

// y = (I - K H) x on three 24-vectors, in place (Joseph factor, Filter.py:384).
template <int ES, int VS>
ESKF_HD void joseph_apply3(double* x, const double* up) {
  double xh[3][7];
#pragma unroll
  for (int v = 0; v < 3; ++v)
#pragma unroll
    for (int mm = 0; mm < 7; ++mm) xh[v][mm] = x[v * VS + ESKF_HSET(mm) * ES];
#pragma unroll
  for (int i = 0; i < 24; ++i) {
    const double cd = up[UP_CD + i];
    double y[3];
#pragma unroll
    for (int v = 0; v < 3; ++v) y[v] = cd * x[v * VS + i * ES];
#pragma unroll
    for (int mm = 0; mm < 7; ++mm) {
      const double k = up[UP_KZ + 7 * i + mm];
#pragma unroll
      for (int v = 0; v < 3; ++v) y[v] -= k * xh[v][mm];
    }
#pragma unroll
    for (int v = 0; v < 3; ++v) x[v * VS + i * ES] = y[v];
  }
}

// Row pass of the update for rows r0..r0+2 (ES = 1):
//   P2 = P1 (I-KH)^T + (K R) K^T ;  P3 = G P2 G^T   (Filter.py:384-390)
// The reset matrix G is block diagonal with 3x3 blocks aligned to the row triples, so both
// G P2 (mixes the three rows held here) and (.) G^T (mixes entries 6:9 / 21:24 of a row)
// are local to the caller.
template <int VS>
ESKF_HD void joseph_rows_finish3(double* x, int r0, const double* up, const double* rd) {
  double xh[3][7], kr[3][7];
#pragma unroll
  for (int v = 0; v < 3; ++v)
#pragma unroll
    for (int mm = 0; mm < 7; ++mm) {
      xh[v][mm] = x[v * VS + ESKF_HSET(mm)];
      const int r = r0 + v;
      const double k = (ESKF_HSET(mm) == r) ? up[UP_KD + mm] : up[UP_KZ + 7 * r + mm];
      kr[v][mm] = k * rd[mm];
    }
  // reset blocks: G = I - [delta_theta / 2]x  (rows 6:9 from delta[6:9], rows 21:24 from delta[21:24])
  const bool mix = (r0 == 6) || (r0 == 21);
  double g[3] = {0.0, 0.0, 0.0};
  if (mix) {
#pragma unroll
    for (int i = 0; i < 3; ++i) g[i] = 0.5 * up[UP_DELTA + r0 + i];
  }
  const double gt[3] = {0.5 * up[UP_DELTA + 6], 0.5 * up[UP_DELTA + 7], 0.5 * up[UP_DELTA + 8]};
  const double gc[3] = {0.5 * up[UP_DELTA + 21], 0.5 * up[UP_DELTA + 22], 0.5 * up[UP_DELTA + 23]};
  double hold[3][6];
#pragma unroll
  for (int i = 0; i < 24; ++i) {
    const double cd = up[UP_CD + i];
    double y[3];
#pragma unroll
    for (int v = 0; v < 3; ++v) y[v] = cd * x[v * VS + i];
    double ki[7];
#pragma unroll
    for (int mm = 0; mm < 7; ++mm) {
      const double kz = up[UP_KZ + 7 * i + mm];
      ki[mm] = kz;
#pragma unroll
      for (int v = 0; v < 3; ++v) y[v] -= kz * xh[v][mm];
    }
    // K R K^T column i: K[i][m] needs the diagonal entries back
    {
      double z[3] = {0.0, 0.0, 0.0};
#pragma unroll
      for (int mm = 0; mm < 7; ++mm) {
        const double k = (ESKF_HSET(mm) == i) ? up[UP_KD + mm] : ki[mm];
#pragma unroll
        for (int v = 0; v < 3; ++v) z[v] += kr[v][mm] * k;
      }
#pragma unroll
      for (int v = 0; v < 3; ++v) y[v] += z[v];
    }
    if (mix) {  // G P2: rows (I - [g]x) applied across the three rows held here
      const double y0 = y[0], y1 = y[1], y2 = y[2];
      // (I - [g]x) = [[1, g2, -g1], [-g2, 1, g0], [g1, -g0, 1]]
      y[0] = y0 + g[2] * y1 - g[1] * y2;
      y[1] = -g[2] * y0 + y1 + g[0] * y2;
      y[2] = g[1] * y0 - g[0] * y1 + y2;
    }
    const bool held = (i >= 6 && i < 9) || (i >= 21);
    if (held) {
      const int hi = (i < 9) ? i - 6 : i - 18;
#pragma unroll
      for (int v = 0; v < 3; ++v) hold[v][hi] = y[v];
    } else {
#pragma unroll
      for (int v = 0; v < 3; ++v) x[v * VS + i] = y[v];
    }
  }
  // (.) G^T on columns 6:9 and 21:24
#pragma unroll
  for (int v = 0; v < 3; ++v) {
    const double a0 = hold[v][0], a1 = hold[v][1], a2 = hold[v][2];
    x[v * VS + 6] = a0 + gt[2] * a1 - gt[1] * a2;
    x[v * VS + 7] = -gt[2] * a0 + a1 + gt[0] * a2;
    x[v * VS + 8] = gt[1] * a0 - gt[0] * a1 + a2;
    const double b0 = hold[v][3], b1 = hold[v][4], b2 = hold[v][5];
    x[v * VS + 21] = b0 + gc[2] * b1 - gc[1] * b2;
    x[v * VS + 22] = -gc[2] * b0 + b1 + gc[0] * b2;
    x[v * VS + 23] = gc[1] * b0 - gc[0] * b1 + b2;
  }
}

// =====================================================================================
// Building blocks of the warp-specialised kernel (eskf_kernel3.cuh): the same arithmetic as
// propagate_scalar, cut along the lines of its scalar roles -- IMU nominal state, camera nominal
// state, Jacobian blocks.  The covariance algebra on the register-resident tile is in eskf_cov3.cuh.
// tests/hostcheck replays them on the CPU against propagate_scalar / fx_apply3 and the oracle.
// =====================================================================================

// "fx3 record": Jacobian blocks in the order the covariance role consumes them.  Element (k, i) of a row
// group lives at BASE + ROWS * k + i: the coefficients of one column k for all rows of the group are
// adjacent, so that the group is applied column by column with 16-byte fetches.
constexpr int FX3_DT = 0;    // dt, pad
constexpr int FX3_H2 = 2;    // rows 21:24, 7 columns {9,10,11,15,19,20,21} x 3 rows (+1 pad):  D (4) then E (3)
constexpr int FX3_H1 = 24;   // rows 18:21, 9 columns 6..14 x 3 rows (+1 pad):                 C1 (3) then C2 (6)
constexpr int FX3_AB = 52;   // rows 3:9,   3 columns 6..8 x 6 rows:                           A rows then B rows
constexpr int FX3_MAIN = 70; // everything below is always written
constexpr int FX3_NP = 70;   // 3x3 (+pad)  Fi[18:21,3:6]   (only with IMU noise in Q, Filter.py:110-117)
constexpr int FX3_NT = 80;   // 3x3 (+pad)  Fi[21:24,3:6]
constexpr int FX3_SIZE = 90;
constexpr int FX3_NPAIR = FX3_SIZE / 2;       // 45
constexpr int FX3_NPAIR_MAIN = FX3_MAIN / 2;  // 35

// Filter._predict_nominal, IMU part (equations.py:72-86; state.py:62-69): p, v, q.
//   R_WB   rot(q) of the pre-step quaternion;  Rn_out  = rot(q+) (the new R_WB_old, Filter.py:227)
ESKF_HD void imu_nominal_step(double* p, double* v, double* q, const double* R_WB, double dt, const double* om_old,
                              const double* acc_old, const double* om, const double* acc, double* R_new) {
  double dth[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) dth[i] = dt * ((om_old[i] + om[i]) / 2.0);
  double Rn[9], RS[9];
  mul_skew(R_WB, dth, RS);
#pragma unroll
  for (int i = 0; i < 9; ++i) Rn[i] = R_WB[i] + RS[i];
  double a0[3], a1[3];
  mv3(R_WB, acc_old, a0);
  mv3(Rn, acc, a1);
  const double hdt2 = dt * dt / 2.0;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double aa = (a0[i] + a1[i]) / 2.0;
    const double vi = v[i];
    p[i] = p[i] + dt * vi + hdt2 * aa;
    v[i] = vi + dt * aa;
  }
  quat_from_matrix(Rn, q);
  quat_to_rot(q, R_new);
}

// Filter._predict_nominal, camera part (equations.py:88-98; state.py:70-74): p_cam, q_cam.
//   v_pre, R_WB   pre-step IMU velocity and rotation;  pk/notch_d at the pre-step (dofs, notch)
ESKF_HD void cam_nominal_step(double* pc, double* qc, const double* v_pre, const double* R_WB, double dt,
                              const double* om_old, const double* om, const double* pk_p, const double* pk_R,
                              const double* pk_z6, double notch_d) {
  double om_avg[3], oxp[3], Roxp[3], omt[3], om_c[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) om_avg[i] = (om_old[i] + om[i]) / 2.0;
  cross3(om_avg, pk_p, oxp);
  mv3(R_WB, oxp, Roxp);
#pragma unroll
  for (int i = 0; i < 3; ++i) omt[i] = om_old[i] + pk_z6[i] * notch_d;
  mtv3(pk_R, omt, om_c);
#pragma unroll
  for (int i = 0; i < 3; ++i) om_c[i] = dt * om_c[i];
  double Rc[9], RcS[9];
  quat_to_rot(qc, Rc);
  mul_skew(Rc, om_c, RcS);
#pragma unroll
  for (int i = 0; i < 9; ++i) Rc[i] = Rc[i] + RcS[i];
#pragma unroll
  for (int i = 0; i < 3; ++i) pc[i] = pc[i] + dt * v_pre[i] + dt * Roxp[i];
  quat_from_matrix(Rc, qc);
}

// ---- probe kinematics / trigonometry cache behind strided views ---------------------------------------
// The Jacobian role keeps (pk, t) in shared memory, element-major over the filters of a CTA (stride ST);
// with ST = 1 the same views sit on top of plain ProbeKin / ProbeTrig structs (host replay).
template <int ST>
struct PKView {  // ProbeKin: p(3) R(9) z6(3)
  double* b;
  ESKF_HD double& p(int i) const { return b[i * ST]; }
  ESKF_HD double& R(int i) const { return b[(3 + i) * ST]; }
  ESKF_HD double& z6(int i) const { return b[(12 + i) * ST]; }
};
template <int ST>
struct TRView {  // ProbeTrig: s1 c1 s2 c2 s3 c3 sd cd ea3(3) eb3(3) ead(3) ebd(3) a1 a2 a3 ad
  double* b;
  ESKF_HD double& sc(int i) const { return b[i * ST]; }  // 0..7: s1 c1 s2 c2 s3 c3 sd cd
  ESKF_HD double& ea3(int i) const { return b[(8 + i) * ST]; }
  ESKF_HD double& eb3(int i) const { return b[(11 + i) * ST]; }
  ESKF_HD double& ead(int i) const { return b[(14 + i) * ST]; }
  ESKF_HD double& ebd(int i) const { return b[(17 + i) * ST]; }
  ESKF_HD double& ang(int i) const { return b[(20 + i) * ST]; }  // a1 a2 a3 ad
};
constexpr int TR_SIZE = 24;
constexpr int PK_SIZE = 15;
static_assert(sizeof(ProbeTrig) == TR_SIZE * sizeof(double) && sizeof(ProbeKin) == PK_SIZE * sizeof(double), "view layout");

// probe_update on views: the sines / cosines whose angle changed are evaluated again, everything that
// depends on them is rebuilt into (pk, t).  Same arithmetic as probe_update / probe_assemble.
template <int ST, int SP>
ESKF_HD void probe_update_v(const Model& m, const double* dofs, const double* notch, const PKView<SP>& k, const TRView<ST>& t) {
  const double ang[4] = {dofs[0], dofs[1], dofs[2], dofs[2] - notch[0]};
  double sc[8];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (ang[j] != t.ang(j)) {
      t.ang(j) = ang[j];
      sincos(ang[j], &sc[2 * j], &sc[2 * j + 1]);
      t.sc(2 * j) = sc[2 * j];
      t.sc(2 * j + 1) = sc[2 * j + 1];
    } else {
      sc[2 * j] = t.sc(2 * j);
      sc[2 * j + 1] = t.sc(2 * j + 1);
    }
  }
  const double s1 = sc[0], c1 = sc[1], s2 = sc[2], c2 = sc[3], s3 = sc[4], c3 = sc[5], sd = sc[6], cd = sc[7];
  const double s1s2 = s1 * s2, c1s2 = c1 * s2;
  const double ea3[3] = {s1s2 * s3 - c1 * c3, s1 * c3 + c1s2 * s3, c2 * s3};
  const double eb3[3] = {s1s2 * c3 + c1 * s3, c1s2 * c3 - s1 * s3, c2 * c3};
  const double ead[3] = {s1s2 * sd - c1 * cd, s1 * cd + c1s2 * sd, c2 * sd};
  const double ebd[3] = {s1s2 * cd + c1 * sd, c1s2 * cd - s1 * sd, c2 * cd};
  const double z6[3] = {-s1 * c2, -c1 * c2, s2};
  const double lq = m.L - dofs[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    t.ea3(i) = ea3[i];
    t.eb3(i) = eb3[i];
    t.ead(i) = ead[i];
    t.ebd(i) = ebd[i];
    k.z6(i) = z6[i];
    k.p(i) = lq * z6[i] + dofs[4] * ea3[i] + dofs[5] * eb3[i];
    k.R(3 * i + 0) = -ead[i];
    k.R(3 * i + 1) = m.sa * z6[i] + m.ca * ebd[i];
    k.R(3 * i + 2) = m.ca * z6[i] - m.sa * ebd[i];
  }
}

// Filter._predict_error (Filter.py:249-342): the Jacobian blocks in the fx3 layout, one function per row
// group, from the buffered R_old / om_old / acc_old and the POST-predict (dofs, notch) whose probe
// kinematics are (pk, t).  fx points at the whole FX3 record (registers: every index is a compile-time
// constant); each function fills its own group.

// rows 3:9 -- A = (-R_old [acc_old]x) dt and B = rot(normalise(quat(w=1, v=dt/2 om_old)))^T (Filter.py:132-134,255)
ESKF_HD void jac_rows_ab(const double* Ro, double dt, const double* om_old, const double* acc_old, double* fx) {
  double T[9];
  mul_skew(Ro, acc_old, T);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int k = 0; k < 3; ++k) fx[FX3_AB + 6 * k + i] = -T[3 * i + k] * dt;
  double qo[4] = {0.5 * dt * om_old[0], 0.5 * dt * om_old[1], 0.5 * dt * om_old[2], 1.0};
  quat_normalise(qo);
  double Rb[9];
  quat_to_rot(qo, Rb);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int k = 0; k < 3; ++k) fx[FX3_AB + 6 * k + 3 + i] = Rb[3 * k + i];  // B(i, k) = Rb(k, i)
}

// dt pair + rows 21:24 -- D = dt d/dq{1,2,3,7} [R(q)^T om_tr] (R^T om_p is constant: no contribution) and
// E = I - dt/2 [a + b]x, a = R_p^T (om_tr + om_p), b = R_p^T (om_old + om_p)
template <int ST, int SP>
ESKF_HD void jac_rows_h2(const Model& m, double notch_d, const PKView<SP>& pk, const TRView<ST>& t, double dt,
                         const double* om_old, const double* sig_om, double* fx) {
  fx[FX3_DT] = dt;
  fx[FX3_DT + 1] = 0.0;
  double wt[3];  // om_tr = om_old - sigma_om (noise symbols evaluated at sigma, quirk Q6)
#pragma unroll
  for (int i = 0; i < 3; ++i) wt[i] = om_old[i] - sig_om[i];
  const double sd = t.sc(6), cd = t.sc(7);
  const double z6[3] = {pk.z6(0), pk.z6(1), pk.z6(2)};
  {
    const double ead[3] = {t.ead(0), t.ead(1), t.ead(2)}, ebd[3] = {t.ebd(0), t.ebd(1), t.ebd(2)};
    const double al = dot3(ead, wt), be = dot3(ebd, wt), ze = dot3(z6, wt);
    const double al1 = ead[1] * wt[0] - ead[0] * wt[1];
    const double be1 = ebd[1] * wt[0] - ebd[0] * wt[1];
    const double ze1 = z6[1] * wt[0] - z6[0] * wt[1];
    const double al2 = -sd * ze, be2 = -cd * ze, ze2 = sd * al + cd * be;
    double* D = fx + FX3_H2;  // D(i, k) at D[3 * k + i]; rows: (-alpha, sa zeta + ca beta, ca zeta - sa beta)
    D[0] = dt * (-al1);
    D[1] = dt * (m.sa * ze1 + m.ca * be1);
    D[2] = dt * (m.ca * ze1 - m.sa * be1);
    D[3] = dt * (-al2);
    D[4] = dt * (m.sa * ze2 + m.ca * be2);
    D[5] = dt * (m.ca * ze2 - m.sa * be2);
    // d/dq3: alpha' = beta, beta' = -alpha, zeta' = 0 ; d/dq7 = - d/dq3
    D[6] = dt * (-be);
    D[7] = dt * (-m.ca * al);
    D[8] = dt * (m.sa * al);
    D[9] = -D[6];
    D[10] = -D[7];
    D[11] = -D[8];
  }
  {
    double ua[3], ub[3], a[3], b[3], R[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) R[i] = pk.R(i);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const double omp = z6[i] * notch_d;
      ua[i] = wt[i] + omp;
      ub[i] = om_old[i] + omp;
    }
    mtv3(R, ua, a);
    mtv3(R, ub, b);
    const double h = 0.5 * dt;
    const double e0 = h * (a[0] + b[0]), e1 = h * (a[1] + b[1]), e2 = h * (a[2] + b[2]);
    double* E = fx + FX3_H2 + 12;  // E(i, k) at E[3 * k + i]
    E[0] = 1.0;
    E[1] = -e2;
    E[2] = e1;
    E[3] = e2;
    E[4] = 1.0;
    E[5] = -e0;
    E[6] = -e1;
    E[7] = e0;
    E[8] = 1.0;
    fx[FX3_H2 + 21] = 0.0;
  }
}

// rows 18:21 -- C1 = -dt R_old [w]x, w = p + om_tr x p (v_tr = p_tr, quirk Q2) and
// C2 = dt R_old (I + [om_tr]x) dp/dq(1..6)
template <int ST, int SP>
ESKF_HD void jac_rows_h1(const Model& m, const double* dofs, const PKView<SP>& pk, const TRView<ST>& t, const double* Ro,
                         double dt, const double* om_old, const double* sig_om, double* fx) {
  double wt[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) wt[i] = om_old[i] - sig_om[i];
  const double p[3] = {pk.p(0), pk.p(1), pk.p(2)};
  {
    double w[3], T[9];
    cross3(wt, p, w);
#pragma unroll
    for (int i = 0; i < 3; ++i) w[i] = p[i] + w[i];
    mul_skew(Ro, w, T);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int k = 0; k < 3; ++k) fx[FX3_H1 + 3 * k + i] = -dt * T[3 * i + k];
  }
  double Mw[9], S[9];
  mul_skew(Ro, wt, S);
#pragma unroll
  for (int i = 0; i < 9; ++i) Mw[i] = dt * (Ro[i] + S[i]);
  const double s1 = t.sc(0), c1 = t.sc(1), s2 = t.sc(2), c2 = t.sc(3), s3 = t.sc(4), c3 = t.sc(5);
  const double lq = m.L - dofs[3];
  const double dz2[3] = {s1 * s2, c1 * s2, c2};  // d z6 / d q2
  const double k2 = dofs[4] * s3 + dofs[5] * c3;
  double col[3];
  col[0] = p[1];
  col[1] = -p[0];
  col[2] = 0.0;
  mv3(Mw, col, fx + FX3_H1 + 9);
#pragma unroll
  for (int i = 0; i < 3; ++i) col[i] = lq * dz2[i] - k2 * pk.z6(i);
  mv3(Mw, col, fx + FX3_H1 + 12);
#pragma unroll
  for (int i = 0; i < 3; ++i) col[i] = dofs[4] * t.eb3(i) - dofs[5] * t.ea3(i);
  mv3(Mw, col, fx + FX3_H1 + 15);
#pragma unroll
  for (int i = 0; i < 3; ++i) col[i] = -pk.z6(i);
  mv3(Mw, col, fx + FX3_H1 + 18);
#pragma unroll
  for (int i = 0; i < 3; ++i) col[i] = t.ea3(i);
  mv3(Mw, col, fx + FX3_H1 + 21);
#pragma unroll
  for (int i = 0; i < 3; ++i) col[i] = t.eb3(i);
  mv3(Mw, col, fx + FX3_H1 + 24);
  fx[FX3_H1 + 27] = 0.0;
}

// rows 18:24 of Fi (only matter when Q[3:6] != 0, Filter.py:110-117)
template <int SP>
ESKF_HD void jac_rows_noise(const PKView<SP>& pk, const double* Ro, double dt, double* fx) {
  double T[9];
  const double p[3] = {pk.p(0), pk.p(1), pk.p(2)};
  mul_skew(Ro, p, T);
#pragma unroll
  for (int i = 0; i < 9; ++i) fx[FX3_NP + i] = dt * T[i];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) fx[FX3_NT + 3 * i + j] = -dt * pk.R(3 * j + i);
  fx[FX3_NP + 9] = 0.0;
  fx[FX3_NT + 9] = 0.0;
}

// 16-byte coefficient pairs of the fx3 record
struct alignas(16) d2 {
  double x, y;
};

// ---- CTA mapping of stacked trajectories (eskf_kernel3, n_traj > 1) --------------------------------------------------
// A CTA follows ONE trajectory's epoch structure, so every trajectory's fpt filters are cut into ceil(fpt / F) CTAs of
// their own, the last one ragged.  A batch of N filters (a shard starts at a trajectory boundary) holds N / fpt whole
// trajectories and, when N % fpt != 0, a partially covered last one: that one gets only the ceil((N % fpt) / F) CTAs that
// hold filters, and they come last, so the decode below is the same for every block and no CTA is empty.
ESKF_HD int64_t stacked_grid(int64_t N, int64_t fpt, int F) {
  const int64_t cpt = (fpt + F - 1) / F;
  return (N / fpt) * cpt + ((N % fpt) + F - 1) / F;
}
// block -> first filter f0, number of filters nf (1..F) and trajectory tl, counted from the batch's first trajectory
ESKF_HD void stacked_cta(int64_t block, int64_t N, int64_t fpt, int F, int64_t& f0, int& nf, int64_t& tl) {
  const int64_t cpt = (fpt + F - 1) / F;
  tl = block / cpt;
  const int64_t ch = block - tl * cpt;
  f0 = tl * fpt + ch * F;
  int64_t left = fpt - ch * F;
  if (N - f0 < left) left = N - f0;
  nf = (int)(left < F ? left : F);
}

}  // namespace eskf
