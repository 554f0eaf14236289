// Covariance algebra of the VI-ESKF hot path on a REGISTER-RESIDENT tile (FP64), the building blocks of
// the covariance role of eskf_kernel3.cuh.  Host/device straight-line code: tests/hostcheck replays the
// eight lanes of a filter on the CPU against the oracle.
//
// Eight lanes own one filter; lane g keeps X[k][v] = P(k, 3g+v), the three columns of state group g of
// the symmetric 24x24 covariance (72 doubles).
//   Filter._predict_error_covariance (Filter.py:344-349):   P' = Fx P Fx^T + Fi Q Fi^T
//       pass 1   T(:, tile) = Fx X                   local; rows go straight to the transposition buffer
//       transposition through shared memory          X[k][v] <- T(3g+v, k)
//       pass 2   X <- Fx X (+ Q terms)               = (Fx T^T)(:, tile) = P'(tile, :)^T = P'(:, tile)
//   Filter.update (Filter.py:351-395), all on the register tile:
//       S columns live in lanes 5..7 (H selects rows/cols {18..23, 15}); K rows use P(h_m, r) = X[h_m][v];
//       W = (I - K H) P is local given K; P' = W (I - K H)^T + (K R) K^T needs W(:, h) and K R; the reset blocks
//       G = I - [delta_theta / 2]x mix rows 6:9 / 21:24 (local) and the columns of lanes 2 and 7 (local).
// The sparse transition matrix is applied with nine (three rows x three columns) independent accumulators
// per row group so that the FP64 pipe always has independent work in flight.
#pragma once
#include "eskf_math.cuh"

#ifndef ESKF_OPT_UPD
#define ESKF_OPT_UPD 1  // hand-pipelined record fetches in the loops of the camera update
#endif
#ifndef ESKF_OPT_FIN14
#define ESKF_OPT_FIN14 0  // Joseph form: both sums of upd3_finish as one rolled loop of fourteen columns
#endif
#ifndef ESKF_OPT_ST2
#define ESKF_OPT_ST2 0  // pass 2: the fetches of the head of the pass spread over its first multiply-adds
#endif
#ifndef ESKF_OPT_QP
#define ESKF_OPT_QP 0  // process-noise diagonal as predicated adds
#endif
#ifndef ESKF_OPT_ST1
#define ESKF_OPT_ST1 1  // pass 1: the stores of the identity rows are spread over the multiply-adds of the other row groups
#endif

namespace eskf {

// N consecutive coefficients starting at the (even) record offset base, held as pairs
template <int PS, int N>
struct Coefs {
  d2 p[(N + 1) / 2];
  ESKF_HD void load(const d2* f2, int base) {
#pragma unroll
    for (int j = 0; j < (N + 1) / 2; ++j) p[j] = f2[(base / 2 + j) * PS];
  }
  ESKF_HD double operator()(int idx) const { return (idx & 1) ? p[idx >> 1].y : p[idx >> 1].x; }
};

// The row groups below fetch their coefficients in windows of two columns (three 16-byte pairs for a
// three-row group): a short live range per window instead of the whole block in registers.

// rows 21:24 (camera orientation error): y[i][v]
template <int PS>
ESKF_HD void fx3_rows_h2(const double (&X)[24][3], const d2* f2, double (&y)[3][3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) y[i][v] = (i == 0) ? 0.0 : X[21 + i][v];  // Fx[22,22] = Fx[23,23] = 1
#pragma unroll
  for (int kb = 0; kb < 7; kb += 2) {
    Coefs<PS, 6> c;  // columns kb, kb + 1
    c.load(f2, FX3_H2 + 3 * kb);
#pragma unroll
    for (int k = kb; k < kb + 2 && k < 7; ++k) {
      const int col = (k < 3) ? 9 + k : (k == 3) ? 15 : 19 + (k - 4);  // D on dofs 1..3 and the notch, E on 19:22 (quirk Q3)
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int v = 0; v < 3; ++v) y[i][v] += c(3 * (k - kb) + i) * X[col][v];
    }
  }
}

// rows 18:21 (camera position error): y[i][v]
template <int PS>
ESKF_HD void fx3_rows_h1(const double (&X)[24][3], const d2* f2, double dt, double (&y)[3][3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) y[i][v] = X[16 + i][v] + dt * X[3 + i][v];  // mis-aligned identity block (quirk Q3)
#pragma unroll
  for (int kb = 0; kb < 9; kb += 2) {  // C1 on theta (6:9), C2 on dofs (9:15)
    Coefs<PS, 6> c;
    c.load(f2, FX3_H1 + 3 * kb);
#pragma unroll
    for (int k = kb; k < kb + 2 && k < 9; ++k)
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int v = 0; v < 3; ++v) y[i][v] += c(3 * (k - kb) + i) * X[6 + k][v];
  }
}

// rows 3:6  v += A theta ; rows 6:9  theta = B theta
template <int PS>
ESKF_HD void fx3_rows_ab(const double (&X)[24][3], const d2* f2, double (&ya)[3][3], double (&yb)[3][3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      ya[i][v] = X[3 + i][v];
      yb[i][v] = 0.0;
    }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    Coefs<PS, 6> c;
    c.load(f2, FX3_AB + 6 * k);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int v = 0; v < 3; ++v) {
        ya[i][v] += c(i) * X[6 + k][v];
        yb[i][v] += c(3 + i) * X[6 + k][v];
      }
  }
}

// Transposed reload between the passes: X[k][v] <- T(3g+v, k) from the rows 3g..3g+2 of the buffer (row
// stride RS doubles, 16-byte aligned), as 16-byte pairs in the order the row groups of pass 2 consume them
// (rows 21:24 first: columns 9..11, 15, 19..23; then rows 18:21: columns 3..18; columns 0..2 last).
template <int RS>
ESKF_HD void fx3_load_transposed(double (&X)[24][3], const double* rows) {
  constexpr int order[12] = {4, 5, 7, 9, 10, 11, 1, 2, 3, 6, 8, 0};
#pragma unroll
  for (int o = 0; o < 12; ++o) {
    const int j = order[o];
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      const d2 t = reinterpret_cast<const d2*>(rows + v * RS)[j];
      X[2 * j][v] = t.x;
      X[2 * j + 1][v] = t.y;
    }
  }
}

// Pass 1: T(:, tile) = Fx X, row i stored as out[i * OS + v] as soon as it is finished (X is not modified;
// the next pass starts from the transposed tile).
// ALL 24 rows are exchanged, the identity rows 9:15 of Fx included.  (T(9:15, :) = P(9:15, :), and a symmetric P would
// let lanes 3 and 4 keep their own tile instead of reloading it -- an earlier version did, and saved 18 stores per lane.
// But the stored matrix is only symmetric up to rounding: with that shortcut the tiles of lanes 3 and 4 follow
// G' = Fx G Fx^T while all others follow G' = Fx G^T Fx^T, which turns the antisymmetric rounding noise of the
// dof / other cross blocks into a symmetric perturbation at every step.  With the default tuning nothing shows; with
// process noise 10x smaller -- a fifth of the BASELINE config-3 grid -- the asymmetry grew tenfold per epoch and the
// filter blew up after 15 updates where the oracle and the first kernel stay together at 1e-10:
// tests/test_hostcheck.py::test_free_running_low_process_noise, tests/test_gpu_full_size.py.)
template <int PS, int OS>
ESKF_HD void fx3_apply_store(const double (&X)[24][3], const d2* f2, double* out) {
  const double dt = f2[(FX3_DT / 2) * PS].x;
  // identity rows of Fx: dofs 9:15 and notch'' 17
#pragma unroll
  for (int i = 9; i < 15; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) out[i * OS + v] = X[i][v];
#pragma unroll
  for (int v = 0; v < 3; ++v) out[17 * OS + v] = X[17][v];
  double y[3][3], z[3][3];
  fx3_rows_h2<PS>(X, f2, y);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) out[(21 + i) * OS + v] = y[i][v];
  fx3_rows_h1<PS>(X, f2, dt, y);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) out[(18 + i) * OS + v] = y[i][v];
#pragma unroll
  for (int i = 0; i < 3; ++i)  // rows 0:3  p += dt v
#pragma unroll
    for (int v = 0; v < 3; ++v) out[i * OS + v] = X[i][v] + dt * X[3 + i][v];
  fx3_rows_ab<PS>(X, f2, y, z);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      out[(3 + i) * OS + v] = y[i][v];
      out[(6 + i) * OS + v] = z[i][v];
    }
#pragma unroll
  for (int v = 0; v < 3; ++v) {  // rows 15:17 notch chain
    out[15 * OS + v] = X[15][v] + dt * X[16][v];
    out[16 * OS + v] = X[16][v] + dt * X[17][v];
  }
}

// Pass 1 with the 72 stores spread over the 222 multiply-adds (ESKF_OPT_ST1): as written above the identity rows leave as
// one burst of 21 stores at the head of the pass, in all covariance warps of the CTA at the same time, and the shared-memory
// queue throttles (ncu: ~8 cycles per store there against ~2 for the stores that sit between multiply-adds).  Same
// operations per accumulator in the same order: bit-identical.
template <int PS, int OS>
ESKF_HD void fx3_apply_store_il(const double (&X)[24][3], const d2* f2, double* out) {
  const double dt = f2[(FX3_DT / 2) * PS].x;
  auto putX = [&](int row) {
#pragma unroll
    for (int v = 0; v < 3; ++v) out[row * OS + v] = X[row][v];
  };
  double y[3][3], z[3][3], w[3][3];
  // rows 21:24; between its seven columns: identity rows 9..14 and 17
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) y[i][v] = (i == 0) ? 0.0 : X[21 + i][v];
#pragma unroll
  for (int kb = 0; kb < 7; kb += 2) {
    Coefs<PS, 6> c;
    c.load(f2, FX3_H2 + 3 * kb);
#if ESKF_OPT_ST1 == 2
    if (kb == 0) {  // (two identity rows behind the first coefficient fetch: something to issue while it is in flight)
      putX(9);
      putX(10);
    }
#endif
#pragma unroll
    for (int k = kb; k < kb + 2 && k < 7; ++k) {
      const int col = (k < 3) ? 9 + k : (k == 3) ? 15 : 19 + (k - 4);
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int v = 0; v < 3; ++v) y[i][v] += c(3 * (k - kb) + i) * X[col][v];
#if ESKF_OPT_ST1 == 2
      if (k < 5) putX(k < 4 ? 11 + k : 17);
#else
      putX(k < 6 ? 9 + k : 17);
#endif
    }
  }
  // rows 18:21; between its nine columns: the finished rows 21:24, rows 0:3 (p += dt v) and the notch chain
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) z[i][v] = X[16 + i][v] + dt * X[3 + i][v];
#pragma unroll
  for (int kb = 0; kb < 9; kb += 2) {
    Coefs<PS, 6> c;
    c.load(f2, FX3_H1 + 3 * kb);
#pragma unroll
    for (int k = kb; k < kb + 2 && k < 9; ++k) {
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int v = 0; v < 3; ++v) z[i][v] += c(3 * (k - kb) + i) * X[6 + k][v];
      if (k < 3) {
#pragma unroll
        for (int v = 0; v < 3; ++v) out[(21 + k) * OS + v] = y[k][v];
      } else if (k < 6) {
#pragma unroll
        for (int v = 0; v < 3; ++v) out[(k - 3) * OS + v] = X[k - 3][v] + dt * X[k][v];
      } else if (k == 6) {
#pragma unroll
        for (int v = 0; v < 3; ++v) out[15 * OS + v] = X[15][v] + dt * X[16][v];
      } else if (k == 7) {
#pragma unroll
        for (int v = 0; v < 3; ++v) out[16 * OS + v] = X[16][v] + dt * X[17][v];
      }
    }
  }
  // rows 3:9; between its three columns: the finished rows 18:21
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      y[i][v] = X[3 + i][v];
      w[i][v] = 0.0;
    }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    Coefs<PS, 6> c;
    c.load(f2, FX3_AB + 6 * k);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int v = 0; v < 3; ++v) {
        y[i][v] += c(i) * X[6 + k][v];
        w[i][v] += c(3 + i) * X[6 + k][v];
      }
#pragma unroll
    for (int v = 0; v < 3; ++v) out[(18 + k) * OS + v] = z[k][v];
  }
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      out[(3 + i) * OS + v] = y[i][v];
      out[(6 + i) * OS + v] = w[i][v];
    }
}

// Pass 2: X <- Fx X in place.
template <int PS>
ESKF_HD void fx3_apply_inplace(double (&X)[24][3], const d2* f2) {
  const double dt = f2[(FX3_DT / 2) * PS].x;
  double y[3][3], ya[3][3], yb[3][3];
  fx3_rows_h2<PS>(X, f2, y);  // reads X[19..21]: before rows 18:21 change
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) X[21 + i][v] = y[i][v];
  fx3_rows_h1<PS>(X, f2, dt, y);  // reads X[3..18]: before rows 3:9 and the notch chain change
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      X[18 + i][v] = y[i][v];
      X[i][v] = X[i][v] + dt * X[3 + i][v];
    }
  fx3_rows_ab<PS>(X, f2, ya, yb);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      X[3 + i][v] = ya[i][v];
      X[6 + i][v] = yb[i][v];
    }
#pragma unroll
  for (int v = 0; v < 3; ++v) {
    X[15][v] = X[15][v] + dt * X[16][v];
    X[16][v] = X[16][v] + dt * X[17][v];
  }
}

// Pass 2 fused with the transposed reload: X <- Fx T^T(:, tile), the operand T(3g+v, k) streamed from the rows 3g..3g+2 of
// the transposition buffer (row stride RS doubles) pair by pair and consumed column by column, so that the 36 fetches of
// the tile are spread over the 222 multiply-adds of the pass instead of preceding them as one burst (during which the FP64
// pipe of the sub-partition idles: all covariance warps of a CTA run the same phase at the same time).  X is write-only
// here.  Every accumulator sees the same operations in the same order as in fx3_apply_inplace after fx3_load_transposed:
// the results are bit-identical (tests/test_hostcheck.py replays both).
template <int PS, int RS>
ESKF_HD void fx3_apply_stream(double (&X)[24][3], const d2* f2, const double* rows) {
  const double dt = f2[(FX3_DT / 2) * PS].x;
  auto ld = [&](int j, double (&lo)[3], double (&hi)[3]) {  // T(3g+v, 2j), T(3g+v, 2j+1)
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      const d2 t = reinterpret_cast<const d2*>(rows + v * RS)[j];
      lo[v] = t.x;
      hi[v] = t.y;
    }
  };
  // multiply-adds of one column k of a three-row group: y[i][v] += c(o + i) x[v]
  auto col3 = [&](int r0, const Coefs<PS, 6>& c, int o, const double (&x)[3]) {
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int v = 0; v < 3; ++v) X[r0 + i][v] += c(o + i) * x[v];
  };
  double o0[3], o1[3], o2[3], o3[3], o4[3], o5[3], o16[3], o17[3], o18[3], o19[3], o22[3], o23[3];
  Coefs<PS, 6> h2a, h2b;
#if ESKF_OPT_ST2
  // The pass starts with the row groups that need the fewest operands -- rows 3:9 on columns 6, 7 want three fetches of the
  // tile -- and the other fetches of the head follow between the multiply-adds (as written before, six fetches of the tile,
  // 18 LDS.128, stood in front of the first multiply-add, in every covariance warp of the CTA at once).  Every accumulator
  // still sees the same operations in the same order.
  {
    double x6[3], x7[3];
    ld(1, o2, o3);
    ld(2, o4, o5);
    ld(3, x6, x7);
    Coefs<PS, 6> ab0, ab1, h1;
    ab0.load(f2, FX3_AB);
    ab1.load(f2, FX3_AB + 6);
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      X[3][v] = o3[v];
      X[4][v] = o4[v];
      X[5][v] = o5[v];
      X[6][v] = 0.0;
      X[7][v] = 0.0;
      X[8][v] = 0.0;
    }
    ld(8, o16, o17);
    ld(9, o18, o19);
    col3(3, ab0, 0, x6);
    col3(6, ab0, 3, x6);
    h1.load(f2, FX3_H1);
    ld(0, o0, o1);
    col3(3, ab1, 0, x7);
    col3(6, ab1, 3, x7);
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      X[18][v] = o16[v] + dt * o3[v];
      X[19][v] = o17[v] + dt * o4[v];
      X[20][v] = o18[v] + dt * o5[v];
      X[16][v] = o16[v] + dt * o17[v];
      X[17][v] = o17[v];
    }
    ld(11, o22, o23);
    col3(18, h1, 0, x6);
    col3(18, h1, 3, x7);
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      X[0][v] = o0[v] + dt * o3[v];
      X[1][v] = o1[v] + dt * o4[v];
      X[2][v] = o2[v] + dt * o5[v];
      X[21][v] = 0.0;
      X[22][v] = o22[v];
      X[23][v] = o23[v];
    }
  }
#else
  ld(1, o2, o3);
  ld(2, o4, o5);
  ld(8, o16, o17);
  ld(9, o18, o19);
  ld(11, o22, o23);
  ld(0, o0, o1);
#pragma unroll
  for (int v = 0; v < 3; ++v) {
    // rows 18:21 start from the mis-aligned identity block (quirk Q3) and dt v
    X[18][v] = o16[v] + dt * o3[v];
    X[19][v] = o17[v] + dt * o4[v];
    X[20][v] = o18[v] + dt * o5[v];
    // rows 21:24: Fx[22,22] = Fx[23,23] = 1
    X[21][v] = 0.0;
    X[22][v] = o22[v];
    X[23][v] = o23[v];
    // rows 0:3  p += dt v
    X[0][v] = o0[v] + dt * o3[v];
    X[1][v] = o1[v] + dt * o4[v];
    X[2][v] = o2[v] + dt * o5[v];
    // rows 3:6 start from v, rows 6:9 from zero
    X[3][v] = o3[v];
    X[4][v] = o4[v];
    X[5][v] = o5[v];
    X[6][v] = 0.0;
    X[7][v] = 0.0;
    X[8][v] = 0.0;
    // notch chain, rows 16 and 17
    X[16][v] = o16[v] + dt * o17[v];
    X[17][v] = o17[v];
  }
  {  // columns 6, 7: C1 (rows 18:21), A and B (rows 3:9)
    double x6[3], x7[3];
    ld(3, x6, x7);
    Coefs<PS, 6> h1, ab;
    h1.load(f2, FX3_H1);
    ab.load(f2, FX3_AB);
    col3(18, h1, 0, x6);
    col3(3, ab, 0, x6);
    col3(6, ab, 3, x6);
    ab.load(f2, FX3_AB + 6);
    col3(18, h1, 3, x7);
    col3(3, ab, 0, x7);
    col3(6, ab, 3, x7);
  }
#endif
  {  // columns 8, 9: C1 / C2, A and B; D on dof 1 (rows 21:24)
    double x8[3], x9[3];
    ld(4, x8, x9);
    Coefs<PS, 6> h1, ab;
    h1.load(f2, FX3_H1 + 6);
    ab.load(f2, FX3_AB + 12);
    h2a.load(f2, FX3_H2);
    col3(18, h1, 0, x8);
    col3(3, ab, 0, x8);
    col3(6, ab, 3, x8);
    col3(18, h1, 3, x9);
    col3(21, h2a, 0, x9);
#pragma unroll
    for (int v = 0; v < 3; ++v) X[9][v] = x9[v];
  }
  {  // columns 10, 11
    double x10[3], x11[3];
    ld(5, x10, x11);
    Coefs<PS, 6> h1;
    h1.load(f2, FX3_H1 + 12);
    h2b.load(f2, FX3_H2 + 6);
    col3(18, h1, 0, x10);
    col3(21, h2a, 3, x10);
    col3(18, h1, 3, x11);
    col3(21, h2b, 0, x11);
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      X[10][v] = x10[v];
      X[11][v] = x11[v];
    }
  }
  {  // columns 12, 13
    double x12[3], x13[3];
    ld(6, x12, x13);
    Coefs<PS, 6> h1;
    h1.load(f2, FX3_H1 + 18);
    col3(18, h1, 0, x12);
    col3(18, h1, 3, x13);
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      X[12][v] = x12[v];
      X[13][v] = x13[v];
    }
  }
  {  // columns 14, 15: last column of C2; D on the notch angle; row 15 of the notch chain
    double x14[3], x15[3];
    ld(7, x14, x15);
    Coefs<PS, 6> h1;
    h1.load(f2, FX3_H1 + 24);
    col3(18, h1, 0, x14);
    col3(21, h2b, 3, x15);
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      X[14][v] = x14[v];
      X[15][v] = x15[v] + dt * o16[v];
    }
  }
  {  // columns 19, 20, 21: E (quirk Q3)
    double x20[3], x21[3];
    ld(10, x20, x21);
    Coefs<PS, 6> h2c, h2d;
    h2c.load(f2, FX3_H2 + 12);
    h2d.load(f2, FX3_H2 + 18);
    col3(21, h2c, 0, o19);
    col3(21, h2c, 3, x20);
    col3(21, h2d, 0, x21);
  }
}

// this lane's share of the diagonal of Fi Q Fi^T: rows 3..14 get qd[r-3] (Fi[3:15,0:12] = I), row 17 gets
// qd[12] (Fi[17,12] = 1); qdv[v] belongs to row 3g+v.  qd(j) = diag(Q)[j].
template <typename QD>
ESKF_HD void fx3_noise_diag(int g, const QD& qd, double (&qdv)[3]) {
#pragma unroll
  for (int v = 0; v < 3; ++v) {
    const int r = 3 * g + v;
    qdv[v] = (r >= 3 && r < 15) ? qd(r - 3) : (r == 17) ? qd(12) : 0.0;
  }
}

// Fi Q Fi^T for the tile of lane group g (Filter.py:349).
// IQ = false compiles the IMU-noise part out (a caller that knows Q[0:6] = 0 for its filters).
template <int PS, bool IQ = true, typename QD>
ESKF_HD void fx3_process_noise(double (&X)[24][3], int g, const d2* f2, const double (&qdv)[3], const QD& qd, bool imu_q) {
  // diagonal entries P'(3g+v, 3g+v) = X[3g+v][v]: every index is a constant
#if ESKF_OPT_QP
  // (predicated adds: four predicates instead of two selects per addend)
#pragma unroll
  for (int j = 1; j < 5; ++j) {
    if (g == j) {
#pragma unroll
      for (int v = 0; v < 3; ++v) X[3 * j + v][v] += qdv[v];
    }
  }
  if (g == 5) X[17][2] += qdv[2];
#else
#pragma unroll
  for (int j = 1; j < 5; ++j)
#pragma unroll
    for (int v = 0; v < 3; ++v) X[3 * j + v][v] += (g == j) ? qdv[v] : 0.0;
  X[17][2] += (g == 5) ? qdv[2] : 0.0;
#endif
  if (IQ && imu_q && (g == 2 || g == 6 || g == 7)) {
    // n_om drives theta (I), p_C (Np) and theta_C (Nt): L Q_om L^T on rows/cols {6:9,18:21,21:24};
    // the diagonal of the theta block was added above.
    auto at = [&](int j) {
      const d2 p = f2[(j >> 1) * PS];
      return (j & 1) ? p.y : p.x;
    };
    double Lr[3][3];
#pragma unroll
    for (int v = 0; v < 3; ++v)
#pragma unroll
      for (int k = 0; k < 3; ++k)
        Lr[v][k] = (g == 2) ? ((k == v) ? 1.0 : 0.0) : (g == 6) ? at(FX3_NP + 3 * v + k) : at(FX3_NT + 3 * v + k);
#pragma unroll
    for (int cb = 0; cb < 3; ++cb) {
      const int c0 = (cb == 0) ? 6 : (cb == 1) ? 18 : 21;
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        double Lc[3];
#pragma unroll
        for (int k = 0; k < 3; ++k)
          Lc[k] = (cb == 0) ? ((k == j) ? 1.0 : 0.0) : (cb == 1) ? at(FX3_NP + 3 * j + k) : at(FX3_NT + 3 * j + k);
#pragma unroll
        for (int v = 0; v < 3; ++v) {
          double acc = 0.0;
#pragma unroll
          for (int k = 0; k < 3; ++k) acc += Lr[v][k] * qd(3 + k) * Lc[k];
          if (!(g == 2 && cb == 0)) X[c0 + j][v] += acc;
        }
      }
    }
  }
}

// ---- camera update on the register tile ------------------------------------------------------------------
// "u3 record": per-filter exchange area of the eight lanes (doubles).  Element j of the record of filter
// q (of QS filters interleaved pair-wise) lives at rec[((j >> 1) * QS) * 2 + (j & 1)], rec already offset
// by 2 * q: the same pair of all QS filters of a warp is one contiguous 16 * QS bytes.  The 24x7 matrices
// are stored TRANSPOSED (7 x 24: element (m, i) at 24 m + i) so that four consecutive rows of one column m
// are two 16-byte fetches; the passes below run column by column over blocks of four rows, twelve
// independent accumulators at a time.
constexpr int U3_S = 0;      // 7x7  S = H P H^T + R         (+1 pad)
constexpr int U3_SINV = 50;  // 7x7  inv(S)                  (+1 pad)
constexpr int U3_K = 100;    // 7x24 K^T
constexpr int U3_WH = 268;   // 7x24 W(:, h_m)^T,  W = (I - K H) P
constexpr int U3_HP = 436;   // 7x24 H P: rows h_m of the prior P (each lane files the entries of its own columns)
constexpr int U3_SIZE = 604;

// The passes over the 24x7 matrices are REAL loops over the measurement index m (a few hundred instructions
// executed seven times instead of several thousand executed once: the update runs once per camera frame and
// straight-line code of that size is instruction-fetch bound); everything indexed by m therefore comes from
// the record, never from a register array.
ESKF_HD int u3_hset(int m) { return (m < 6) ? 18 + m : 15; }

template <int QS>
ESKF_HD double& u3_at(double* rec, int j) {
  return rec[((j >> 1) * QS) * 2 + (j & 1)];
}
template <int QS>
ESKF_HD double u3_get(const double* rec, int j) {
  return rec[((j >> 1) * QS) * 2 + (j & 1)];
}
// four consecutive record elements starting at the even element j
template <int QS>
ESKF_HD void u3_get4(const double* rec, int j, double (&o)[4]) {
  const d2* r2 = reinterpret_cast<const d2*>(rec);
  const d2 a = r2[(j >> 1) * QS], b = r2[((j >> 1) + 1) * QS];
  o[0] = a.x;
  o[1] = a.y;
  o[2] = b.x;
  o[3] = b.y;
}

// owner of measurement row m: column h_m = ESKF_HSET(m) belongs to lane h_m / 3, tile column h_m % 3
// U0a: lanes 5..7 publish their columns of S (Filter.py:355); every lane files H P for its own columns.
//
// ORIENTATION.  The reference's covariance is symmetric only up to ITS rounding, and after an ill-conditioned update that
// is not small: 2.6e-11 relative at a point of the BASELINE tuning grid, where reading the other triangle moves the next
// update by 3e-8.  The tile is the transpose of the reference's matrix, X[k][v] = P(3g+v, k), whenever an update runs
// (eskf_kernel3.cuh keeps it that way: every propagation flips the orientation, and an odd number of them is followed by
// one explicit transposition).  With that orientation rows h of the tile are the reference's P H^T (the operand of the
// gain), W = (I - K H) X and X' = W (I - K H)^T + K R K^T are the transposes of the reference's products, and the one
// thing that must be turned around is S: the tile entry X[h_i][h_m] is P(h_m, h_i) = S(m, i).  The record keeps the tile's
// view (S^T); the inverse routines deliver inv(S): on the device the Gauss-Jordan elimination runs on the record and writes
// its result transposed (inv7_group3), on the host inv7 is given the transposed record.  (Inverting S^T and transposing is
// not the same rounding as inverting S: it yields a good LEFT inverse, K S = P H^T, which is what the first update with
// its prior >> R needs -- eliminating S itself was off by 3e-8 there.)
// (tests/test_hostcheck.py::test_lockstep_ill_conditioned_tuning: 1e-14 with, 3e-8 without.)
template <int QS>
ESKF_HD void upd3_publish_S(const double (&X)[24][3], int g, const double* rd, double* rec) {
#pragma unroll
  for (int m = 0; m < 7; ++m) {
    const int h = ESKF_HSET(m);
#if !ESKF_OPT_UPD  // (with ESKF_OPT_UPD the inverse reads S from the H P record: S^T(i, m) = H P(i, h_m) + [i == m] R_m)
    if (g == h / 3) {
#pragma unroll
      for (int i = 0; i < 7; ++i) u3_at<QS>(rec, U3_S + 7 * i + m) = X[ESKF_HSET(i)][h % 3] + ((i == m) ? rd[m] : 0.0);
    }
#endif
#pragma unroll
    for (int v = 0; v < 3; ++v) u3_at<QS>(rec, U3_HP + 24 * m + 3 * g + v) = X[h][v];
  }
}

// U1: gain rows 3g..3g+2  K = (P H^T) inv(S)  (Filter.py:357), published; delta = K res for the same rows.
template <int QS>
ESKF_HD void upd3_gain(int g, double* rec, const double* res, double (&K)[3][7], double (&dl)[3]) {
  // K(r, :) = sum_j P(r, h_j) inv(S)(j, :),  P(r, h_j) = P(h_j, r) = H P(j, r): everything comes from the record,
  // the tile is not touched.  Two sweeps over the rows of inv(S) (columns 0..3, then 4..6): twelve / nine
  // independent accumulators each.
#pragma unroll
  for (int v = 0; v < 3; ++v)
#pragma unroll
    for (int m = 0; m < 7; ++m) K[v][m] = 0.0;
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int m0 = half ? 4 : 0, m1 = half ? 7 : 4;
#pragma unroll
    for (int j = 0; j < 7; ++j) {
      double ph[3], si[4];
#pragma unroll
      for (int v = 0; v < 3; ++v) ph[v] = u3_get<QS>(rec, U3_HP + 24 * j + 3 * g + v);
#pragma unroll
      for (int m = m0; m < m1; ++m) si[m - m0] = u3_get<QS>(rec, U3_SINV + 7 * j + m);
#pragma unroll
      for (int v = 0; v < 3; ++v)
#pragma unroll
        for (int m = m0; m < m1; ++m) K[v][m] += ph[v] * si[m - m0];
    }
  }
#pragma unroll
  for (int v = 0; v < 3; ++v) {
    dl[v] = 0.0;
#pragma unroll
    for (int m = 0; m < 7; ++m) {
      dl[v] += K[v][m] * res[m];
      u3_at<QS>(rec, U3_K + 24 * m + 3 * g + v) = K[v][m];
    }
  }
}

// NIS r^T inv(S) r of the update (eskf_keep_consistency): the residual and the inverse upd3_gain used, from the record
template <int QS>
ESKF_HD double upd3_nis(const double* rec, const double* res) {
  double nis = 0.0;
#pragma unroll
  for (int j = 0; j < 7; ++j) {
    double t = 0.0;
#pragma unroll
    for (int m = 0; m < 7; ++m) t += u3_get<QS>(rec, U3_SINV + 7 * j + m) * res[m];
    nis += res[j] * t;
  }
  return nis;
}

// U2a: X <- (I - K H) X  (Joseph factor, Filter.py:384), then lanes 5..7 publish the columns h_m of W.
// The diagonal entries of I - K H are formed first, 1 - K[h_a][a], exactly as the reference's I - K @ H does:
// with a prior >> R they are O(1e-12) and everything they multiply is cancellation dominated, so the order
// of the roundings is kept (tests/test_conditioning.py).
template <int QS>
ESKF_HD void upd3_w_pass(double (&X)[24][3], int g, double* rec) {
  // rows outside H (0..14, 16, 17): column by column of K, four rows at a time, X[i][v] -= K(i, m) P(h_m, j_v)
#if ESKF_OPT_UPD
  // Software pipelined by hand: the fetches of a block are issued two blocks ahead of the multiply-adds that use them, and
  // those of the first blocks of column m + 1 at the end of column m.  (ptxas keeps the order of the fetches it is given: as
  // written below -- fetch, use, fetch, use through ONE scratch quad -- every 16-byte fetch exposed its full latency, 12
  // times per column: 667 cycles per column for 144 cycles of FP64 issue.)  Same operations in the same order per element.
  {
    double xh[3], ka[4], kb[4], kc[4];
    auto pre = [&](int m) {
#pragma unroll
      for (int v = 0; v < 3; ++v) xh[v] = u3_get<QS>(rec, U3_HP + 24 * m + 3 * g + v);
      u3_get4<QS>(rec, U3_K + 24 * m + 0, ka);
      u3_get4<QS>(rec, U3_K + 24 * m + 4, kb);
    };
    auto blk = [&](int ib, const double (&k)[4], const double (&x)[3]) {
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int v = 0; v < 3; ++v) X[ib + r][v] -= k[r] * x[v];
    };
    pre(0);
#pragma unroll 1
    for (int m = 0; m < 7; ++m) {
      const double x[3] = {xh[0], xh[1], xh[2]};
      u3_get4<QS>(rec, U3_K + 24 * m + 8, kc);
      blk(0, ka, x);
      u3_get4<QS>(rec, U3_K + 24 * m + 12, ka);  // rows 12..15 (15 is an H row)
      blk(4, kb, x);
      u3_get4<QS>(rec, U3_K + 24 * m + 16, kb);  // rows 16, 17 (18, 19 are H rows)
      blk(8, kc, x);
      const double k12[3] = {ka[0], ka[1], ka[2]}, k16[2] = {kb[0], kb[1]};
      pre(m < 6 ? m + 1 : 6);
#pragma unroll
      for (int v = 0; v < 3; ++v) {
        X[12][v] -= k12[0] * x[v];
        X[13][v] -= k12[1] * x[v];
        X[14][v] -= k12[2] * x[v];
        X[16][v] -= k16[0] * x[v];
        X[17][v] -= k16[1] * x[v];
      }
    }
  }
#else
#pragma unroll 1
  for (int m = 0; m < 7; ++m) {
    double xh[3];
#pragma unroll
    for (int v = 0; v < 3; ++v) xh[v] = u3_get<QS>(rec, U3_HP + 24 * m + 3 * g + v);
#pragma unroll
    for (int ib = 0; ib < 12; ib += 4) {
      double k[4];
      u3_get4<QS>(rec, U3_K + 24 * m + ib, k);
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int v = 0; v < 3; ++v) X[ib + r][v] -= k[r] * xh[v];
    }
    double k[4], k2[4];
    u3_get4<QS>(rec, U3_K + 24 * m + 12, k);   // rows 12..15 (15 is an H row)
    u3_get4<QS>(rec, U3_K + 24 * m + 16, k2);  // rows 16, 17 (18, 19 are H rows)
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      X[12][v] -= k[0] * xh[v];
      X[13][v] -= k[1] * xh[v];
      X[14][v] -= k[2] * xh[v];
      X[16][v] -= k2[0] * xh[v];
      X[17][v] -= k2[1] * xh[v];
    }
  }
#endif
  // the seven rows h_a themselves (they still hold the prior)
  double w[7][3];
#pragma unroll
  for (int a = 0; a < 7; ++a) {
    const int i = ESKF_HSET(a);
    double k[7];
#pragma unroll
    for (int m = 0; m < 7; ++m) k[m] = u3_get<QS>(rec, U3_K + 24 * m + i);
    const double cd = 1.0 - k[a];
#pragma unroll
    for (int v = 0; v < 3; ++v) w[a][v] = cd * X[i][v];
#pragma unroll
    for (int m = 0; m < 7; ++m) {
      if (m == a) continue;
#pragma unroll
      for (int v = 0; v < 3; ++v) w[a][v] -= k[m] * X[ESKF_HSET(m)][v];
    }
  }
#pragma unroll
  for (int a = 0; a < 7; ++a)
#pragma unroll
    for (int v = 0; v < 3; ++v) X[ESKF_HSET(a)][v] = w[a][v];
#pragma unroll
  for (int m = 0; m < 7; ++m) {
    const int h = ESKF_HSET(m);
    if (g == h / 3) {
      d2* r2 = reinterpret_cast<d2*>(rec);
#pragma unroll
      for (int i = 0; i < 24; i += 2) r2[((U3_WH + 24 * m + i) >> 1) * QS] = d2{X[i][h % 3], X[i + 1][h % 3]};
    }
  }
}

// U2b: X <- W (I - K H)^T + (K R) K^T for the tile columns j = 3g+v  (Filter.py:384):
//   W(:,j) (1 - K[j][a]) - sum_{m != a} W(:,h_m) K[j][m] + sum_m K(:,m) (R_m K[j][m])
// then the reset P <- G P G^T with G = I - [delta_theta / 2]x on 6:9 and 21:24 (Filter.py:386-390).
//   rd[m * RDS] = diag(R)[m]: read from memory inside the loop over m (a register array cannot be indexed by m)
//   dth[i * DS], dthc[i * DS]: the error-state rotations of the reset, read AFTER the loops (twelve registers less across them)
template <int QS, int RDS, int DS>
ESKF_HD void upd3_finish(double (&X)[24][3], int g, const double* rec, const double* rd, const double* dth,
                         const double* dthc) {
  // (1 - K[j][a]) for a column j = h_a measured directly, 1 otherwise: lanes 5 (column 15), 6 and 7
  double cdv[3];
#pragma unroll
  for (int v = 0; v < 3; ++v) {
    const int j = 3 * g + v;
    const int a = (j >= 18) ? j - 18 : 6;  // only used when j is in H
    const double k = u3_get<QS>(rec, U3_K + 24 * a + j);
    cdv[v] = (j >= 18 || j == 15) ? 1.0 - k : 1.0;
  }
#pragma unroll
  for (int i = 0; i < 24; ++i)
#pragma unroll
    for (int v = 0; v < 3; ++v) X[i][v] = cdv[v] * X[i][v];
#if ESKF_OPT_UPD && ESKF_OPT_FIN14
  {  // both sums as ONE rolled loop of fourteen columns (t < 7: - W(:,h_t) K[j][t] with the measured column masked;
     // t >= 7: + K(:,m) R_m K[j][m]): one loop body in the instruction cache and no drain / refill of the hand-made
     // pipeline between the two sweeps.  fma(w, -z, x) is the same rounding as x - w z: bit-identical to the two sweeps.
    double kv[3], rdm = 0.0, ba[4], bb[4], bc[4];
    auto pre = [&](int t) {
      const int m = t < 7 ? t : t - 7;
      const int base = t < 7 ? U3_WH : U3_K;
#pragma unroll
      for (int v = 0; v < 3; ++v) kv[v] = u3_get<QS>(rec, U3_K + 24 * m + 3 * g + v);
      rdm = rd[m * RDS];
      u3_get4<QS>(rec, base + 24 * m + 0, ba);
      u3_get4<QS>(rec, base + 24 * m + 4, bb);
    };
    auto blk = [&](int ib, const double (&w)[4], const double (&z)[3]) {
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int v = 0; v < 3; ++v) X[ib + r][v] += w[r] * z[v];
    };
    pre(0);
#pragma unroll 1
    for (int t = 0; t < 14; ++t) {
      const int m = t < 7 ? t : t - 7;
      const int base = t < 7 ? U3_WH : U3_K;
      double z[3];
#pragma unroll
      for (int v = 0; v < 3; ++v) z[v] = (t < 7) ? ((u3_hset(m) == 3 * g + v) ? -0.0 : -kv[v]) : rdm * kv[v];
      u3_get4<QS>(rec, base + 24 * m + 8, bc);
      blk(0, ba, z);
      u3_get4<QS>(rec, base + 24 * m + 12, ba);
      blk(4, bb, z);
      u3_get4<QS>(rec, base + 24 * m + 16, bb);
      blk(8, bc, z);
      u3_get4<QS>(rec, base + 24 * m + 20, bc);
      blk(12, ba, z);
      const double b16[4] = {bb[0], bb[1], bb[2], bb[3]}, b20[4] = {bc[0], bc[1], bc[2], bc[3]};
      pre(t < 13 ? t + 1 : 13);
      blk(16, b16, z);
      blk(20, b20, z);
    }
  }
#elif ESKF_OPT_UPD
  {  // software pipelined by hand (see upd3_w_pass): fetches two blocks ahead, the next column's first blocks at the end
    double kv[3], rdm, ba[4], bb[4], bc[4];
    auto blk = [&](int ib, const double (&w)[4], const double (&z)[3], bool sub) {
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int v = 0; v < 3; ++v) {
          if (sub)
            X[ib + r][v] -= w[r] * z[v];
          else
            X[ib + r][v] += w[r] * z[v];
        }
    };
    // pass over m of ONE of the two sums: base = U3_WH (sub) or U3_K (add)
    auto sweep = [&](int base, bool sub) {
      auto pre = [&](int m) {
#pragma unroll
        for (int v = 0; v < 3; ++v) kv[v] = u3_get<QS>(rec, U3_K + 24 * m + 3 * g + v);
        if (!sub) rdm = rd[m * RDS];
        u3_get4<QS>(rec, base + 24 * m + 0, ba);
        u3_get4<QS>(rec, base + 24 * m + 4, bb);
      };
      pre(0);
#pragma unroll 1
      for (int m = 0; m < 7; ++m) {
        double z[3];
#pragma unroll
        for (int v = 0; v < 3; ++v) z[v] = sub ? ((u3_hset(m) == 3 * g + v) ? 0.0 : kv[v]) : rdm * kv[v];
        u3_get4<QS>(rec, base + 24 * m + 8, bc);
        blk(0, ba, z, sub);
        u3_get4<QS>(rec, base + 24 * m + 12, ba);
        blk(4, bb, z, sub);
        u3_get4<QS>(rec, base + 24 * m + 16, bb);
        blk(8, bc, z, sub);
        u3_get4<QS>(rec, base + 24 * m + 20, bc);
        blk(12, ba, z, sub);
        const double b16[4] = {bb[0], bb[1], bb[2], bb[3]}, b20[4] = {bc[0], bc[1], bc[2], bc[3]};
        pre(m < 6 ? m + 1 : 6);
        blk(16, b16, z, sub);
        blk(20, b20, z, sub);
      }
    };
    sweep(U3_WH, true);
    sweep(U3_K, false);
  }
#else
#pragma unroll 1
  for (int m = 0; m < 7; ++m) {
    double kz[3];
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      const double k = u3_get<QS>(rec, U3_K + 24 * m + 3 * g + v);
      kz[v] = (u3_hset(m) == 3 * g + v) ? 0.0 : k;
    }
#pragma unroll
    for (int ib = 0; ib < 24; ib += 4) {
      double wh[4];
      u3_get4<QS>(rec, U3_WH + 24 * m + ib, wh);
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int v = 0; v < 3; ++v) X[ib + r][v] -= wh[r] * kz[v];
    }
  }
#pragma unroll 1
  for (int m = 0; m < 7; ++m) {
    double kjr[3];
#pragma unroll
    for (int v = 0; v < 3; ++v) kjr[v] = rd[m * RDS] * u3_get<QS>(rec, U3_K + 24 * m + 3 * g + v);
#pragma unroll
    for (int ib = 0; ib < 24; ib += 4) {
      double k[4];
      u3_get4<QS>(rec, U3_K + 24 * m + ib, k);
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int v = 0; v < 3; ++v) X[ib + r][v] += k[r] * kjr[v];
    }
  }
#endif
#if ESKF_OPT_UPD && defined(__CUDA_ARCH__)
  asm volatile("" ::: "memory");  // the reset operands are fetched here, not before the loops
#endif
  const double gt[3] = {0.5 * dth[0], 0.5 * dth[DS], 0.5 * dth[2 * DS]};
  const double gc[3] = {0.5 * dthc[0], 0.5 * dthc[DS], 0.5 * dthc[2 * DS]};
  // G P: rows 6:9 and 21:24 of every column;  (I - [g]x) = [[1, g2, -g1], [-g2, 1, g0], [g1, -g0, 1]]
#pragma unroll
  for (int v = 0; v < 3; ++v) {
    const double a0 = X[6][v], a1 = X[7][v], a2 = X[8][v];
    X[6][v] = a0 + gt[2] * a1 - gt[1] * a2;
    X[7][v] = -gt[2] * a0 + a1 + gt[0] * a2;
    X[8][v] = gt[1] * a0 - gt[0] * a1 + a2;
    const double b0 = X[21][v], b1 = X[22][v], b2 = X[23][v];
    X[21][v] = b0 + gc[2] * b1 - gc[1] * b2;
    X[22][v] = -gc[2] * b0 + b1 + gc[0] * b2;
    X[23][v] = gc[1] * b0 - gc[0] * b1 + b2;
  }
  // (.) G^T: the three columns of lane 2 (6:9) and lane 7 (21:24)
  if (g == 2 || g == 7) {
    const double h0 = (g == 2) ? gt[0] : gc[0], h1 = (g == 2) ? gt[1] : gc[1], h2 = (g == 2) ? gt[2] : gc[2];
#pragma unroll
    for (int i = 0; i < 24; ++i) {
      const double a0 = X[i][0], a1 = X[i][1], a2 = X[i][2];
      X[i][0] = a0 + h2 * a1 - h1 * a2;
      X[i][1] = -h2 * a0 + a1 + h0 * a2;
      X[i][2] = h1 * a0 - h0 * a1 + a2;
    }
  }
}

}  // namespace eskf
