// The persistent VI-ESKF kernel for sm_100a (one template instance per CTA shape).
//
// One CTA owns F filters for a whole call (a whole trajectory in eskf_run):
//   * warp 0 is the SCALAR role, one lane per filter: nominal state, probe
//     kinematics and the Jacobian blocks (Filter._predict_nominal /
//     _predict_error, Filter.py:232-342) live in its registers;
//   * the other warps are the COVARIANCE role, eight lanes per filter, lane g
//     owning the 3 columns (column pass) / 3 rows (row pass) of state group g
//     of the 24x24 covariance, which stays in shared memory for the whole
//     trajectory (Filter._predict_error_covariance, Filter.py:344-349, and the
//     gain / Joseph / reset algebra of Filter.update, Filter.py:355-390).
// The nominal propagation never reads P, so the scalar role runs one step
// ahead of the covariance role through a double-buffered Jacobian record; the
// two meet at one __syncthreads per step and at the camera update.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/eskf.h"
#include "eskf_math.cuh"
#include "eskf_rng.cuh"

namespace eskf {

constexpr int P_RS = 25;             // padded row stride of P in shared memory: conflict free for the
constexpr int P_STRIDE = 24 * P_RS;  // column pass AND the row pass (see DESIGN.md, "bank layout")
constexpr int UP_OK2 = UP_SIZE;      // combined "apply this update" flag (written by the covariance role)
constexpr int SCR_STRIDE = UP_SIZE + 2;  // union {2 x fx record, update record}; even => 16 B aligned rows
static_assert(2 * FX_STRIDE <= SCR_STRIDE, "fx double buffer must fit the scratch union");
constexpr int SM_PER_FILTER = P_STRIDE + SCR_STRIDE + PAR_STRIDE;  // doubles of shared memory per filter

struct KArgs {
  double* x;
  double* P;
  double* u;
  double* Ro;
  int32_t* status;
  const double* par;  // [N,PAR_STRIDE]
  int64_t N;
  Model model;
  int64_t T, E;
  int n_traj;
  int64_t filters_per_traj;
  int64_t filter_id0;
  const double* dt;
  const double* om_acc;
  int stream_per_filter;
  const int32_t* n_prop;
  const double* cam;
  const double* notch;
  int meas_per_filter;
  int do_update;
  const double* cam_ref;
  const double* imu_ref;
  double gt_dofs[6];
  double* K_out;
  double* stats_out;
  double* stats_sum;
  double* trace;  // [N,T,26] or nullptr
  uint64_t seed;
  double imu_noise[6];
  double cam_noise[7];
  int noise_on;
  int noise_free0;
  int noise_mod;  // > 0: noise id = global id % noise_mod
  // pre- / post-pass mode of eskf_run (eskf_kernel3 only; see eskf_pp.cuh): per-filter streams prepared by a pre-pass
  // kernel and per-epoch snapshots for the statistics post-pass, so that neither the Monte-Carlo generator nor the
  // Euler angles of Filter.calculate_update_mse run inside the persistent kernel
  const double* imu_pf;   // [T][N][6]  noisy IMU samples per filter, or nullptr
  const double* meas_pf;  // [E][N][8]  noisy camera measurement (pos 3, quat 4, notch) per filter, or nullptr
  double* snap;           // [E][N][14] v(3) q(4) p_cam(3) q_cam(4) after every update, or nullptr
  double* fx_dump;        // [N][FX3_SIZE] Jacobian record of the filter's LAST executed IMU step of the launch (eskf_get_jacobians), or nullptr
  // (members added below this line keep the parameter offsets of the ones above: the production instantiation does not move)
  double* cons;           // [E][CONS_SIZE][N] consistency record of every update (eskf_keep_consistency, eskf_math.cuh), or nullptr
  // a segment of the trajectory (eskf_run_epochs; eskf_kernel3, MODE bit 2 only): epochs [e_base, e_base + E) of streams whose
  // per-epoch rows are E_all long, trajectory t starting at step k_base[t]; the per-filter accumulators the statistics row
  // cannot hold come from carry_in and go to carry_out ([N][ESKF_NCARRY], either may be nullptr)
  const int64_t* k_base;
  int64_t e_base, E_all;
  const double* carry_in;
  double* carry_out;
  // simulated frame loss (eskf_set_meas_dropout; eskf_kernel3 export instantiations only): [n_traj][E_all] (E_all = E outside a
  // segment) drop probabilities of every epoch, indexed like the per-epoch streams, or nullptr
  const double* drop_p;
};

// one FilterTraj row's worth of nominal state in the layout of x (include/eskf.h)
__device__ __forceinline__ void trace_row(double* r, const Nominal& s) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    r[i] = s.p[i];
    r[3 + i] = s.v[i];
    r[16 + i] = s.notch[i];
    r[19 + i] = s.pc[i];
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    r[6 + i] = s.q[i];
    r[22 + i] = s.qc[i];
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) r[10 + i] = s.dofs[i];
}

__device__ __forceinline__ void euler_xyz_deg(const double* q, double* e) {
  // Rotation.as_euler("xyz", degrees=True) away from gimbal lock (Quaternion.py:121-123)
  double R[9];
  quat_to_rot(q, R);
  const double r2d = 57.295779513082320876798154814105;
  e[0] = atan2(R[7], R[8]) * r2d;
  e[1] = -asin(fmin(1.0, fmax(-1.0, R[6]))) * r2d;
  e[2] = atan2(R[3], R[0]) * r2d;
}

// inv(S), S = H P H^T + R (Filter.py:355-357), by the eight lanes of a filter group: lane c < 7 owns
// column c of [S | I].  LU with partial pivoting + back substitution, the same operations in the same
// order as eskf::inv7 (the host-checkable restatement of np.linalg.inv -> LAPACK gesv); multipliers
// and U entries travel by width-8 shuffles.  Returns false for an exactly singular / non-finite S.
template <int RS>
__device__ __forceinline__ bool inv7_group(const double* Pf, const double* rd, int g, double* up) {
  const unsigned FULL = 0xffffffffu;
  const int c = (g < 7) ? g : 6;
  double a[7], b[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) {
    a[i] = Pf[ESKF_HSET(i) * RS + ESKF_HSET(c)] + ((i == c) ? rd[c] : 0.0);
    b[i] = (i == c) ? 1.0 : 0.0;
  }
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    int piv = k;
    double best = fabs(a[k]);
#pragma unroll
    for (int i = k + 1; i < 7; ++i) {
      const double v = fabs(a[i]);
      if (v > best) {
        best = v;
        piv = i;
      }
    }
    piv = __shfl_sync(FULL, piv, k, 8);
    best = __shfl_sync(FULL, best, k, 8);
    ok = ok && (best != 0.0);
#pragma unroll
    for (int i = k + 1; i < 7; ++i) {
      if (piv == i) {
        double t = a[k];
        a[k] = a[i];
        a[i] = t;
        t = b[k];
        b[k] = b[i];
        b[i] = t;
      }
    }
    const double rp = 1.0 / a[k];
#pragma unroll
    for (int i = k + 1; i < 7; ++i) {
      const double l = __shfl_sync(FULL, a[i] * rp, k, 8);
      a[i] -= l * a[k];
      b[i] -= l * b[k];
    }
  }
#pragma unroll
  for (int i = 6; i >= 0; --i) {
    double v = b[i];
#pragma unroll
    for (int k = i + 1; k < 7; ++k) {
      const double uik = __shfl_sync(FULL, a[i], k, 8);
      v -= uik * b[k];
    }
    const double uii = __shfl_sync(FULL, a[i], i, 8);
    b[i] = v * (1.0 / uii);
  }
  double chk = 0.0;
#pragma unroll
  for (int i = 0; i < 7; ++i) chk += b[i] * 0.0;  // NaN / inf detector
  ok = ok && (chk == 0.0);
  if (g < 7) {
#pragma unroll
    for (int i = 0; i < 7; ++i) up[UP_SINV + 7 * i + c] = b[i];
  }
  const unsigned bal = __ballot_sync(FULL, ok);
  const unsigned lane = threadIdx.x & 31u;
  return ((bal >> (lane & 24u)) & 0xffu) == 0xffu;
}

template <int F>
__global__ void __launch_bounds__(32 + 8 * F, 1) eskf_kernel(const __grid_constant__ KArgs a) {
  extern __shared__ __align__(16) double smem[];
  double* sP = smem;                     // [F][P_STRIDE]
  double* sScr = sP + F * P_STRIDE;      // [F][SCR_STRIDE]
  double* sPar = sScr + F * SCR_STRIDE;  // [F][PAR_STRIDE]

  const int tid = threadIdx.x;
  constexpr int nthr = 32 + 8 * F;
  const int64_t f0 = (int64_t)blockIdx.x * F;  // first local filter of this CTA
  const int nf = (int)((a.N - f0) < F ? (a.N - f0) : F);

  // ---- load P and the parameter rows (coalesced) ----
  for (int idx = tid; idx < F * 576; idx += nthr) {
    const int f = idx / 576, r = idx - f * 576;
    const int i = r / 24, j = r - i * 24;
    sP[f * P_STRIDE + i * P_RS + j] = (f < nf) ? a.P[(f0 + f) * 576 + r] : ((i == j) ? 1.0 : 0.0);
  }
  for (int idx = tid; idx < F * PAR_STRIDE; idx += nthr) {
    const int f = idx / PAR_STRIDE, r = idx - f * PAR_STRIDE;
    const int64_t row = (f < nf) ? (f0 + f) : f0;
    sPar[idx] = (r < PAR_SIZE) ? a.par[row * PAR_STRIDE + r] : 0.0;
  }

  const bool is_scalar = tid < 32;
  const bool s_active = is_scalar && tid < nf;
  const int ct = tid - 32;
  const int cf = ct >> 3;  // filter of this covariance lane (padded filters run on an identity P, never stored)
  const int cg = ct & 7;   // state group owned
  // the eight lanes of a filter group always take the same branches: group-level barriers use this mask
  const unsigned gmask = 0xffu << (tid & 24);

  // trajectory of this CTA (all filters of a CTA share it: host guarantees filters_per_traj % F == 0)
  const int64_t gid0 = a.filter_id0 + f0;
  const int64_t traj = (a.n_traj > 1) ? (gid0 / a.filters_per_traj) : 0;
  const int32_t* n_prop = a.n_prop ? a.n_prop + traj * a.E : nullptr;
  const double* dtp = a.dt ? a.dt + traj * a.T : nullptr;

  // ---- scalar role state ----
  Nominal s;
  ProbeKin pk;
  ProbeTrig ptr;
  bool after_update = true;  // R_WB must be recomputed from q (R_old may be stale, quirk Q8)
  int32_t st = 0;
  double sig_om[3] = {0, 0, 0};
  double mse_last = 0.0, mse_sum = 0.0, n_upd = 0.0;
  const double* oap = nullptr;
  const int64_t gid = a.noise_mod > 0 ? (gid0 + tid) % a.noise_mod : gid0 + tid;  // id the noise is keyed by
  bool noisy = false;
  if (s_active) {
    const double* xg = a.x + (f0 + tid) * NX;
    const double* ug = a.u + (f0 + tid) * 6;
    const double* rg = a.Ro + (f0 + tid) * 9;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      s.p[i] = xg[i];
      s.v[i] = xg[3 + i];
      s.notch[i] = xg[16 + i];
      s.pc[i] = xg[19 + i];
      s.om_old[i] = ug[i];
      s.acc_old[i] = ug[3 + i];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      s.q[i] = xg[6 + i];
      s.qc[i] = xg[22 + i];
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) s.dofs[i] = xg[10 + i];
#pragma unroll
    for (int i = 0; i < 9; ++i) s.R_old[i] = rg[i];
    st = a.status[f0 + tid];
    probe_eval(a.model, s.dofs, s.notch, pk, ptr);
    const int64_t row = f0 + tid;
#pragma unroll
    for (int i = 0; i < 3; ++i) sig_om[i] = a.par[row * PAR_STRIDE + PAR_SIGOM + i];
    oap = a.om_acc ? (a.stream_per_filter ? a.om_acc + (f0 + tid) * a.T * 6 : a.om_acc + traj * a.T * 6) : nullptr;
    noisy = a.noise_on && !(a.noise_free0 && gid == 0);
  }
  __syncthreads();

  double* Pf = sP + cf * P_STRIDE;
  double* scr_c = sScr + cf * SCR_STRIDE;
  const double* par_c = sPar + cf * PAR_STRIDE;
  bool imu_q = false;
  if (!is_scalar) {
    imu_q = (par_c[PAR_QD + 3] != 0.0) || (par_c[PAR_QD + 4] != 0.0) || (par_c[PAR_QD + 5] != 0.0);
  } else if (s_active) {
    const double* par_s = sPar + tid * PAR_STRIDE;
    imu_q = (par_s[PAR_QD + 3] != 0.0) || (par_s[PAR_QD + 4] != 0.0) || (par_s[PAR_QD + 5] != 0.0);
  }

  int64_t k = 0;  // step index within the trajectory
  for (int64_t e = 0; e < a.E; ++e) {
    const int n = n_prop ? n_prop[e] : (int)a.T;
    // ---- IMU propagation: scalar role one step ahead of the covariance role ----
    for (int it = 0; it <= n; ++it) {
      if (is_scalar) {
        if (s_active && it < n) {
          const int64_t kk = k + it;
          const double dt = dtp[kk];
          double om[3], acc[3];
#pragma unroll
          for (int i = 0; i < 3; ++i) {
            om[i] = oap[kk * 6 + i];
            acc[i] = oap[kk * 6 + 3 + i];
          }
          if (noisy) {
            double z[8];
            normal8(a.seed, (uint64_t)gid, (uint64_t)kk, RNG_KIND_IMU, z);
#pragma unroll
            for (int i = 0; i < 3; ++i) {
              om[i] += a.imu_noise[i] * z[i];
              acc[i] += a.imu_noise[3 + i] * z[3 + i];
            }
          }
          double Rq[9];
          if (after_update) {
            quat_to_rot(s.q, Rq);
          } else {
#pragma unroll
            for (int i = 0; i < 9; ++i) Rq[i] = s.R_old[i];
          }
          after_update = false;
#ifndef ESKF_EXP_NO_SCALAR  // (profiling experiment switch: time the covariance role alone)
          propagate_scalar(a.model, s, pk, ptr, Rq, dt, om, acc, sig_om, imu_q,
                           sScr + tid * SCR_STRIDE + (it & 1) * FX_STRIDE);
#endif
          if (a.trace) trace_row(a.trace + ((f0 + tid) * a.T + kk) * NX, s);
        }
      } else if (it >= 1) {
#ifndef ESKF_EXP_NO_COV  // (profiling experiment switch: time the scalar role alone)
        const double* fx = scr_c + ((it - 1) & 1) * FX_STRIDE;
        fx_apply3<P_RS, 1>(Pf + 3 * cg, fx);  // T = Fx P      (columns 3g..3g+2)
        __syncwarp(gmask);
        fx_apply3<1, P_RS>(Pf + 3 * cg * P_RS, fx);  // P' = T Fx^T   (rows 3g..3g+2)
        add_process_noise3<1, P_RS>(Pf + 3 * cg * P_RS, 3 * cg, fx, par_c + PAR_QD, imu_q);
        __syncwarp(gmask);
#endif
      }
      __syncthreads();
    }
    k += n;

    if (!a.do_update) continue;
    // ---- camera update (Filter.update, Filter.py:351-395) ----
    // phase U0: scalar role -> residual; covariance role -> inv(S)
    bool inv_ok = false;
    if (is_scalar) {
      if (tid < F) {
        double* up = sScr + tid * SCR_STRIDE;
        bool ok = false;
        if (s_active) {
          const int64_t mrow = a.meas_per_filter ? (f0 + tid) : (traj * a.E + e);
          double cam[7];
#pragma unroll
          for (int i = 0; i < 7; ++i) cam[i] = a.cam[mrow * 7 + i];
          double notch = a.notch[mrow];
          if (noisy) {
            double z[8];
            normal8(a.seed, (uint64_t)gid, (uint64_t)e, RNG_KIND_CAM, z);
            double dth[3];
#pragma unroll
            for (int i = 0; i < 3; ++i) {
              cam[i] += a.cam_noise[i] * z[i];
              dth[i] = a.cam_noise[3 + i] * z[3 + i];
            }
            // orientation noise: small body rotation of the measured quaternion (its norm is kept)
            double dq[4], qn[4];
            quat_about_axis(sqrt(dth[0] * dth[0] + dth[1] * dth[1] + dth[2] * dth[2]), dth, dq);
            const double nq = sqrt(cam[3] * cam[3] + cam[4] * cam[4] + cam[5] * cam[5] + cam[6] * cam[6]);
            quat_mul(cam + 3, dq, qn);
#pragma unroll
            for (int i = 0; i < 4; ++i) cam[3 + i] = qn[i] * nq;
            notch += a.cam_noise[6] * z[6];
          }
          ok = update_residual(s, cam, cam + 3, notch, up + UP_RES);
          if (!ok) st |= ESKF_STATUS_ASIN_DOMAIN;
        }
        up[UP_OK] = ok ? 1.0 : 0.0;
      }
    } else {
      inv_ok = inv7_group<P_RS>(Pf, par_c + PAR_RD, cg, scr_c);
    }
    __syncthreads();
    // phase U1: gain rows, delta
    bool upd_c = false;
    if (!is_scalar) {
      upd_c = inv_ok && (scr_c[UP_OK] != 0.0);
      if (upd_c) gain_rows3<P_RS>(Pf, 3 * cg, scr_c);
      if (cg == 0) scr_c[UP_OK2] = upd_c ? 1.0 : 0.0;
    }
    __syncthreads();
    // phase U2: scalar role injects the error state; covariance role does Joseph + reset
    if (is_scalar) {
      if (s_active) {
        const double* up = sScr + tid * SCR_STRIDE;
        if (up[UP_OK2] != 0.0) {
          double d[24];
#pragma unroll
          for (int i = 0; i < 24; ++i) d[i] = up[UP_DELTA + i];
          inject_error(a.model, s, d);
          probe_update(a.model, s.dofs, s.notch, pk, ptr);
          after_update = true;
          n_upd += 1.0;
          if (a.trace && k > 0) trace_row(a.trace + ((f0 + tid) * a.T + k - 1) * NX, s);  // FilterTraj.append_updated_states
        } else {
          st |= ESKF_STATUS_UPDATE_SKIPPED;
        }
        if (a.cam_ref && a.imu_ref) {  // Filter.calculate_update_mse (Filter.py:397-418)
          const double* cr = a.cam_ref + (traj * a.E + e) * 6;
          const double* ir = a.imu_ref + (traj * a.E + e) * 6;
          double ec[3], ei[3], acc = 0.0;
          euler_xyz_deg(s.qc, ec);
          euler_xyz_deg(s.q, ei);
#pragma unroll
          for (int i = 0; i < 3; ++i) {
            const double d0 = cr[i] - s.pc[i], d1 = cr[3 + i] - ec[i];
            const double d2 = s.v[i] - ir[i], d3 = ei[i] - ir[3 + i];
            acc += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
          }
          mse_last = acc / 12.0;
          mse_sum += mse_last;
        }
      }
    } else if (upd_c) {
      if (a.K_out && cf < nf) {
#pragma unroll
        for (int v = 0; v < 3; ++v) {
          const int r = 3 * cg + v;
#pragma unroll
          for (int m = 0; m < 7; ++m)
            a.K_out[((f0 + cf) * 24 + r) * 7 + m] = (ESKF_HSET(m) == r) ? scr_c[UP_KD + m] : scr_c[UP_KZ + 7 * r + m];
        }
      }
      joseph_apply3<P_RS, 1>(Pf + 3 * cg, scr_c);  // (I-KH) P
      __syncwarp(gmask);
      joseph_rows_finish3<P_RS>(Pf + 3 * cg * P_RS, 3 * cg, scr_c, par_c + PAR_RD);  // (.)(I-KH)^T + K R K^T, reset
      __syncwarp(gmask);
    }
    __syncthreads();  // the update record shares storage with the fx buffers
  }

  // ---- write back ----
  for (int idx = tid; idx < nf * 576; idx += nthr) {
    const int f = idx / 576, r = idx - f * 576;
    const int i = r / 24, j = r - i * 24;
    a.P[(f0 + f) * 576 + r] = sP[f * P_STRIDE + i * P_RS + j];
  }
  if (s_active) {
    double* xg = a.x + (f0 + tid) * NX;
    double* ug = a.u + (f0 + tid) * 6;
    double* rg = a.Ro + (f0 + tid) * 9;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      xg[i] = s.p[i];
      xg[3 + i] = s.v[i];
      xg[16 + i] = s.notch[i];
      xg[19 + i] = s.pc[i];
      ug[i] = s.om_old[i];
      ug[3 + i] = s.acc_old[i];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      xg[6 + i] = s.q[i];
      xg[22 + i] = s.qc[i];
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) xg[10 + i] = s.dofs[i];
#pragma unroll
    for (int i = 0; i < 9; ++i) rg[i] = s.R_old[i];
    a.status[f0 + tid] = st;
  }
  if ((a.stats_out || a.stats_sum) && is_scalar) {
    double row[ESKF_NSTAT];
#pragma unroll
    for (int i = 0; i < ESKF_NSTAT; ++i) row[i] = 0.0;
    if (s_active) {
      double acc = 0.0;
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        const double d = s.dofs[i] - a.gt_dofs[i];
        row[i] = d * d;
        acc += d * d;
      }
      row[6] = acc / 6.0;  // Filter.calculate_dof_metric (Filter.py:452-455)
      row[7] = mse_last;
      row[8] = mse_sum;
      row[9] = n_upd;
      row[10] = (double)st;
      row[11] = 1.0;  // filter count
      if (a.stats_out) {
#pragma unroll
        for (int i = 0; i < ESKF_NSTAT; ++i) a.stats_out[(f0 + tid) * ESKF_NSTAT + i] = row[i];
      }
    }
    if (a.stats_sum) {
      // warp tree reduction, then one atomic per CTA and statistic
#pragma unroll
      for (int i = 0; i < ESKF_NSTAT; ++i) {
        double v = row[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (tid == 0) atomicAdd(a.stats_sum + i, v);
      }
    }
  }
}

// host-side launcher, one per instantiated CTA shape (defined in eskf_launch.cu)
template <int F>
cudaError_t launch_eskf_kernel(const KArgs& a, cudaStream_t stream);

}  // namespace eskf
