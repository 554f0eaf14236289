// C ABI of the B200 batched VI-ESKF engine (see include/eskf.h) and its small utility kernels.
// The persistent kernel itself lives in eskf_kernel.cuh and is instantiated per CTA shape in
// eskf_launch.cu.
#include <nvtx3/nvToolsExt.h>  // header-only NVTX v3: ranges cost nothing unless a profiler is attached (SURVEY section 5)
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "eskf_kernel3.cuh"

using namespace eskf;

namespace eskf {
#define ESKF_DECL(F) template <> cudaError_t launch_eskf_kernel<F>(const KArgs& a, cudaStream_t stream);
ESKF_DECL(4) ESKF_DECL(28)
#undef ESKF_DECL
#define ESKF_DECL3(F) template <> cudaError_t launch_eskf_kernel3<F>(const KArgs& a, cudaStream_t stream);
ESKF_DECL3(4) ESKF_DECL3(8) ESKF_DECL3(16) ESKF_DECL3(28)
#undef ESKF_DECL3
}  // namespace eskf

namespace {

// ---- small utility kernels ----
__global__ void bcast_rows_kernel(double* dst, const double* src, int64_t n, int w) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * w) return;
  dst[i] = src[i % w];
}
__global__ void rot_from_state_kernel(double* Ro, const double* x, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double R[9];
  quat_to_rot(x + i * NX + 6, R);
  for (int j = 0; j < 9; ++j) Ro[i * 9 + j] = R[j];
}
__global__ void fill_par_kernel(double* par, const double* q, int64_t nq, const double* r, int64_t nr, const double* s,
                                int64_t ns, int64_t rows) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows) return;
  double* p = par + i * PAR_STRIDE;
  if (q)
    for (int j = 0; j < 13; ++j) p[PAR_QD + j] = q[(nq == 1 ? 0 : i) * 13 + j];
  if (r)
    for (int j = 0; j < 7; ++j) p[PAR_RD + j] = r[(nr == 1 ? 0 : i) * 7 + j];
  if (s)
    for (int j = 0; j < 3; ++j) p[PAR_SIGOM + j] = s[(ns == 1 ? 0 : i) * 3 + j];
  p[PAR_SIZE] = 0.0;
}

// FP64 FMA throughput probe: ILP independent DFMA chains per thread, nothing else in the loop.
// Used by bench.py to measure the roofline denominator (MEASURED_PEAKS.json has no FP64 figure).
template <int ILP>
__global__ void dfma_peak_kernel(double* out, int iters, double a, double b) {
  double acc[ILP];
#pragma unroll
  for (int i = 0; i < ILP; ++i) acc[i] = (double)(threadIdx.x + i);
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < ILP; ++i) acc[i] = fma(acc[i], a, b);
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < ILP; ++i) s += acc[i];
  if (s == 123.456) out[0] = s;  // keeps the chain alive without a store in the common case
}

// eskf_noise_dump: the standard normals of (filter, step, kind), exactly as the persistent kernels draw them; for
// RNG_KIND_DROP the dropout uniform of (filter, epoch) in z[0] and zeros; for RNG_KIND_OUTLIER the outlier uniform in z[0]
// and the seven offset normals in z[1..7]
__global__ void noise_dump_kernel(double* out, uint64_t seed, int64_t filter_id0, int64_t n_filters, int64_t step0, int64_t n_steps,
                                  uint32_t kind) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_filters * n_steps) return;
  const int64_t f = i / n_steps, k = i - f * n_steps;
  double z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (kind == RNG_KIND_DROP) {
    z[0] = drop_uniform(seed, (uint64_t)(filter_id0 + f), (uint64_t)(step0 + k));
  } else if (kind == RNG_KIND_OUTLIER) {
    double w[8];
    normal8(seed, (uint64_t)(filter_id0 + f), (uint64_t)(step0 + k), kind, w);
    z[0] = outlier_uniform(seed, (uint64_t)(filter_id0 + f), (uint64_t)(step0 + k));
    for (int j = 0; j < 7; ++j) z[1 + j] = w[j];
  } else {
    normal8(seed, (uint64_t)(filter_id0 + f), (uint64_t)(step0 + k), kind, z);
  }
  for (int j = 0; j < 8; ++j) out[i * 8 + j] = z[j];
}

// ---- pre- / post-pass of eskf_run (KArgs::imu_pf / meas_pf / snap) -------------------------------------------------
// The Monte-Carlo generator and the Euler angles of Filter.calculate_update_mse are throughput work with no dependence on
// the filters' recursion.  Inside the persistent kernel they ran on ONE warp of every CTA and slowed the whole CTA through
// that warp's sub-partition (12 % of the launch at 4096 filters, profiles/r02_*); as separate, fully parallel kernels they
// cost a few per cent of that.  Same generator, same operations in the same order: the results are bit-identical
// (tests/test_gpu_noise.py compares both paths).
// A segment of the trajectory (eskf_run_epochs) indexes the buffers by the segment's steps and epochs (T, E) and the streams
// and the noise counter by global step and epoch: trajectory t's step j is global step k0[t] + j (k0 = nullptr: 0) of the
// T_all-long stream, epoch e is global epoch e0 + e of the E_all-long ones.
struct PPArgs {
  int64_t N, T, E;
  int n_traj;
  int64_t fpt, filter_id0;
  uint64_t seed;
  double imu_noise[6], cam_noise[7];
  int noise_on, noise_free0, noise_mod, per_filter;
  const int64_t* k0;
  int64_t T_all, E_all, e0;
};

__device__ __forceinline__ void pp_ids(const PPArgs& p, int64_t f, int64_t& traj, int64_t& gid, bool& noisy) {
  const int64_t g = p.filter_id0 + f;
  traj = (p.n_traj > 1) ? g / p.fpt : 0;
  gid = p.noise_mod > 0 ? g % p.noise_mod : g;
  noisy = p.noise_on && !(p.noise_free0 && gid == 0);
}

// out[(j N + f) 6 + i]: IMU sample of step j as filter f sees it (role3_stage::stage_sample)
__global__ void pp_imu_kernel(double* __restrict__ out, const double* __restrict__ om_acc, const PPArgs p) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= p.T * p.N) return;
  const int64_t j = idx / p.N, f = idx - j * p.N;
  int64_t traj, gid;
  bool noisy;
  pp_ids(p, f, traj, gid, noisy);
  const int64_t g = (p.k0 ? p.k0[traj] : 0) + j;  // global step
  if (g >= p.T_all) return;  // (past the end of this trajectory's stream: never read)
  const double* src = p.per_filter ? om_acc + (f * p.T_all + g) * 6 : om_acc + (traj * p.T_all + g) * 6;
  double u[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) u[i] = src[i];
  if (noisy) {
    double z[8];
    normal8(p.seed, (uint64_t)gid, (uint64_t)g, RNG_KIND_IMU, z);
#pragma unroll
    for (int i = 0; i < 6; ++i) u[i] += p.imu_noise[i] * z[i];
  }
  double* dst = out + idx * 6;
#pragma unroll
  for (int i = 0; i < 6; ++i) dst[i] = u[i];
}

// out[(e N + f) 8 + i]: camera measurement of epoch e as filter f sees it: position, raw quaternion, notch angle
// (role3_stage::stage_meas)
__global__ void pp_meas_kernel(double* __restrict__ out, const double* __restrict__ camm, const double* __restrict__ notchm,
                               const PPArgs p) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= p.E * p.N) return;
  const int64_t e = idx / p.N, f = idx - e * p.N;
  int64_t traj, gid;
  bool noisy;
  pp_ids(p, f, traj, gid, noisy);
  const int64_t eg = p.e0 + e;  // global epoch
  const int64_t mrow = traj * p.E_all + eg;
  double cam[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) cam[i] = camm[mrow * 7 + i];
  double notch = notchm[mrow];
  if (noisy) {
    double z[8];
    normal8(p.seed, (uint64_t)gid, (uint64_t)eg, RNG_KIND_CAM, z);
    double dth[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      cam[i] += p.cam_noise[i] * z[i];
      dth[i] = p.cam_noise[3 + i] * z[3 + i];
    }
    double dq[4], qn[4];
    quat_about_axis(sqrt(dth[0] * dth[0] + dth[1] * dth[1] + dth[2] * dth[2]), dth, dq);
    const double nq = sqrt(cam[3] * cam[3] + cam[4] * cam[4] + cam[5] * cam[5] + cam[6] * cam[6]);
    quat_mul(cam + 3, dq, qn);
#pragma unroll
    for (int i = 0; i < 4; ++i) cam[3 + i] = qn[i] * nq;
    notch += p.cam_noise[6] * z[6];
  }
  double* dst = out + idx * 8;
#pragma unroll
  for (int i = 0; i < 7; ++i) dst[i] = cam[i];
  dst[7] = notch;
}

// Filter.calculate_update_mse (Filter.py:397-418) from the per-epoch snapshots snap[(e N + f) 14]: v q p_cam q_cam after
// every update.  Stage 1, one thread per (epoch, filter): the two squared-error sums of the epoch (the same operations as
// role3_stage's flush_stats), written over the first two entries of the snapshot.  Stage 2, one thread per filter: the
// running sums over the epochs IN ORDER (the same additions as in the kernel), rows [7] (last epoch) and [8] (sum over
// the epochs) of the statistics, and their contribution to stats_sum.  A segment of the trajectory continues the sums of
// carry_in and leaves them in carry_out ([N][ESKF_NCARRY], entries 0 and 1; either may be nullptr).
__global__ void pp_stats1_kernel(double* __restrict__ snap, const double* __restrict__ cam_ref,
                                 const double* __restrict__ imu_ref, const PPArgs p) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= p.E * p.N) return;
  const int64_t e = idx / p.N, f = idx - e * p.N;
  int64_t traj, gid;
  bool noisy;
  pp_ids(p, f, traj, gid, noisy);
  double* xs = snap + idx * 14;
  const double* ir = imu_ref + (traj * p.E_all + p.e0 + e) * 6;
  const double* cr = cam_ref + (traj * p.E_all + p.e0 + e) * 6;
  double xr[14];
#pragma unroll
  for (int i = 0; i < 14; ++i) xr[i] = xs[i];
  double ei[3], ec[3], accA = 0.0, accB = 0.0;
  euler_xyz_deg(xr + 3, ei);
  euler_xyz_deg(xr + 10, ec);
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double d2_ = xr[i] - ir[i], d3 = ei[i] - ir[3 + i];
    accA += d2_ * d2_ + d3 * d3;
    const double d0 = cr[i] - xr[7 + i], d1 = cr[3 + i] - ec[i];
    accB += d0 * d0 + d1 * d1;
  }
  xs[0] = accA;
  xs[1] = accB;
}

__global__ void pp_stats2_kernel(const double* __restrict__ snap, double* stats_out, double* stats_sum, const PPArgs p,
                                 const double* carry_in, double* carry_out) {
  const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  double r7 = 0.0, r8 = 0.0;
  if (f < p.N) {
    double mseA_last = 0.0, mseA_sum = 0.0, mseB_last = 0.0, mseB_sum = 0.0;
    if (carry_in) {
      mseA_sum = carry_in[f * ESKF_NCARRY + 0];
      mseB_sum = carry_in[f * ESKF_NCARRY + 1];
    }
    for (int64_t e = 0; e < p.E; ++e) {
      const double* xs = snap + (e * p.N + f) * 14;
      mseA_last = xs[0];
      mseA_sum += mseA_last;
      mseB_last = xs[1];
      mseB_sum += mseB_last;
    }
    r7 = (mseA_last + mseB_last) / 12.0;
    r8 = (mseA_sum + mseB_sum) / 12.0;
    if (carry_out) {
      carry_out[f * ESKF_NCARRY + 0] = mseA_sum;
      carry_out[f * ESKF_NCARRY + 1] = mseB_sum;
    }
    if (stats_out) {
      stats_out[f * ESKF_NSTAT + 7] = r7;
      stats_out[f * ESKF_NSTAT + 8] = r8;
    }
  }
  if (stats_sum) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      r7 += __shfl_xor_sync(0xffffffffu, r7, o);
      r8 += __shfl_xor_sync(0xffffffffu, r8, o);
    }
    if ((threadIdx.x & 31) == 0) {
      atomicAdd(stats_sum + 7, r7);
      atomicAdd(stats_sum + 8, r8);
    }
  }
}

// ---- segments of the trajectory (eskf_run_epochs) --------------------------------------------------------------------
// kb[t] and kb[n_traj + t]: the global steps at which trajectory t's epochs e0 and e1 start, k(e) = sum over e' < e of
// n_prop[t, e'] clamped as epoch_steps3 clamps every epoch (a negative entry counts 0 steps, none goes past T).  Clamping
// each term to what is left makes the running sum saturate at T, so k(e) = min(T, sum of max(n_prop, 0)): an exact integer
// reduction.  The one definition of a segment's first step, for the persistent kernel (KArgs::k_base) and the pre-pass.
__global__ void __launch_bounds__(256) seg_base_kernel(const int32_t* __restrict__ n_prop, int64_t E, int64_t T, int64_t e0,
                                                       int64_t e1, int n_traj, int64_t* __restrict__ kb) {
  __shared__ long long sh[2][256];
  const int t = blockIdx.x;
  const int32_t* np_ = n_prop + (int64_t)t * E;
  long long s0 = 0, s1 = 0;
  for (int64_t e = threadIdx.x; e < e1; e += 256) {
    const long long n = np_[e] > 0 ? np_[e] : 0;
    if (e < e0) s0 += n;
    s1 += n;
  }
  sh[0][threadIdx.x] = s0;
  sh[1][threadIdx.x] = s1;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
      sh[0][threadIdx.x] += sh[0][threadIdx.x + o];
      sh[1][threadIdx.x] += sh[1][threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    kb[t] = sh[0][0] < T ? sh[0][0] : T;
    kb[n_traj + t] = sh[1][0] < T ? sh[1][0] : T;
  }
}

// ---- reduction of the statistics rows (the vector a multi-GPU launcher all-reduces) -----------------------------------
// stats_sum of eskf_run, from the per-filter rows, DETERMINISTICALLY (fixed summation tree, no atomics: the same bits
// whatever the CTA scheduling) and MASKED: a filter that diverged (non-finite row) or whose status word is set would
// otherwise turn the reduced vector of a million healthy filters into NaN.  [0:10] sums over the healthy filters,
// [10] filters with a non-zero status, [11] healthy filters (the divisor of every mean), [12] non-finite filters.
// Every reduction of the rows or of the consistency records takes its blocks from a GroupMap (eskf_set_groups): with one
// group, ceil(N / RED_ROWS) blocks of RED_ROWS rows, the ungrouped sums; with groups, per group (group_block, eskf_math.cuh),
// and the final kernels add the blocks of each group in order.  The same fixed trees either way.
constexpr int RED_ROWS = 4096;  // rows per block
struct GroupMap {
  int64_t N, id0, g;  // filters, global id of the first one, group size (0: one group)
  int64_t G, nblk;    // local groups, reduction blocks
};
__host__ __device__ inline GroupMap group_map(int64_t N, int64_t id0, int64_t g) {
  return GroupMap{N, id0, g, g > 0 ? (id0 + N - 1) / g - id0 / g + 1 : 1, group_blocks(N, id0, g, RED_ROWS)};
}
// the blocks b0 .. b1 - 1 of local group k
__device__ __forceinline__ void group_range(const GroupMap& m, int64_t k, int64_t& b0, int64_t& b1) {
  b0 = group_blocks(group_row0(k, m.N, m.id0, m.g), m.id0, m.g, RED_ROWS);
  b1 = group_blocks(group_row0(k + 1, m.N, m.id0, m.g), m.id0, m.g, RED_ROWS);
}
__global__ void stats_partial_kernel(const double* __restrict__ rows, const int32_t* __restrict__ status, const GroupMap m,
                                     double* __restrict__ partial) {
  __shared__ double sh[256][13];
  int64_t r0, r1, k;
  group_block(blockIdx.x, m.N, m.id0, m.g, RED_ROWS, r0, r1, k);
  double acc[13];
#pragma unroll
  for (int i = 0; i < 13; ++i) acc[i] = 0.0;
  for (int64_t r = r0 + threadIdx.x; r < r1; r += 256) {
    const double* row = rows + r * ESKF_NSTAT;
    double v[10], chk = 0.0;
#pragma unroll
    for (int i = 0; i < 10; ++i) {
      v[i] = row[i];
      chk += v[i] * 0.0;  // NaN / inf detector
    }
    const bool fin = (chk == 0.0), flagged = status[r] != 0;
    if (fin && !flagged) {
#pragma unroll
      for (int i = 0; i < 10; ++i) acc[i] += v[i];
      acc[11] += 1.0;
    }
    if (flagged) acc[10] += 1.0;
    if (!fin) acc[12] += 1.0;
  }
#pragma unroll
  for (int i = 0; i < 13; ++i) sh[threadIdx.x][i] = acc[i];
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
#pragma unroll
      for (int i = 0; i < 13; ++i) sh[threadIdx.x][i] += sh[threadIdx.x + o][i];
    }
    __syncthreads();
  }
  if (threadIdx.x < ESKF_NSTAT) partial[(int64_t)blockIdx.x * ESKF_NSTAT + threadIdx.x] = threadIdx.x < 13 ? sh[0][threadIdx.x] : 0.0;
}
// out [G][ESKF_NSTAT]: the blocks of each group added in order
__global__ void stats_final_kernel(const double* __restrict__ partial, const GroupMap m, double* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, k = idx / ESKF_NSTAT, i = idx - k * ESKF_NSTAT;
  if (k >= m.G) return;
  int64_t b0, b1;
  group_range(m, k, b0, b1);
  double a = 0.0;
  for (int64_t b = b0; b < b1; ++b) a += partial[b * ESKF_NSTAT + i];
  out[idx] = a;
}

// ---- filter consistency (eskf_keep_consistency): post-pass over the records the export instantiation filed ------------
// cons_eval_kernel, one thread per (epoch, filter): NIS as filed, NEES of the estimated DOFs from the posterior DOFs and DOF
// block (nees_dofs, eskf_math.cuh); NaN for an update that was not applied and for any non-finite value.  Writes the
// filter-major outputs [N, E] and both values back into the record (CONS_NIS, CONS_NEES) for the epoch reduction.
// An update rejected by the innovation gate keeps the NIS the gate compared and, like a dropped measurement, the NEES of
// the prior.
struct ConsArgs {
  int64_t N, E;
  double gt[6];
  int frozen_mask;
  const double* gate;  // [N] the innovation-gate thresholds of the run that filed the records (a snapshot), or nullptr
};
__global__ void cons_eval_kernel(double* __restrict__ rec, double* __restrict__ nis, double* __restrict__ nees, const ConsArgs p) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= p.E * p.N) return;
  const int64_t e = idx / p.N, f = idx - e * p.N;
  double* r = rec + e * CONS_SIZE * p.N + f;  // element j at r[j N]
  const double flag = r[CONS_NEES * p.N];
  // (a dropped measurement or a rejected update: the NEES of the prior)
  const bool applied = flag == 1.0, dropped = flag == 2.0, rejected = flag == 3.0;
  double eps[6], B[36];
#pragma unroll
  for (int i = 0; i < 6; ++i) eps[i] = r[(CONS_DOFS + i) * p.N] - p.gt[i];
#pragma unroll
  for (int i = 0; i < 36; ++i) B[i] = r[(CONS_B + i) * p.N];
  double vn = r[CONS_NIS * p.N];
  double ve = nees_dofs(B, eps, p.frozen_mask);
  if (!rejected && (!applied || !isfinite(vn))) vn = NAN;
  if (!(applied || dropped || rejected) || !isfinite(ve)) ve = NAN;
  nis[f * p.E + e] = vn;
  nees[f * p.E + e] = ve;
  r[CONS_NIS * p.N] = dropped ? -INFINITY : vn;  // (-inf marks the dropped ones for the reductions: a NIS is never infinite)
  r[CONS_NEES * p.N] = ve;
}

// epoch_sum [E][ESKF_NCONS], deterministically like stats_sum: block b of epoch e sums the finite values of the filters of
// block b of the map through a fixed tree, cons_final_kernel adds the blocks of an epoch (of each group) in order.
// [0] finite NIS, [1] sum, [2] sum of squares, [3..5] the same for the NEES, [6] filters whose NIS (measurement not dropped) or
// (d > 0) NEES is NaN, [7] filters whose measurement was dropped.
__global__ void cons_partial_kernel(const double* __restrict__ rec, const GroupMap m, int with_nees, double* __restrict__ partial) {
  __shared__ double sh[256][8];
  const int64_t N = m.N, e = blockIdx.x / m.nblk, b = blockIdx.x - e * m.nblk;
  int64_t r0, r1, k;
  group_block(b, N, m.id0, m.g, RED_ROWS, r0, r1, k);
  const double* vn = rec + e * CONS_SIZE * N + CONS_NIS * N;
  const double* ve = rec + e * CONS_SIZE * N + CONS_NEES * N;
  double acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.0;
  for (int64_t r = r0 + threadIdx.x; r < r1; r += 256) {
    const double a = vn[r], c = ve[r];
    const bool fa = isfinite(a), fc = isfinite(c), dr = a == -INFINITY;
    if (fa) {
      acc[0] += 1.0;
      acc[1] += a;
      acc[2] += a * a;
    }
    if (fc) {
      acc[3] += 1.0;
      acc[4] += c;
      acc[5] += c * c;
    }
    if ((!fa && !dr) || (with_nees && !fc)) acc[6] += 1.0;
    if (dr) acc[7] += 1.0;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) sh[threadIdx.x][i] = acc[i];
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
#pragma unroll
      for (int i = 0; i < 8; ++i) sh[threadIdx.x][i] += sh[threadIdx.x + o][i];
    }
    __syncthreads();
  }
  if (threadIdx.x < ESKF_NCONS) partial[(int64_t)blockIdx.x * ESKF_NCONS + threadIdx.x] = sh[0][threadIdx.x];
}
// out [G][E][width] from the partial rows [E][nblk][width] of cons_partial_kernel (width ESKF_NCONS) or dof_partial_kernel
// (ESKF_NDOFSUM): the blocks of an epoch and group added in order
__global__ void cons_final_kernel(const double* __restrict__ partial, const GroupMap m, int64_t E, int width, double* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= m.G * E * width) return;
  const int64_t k = idx / (E * width), e = (idx - k * E * width) / width, i = idx - (k * E + e) * width;
  int64_t b0, b1;
  group_range(m, k, b0, b1);
  double a = 0.0;
  for (int64_t b = b0; b < b1; ++b) a += partial[(e * m.nblk + b) * width + i];
  out[idx] = a;
}

// ---- per-DOF history and Monte-Carlo envelope: a second post-pass over the consistency records, run by the getters --------
// (eskf_get_dof_history / eskf_get_dof_envelope) on the records of the last run, never by eskf_run itself.
// dof_history_kernel: filter rows f0 .. f0 + nf - 1 of dofs / var [N][E][6] (either may be nullptr; row f0 at index 0).  A
// block transposes a tile of 32 filters x 8 epochs through shared memory: every warp reads 32 consecutive filters of one
// record element (256 B), and writes runs of 48 consecutive doubles (8 epochs of one filter).
constexpr int HT_F = 32, HT_E = 8;
__global__ void __launch_bounds__(256) dof_history_kernel(const double* __restrict__ rec, int64_t N, int64_t E, int64_t f0,
                                                          int64_t nf, double* __restrict__ dofs, double* __restrict__ var) {
  __shared__ double sd[HT_F][HT_E * 6 + 1], sv[HT_F][HT_E * 6 + 1];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int64_t fb = (int64_t)blockIdx.x * HT_F;
  for (int64_t e0 = (int64_t)blockIdx.y * HT_E; e0 < E; e0 += (int64_t)gridDim.y * HT_E) {
    const int64_t f = fb + tx, e = e0 + ty;
    if (f < nf && e < E) {
      const double* r = rec + e * CONS_SIZE * N + f0 + f;
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        if (dofs) sd[tx][6 * ty + i] = r[(CONS_DOFS + i) * N];
        if (var) sv[tx][6 * ty + i] = r[(CONS_B + 7 * i) * N];
      }
    }
    __syncthreads();
    const int nc = 6 * (int)(E - e0 < HT_E ? E - e0 : HT_E);
    for (int k = threadIdx.x; k < HT_F * HT_E * 6; k += 256) {
      const int lf = k / (HT_E * 6), c = k - lf * (HT_E * 6);
      if (fb + lf < nf && c < nc) {
        const int64_t o = ((fb + lf) * E + e0) * 6 + c;
        if (dofs) dofs[o] = sd[lf][c];
        if (var) var[o] = sv[lf][c];
      }
    }
    __syncthreads();
  }
}

// dof_partial_kernel: the envelope rows [E][ESKF_NDOFSUM] deterministically, as cons_partial_kernel does the epoch sums:
// block b of epoch e takes the filters of block b of the map.  Each filter's DSUM_USED terms (dof_terms) do not fit
// a per-thread accumulator, so every warp reduces the terms of its 32 filters at once, over fixed trees: recursive halving
// over the lanes for each full group of 32 columns (after five exchange steps lane l holds the warp's sum of column
// 32 g + l), an xor butterfly for each of the remaining columns (lane c - 64 keeps column c).  Every lane accumulates its
// columns over the warp's rows in order, and the eight warps are added in order at the end.  cons_final_kernel adds the
// blocks.
// A dropped measurement (CONS_NIS = -inf, cons_eval_kernel) lets the filter contribute its prior and counts in column DSUM_DROP.
// So does an update rejected by the innovation gate, in column DSUM_REJ: its NIS exceeds the threshold of the run that filed
// the record (ConsArgs::gate, the kernel's own comparison of the same values), an applied update's does not.
__global__ void __launch_bounds__(256) dof_partial_kernel(const double* __restrict__ rec, const ConsArgs p, const GroupMap m,
                                                          double* __restrict__ partial) {
  constexpr int W = DSUM_REJ + 1;  // reduced columns
  constexpr int NG = W / 32;  // full column groups; the tail W - 32 NG < 32 columns
  static_assert(W - 32 * NG < 32 && DSUM_DROP >= DSUM_USED && DSUM_REJ == DSUM_DROP + 1, "tail");
  __shared__ double sh[8][32 * (NG + 1)];
  const int64_t e = blockIdx.x / m.nblk, b = blockIdx.x - e * m.nblk;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int64_t rb, r1, k;
  group_block(b, m.N, m.id0, m.g, RED_ROWS, rb, r1, k);
  const double* re = rec + e * CONS_SIZE * p.N + rb;  // (rows counted from the block's first one)
  const int nr = (int)(r1 - rb);
  double acc[NG + 1];
#pragma unroll
  for (int g = 0; g <= NG; ++g) acc[g] = 0.0;
  for (int r0 = 32 * w; r0 < nr; r0 += 256) {  // (warp-uniform)
    const int r = r0 + lane;
    double t[W];
#pragma unroll
    for (int c = 0; c < W; ++c) t[c] = 0.0;
    if (r < nr) {
      double eps[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) eps[i] = re[(CONS_DOFS + i) * p.N + r] - p.gt[i];
      const double vn = re[CONS_NIS * p.N + r];
      const bool dr = vn == -INFINITY;
      dof_terms(dr ? 0.0 : vn, eps, re + CONS_B * p.N + r, p.N, p.frozen_mask, t);
      t[DSUM_DROP] = dr ? 1.0 : 0.0;
      t[DSUM_REJ] = (p.gate && vn > p.gate[rb + r]) ? 1.0 : 0.0;
    }
    // (the tail first, then the groups from the last: fewer terms live at once)
#pragma unroll
    for (int c = 32 * NG; c < W; ++c) {
      double v = t[c];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == c - 32 * NG) acc[NG] += v;
    }
#pragma unroll
    for (int g = NG - 1; g >= 0; --g) {
      double* v = t + 32 * g;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const bool up = (lane & o) != 0;  // keeps the upper half of the columns, sends the lower one
#pragma unroll
        for (int j = 0; j < o; ++j) {
          const double keep = up ? v[j + o] : v[j], send = up ? v[j] : v[j + o];
          v[j] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
      }
      acc[g] += v[0];
    }
  }
#pragma unroll
  for (int g = 0; g <= NG; ++g) sh[w][32 * g + lane] = acc[g];
  __syncthreads();
  if (threadIdx.x < ESKF_NDOFSUM) {
    double a = 0.0;
    if (threadIdx.x < W)
      for (int k = 0; k < 8; ++k) a += sh[k][threadIdx.x];
    partial[(int64_t)blockIdx.x * ESKF_NDOFSUM + threadIdx.x] = a;
  }
}
static_assert(DSUM_USED <= ESKF_NDOFSUM && ESKF_NDOFSUM <= 256, "envelope row");

// Filter.Fx (24 x 24) and Filter.Fi (24 x 13) as the reference assembles them (Filter.py:249-342), from the fx3 record the
// producer roles filed for the last IMU step of a launch (KArgs::fx_dump): the dense matrices the register-tile algebra of
// eskf_cov3.cuh applies implicitly.
__global__ void expand_jac_kernel(const double* __restrict__ rec, int64_t n, double* __restrict__ Fx, double* __restrict__ Fi) {
  const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  const double* r = rec + f * FX3_SIZE;
  if (Fx) {
    double* M = Fx + f * 576;
    for (int i = 0; i < 576; ++i) M[i] = 0.0;
    for (int i = 0; i < 24; ++i) M[i * 24 + i] = 1.0;
    const double dt = r[FX3_DT];
    for (int i = 0; i < 3; ++i) {
      M[i * 24 + 3 + i] = dt;  // Filter.py:252
      for (int k = 0; k < 3; ++k) {
        M[(3 + i) * 24 + 6 + k] = r[FX3_AB + 6 * k + i];      // Filter.py:253
        M[(6 + i) * 24 + 6 + k] = r[FX3_AB + 6 * k + 3 + i];  // Filter.py:255
      }
    }
    M[15 * 24 + 16] += dt;  // notch chain, Filter.py:257-258
    M[16 * 24 + 17] += dt;
    // rows 18:24: Fx[18:24, 0:22] = jacobian (Filter.py:279-285: columns 0..21 are overwritten, 22 and 23 keep the identity)
    for (int i = 18; i < 24; ++i)
      for (int j = 0; j < 22; ++j) M[i * 24 + j] = 0.0;
    for (int i = 0; i < 3; ++i) {
      M[(18 + i) * 24 + 3 + i] = dt;
      for (int k = 0; k < 9; ++k) M[(18 + i) * 24 + 6 + k] = r[FX3_H1 + 3 * k + i];
      M[(18 + i) * 24 + 16 + i] = 1.0;  // the mis-aligned identity block (quirk Q3)
      for (int k = 0; k < 7; ++k) {
        const int col = (k < 3) ? 9 + k : (k == 3) ? 15 : 19 + (k - 4);
        M[(21 + i) * 24 + col] = r[FX3_H2 + 3 * k + i];
      }
    }
  }
  if (Fi) {
    double* M = Fi + f * 312;
    for (int i = 0; i < 312; ++i) M[i] = 0.0;
    for (int i = 0; i < 12; ++i) M[(3 + i) * 13 + i] = 1.0;  // Filter.py:262-263
    M[17 * 13 + 12] = 1.0;
    for (int i = 0; i < 3; ++i)
      for (int k = 0; k < 3; ++k) {
        M[(18 + i) * 13 + 3 + k] = r[FX3_NP + 3 * i + k];
        M[(21 + i) * 13 + 3 + k] = r[FX3_NT + 3 * i + k];
      }
  }
}

thread_local std::string g_err;

// NVTX range for the lifetime of a scope (nsys / ncu --nvtx timelines: eskf_run and its pre- / post-pass, eskf_propagate,
// eskf_update, eskf_prepass; the reference's only instrumentation is the disabled timer at Imu.py:256,271)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

}  // namespace

// ---------------------------------------------------------------------------------------------
// 0..8: arguments / results of the calls; 9..11: pre- / post-pass buffers of eskf_run; 12: partial sums; 13: first steps of a
// segment (seg_base_kernel); 14, 15: host carry of eskf_run_epochs; 16: partial sums of the grouped statistics
constexpr int N_STAGE = 17;
struct eskf_handle {
  int device = 0;
  cudaStream_t stream = nullptr;
  int64_t N = 0;
  Model model{};
  double *x = nullptr, *P = nullptr, *u = nullptr, *Ro = nullptr, *par = nullptr;
  int32_t* status = nullptr;
  // grow-only device staging for host-side arguments / results
  void* stage[N_STAGE] = {};
  size_t stage_sz[N_STAGE] = {};
  double* stats_sum_dev = nullptr;
  int64_t launches = 0;
  int fpc = 0;  // filters per CTA (0 = automatic)
  int variant = 0;  // 0 = default (eskf_kernel3), 1 = eskf_kernel (first version, kept for A/B measurements), 3 = eskf_kernel3
  int sm_count = 148;
  double* fxrec = nullptr;  // [N][FX3_SIZE] Jacobian record of the last step (eskf_keep_jacobians), or nullptr
  size_t pp_budget = 0;  // bytes the pre- / post-pass buffers of one eskf_run may take (0: everything inside the kernel)
  // filter consistency (eskf_keep_consistency): the records of one run [E][CONS_SIZE][N] and the results of the last run,
  // one buffer: nis [N][E], nees [N][E], epoch_sum [E][ESKF_NCONS], the partial sums of the reduction, then the envelope row
  // [E][ESKF_NDOFSUM] and its partial sums (eskf_get_dof_envelope)
  bool cons_on = false;
  int64_t cons_E = -1;  // epochs of the last run that filed them (-1: none since eskf_keep_consistency)
  double *cons_rec = nullptr, *cons_out = nullptr;
  size_t cons_rec_sz = 0, cons_out_sz = 0;
  ConsArgs cons_args{};  // gt_dofs and frozen mask of the last run that filed them
  // filter groups (eskf_set_groups): the group size of the next run, and the block map of the last run's filters, with
  // which eskf_get_group_sums reduces its results.  grp_stats [G][ESKF_NSTAT]: the last run's statistics per group (valid
  // when grp_stats_ok); grp_buf: partial sums and host staging of eskf_get_group_sums
  int64_t groups = 0;
  GroupMap run_groups{};
  bool grp_stats_ok = false;
  double *grp_stats = nullptr, *grp_buf = nullptr;
  size_t grp_stats_sz = 0, grp_buf_sz = 0;
  // simulated frame loss (eskf_set_meas_dropout): drop probabilities [drop_nt][drop_E] of every later run, on (drop_nt > 0) or off
  double* drop_p = nullptr;
  size_t drop_sz = 0;
  int64_t drop_nt = 0, drop_E = 0;
  // simulated outlier frames (eskf_set_meas_outliers): probabilities [out_nt][out_E] and offset std of every later run, on
  // (out_nt > 0) or off
  double* out_p = nullptr;
  size_t out_sz = 0;
  int64_t out_nt = 0, out_E = 0;
  double out_std[7] = {0, 0, 0, 0, 0, 0, 0};
  // innovation gate (eskf_set_innovation_gate): gate[0, N) the thresholds of every later run, on (gate_on) or off;
  // gate[N, 2N) a snapshot of those the last run with consistency records used (ConsArgs::gate, read by the getters)
  double* gate = nullptr;
  bool gate_on = false;
};

#define CK(call)                                                  \
  do {                                                            \
    cudaError_t e_ = (call);                                      \
    if (e_ != cudaSuccess) {                                      \
      g_err = std::string(#call) + ": " + cudaGetErrorString(e_); \
      return ESKF_ECUDA;                                          \
    }                                                             \
  } while (0)

static int stage_reserve(eskf_t* h, int slot, size_t bytes) {
  if (h->stage_sz[slot] >= bytes) return ESKF_OK;
  if (h->stage[slot]) CK(cudaFree(h->stage[slot]));
  h->stage[slot] = nullptr;
  h->stage_sz[slot] = 0;
  CK(cudaMalloc(&h->stage[slot], bytes));
  h->stage_sz[slot] = bytes;
  return ESKF_OK;
}

// host pointer -> copied into a staging slot on the handle's stream; device pointer -> used as is
static int stage_in(eskf_t* h, int slot, const void* src, size_t bytes, int mem, const void** out) {
  *out = nullptr;
  if (!src || bytes == 0) return ESKF_OK;
  if (mem == ESKF_MEM_DEVICE) {
    *out = src;
    return ESKF_OK;
  }
  int rc = stage_reserve(h, slot, bytes);
  if (rc) return rc;
  CK(cudaMemcpyAsync(h->stage[slot], src, bytes, cudaMemcpyHostToDevice, h->stream));
  *out = h->stage[slot];
  return ESKF_OK;
}

// grow-only device buffer *p of *sz bytes: the new one is allocated before the old one is released, so that a request that
// does not fit (ESKF_ENOMEM) leaves the old content readable
static int grow(double** p, size_t* sz, size_t bytes, const char* what) {
  if (*sz >= bytes) return ESKF_OK;
  void* n = nullptr;
  const cudaError_t err = cudaMalloc(&n, bytes);
  if (err != cudaSuccess) {
    cudaGetLastError();  // (an allocation failure is not sticky: clear it for the launches of later calls)
    g_err = std::string(what) + ": " + std::to_string((unsigned long long)bytes) + " bytes do not fit in device memory: " +
            cudaGetErrorString(err);
    return err == cudaErrorMemoryAllocation ? ESKF_ENOMEM : ESKF_ECUDA;
  }
  CK(cudaFree(*p));
  *p = (double*)n;
  *sz = bytes;
  return ESKF_OK;
}

// the buffers of the consistency records and results of a run over E epochs.  Both are allocated before an old one is
// released, so that a run that does not fit (ESKF_ENOMEM) leaves the results of the last run readable.
static int64_t cons_nblk(const eskf_t* h) { return (h->N + RED_ROWS - 1) / RED_ROWS; }
static int cons_reserve(eskf_t* h, int64_t E) {
  const size_t n = (size_t)h->N, e = (size_t)E;
  const size_t rb = e * CONS_SIZE * n * sizeof(double);
  const size_t nb = (size_t)cons_nblk(h);
  const size_t ob = (2 * n * e + (e + nb * e) * (ESKF_NCONS + ESKF_NDOFSUM)) * sizeof(double);
  void *nr = nullptr, *no = nullptr;
  cudaError_t err = cudaSuccess;
  if (rb > h->cons_rec_sz) err = cudaMalloc(&nr, rb);
  if (err == cudaSuccess && ob > h->cons_out_sz) err = cudaMalloc(&no, ob);
  if (err != cudaSuccess) {
    cudaGetLastError();  // (an allocation failure is not sticky: clear it for the launches of later calls)
    cudaFree(nr);
    g_err = "eskf_run: the consistency records of " + std::to_string((long long)h->N) + " filters x " +
            std::to_string((long long)E) + " epochs (" + std::to_string((unsigned long long)(rb + ob)) +
            " bytes) do not fit in device memory: " + cudaGetErrorString(err);
    return err == cudaErrorMemoryAllocation ? ESKF_ENOMEM : ESKF_ECUDA;
  }
  if (nr) {
    CK(cudaFree(h->cons_rec));
    h->cons_rec = (double*)nr;
    h->cons_rec_sz = rb;
  }
  if (no) {
    CK(cudaFree(h->cons_out));
    h->cons_out = (double*)no;
    h->cons_out_sz = ob;
  }
  return ESKF_OK;
}

// default of eskf_set_prepass_budget: memory the pre- / post-pass buffers of one eskf_run may take (ESKF_B200_PP_MAX_BYTES;
// 0 switches the mode off and the generator / the statistics run inside the persistent kernel as in round 1)
static size_t pp_budget_bytes() {
  static const size_t v = [] {
    const char* e = getenv("ESKF_B200_PP_MAX_BYTES");
    return e ? (size_t)strtoull(e, nullptr, 10) : ((size_t)32 << 30);
  }();
  return v;
}

static const int kShapes1[] = {28, 4};  // eskf_kernel  (v1: the first correct path, kept as an A/B and test variant only)
static const int kShapes3[] = {28, 16, 8, 4};              // eskf_kernel3

static int kernel_of(const eskf_t* h) { return h->variant == 1 ? 1 : 3; }

// Filters per CTA.  A CTA follows ONE trajectory's epoch structure: eskf_kernel3 cuts every trajectory's filters into
// CTAs of their own (ragged last CTA per trajectory), the first kernel needs a shape that divides filters_per_traj.
// Every shape runs one CTA per SM (registers / shared memory) and a wave of CTAs takes about the same time whatever
// its shape (per-step latency bound, profiles/r01_*): the automatic choice minimises the number of waves and then
// prefers the larger shape.
static int pick_fpc(const eskf_t* h, int64_t fpt, bool multi_traj) {
  const bool k3 = kernel_of(h) == 3;
  auto fits = [&](int c) { return !multi_traj || k3 || (fpt % c) == 0; };
  const int* shapes = kernel_of(h) == 3 ? kShapes3 : kShapes1;
  const int ns = kernel_of(h) == 3 ? 4 : 2;
  if (h->fpc > 0) {
    for (int i = 0; i < ns; ++i)
      if (shapes[i] == h->fpc && fits(shapes[i])) return shapes[i];
  }
  int best = 0;
  int64_t best_waves = 0;
  for (int i = 0; i < ns; ++i) {  // descending
    const int c = shapes[i];
    if (!fits(c)) continue;
    const int64_t ctas = (multi_traj && k3) ? stacked_grid(h->N, fpt, c) : (h->N + c - 1) / c;
    const int64_t waves = (ctas + h->sm_count - 1) / h->sm_count;
    if (best == 0 || waves < best_waves) {
      best = c;
      best_waves = waves;
    }
  }
  return best;
}

static int launch(eskf_t* h, const KArgs& a, int64_t fpt, bool multi_traj) {
  cudaError_t e;
  const int fpc = pick_fpc(h, fpt, multi_traj);
  if (kernel_of(h) == 3) {
    switch (fpc) {
      case 28: e = launch_eskf_kernel3<28>(a, h->stream); break;
      case 16: e = launch_eskf_kernel3<16>(a, h->stream); break;
      case 8: e = launch_eskf_kernel3<8>(a, h->stream); break;
      case 4: e = launch_eskf_kernel3<4>(a, h->stream); break;
      default:
        g_err = "filters_per_traj must be a multiple of 4 when several trajectories are stacked";
        return ESKF_EINVAL;
    }
  } else {
    switch (fpc) {
      case 28: e = launch_eskf_kernel<28>(a, h->stream); break;
      case 4: e = launch_eskf_kernel<4>(a, h->stream); break;
      default:
        g_err = "filters_per_traj must be a multiple of 4 when several trajectories are stacked";
        return ESKF_EINVAL;
    }
  }
  if (e != cudaSuccess) {
    g_err = std::string("eskf_kernel launch: ") + cudaGetErrorString(e);
    return ESKF_ECUDA;
  }
  h->launches += 1;
  return ESKF_OK;
}

static void base_args(const eskf_t* h, KArgs& a) {
  memset(&a, 0, sizeof(a));
  a.x = h->x;
  a.P = h->P;
  a.u = h->u;
  a.Ro = h->Ro;
  a.status = h->status;
  a.par = h->par;
  a.N = h->N;
  a.model = h->model;
  a.n_traj = 1;
  a.filters_per_traj = h->N;
  a.fx_dump = h->fxrec;
}

extern "C" {
static int create_alloc(eskf_t* h, const eskf_model_t* model, int64_t n_filters, int device, void* cuda_stream);

const char* eskf_last_error(void) { return g_err.c_str(); }
const char* eskf_version(void) { return "eskf_b200 0.3 (sm_100a)"; }

int eskf_create(const eskf_model_t* model, int64_t n_filters, int device, void* cuda_stream, eskf_t** out) {
  if (!model || !out || n_filters <= 0) {
    g_err = "eskf_create: bad argument";
    return ESKF_EINVAL;
  }
  CK(cudaSetDevice(device));
  eskf_t* h = new eskf_handle();
  const int rc_alloc = create_alloc(h, model, n_filters, device, cuda_stream);
  if (rc_alloc != ESKF_OK) {
    const std::string keep = g_err;  // (eskf_destroy does not touch it, but keep the first error whatever happens)
    eskf_destroy(h);
    g_err = keep;
    return rc_alloc;
  }
  *out = h;
  return ESKF_OK;
}

static int create_alloc(eskf_t* h, const eskf_model_t* model, int64_t n_filters, int device, void* cuda_stream) {
  h->device = device;
  h->stream = (cudaStream_t)cuda_stream;
  h->N = n_filters;
  h->model.L = model->scope_length;
  h->model.sa = sin(model->cam_angle_rad);
  h->model.ca = cos(model->cam_angle_rad);
  h->model.frozen_mask = model->frozen_mask;
  h->model.flags = model->flags;
  int smc = 0;
  CK(cudaDeviceGetAttribute(&smc, cudaDevAttrMultiProcessorCount, device));
  h->sm_count = smc > 0 ? smc : 148;
  h->pp_budget = pp_budget_bytes();
  h->run_groups = group_map(n_filters, 0, 0);
  const size_t n = (size_t)n_filters;
  CK(cudaMalloc(&h->x, n * NX * sizeof(double)));
  CK(cudaMalloc(&h->P, n * 576 * sizeof(double)));
  CK(cudaMalloc(&h->u, n * 6 * sizeof(double)));
  CK(cudaMalloc(&h->Ro, n * 9 * sizeof(double)));
  CK(cudaMalloc(&h->par, n * PAR_STRIDE * sizeof(double)));
  CK(cudaMalloc(&h->status, n * sizeof(int32_t)));
  CK(cudaMalloc(&h->stats_sum_dev, ESKF_NSTAT * sizeof(double)));
  CK(cudaMemsetAsync(h->x, 0, n * NX * sizeof(double), h->stream));
  CK(cudaMemsetAsync(h->P, 0, n * 576 * sizeof(double), h->stream));
  CK(cudaMemsetAsync(h->u, 0, n * 6 * sizeof(double), h->stream));
  CK(cudaMemsetAsync(h->Ro, 0, n * 9 * sizeof(double), h->stream));
  CK(cudaMemsetAsync(h->par, 0, n * PAR_STRIDE * sizeof(double), h->stream));
  CK(cudaMemsetAsync(h->status, 0, n * sizeof(int32_t), h->stream));
  return ESKF_OK;
}

int eskf_destroy(eskf_t* h) {
  if (!h) return ESKF_OK;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  cudaFree(h->x);
  cudaFree(h->P);
  cudaFree(h->u);
  cudaFree(h->Ro);
  cudaFree(h->par);
  cudaFree(h->status);
  cudaFree(h->stats_sum_dev);
  cudaFree(h->fxrec);
  cudaFree(h->cons_rec);
  cudaFree(h->cons_out);
  cudaFree(h->grp_stats);
  cudaFree(h->grp_buf);
  cudaFree(h->drop_p);
  cudaFree(h->out_p);
  cudaFree(h->gate);
  for (int i = 0; i < N_STAGE; ++i)
    if (h->stage[i]) cudaFree(h->stage[i]);
  delete h;
  return ESKF_OK;
}

static int set_rows(eskf_t* h, int slot, double* dst, const double* src, int64_t rows, int w, int mem) {
  if (!src) return ESKF_OK;
  if (rows != 1 && rows != h->N) {
    g_err = "leading dimension must be 1 or n_filters";
    return ESKF_EINVAL;
  }
  const size_t bytes = (size_t)rows * w * sizeof(double);
  if (rows == h->N) {
    CK(cudaMemcpyAsync(dst, src, bytes, mem == ESKF_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice,
                       h->stream));
    return ESKF_OK;
  }
  const void* d = nullptr;
  int rc = stage_in(h, slot, src, bytes, mem, &d);
  if (rc) return rc;
  const int64_t tot = h->N * w;
  bcast_rows_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, h->stream>>>(dst, (const double*)d, h->N, w);
  CK(cudaGetLastError());
  h->launches += 1;
  return ESKF_OK;
}

int eskf_set_state(eskf_t* h, const double* x, int64_t nx, const double* P, int64_t nP, const double* u_old,
                   int64_t nu, const double* R_old, int64_t nR, int mem) {
  if (!h) return ESKF_EINVAL;
  CK(cudaSetDevice(h->device));
  int rc;
  if ((rc = set_rows(h, 0, h->x, x, nx, NX, mem))) return rc;
  if ((rc = set_rows(h, 1, h->P, P, nP, 576, mem))) return rc;
  if ((rc = set_rows(h, 2, h->u, u_old, nu, 6, mem))) return rc;
  if (R_old) {
    if ((rc = set_rows(h, 3, h->Ro, R_old, nR, 9, mem))) return rc;
  } else if (x) {
    rot_from_state_kernel<<<(unsigned)((h->N + 255) / 256), 256, 0, h->stream>>>(h->Ro, h->x, h->N);
    CK(cudaGetLastError());
    h->launches += 1;
  }
  if (x) CK(cudaMemsetAsync(h->status, 0, (size_t)h->N * sizeof(int32_t), h->stream));
  return ESKF_OK;
}

int eskf_set_noise(eskf_t* h, const double* Qdiag, int64_t nq, const double* Rdiag, int64_t nr,
                   const double* sigma_om, int64_t ns, int mem) {
  if (!h) return ESKF_EINVAL;
  CK(cudaSetDevice(h->device));
  auto bad = [&](const double* p, int64_t n) { return p && n != 1 && n != h->N; };
  if (bad(Qdiag, nq) || bad(Rdiag, nr) || bad(sigma_om, ns)) {
    g_err = "eskf_set_noise: leading dimension must be 1 or n_filters";
    return ESKF_EINVAL;
  }
  const void *dq = nullptr, *dr = nullptr, *ds = nullptr;
  int rc;
  if ((rc = stage_in(h, 0, Qdiag, (size_t)nq * 13 * sizeof(double), mem, &dq))) return rc;
  if ((rc = stage_in(h, 1, Rdiag, (size_t)nr * 7 * sizeof(double), mem, &dr))) return rc;
  if ((rc = stage_in(h, 2, sigma_om, (size_t)ns * 3 * sizeof(double), mem, &ds))) return rc;
  // the parameter table always has N rows; a broadcast simply fills every row
  fill_par_kernel<<<(unsigned)((h->N + 127) / 128), 128, 0, h->stream>>>(h->par, (const double*)dq, nq, (const double*)dr,
                                                                       nr, (const double*)ds, ns, h->N);
  CK(cudaGetLastError());
  h->launches += 1;
  return ESKF_OK;
}

int eskf_propagate(eskf_t* h, const double* dt, const double* om_acc, int64_t T, int per_filter, int mem) {
  NvtxRange nvtx_("eskf_propagate");
  if (!h || !dt || !om_acc || T < 0) {
    g_err = "eskf_propagate: bad argument";
    return ESKF_EINVAL;
  }
  if (T == 0) return ESKF_OK;
  CK(cudaSetDevice(h->device));
  const void *ddt = nullptr, *doa = nullptr;
  int rc;
  if ((rc = stage_in(h, 0, dt, (size_t)T * sizeof(double), mem, &ddt))) return rc;
  if ((rc = stage_in(h, 1, om_acc, (size_t)(per_filter ? h->N : 1) * T * 6 * sizeof(double), mem, &doa))) return rc;
  KArgs a;
  base_args(h, a);
  a.T = T;
  a.E = 1;
  a.dt = (const double*)ddt;
  a.om_acc = (const double*)doa;
  a.stream_per_filter = per_filter ? 1 : 0;
  a.do_update = 0;
  return launch(h, a, h->N, false);
}

int eskf_update(eskf_t* h, const double* cam, const double* notch, int per_filter, double* K_out, int mem) {
  NvtxRange nvtx_("eskf_update");
  if (!h || !cam || !notch) {
    g_err = "eskf_update: bad argument";
    return ESKF_EINVAL;
  }
  CK(cudaSetDevice(h->device));
  const int64_t rows = per_filter ? h->N : 1;
  const void *dc = nullptr, *dn = nullptr;
  int rc;
  if ((rc = stage_in(h, 0, cam, (size_t)rows * 7 * sizeof(double), mem, &dc))) return rc;
  if ((rc = stage_in(h, 1, notch, (size_t)rows * sizeof(double), mem, &dn))) return rc;
  double* dK = nullptr;
  const size_t kb = (size_t)h->N * 168 * sizeof(double);
  if (K_out) {
    if (mem == ESKF_MEM_DEVICE) {
      dK = K_out;
    } else {
      if ((rc = stage_reserve(h, 2, kb))) return rc;
      dK = (double*)h->stage[2];
    }
    CK(cudaMemsetAsync(dK, 0, kb, h->stream));
  }
  KArgs a;
  base_args(h, a);
  a.T = 0;
  a.E = 1;
  a.cam = (const double*)dc;
  a.notch = (const double*)dn;
  a.meas_per_filter = per_filter ? 1 : 0;
  a.do_update = 1;
  a.K_out = dK;
  if ((rc = launch(h, a, h->N, false))) return rc;
  if (K_out && mem == ESKF_MEM_HOST) {
    CK(cudaMemcpyAsync(K_out, dK, kb, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  return ESKF_OK;
}

// eskf_run and eskf_run_epochs: epochs [e0, e1) of the trajectory in `sp`.  `whole` (eskf_run) makes the launch eskf_run has
// always made.  A segment -- a range other than [0, E), or a carry -- runs the instantiation with MODE bit 2: every CTA rebases
// onto its trajectory's first step (k_base, seg_base_kernel) and the range's first epoch, the pre- and post-pass buffers and the
// consistency records are sized by the segment, and the accumulators come from / go to the carry.
static int run_epochs(eskf_t* h, const eskf_streams_t* sp, int64_t e0, int64_t e1, const double* carry_in, double* carry_out,
                      double* stats_out, double* stats_sum, int mem, bool whole) {
  const std::string fn = whole ? "eskf_run" : "eskf_run_epochs";
  NvtxRange nvtx_(fn.c_str());
  if (!h || !sp || !sp->dt || !sp->om_acc || !sp->n_prop || !sp->cam || !sp->notch || sp->n_traj < 1) {
    g_err = fn + ": bad argument";
    return ESKF_EINVAL;
  }
  CK(cudaSetDevice(h->device));
  const int smem_kind = sp->mem;
  const int64_t T = sp->n_steps, E = sp->n_epochs, nt = sp->n_traj;
  const int64_t fpt = nt > 1 ? sp->filters_per_traj : h->N;
  if (T < 0 || E < 0 || sp->filter_id0 < 0) {
    g_err = fn + ": n_steps, n_epochs and filter_id0 must not be negative";
    return ESKF_EINVAL;
  }
  if (nt > 1) {
    // the kernels pick the trajectory of a filter from its GLOBAL id: (filter_id0 + f) / filters_per_traj
    if (fpt <= 0 || (sp->filter_id0 % fpt) != 0) {
      g_err = fn + ": filter_id0 must be a multiple of filters_per_traj (a shard starts at a trajectory boundary)";
      return ESKF_EINVAL;
    }
    if (sp->filter_id0 + h->N > nt * fpt) {
      g_err = fn + ": filter_id0 + n_filters exceeds n_traj * filters_per_traj (the streams of " +
              std::to_string((long long)nt) + " trajectories do not cover these filters)";
      return ESKF_EINVAL;
    }
  }
  if (smem_kind == ESKF_MEM_HOST) {  // (device-resident streams: the kernels clamp every epoch to what is left, epoch_steps3)
    for (int64_t tr = 0; tr < nt; ++tr) {
      int64_t tot = 0;
      for (int64_t e = 0; e < E; ++e) {
        const int32_t np_ = sp->n_prop[tr * E + e];
        if (np_ < 0) {
          g_err = fn + ": negative n_prop entry";
          return ESKF_EINVAL;
        }
        tot += np_;
      }
      if (tot > T) {
        g_err = fn + ": sum(n_prop) = " + std::to_string((long long)tot) + " exceeds n_steps = " + std::to_string((long long)T);
        return ESKF_EINVAL;
      }
    }
  }
  if (!whole) {
    if (e0 < 0 || e0 > e1 || e1 > E) {
      g_err = fn + ": epoch range [" + std::to_string((long long)e0) + ", " + std::to_string((long long)e1) +
              ") is not within [0, n_epochs = " + std::to_string((long long)E) + "]";
      return ESKF_EINVAL;
    }
    if (kernel_of(h) != 3) {
      g_err = fn + ": segments need the default kernel (eskf_set_variant(h, 1) selects the first one)";
      return ESKF_EINVAL;
    }
  }
  if (h->drop_nt > 0) {
    if (kernel_of(h) != 3) {
      g_err = fn + ": measurement dropout needs the default kernel (eskf_set_variant(h, 1) selects the first one)";
      return ESKF_EINVAL;
    }
    if (h->drop_nt != nt || h->drop_E != E) {
      g_err = fn + ": the dropout probabilities are [" + std::to_string((long long)h->drop_nt) + ", " +
              std::to_string((long long)h->drop_E) + "], the streams [n_traj = " + std::to_string((long long)nt) +
              ", n_epochs = " + std::to_string((long long)E) + "]";
      return ESKF_EINVAL;
    }
  }
  if (h->out_nt > 0) {
    if (kernel_of(h) != 3) {
      g_err = fn + ": simulated outlier frames need the default kernel (eskf_set_variant(h, 1) selects the first one)";
      return ESKF_EINVAL;
    }
    if (h->out_nt != nt || h->out_E != E) {
      g_err = fn + ": the outlier probabilities are [" + std::to_string((long long)h->out_nt) + ", " +
              std::to_string((long long)h->out_E) + "], the streams [n_traj = " + std::to_string((long long)nt) +
              ", n_epochs = " + std::to_string((long long)E) + "]";
      return ESKF_EINVAL;
    }
  }
  if (h->gate_on && kernel_of(h) != 3) {
    g_err = fn + ": the innovation gate needs the default kernel (eskf_set_variant(h, 1) selects the first one)";
    return ESKF_EINVAL;
  }
  const size_t cb = (size_t)h->N * ESKF_NCARRY * sizeof(double);
  if (!whole && e0 == e1) {  // an empty range launches nothing: the carry passes through, the statistics are not written
    if (carry_out && carry_out != carry_in) {
      if (mem == ESKF_MEM_DEVICE) {
        if (carry_in) CK(cudaMemcpyAsync(carry_out, carry_in, cb, cudaMemcpyDeviceToDevice, h->stream));
        else CK(cudaMemsetAsync(carry_out, 0, cb, h->stream));
      } else if (carry_in) {
        memcpy(carry_out, carry_in, cb);
      } else {
        memset(carry_out, 0, cb);
      }
    }
    if (h->cons_on) h->cons_E = 0;
    h->run_groups = group_map(h->N, sp->filter_id0, h->groups);  // (a run of no epochs: its groups, and no statistics rows)
    h->grp_stats_ok = false;
    return ESKF_OK;
  }
  const int64_t Es = e1 - e0;  // epochs of this launch
  const bool seg = !whole && (e0 > 0 || e1 < E || carry_in || carry_out);
  int rc;
  if (h->cons_on) {
    if (kernel_of(h) != 3) {
      g_err = fn + ": filter consistency needs the default kernel (eskf_set_variant(h, 1) selects the first one)";
      return ESKF_EINVAL;
    }
    if ((rc = cons_reserve(h, Es))) return rc;
    h->cons_E = -1;  // (valid again once this run has filed its records)
  }
  const void *ddt, *doa, *dnp, *dcam, *dno, *dcr, *dir;
  if ((rc = stage_in(h, 0, sp->dt, (size_t)nt * T * sizeof(double), smem_kind, &ddt))) return rc;
  if ((rc = stage_in(h, 1, sp->om_acc, (size_t)nt * T * 6 * sizeof(double), smem_kind, &doa))) return rc;
  if ((rc = stage_in(h, 2, sp->n_prop, (size_t)nt * E * sizeof(int32_t), smem_kind, &dnp))) return rc;
  if ((rc = stage_in(h, 3, sp->cam, (size_t)nt * E * 7 * sizeof(double), smem_kind, &dcam))) return rc;
  if ((rc = stage_in(h, 4, sp->notch, (size_t)nt * E * sizeof(double), smem_kind, &dno))) return rc;
  if ((rc = stage_in(h, 5, sp->cam_ref, (size_t)nt * E * 6 * sizeof(double), smem_kind, &dcr))) return rc;
  if ((rc = stage_in(h, 6, sp->imu_ref, (size_t)nt * E * 6 * sizeof(double), smem_kind, &dir))) return rc;
  double* dstats = nullptr;  // the per-filter rows live on the device whenever any statistic is wanted: stats_sum is reduced
  const size_t sb = (size_t)h->N * ESKF_NSTAT * sizeof(double);  // from them after the launch (stats_partial_kernel)
  if (stats_out || stats_sum) {
    if (stats_out && mem == ESKF_MEM_DEVICE) {
      dstats = stats_out;
    } else {
      if ((rc = stage_reserve(h, 7, sb))) return rc;
      dstats = (double*)h->stage[7];
    }
  }
  // with groups (eskf_set_groups), the statistics rows are also reduced per group: the buffers are reserved before anything
  // is launched
  const GroupMap gm = group_map(h->N, sp->filter_id0, h->groups);
  const bool grp_stats = h->groups > 0 && dstats;
  if (grp_stats) {
    if ((rc = stage_reserve(h, 16, (size_t)gm.nblk * ESKF_NSTAT * sizeof(double)))) return rc;
    const double* old = h->grp_stats;
    if ((rc = grow(&h->grp_stats, &h->grp_stats_sz, (size_t)gm.G * ESKF_NSTAT * sizeof(double), fn.c_str()))) return rc;
    if (h->grp_stats != old) h->grp_stats_ok = false;  // (the last run's rows went with the old buffer)
  }
  double* dtrace = nullptr;
  const size_t tb = (size_t)h->N * (size_t)T * NX * sizeof(double);
  if (sp->trace_x) {
    if (smem_kind == ESKF_MEM_DEVICE) {
      dtrace = sp->trace_x;
    } else {
      if ((rc = stage_reserve(h, 8, tb))) return rc;
      dtrace = (double*)h->stage[8];
      // rows the kernels do not write (steps a trajectory does not execute) keep the caller's content, as in place
      CK(cudaMemcpyAsync(dtrace, sp->trace_x, tb, cudaMemcpyHostToDevice, h->stream));
    }
  }
  double* dsum = nullptr;
  if (stats_sum) dsum = (mem == ESKF_MEM_DEVICE) ? stats_sum : h->stats_sum_dev;
  const void* dcin = nullptr;
  double* dcout = nullptr;
  int64_t* kb = nullptr;  // [2][n_traj]: first step of every trajectory's epoch e0, then of its epoch e1
  if (seg) {
    if ((rc = stage_in(h, 14, carry_in, cb, mem, &dcin))) return rc;
    if (carry_out) {
      if (mem == ESKF_MEM_DEVICE) {
        dcout = carry_out;
      } else {
        if ((rc = stage_reserve(h, 15, cb))) return rc;
        dcout = (double*)h->stage[15];
      }
    }
    if ((rc = stage_reserve(h, 13, (size_t)2 * nt * sizeof(int64_t)))) return rc;
    kb = (int64_t*)h->stage[13];
    seg_base_kernel<<<(unsigned)nt, 256, 0, h->stream>>>((const int32_t*)dnp, E, T, e0, e1, (int)nt, kb);
    CK(cudaGetLastError());
    h->launches += 1;
  }
  KArgs a;
  base_args(h, a);
  a.T = T;
  a.E = whole ? E : Es;
  if (seg) {
    a.k_base = kb;
    a.e_base = e0;
    a.E_all = E;
    a.carry_in = (const double*)dcin;
    a.carry_out = dcout;
  }
  a.n_traj = (int)nt;
  a.filters_per_traj = fpt;
  a.filter_id0 = sp->filter_id0;
  a.dt = (const double*)ddt;
  a.om_acc = (const double*)doa;
  a.n_prop = (const int32_t*)dnp;
  a.cam = (const double*)dcam;
  a.notch = (const double*)dno;
  a.cam_ref = (const double*)dcr;
  a.imu_ref = (const double*)dir;
  for (int i = 0; i < 6; ++i) a.gt_dofs[i] = sp->gt_dofs[i];
  a.do_update = 1;
  a.stats_out = dstats;
  a.stats_sum = nullptr;  // (the kernels' own atomic sums are not used any more: see stats_partial_kernel)
  a.trace = dtrace;
  a.cons = (h->cons_on && E > 0) ? h->cons_rec : nullptr;
  a.drop_p = h->drop_nt > 0 ? h->drop_p : nullptr;
  a.out_p = h->out_nt > 0 ? h->out_p : nullptr;
  for (int i = 0; i < 7; ++i) a.out_std[i] = h->out_std[i];
  a.nis_gate = h->gate_on ? h->gate : nullptr;
  a.seed = sp->seed;
  a.noise_free0 = sp->noise_free_filter0;
  a.noise_mod = sp->noise_id_modulus;
  for (int i = 0; i < 6; ++i) {
    a.imu_noise[i] = sp->imu_noise_std[i];
    if (a.imu_noise[i] != 0.0) a.noise_on = 1;
  }
  for (int i = 0; i < 7; ++i) {
    a.cam_noise[i] = sp->cam_noise_std[i];
    if (a.cam_noise[i] != 0.0) a.noise_on = 1;
  }
  // ---- pre- / post-pass mode (eskf_kernel3, F = 28 and the smaller shapes alike): see PPArgs above ----
  bool pp_stats = false;
  PPArgs pp;
  memset(&pp, 0, sizeof(pp));
#if ESKF_OPT_PP
  if (kernel_of(h) == 3 && h->pp_budget > 0 && T > 0 && a.E > 0) {
    // a segment's sample buffer holds the most steps any trajectory takes in it, plus the sample the STAGER stages ahead
    int64_t Ts = T;
    if (seg && a.noise_on) {
      int64_t most = 0;
      if (smem_kind == ESKF_MEM_HOST) {  // (validated above: no negative entry, no sum past n_steps)
        for (int64_t tr = 0; tr < nt; ++tr) {
          int64_t n = 0;
          for (int64_t e = e0; e < e1; ++e) n += sp->n_prop[tr * E + e];
          most = n > most ? n : most;
        }
      } else {  // device-resident n_prop: read the segment's first steps back (the call synchronises here)
        std::vector<int64_t> hk((size_t)(2 * nt));
        CK(cudaMemcpyAsync(hk.data(), kb, hk.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        for (int64_t tr = 0; tr < nt; ++tr) most = hk[nt + tr] - hk[tr] > most ? hk[nt + tr] - hk[tr] : most;
      }
      Ts = most + 1;
    }
    pp.N = h->N;
    pp.T = Ts;
    pp.E = a.E;
    pp.k0 = kb;
    pp.T_all = T;
    pp.E_all = E;
    pp.e0 = seg ? e0 : 0;
    pp.n_traj = (int)nt;
    pp.fpt = fpt;
    pp.filter_id0 = sp->filter_id0;
    pp.seed = sp->seed;
    for (int i = 0; i < 6; ++i) pp.imu_noise[i] = a.imu_noise[i];
    for (int i = 0; i < 7; ++i) pp.cam_noise[i] = a.cam_noise[i];
    pp.noise_on = a.noise_on;
    pp.noise_free0 = a.noise_free0;
    pp.noise_mod = a.noise_mod;
    pp.per_filter = 0;
    const bool want_stats = dcr && dir && dstats;
    const size_t b_imu = a.noise_on ? (size_t)h->N * Ts * 6 * sizeof(double) : 0;
    const size_t b_meas = a.noise_on ? (size_t)h->N * a.E * 8 * sizeof(double) : 0;
    const size_t b_snap = want_stats ? (size_t)h->N * a.E * 14 * sizeof(double) : 0;
    if (b_imu + b_meas + b_snap <= h->pp_budget) {
      if (a.noise_on) {
        if ((rc = stage_reserve(h, 9, b_imu))) return rc;
        if ((rc = stage_reserve(h, 10, b_meas))) return rc;
        const int64_t n1 = h->N * Ts, n2 = h->N * a.E;
        NvtxRange nvtx_pp("eskf_run: Monte-Carlo pre-pass");
        pp_imu_kernel<<<(unsigned)((n1 + 255) / 256), 256, 0, h->stream>>>((double*)h->stage[9], a.om_acc, pp);
        pp_meas_kernel<<<(unsigned)((n2 + 255) / 256), 256, 0, h->stream>>>((double*)h->stage[10], a.cam, a.notch, pp);
        CK(cudaGetLastError());
        h->launches += 2;
        a.imu_pf = (const double*)h->stage[9];
        a.meas_pf = (const double*)h->stage[10];
      }
      if (want_stats) {
        if ((rc = stage_reserve(h, 11, b_snap))) return rc;
        a.snap = (double*)h->stage[11];
        pp_stats = true;
      }
    }
  }
#endif
  h->run_groups = gm;  // (the results of this run are reduced with its groups, whatever eskf_set_groups says later)
  h->grp_stats_ok = false;
  {
    NvtxRange nvtx_k("eskf_run: persistent kernel");
    if ((rc = launch(h, a, fpt, nt > 1))) return rc;
  }
  if (pp_stats) {
    NvtxRange nvtx_ps("eskf_run: statistics post-pass");
    const int64_t n2 = h->N * a.E;
    pp_stats1_kernel<<<(unsigned)((n2 + 127) / 128), 128, 0, h->stream>>>(a.snap, a.cam_ref, a.imu_ref, pp);
    pp_stats2_kernel<<<(unsigned)((h->N + 63) / 64), 64, 0, h->stream>>>(a.snap, dstats, nullptr, pp, a.carry_in, a.carry_out);
    CK(cudaGetLastError());
    h->launches += 2;
  }
  if (dsum) {
    const GroupMap one = group_map(h->N, 0, 0);
    if ((rc = stage_reserve(h, 12, (size_t)one.nblk * ESKF_NSTAT * sizeof(double)))) return rc;
    NvtxRange nvtx_red("eskf_run: statistics reduction");
    stats_partial_kernel<<<(unsigned)one.nblk, 256, 0, h->stream>>>(dstats, h->status, one, (double*)h->stage[12]);
    stats_final_kernel<<<1, 32, 0, h->stream>>>((const double*)h->stage[12], one, dsum);
    CK(cudaGetLastError());
    h->launches += 2;
  }
  if (grp_stats) {
    NvtxRange nvtx_red("eskf_run: statistics reduction per group");
    stats_partial_kernel<<<(unsigned)gm.nblk, 256, 0, h->stream>>>(dstats, h->status, gm, (double*)h->stage[16]);
    stats_final_kernel<<<(unsigned)((gm.G * ESKF_NSTAT + 127) / 128), 128, 0, h->stream>>>((const double*)h->stage[16], gm,
                                                                                          h->grp_stats);
    CK(cudaGetLastError());
    h->launches += 2;
    h->grp_stats_ok = true;
  }
  if (h->cons_on) {
    const int64_t E = a.E;  // (a segment's records: its epochs only)
    if (E > 0) {
      NvtxRange nvtx_c("eskf_run: consistency post-pass");
      double* nis = h->cons_out;
      double* nees = nis + h->N * E;
      double* esum = nees + h->N * E;
      double* part = esum + E * ESKF_NCONS;
      ConsArgs ca;
      ca.N = h->N;
      ca.E = E;
      for (int i = 0; i < 6; ++i) ca.gt[i] = sp->gt_dofs[i];
      ca.frozen_mask = h->model.frozen_mask & 63;
      ca.gate = nullptr;
      if (h->gate_on) {  // (the getters answer from the thresholds this run compared, whatever is set later)
        CK(cudaMemcpyAsync(h->gate + h->N, h->gate, (size_t)h->N * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
        ca.gate = h->gate + h->N;
      }
      const int64_t n2 = h->N * E;
      const GroupMap one = group_map(h->N, 0, 0);
      cons_eval_kernel<<<(unsigned)((n2 + 127) / 128), 128, 0, h->stream>>>(h->cons_rec, nis, nees, ca);
      cons_partial_kernel<<<(unsigned)(one.nblk * E), 256, 0, h->stream>>>(h->cons_rec, one, ca.frozen_mask != 63, part);
      cons_final_kernel<<<(unsigned)((E * ESKF_NCONS + 127) / 128), 128, 0, h->stream>>>(part, one, E, ESKF_NCONS, esum);
      CK(cudaGetLastError());
      h->launches += 3;
      h->cons_args = ca;  // (for the envelope of eskf_get_dof_envelope)
    }
    h->cons_E = E;
  }
  if (dtrace && smem_kind == ESKF_MEM_HOST) {
    CK(cudaMemcpyAsync(sp->trace_x, dtrace, tb, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  if (mem == ESKF_MEM_HOST && (stats_out || stats_sum || dcout)) {
    if (stats_out) CK(cudaMemcpyAsync(stats_out, dstats, sb, cudaMemcpyDeviceToHost, h->stream));
    if (stats_sum) CK(cudaMemcpyAsync(stats_sum, dsum, ESKF_NSTAT * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (dcout) CK(cudaMemcpyAsync(carry_out, dcout, cb, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  return ESKF_OK;
}

int eskf_run(eskf_t* h, const eskf_streams_t* sp, double* stats_out, double* stats_sum, int mem) {
  return run_epochs(h, sp, 0, sp ? sp->n_epochs : 0, nullptr, nullptr, stats_out, stats_sum, mem, true);
}

int eskf_run_epochs(eskf_t* h, const eskf_streams_t* sp, int64_t epoch_begin, int64_t epoch_end, const double* carry_in,
                    double* carry_out, double* stats_out, double* stats_sum, int mem) {
  return run_epochs(h, sp, epoch_begin, epoch_end, carry_in, carry_out, stats_out, stats_sum, mem, false);
}


int eskf_get_state(eskf_t* h, double* x, double* P, double* u_old, double* R_old, int32_t* status, int mem) {
  if (!h) return ESKF_EINVAL;
  CK(cudaSetDevice(h->device));
  const cudaMemcpyKind kd = (mem == ESKF_MEM_HOST) ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  const size_t n = (size_t)h->N;
  if (x) CK(cudaMemcpyAsync(x, h->x, n * NX * sizeof(double), kd, h->stream));
  if (P) CK(cudaMemcpyAsync(P, h->P, n * 576 * sizeof(double), kd, h->stream));
  if (u_old) CK(cudaMemcpyAsync(u_old, h->u, n * 6 * sizeof(double), kd, h->stream));
  if (R_old) CK(cudaMemcpyAsync(R_old, h->Ro, n * 9 * sizeof(double), kd, h->stream));
  if (status) CK(cudaMemcpyAsync(status, h->status, n * sizeof(int32_t), kd, h->stream));
  if (mem == ESKF_MEM_HOST) CK(cudaStreamSynchronize(h->stream));
  return ESKF_OK;
}

int eskf_sync(eskf_t* h) {
  if (!h) return ESKF_EINVAL;
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->stream));
  return ESKF_OK;
}

int eskf_fp64_peak(int device, void* cuda_stream, int repeats, double* tflops_out, double* ms_out) {
  if (!tflops_out || repeats < 1) return ESKF_EINVAL;
  CK(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  int smc = 0;
  CK(cudaDeviceGetAttribute(&smc, cudaDevAttrMultiProcessorCount, device));
  double* d = nullptr;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  constexpr int ILP = 16;
  const int blocks = smc * 8, threads = 256, iters = 1 << 14;
  double best = 1e30;
  auto body = [&]() -> int {  // (every resource is released below whichever call fails)
    CK(cudaMalloc(&d, 64));
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    dfma_peak_kernel<ILP><<<blocks, threads, 0, st>>>(d, iters, 1.0000001, 1e-9);  // warm-up
    for (int r = 0; r < repeats; ++r) {
      CK(cudaEventRecord(e0, st));
      dfma_peak_kernel<ILP><<<blocks, threads, 0, st>>>(d, iters, 1.0000001, 1e-9);
      CK(cudaEventRecord(e1, st));
      CK(cudaEventSynchronize(e1));
      float ms = 0.f;
      CK(cudaEventElapsedTime(&ms, e0, e1));
      if (ms < best) best = ms;
    }
    CK(cudaGetLastError());
    return ESKF_OK;
  };
  const int rc = body();
  if (e0) cudaEventDestroy(e0);
  if (e1) cudaEventDestroy(e1);
  if (d) cudaFree(d);
  if (rc) return rc;
  const double flops = 2.0 * ILP * (double)iters * blocks * threads;
  *tflops_out = flops / (best * 1e-3) * 1e-12;
  if (ms_out) *ms_out = best;
  return ESKF_OK;
}

int eskf_noise_dump(int device, void* cuda_stream, uint64_t seed, int64_t filter_id0, int64_t n_filters, int64_t step0,
                    int64_t n_steps, int kind, double* out, int mem) {
  if (!out || n_filters <= 0 || n_steps <= 0 ||
      (kind != (int)RNG_KIND_IMU && kind != (int)RNG_KIND_CAM && kind != (int)RNG_KIND_DROP && kind != (int)RNG_KIND_OUTLIER)) {
    g_err = "eskf_noise_dump: bad argument";
    return ESKF_EINVAL;
  }
  CK(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const int64_t tot = n_filters * n_steps;
  const size_t bytes = (size_t)tot * 8 * sizeof(double);
  double* d = out;
  if (mem == ESKF_MEM_HOST) CK(cudaMalloc(&d, bytes));
  auto body = [&]() -> int {
    noise_dump_kernel<<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(d, seed, filter_id0, n_filters, step0, n_steps, (uint32_t)kind);
    CK(cudaGetLastError());
    if (mem == ESKF_MEM_HOST) {
      CK(cudaMemcpyAsync(out, d, bytes, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
    }
    return ESKF_OK;
  };
  const int rc = body();
  if (mem == ESKF_MEM_HOST) cudaFree(d);
  return rc;
}

int eskf_set_meas_dropout(eskf_t* h, const double* prob, int64_t n_traj, int64_t n_epochs, int mem) {
  if (!h || (mem != ESKF_MEM_HOST && mem != ESKF_MEM_DEVICE)) {
    g_err = "eskf_set_meas_dropout: bad argument";
    return ESKF_EINVAL;
  }
  if (!prob) {
    h->drop_nt = h->drop_E = 0;
    return ESKF_OK;
  }
  if (n_traj < 1 || n_epochs < 0) {
    g_err = "eskf_set_meas_dropout: n_traj must be positive and n_epochs non-negative";
    return ESKF_EINVAL;
  }
  CK(cudaSetDevice(h->device));
  const size_t n = (size_t)n_traj * (size_t)n_epochs, bytes = n * sizeof(double);
  std::vector<double> hp;
  const double* v = prob;
  if (mem == ESKF_MEM_DEVICE && n > 0) {  // (read back to validate: a synchronous call, not a hot path)
    hp.resize(n);
    CK(cudaMemcpyAsync(hp.data(), prob, bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    v = hp.data();
  }
  for (size_t i = 0; i < n; ++i)
    if (!(v[i] >= 0.0 && v[i] <= 1.0)) {  // (false for NaN)
      g_err = "eskf_set_meas_dropout: entry " + std::to_string((unsigned long long)i) + " = " + std::to_string(v[i]) +
              " is not a probability in [0, 1]";
      return ESKF_EINVAL;
    }
  int rc = grow(&h->drop_p, &h->drop_sz, bytes > 0 ? bytes : sizeof(double), "eskf_set_meas_dropout");
  if (rc) return rc;
  if (n > 0) {  // (from the validated host values; the source may go away on return)
    CK(cudaMemcpyAsync(h->drop_p, v, bytes, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  h->drop_nt = n_traj;
  h->drop_E = n_epochs;
  return ESKF_OK;
}

int eskf_set_meas_outliers(eskf_t* h, const double* prob, int64_t n_traj, int64_t n_epochs, const double* std_, int mem) {
  if (!h || (mem != ESKF_MEM_HOST && mem != ESKF_MEM_DEVICE)) {
    g_err = "eskf_set_meas_outliers: bad argument";
    return ESKF_EINVAL;
  }
  if (!prob) {
    h->out_nt = h->out_E = 0;
    return ESKF_OK;
  }
  if (n_traj < 1 || n_epochs < 0) {
    g_err = "eskf_set_meas_outliers: n_traj must be positive and n_epochs non-negative";
    return ESKF_EINVAL;
  }
  if (!std_) {
    g_err = "eskf_set_meas_outliers: std (7 values) is required with a probability table";
    return ESKF_EINVAL;
  }
  for (int i = 0; i < 7; ++i)
    if (!(std_[i] >= 0.0 && std_[i] < INFINITY)) {  // (false for NaN)
      g_err = "eskf_set_meas_outliers: std[" + std::to_string(i) + "] = " + std::to_string(std_[i]) +
              " is not finite and non-negative";
      return ESKF_EINVAL;
    }
  CK(cudaSetDevice(h->device));
  const size_t n = (size_t)n_traj * (size_t)n_epochs, bytes = n * sizeof(double);
  std::vector<double> hp;
  const double* v = prob;
  if (mem == ESKF_MEM_DEVICE && n > 0) {  // (read back to validate: a synchronous call, not a hot path)
    hp.resize(n);
    CK(cudaMemcpyAsync(hp.data(), prob, bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    v = hp.data();
  }
  for (size_t i = 0; i < n; ++i)
    if (!(v[i] >= 0.0 && v[i] <= 1.0)) {  // (false for NaN)
      g_err = "eskf_set_meas_outliers: entry " + std::to_string((unsigned long long)i) + " = " + std::to_string(v[i]) +
              " is not a probability in [0, 1]";
      return ESKF_EINVAL;
    }
  int rc = grow(&h->out_p, &h->out_sz, bytes > 0 ? bytes : sizeof(double), "eskf_set_meas_outliers");
  if (rc) return rc;
  if (n > 0) {  // (from the validated host values; the source may go away on return)
    CK(cudaMemcpyAsync(h->out_p, v, bytes, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  h->out_nt = n_traj;
  h->out_E = n_epochs;
  for (int i = 0; i < 7; ++i) h->out_std[i] = std_[i];
  return ESKF_OK;
}

int eskf_set_innovation_gate(eskf_t* h, const double* nis_max, int64_t n, int mem) {
  if (!h || (mem != ESKF_MEM_HOST && mem != ESKF_MEM_DEVICE)) {
    g_err = "eskf_set_innovation_gate: bad argument";
    return ESKF_EINVAL;
  }
  if (!nis_max) {
    h->gate_on = false;
    return ESKF_OK;
  }
  if (n != 1 && n != h->N) {
    g_err = "eskf_set_innovation_gate: n must be 1 or n_filters";
    return ESKF_EINVAL;
  }
  CK(cudaSetDevice(h->device));
  std::vector<double> hv((size_t)n);
  if (mem == ESKF_MEM_DEVICE) {  // (read back to validate: a synchronous call, not a hot path)
    CK(cudaMemcpyAsync(hv.data(), nis_max, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  } else {
    memcpy(hv.data(), nis_max, (size_t)n * sizeof(double));
  }
  for (int64_t i = 0; i < n; ++i)
    if (!(hv[i] >= 0.0)) {  // (false for NaN; +inf passes: that filter is never gated)
      g_err = "eskf_set_innovation_gate: entry " + std::to_string((long long)i) + " = " + std::to_string(hv[i]) +
              " is not a threshold >= 0";
      return ESKF_EINVAL;
    }
  if (n == 1) hv.assign((size_t)h->N, hv[0]);
  if (!h->gate) {  // (thresholds and the snapshot of the last run's; allocated once, kept when the gate is switched off)
    void* g = nullptr;
    const cudaError_t err = cudaMalloc(&g, (size_t)h->N * 2 * sizeof(double));
    if (err != cudaSuccess) {
      cudaGetLastError();
      g_err = std::string("eskf_set_innovation_gate: ") + cudaGetErrorString(err);
      return err == cudaErrorMemoryAllocation ? ESKF_ENOMEM : ESKF_ECUDA;
    }
    h->gate = (double*)g;
  }
  CK(cudaMemcpyAsync(h->gate, hv.data(), (size_t)h->N * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->gate_on = true;
  return ESKF_OK;
}

int64_t eskf_launch_count(const eskf_t* h) { return h ? h->launches : 0; }

int eskf_set_variant(eskf_t* h, int variant) {
  if (!h || (variant != 0 && variant != 1 && variant != 3)) return ESKF_EINVAL;
  if (variant == 1 && h->cons_on) {
    g_err = "eskf_set_variant: filter consistency is on (default kernel only)";
    return ESKF_EINVAL;
  }
  h->variant = variant;
  return ESKF_OK;
}

int eskf_keep_jacobians(eskf_t* h, int on) {
  if (!h) return ESKF_EINVAL;
  CK(cudaSetDevice(h->device));
  if (on && !h->fxrec) {
    CK(cudaMalloc(&h->fxrec, (size_t)h->N * FX3_SIZE * sizeof(double)));
    CK(cudaMemsetAsync(h->fxrec, 0, (size_t)h->N * FX3_SIZE * sizeof(double), h->stream));
  } else if (!on && h->fxrec) {
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaFree(h->fxrec));
    h->fxrec = nullptr;
  }
  return ESKF_OK;
}

int eskf_get_jacobians(eskf_t* h, double* Fx, double* Fi, int mem) {
  if (!h) return ESKF_EINVAL;
  if (!h->fxrec || kernel_of(h) != 3) {
    g_err = "eskf_get_jacobians: call eskf_keep_jacobians(h, 1) before the propagation (default kernel only)";
    return ESKF_EINVAL;
  }
  CK(cudaSetDevice(h->device));
  const size_t bx = (size_t)h->N * 576 * sizeof(double), bi = (size_t)h->N * 312 * sizeof(double);
  double *dFx = Fx, *dFi = Fi;
  int rc;
  if (mem == ESKF_MEM_HOST) {
    if (Fx) {
      if ((rc = stage_reserve(h, 2, bx))) return rc;
      dFx = (double*)h->stage[2];
    }
    if (Fi) {
      if ((rc = stage_reserve(h, 3, bi))) return rc;
      dFi = (double*)h->stage[3];
    }
  }
  expand_jac_kernel<<<(unsigned)((h->N + 127) / 128), 128, 0, h->stream>>>(h->fxrec, h->N, dFx, dFi);
  CK(cudaGetLastError());
  h->launches += 1;
  if (mem == ESKF_MEM_HOST) {
    if (Fx) CK(cudaMemcpyAsync(Fx, dFx, bx, cudaMemcpyDeviceToHost, h->stream));
    if (Fi) CK(cudaMemcpyAsync(Fi, dFi, bi, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  return ESKF_OK;
}

int eskf_keep_consistency(eskf_t* h, int on) {
  if (!h) return ESKF_EINVAL;
  if (on && kernel_of(h) != 3) {
    g_err = "eskf_keep_consistency: default kernel only (eskf_set_variant(h, 1) selects the first one)";
    return ESKF_EINVAL;
  }
  CK(cudaSetDevice(h->device));
  h->cons_on = on != 0;
  h->cons_E = -1;
  if (!on && (h->cons_rec || h->cons_out)) {
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaFree(h->cons_rec));
    CK(cudaFree(h->cons_out));
    h->cons_rec = h->cons_out = nullptr;
    h->cons_rec_sz = h->cons_out_sz = 0;
  }
  return ESKF_OK;
}

int eskf_get_consistency(eskf_t* h, double* nis, double* nees, double* epoch_sum, int64_t* n_epochs, int mem) {
  if (!h) return ESKF_EINVAL;
  if (h->cons_E < 0) {
    g_err = "eskf_get_consistency: no eskf_run since eskf_keep_consistency(h, 1)";
    return ESKF_EINVAL;
  }
  const int64_t E = h->cons_E;
  if (n_epochs) *n_epochs = E;
  if (E == 0) return ESKF_OK;
  CK(cudaSetDevice(h->device));
  const cudaMemcpyKind kd = (mem == ESKF_MEM_HOST) ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  const size_t nb = (size_t)h->N * E * sizeof(double);
  const double* src = h->cons_out;
  if (nis) CK(cudaMemcpyAsync(nis, src, nb, kd, h->stream));
  if (nees) CK(cudaMemcpyAsync(nees, src + h->N * E, nb, kd, h->stream));
  if (epoch_sum) CK(cudaMemcpyAsync(epoch_sum, src + 2 * h->N * E, (size_t)E * ESKF_NCONS * sizeof(double), kd, h->stream));
  if (mem == ESKF_MEM_HOST) CK(cudaStreamSynchronize(h->stream));
  return ESKF_OK;
}

// the epochs of the last run that filed consistency records, or ESKF_EINVAL (shared by the getters of its records)
static int cons_epochs(eskf_t* h, const char* what, int mem, int64_t* n_epochs, int64_t* E) {
  if (!h || (mem != ESKF_MEM_HOST && mem != ESKF_MEM_DEVICE)) return ESKF_EINVAL;
  if (h->cons_E < 0) {
    g_err = std::string(what) + ": no eskf_run since eskf_keep_consistency(h, 1)";
    return ESKF_EINVAL;
  }
  *E = h->cons_E;
  if (n_epochs) *n_epochs = *E;
  return ESKF_OK;
}

constexpr size_t DOF_STAGE_BYTES = (size_t)64 << 20;  // staging of eskf_get_dof_history into host memory

int eskf_get_dof_history(eskf_t* h, double* dofs, double* var, int64_t* n_epochs, int mem) {
  int64_t E;
  int rc = cons_epochs(h, "eskf_get_dof_history", mem, n_epochs, &E);
  if (rc || E == 0 || (!dofs && !var)) return rc;
  CK(cudaSetDevice(h->device));
  const int64_t row = 6 * E;  // doubles per filter and array
  const unsigned gy = (unsigned)((E + HT_E - 1) / HT_E < 65535 ? (E + HT_E - 1) / HT_E : 65535);
  auto launch = [&](int64_t f0, int64_t nf, double* d, double* v) {
    dof_history_kernel<<<dim3((unsigned)((nf + HT_F - 1) / HT_F), gy), 256, 0, h->stream>>>(h->cons_rec, h->N, E, f0, nf, d, v);
    h->launches += 1;
  };
  if (mem == ESKF_MEM_DEVICE) {
    launch(0, h->N, dofs, var);
    CK(cudaGetLastError());
    return ESKF_OK;
  }
  // host destination: filter rows a chunk at a time through a staging buffer of at most DOF_STAGE_BYTES (the whole history
  // of a large batch, N * E * 96 bytes, need not fit in device memory); one row per chunk at least
  const int64_t arrays = (dofs ? 1 : 0) + (var ? 1 : 0);
  int64_t chunk = (int64_t)(DOF_STAGE_BYTES / ((size_t)arrays * row * sizeof(double)));
  chunk = chunk < 1 ? 1 : (chunk > h->N ? h->N : chunk);
  if ((rc = stage_reserve(h, 2, (size_t)(arrays * chunk * row) * sizeof(double)))) return rc;
  double* sd = dofs ? (double*)h->stage[2] : nullptr;
  double* sv = var ? (double*)h->stage[2] + (dofs ? chunk * row : 0) : nullptr;
  for (int64_t f0 = 0; f0 < h->N; f0 += chunk) {
    const int64_t nf = h->N - f0 < chunk ? h->N - f0 : chunk;
    const size_t nb = (size_t)(nf * row) * sizeof(double);
    launch(f0, nf, sd, sv);
    CK(cudaGetLastError());
    if (dofs) CK(cudaMemcpyAsync(dofs + f0 * row, sd, nb, cudaMemcpyDeviceToHost, h->stream));
    if (var) CK(cudaMemcpyAsync(var + f0 * row, sv, nb, cudaMemcpyDeviceToHost, h->stream));
  }
  CK(cudaStreamSynchronize(h->stream));
  return ESKF_OK;
}

int eskf_get_dof_envelope(eskf_t* h, double* dof_sum, int64_t* n_epochs, int mem) {
  int64_t E;
  int rc = cons_epochs(h, "eskf_get_dof_envelope", mem, n_epochs, &E);
  if (rc || E == 0 || !dof_sum) return rc;
  CK(cudaSetDevice(h->device));
  const GroupMap one = group_map(h->N, 0, 0);
  double* row = h->cons_out + 2 * h->N * E + (E + one.nblk * E) * ESKF_NCONS;  // (the layout of cons_reserve)
  double* part = row + E * ESKF_NDOFSUM;
  dof_partial_kernel<<<(unsigned)(one.nblk * E), 256, 0, h->stream>>>(h->cons_rec, h->cons_args, one, part);
  cons_final_kernel<<<(unsigned)((E * ESKF_NDOFSUM + 127) / 128), 128, 0, h->stream>>>(part, one, E, ESKF_NDOFSUM, row);
  CK(cudaGetLastError());
  h->launches += 2;
  const cudaMemcpyKind kd = (mem == ESKF_MEM_HOST) ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  CK(cudaMemcpyAsync(dof_sum, row, (size_t)E * ESKF_NDOFSUM * sizeof(double), kd, h->stream));
  if (mem == ESKF_MEM_HOST) CK(cudaStreamSynchronize(h->stream));
  return ESKF_OK;
}

int eskf_set_groups(eskf_t* h, int64_t group_size) {
  if (!h || group_size < 0) {
    g_err = "eskf_set_groups: group_size must be 0 (no groups) or positive";
    return ESKF_EINVAL;
  }
  h->groups = group_size;
  return ESKF_OK;
}

int eskf_get_group_sums(eskf_t* h, double* stats_sum, double* epoch_sum, double* dof_sum, int64_t* group0, int64_t* n_groups,
                        int64_t* n_epochs, int mem) {
  if (!h || (mem != ESKF_MEM_HOST && mem != ESKF_MEM_DEVICE)) {
    g_err = "eskf_get_group_sums: bad argument";
    return ESKF_EINVAL;
  }
  const GroupMap m = h->run_groups;
  if (stats_sum && !h->grp_stats_ok) {
    g_err = "eskf_get_group_sums: the last eskf_run produced no statistics rows or ran without groups (eskf_set_groups)";
    return ESKF_EINVAL;
  }
  int64_t E = 0;
  if (epoch_sum || dof_sum) {
    const int rc = cons_epochs(h, "eskf_get_group_sums", mem, nullptr, &E);
    if (rc) return rc;
  }
  if (group0) *group0 = m.g > 0 ? m.id0 / m.g : 0;
  if (n_groups) *n_groups = m.G;
  if (n_epochs) *n_epochs = h->cons_E > 0 ? h->cons_E : 0;
  if (!stats_sum && !((epoch_sum || dof_sum) && E > 0)) return ESKF_OK;
  CK(cudaSetDevice(h->device));
  const bool host = mem == ESKF_MEM_HOST;
  const cudaMemcpyKind kd = host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  // scratch: the partial sums of the rows asked for ([E][nblk][width]) and, for a host destination, their [G][E][width]
  const size_t wc = epoch_sum && E > 0 ? ESKF_NCONS : 0, wd = dof_sum && E > 0 ? ESKF_NDOFSUM : 0;
  const size_t pb = (size_t)E * m.nblk, ob = host ? (size_t)m.G * E : 0;
  if (pb > (size_t)INT32_MAX) {  // (one block per epoch and reduction block: the grid's x dimension)
    g_err = "eskf_get_group_sums: " + std::to_string((unsigned long long)pb) + " reduction blocks (epochs x blocks of the groups) " +
            "exceed the grid limit of 2^31 - 1: take larger groups, or fewer epochs per segment";
    return ESKF_EINVAL;
  }
  int rc = grow(&h->grp_buf, &h->grp_buf_sz, ((pb + ob) * (wc + wd)) * sizeof(double), "eskf_get_group_sums");
  if (rc) return rc;
  double* part = h->grp_buf;
  double* stage = part + pb * (wc + wd);
  if (stats_sum) CK(cudaMemcpyAsync(stats_sum, h->grp_stats, (size_t)m.G * ESKF_NSTAT * sizeof(double), kd, h->stream));
  if (wc) {
    double* out = host ? stage : epoch_sum;
    cons_partial_kernel<<<(unsigned)pb, 256, 0, h->stream>>>(h->cons_rec, m, h->cons_args.frozen_mask != 63, part);
    cons_final_kernel<<<(unsigned)((m.G * E * ESKF_NCONS + 127) / 128), 128, 0, h->stream>>>(part, m, E, ESKF_NCONS, out);
    CK(cudaGetLastError());
    h->launches += 2;
    if (host) CK(cudaMemcpyAsync(epoch_sum, out, ob * ESKF_NCONS * sizeof(double), kd, h->stream));
  }
  if (wd) {
    double* p = part + pb * wc;
    double* out = host ? stage + ob * wc : dof_sum;
    dof_partial_kernel<<<(unsigned)pb, 256, 0, h->stream>>>(h->cons_rec, h->cons_args, m, p);
    cons_final_kernel<<<(unsigned)((m.G * E * ESKF_NDOFSUM + 127) / 128), 128, 0, h->stream>>>(p, m, E, ESKF_NDOFSUM, out);
    CK(cudaGetLastError());
    h->launches += 2;
    if (host) CK(cudaMemcpyAsync(dof_sum, out, ob * ESKF_NDOFSUM * sizeof(double), kd, h->stream));
  }
  if (host) CK(cudaStreamSynchronize(h->stream));
  return ESKF_OK;
}

int eskf_set_prepass_budget(eskf_t* h, int64_t bytes) {
  if (!h || bytes < 0) return ESKF_EINVAL;
  h->pp_budget = (size_t)bytes;
  return ESKF_OK;
}

int eskf_set_tuning(eskf_t* h, int filters_per_cta) {
  if (!h || filters_per_cta < 0) return ESKF_EINVAL;
  h->fpc = filters_per_cta;
  return ESKF_OK;
}

}  // extern "C"
