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

// eskf_noise_dump: the standard normals of (filter, step, kind), exactly as the persistent kernels draw them
__global__ void noise_dump_kernel(double* out, uint64_t seed, int64_t filter_id0, int64_t n_filters, int64_t step0, int64_t n_steps,
                                  uint32_t kind) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_filters * n_steps) return;
  const int64_t f = i / n_steps, k = i - f * n_steps;
  double z[8];
  normal8(seed, (uint64_t)(filter_id0 + f), (uint64_t)(step0 + k), kind, z);
  for (int j = 0; j < 8; ++j) out[i * 8 + j] = z[j];
}

// ---- pre- / post-pass of eskf_run (KArgs::imu_pf / meas_pf / snap) -------------------------------------------------
// The Monte-Carlo generator and the Euler angles of Filter.calculate_update_mse are throughput work with no dependence on
// the filters' recursion.  Inside the persistent kernel they ran on ONE warp of every CTA and slowed the whole CTA through
// that warp's sub-partition (12 % of the launch at 4096 filters, profiles/r02_*); as separate, fully parallel kernels they
// cost a few per cent of that.  Same generator, same operations in the same order: the results are bit-identical
// (tests/test_gpu_noise.py compares both paths).
struct PPArgs {
  int64_t N, T, E;
  int n_traj;
  int64_t fpt, filter_id0;
  uint64_t seed;
  double imu_noise[6], cam_noise[7];
  int noise_on, noise_free0, noise_mod, per_filter;
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
  const double* src = p.per_filter ? om_acc + (f * p.T + j) * 6 : om_acc + (traj * p.T + j) * 6;
  double u[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) u[i] = src[i];
  if (noisy) {
    double z[8];
    normal8(p.seed, (uint64_t)gid, (uint64_t)j, RNG_KIND_IMU, z);
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
  const int64_t mrow = traj * p.E + e;
  double cam[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) cam[i] = camm[mrow * 7 + i];
  double notch = notchm[mrow];
  if (noisy) {
    double z[8];
    normal8(p.seed, (uint64_t)gid, (uint64_t)e, RNG_KIND_CAM, z);
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
// the epochs) of the statistics, and their contribution to stats_sum.
__global__ void pp_stats1_kernel(double* __restrict__ snap, const double* __restrict__ cam_ref,
                                 const double* __restrict__ imu_ref, const PPArgs p) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= p.E * p.N) return;
  const int64_t e = idx / p.N, f = idx - e * p.N;
  int64_t traj, gid;
  bool noisy;
  pp_ids(p, f, traj, gid, noisy);
  double* xs = snap + idx * 14;
  const double* ir = imu_ref + (traj * p.E + e) * 6;
  const double* cr = cam_ref + (traj * p.E + e) * 6;
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

__global__ void pp_stats2_kernel(const double* __restrict__ snap, double* stats_out, double* stats_sum, const PPArgs p) {
  const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  double r7 = 0.0, r8 = 0.0;
  if (f < p.N) {
    double mseA_last = 0.0, mseA_sum = 0.0, mseB_last = 0.0, mseB_sum = 0.0;
    for (int64_t e = 0; e < p.E; ++e) {
      const double* xs = snap + (e * p.N + f) * 14;
      mseA_last = xs[0];
      mseA_sum += mseA_last;
      mseB_last = xs[1];
      mseB_sum += mseB_last;
    }
    r7 = (mseA_last + mseB_last) / 12.0;
    r8 = (mseA_sum + mseB_sum) / 12.0;
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

// ---- reduction of the statistics rows (the vector a multi-GPU launcher all-reduces) -----------------------------------
// stats_sum of eskf_run, from the per-filter rows, DETERMINISTICALLY (fixed summation tree, no atomics: the same bits
// whatever the CTA scheduling) and MASKED: a filter that diverged (non-finite row) or whose status word is set would
// otherwise turn the reduced vector of a million healthy filters into NaN.  [0:10] sums over the healthy filters,
// [10] filters with a non-zero status, [11] healthy filters (the divisor of every mean), [12] non-finite filters.
constexpr int RED_ROWS = 4096;  // rows per block
__global__ void stats_partial_kernel(const double* __restrict__ rows, const int32_t* __restrict__ status, int64_t n,
                                     double* __restrict__ partial) {
  __shared__ double sh[256][13];
  const int64_t r0 = (int64_t)blockIdx.x * RED_ROWS;
  double acc[13];
#pragma unroll
  for (int i = 0; i < 13; ++i) acc[i] = 0.0;
  for (int64_t r = r0 + threadIdx.x; r < r0 + RED_ROWS && r < n; r += 256) {
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
__global__ void stats_final_kernel(const double* __restrict__ partial, int64_t nblk, double* __restrict__ out) {
  if (threadIdx.x >= ESKF_NSTAT) return;
  double a = 0.0;
  for (int64_t b = 0; b < nblk; ++b) a += partial[b * ESKF_NSTAT + threadIdx.x];
  out[threadIdx.x] = a;
}

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
constexpr int N_STAGE = 13;  // 0..8: arguments / results of the calls; 9..11: pre- / post-pass buffers of eskf_run; 12: partial sums
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

int eskf_run(eskf_t* h, const eskf_streams_t* sp, double* stats_out, double* stats_sum, int mem) {
  NvtxRange nvtx_("eskf_run");
  if (!h || !sp || !sp->dt || !sp->om_acc || !sp->n_prop || !sp->cam || !sp->notch || sp->n_traj < 1) {
    g_err = "eskf_run: bad argument";
    return ESKF_EINVAL;
  }
  CK(cudaSetDevice(h->device));
  const int smem_kind = sp->mem;
  const int64_t T = sp->n_steps, E = sp->n_epochs, nt = sp->n_traj;
  const int64_t fpt = nt > 1 ? sp->filters_per_traj : h->N;
  if (T < 0 || E < 0 || sp->filter_id0 < 0) {
    g_err = "eskf_run: n_steps, n_epochs and filter_id0 must not be negative";
    return ESKF_EINVAL;
  }
  if (nt > 1) {
    // the kernels pick the trajectory of a filter from its GLOBAL id: (filter_id0 + f) / filters_per_traj
    if (fpt <= 0 || (sp->filter_id0 % fpt) != 0) {
      g_err = "eskf_run: filter_id0 must be a multiple of filters_per_traj (a shard starts at a trajectory boundary)";
      return ESKF_EINVAL;
    }
    if (sp->filter_id0 + h->N > nt * fpt) {
      g_err = "eskf_run: filter_id0 + n_filters exceeds n_traj * filters_per_traj (the streams of " +
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
          g_err = "eskf_run: negative n_prop entry";
          return ESKF_EINVAL;
        }
        tot += np_;
      }
      if (tot > T) {
        g_err = "eskf_run: sum(n_prop) = " + std::to_string((long long)tot) + " exceeds n_steps = " + std::to_string((long long)T);
        return ESKF_EINVAL;
      }
    }
  }
  const void *ddt, *doa, *dnp, *dcam, *dno, *dcr, *dir;
  int rc;
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
  KArgs a;
  base_args(h, a);
  a.T = T;
  a.E = E;
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
  if (kernel_of(h) == 3 && h->pp_budget > 0 && T > 0 && E > 0) {
    pp.N = h->N;
    pp.T = T;
    pp.E = E;
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
    const size_t b_imu = a.noise_on ? (size_t)h->N * T * 6 * sizeof(double) : 0;
    const size_t b_meas = a.noise_on ? (size_t)h->N * E * 8 * sizeof(double) : 0;
    const size_t b_snap = want_stats ? (size_t)h->N * E * 14 * sizeof(double) : 0;
    if (b_imu + b_meas + b_snap <= h->pp_budget) {
      if (a.noise_on) {
        if ((rc = stage_reserve(h, 9, b_imu))) return rc;
        if ((rc = stage_reserve(h, 10, b_meas))) return rc;
        const int64_t n1 = h->N * T, n2 = h->N * E;
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
  {
    NvtxRange nvtx_k("eskf_run: persistent kernel");
    if ((rc = launch(h, a, fpt, nt > 1))) return rc;
  }
  if (pp_stats) {
    NvtxRange nvtx_ps("eskf_run: statistics post-pass");
    const int64_t n2 = h->N * E;
    pp_stats1_kernel<<<(unsigned)((n2 + 127) / 128), 128, 0, h->stream>>>(a.snap, a.cam_ref, a.imu_ref, pp);
    pp_stats2_kernel<<<(unsigned)((h->N + 63) / 64), 64, 0, h->stream>>>(a.snap, dstats, nullptr, pp);
    CK(cudaGetLastError());
    h->launches += 2;
  }
  if (dsum) {
    const int64_t nblk = (h->N + RED_ROWS - 1) / RED_ROWS;
    if ((rc = stage_reserve(h, 12, (size_t)nblk * ESKF_NSTAT * sizeof(double)))) return rc;
    NvtxRange nvtx_red("eskf_run: statistics reduction");
    stats_partial_kernel<<<(unsigned)nblk, 256, 0, h->stream>>>(dstats, h->status, h->N, (double*)h->stage[12]);
    stats_final_kernel<<<1, 32, 0, h->stream>>>((const double*)h->stage[12], nblk, dsum);
    CK(cudaGetLastError());
    h->launches += 2;
  }
  if (dtrace && smem_kind == ESKF_MEM_HOST) {
    CK(cudaMemcpyAsync(sp->trace_x, dtrace, tb, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  if (mem == ESKF_MEM_HOST && (stats_out || stats_sum)) {
    if (stats_out) CK(cudaMemcpyAsync(stats_out, dstats, sb, cudaMemcpyDeviceToHost, h->stream));
    if (stats_sum) CK(cudaMemcpyAsync(stats_sum, dsum, ESKF_NSTAT * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  return ESKF_OK;
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
  if (!out || n_filters <= 0 || n_steps <= 0 || (kind != (int)RNG_KIND_IMU && kind != (int)RNG_KIND_CAM)) {
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

int64_t eskf_launch_count(const eskf_t* h) { return h ? h->launches : 0; }

int eskf_set_variant(eskf_t* h, int variant) {
  if (!h || (variant != 0 && variant != 1 && variant != 3)) return ESKF_EINVAL;
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
