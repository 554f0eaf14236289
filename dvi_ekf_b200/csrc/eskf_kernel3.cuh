// eskf_kernel3: the warp-specialised persistent VI-ESKF kernel for sm_100a, covariance resident in
// registers for the propagation AND the camera update.
//
// One CTA owns F filters for a whole launch (a whole trajectory in eskf_run).  Warps are roles:
//   warp 0  IMU     lane = filter: p, v, q of the nominal state (Filter._predict_nominal, Filter.py:232-247,
//                   equations.py:72-86) and R_WB_old (Filter.py:227)
//   warp 1  CAMERA  lane = filter: p_cam, q_cam (equations.py:88-98), rows 18:21 of Fx (Filter.py:283-321, second half of
//                   the Jacobian work: it waits for JACOB's probe kinematics of the step at a two-warp barrier),
//                   the measurement residual (Filter.py:363-375), status word
//   warp 3  JACOB   lane = filter: dofs, notch chain, probe forward kinematics (Probe.py:470-480) and the
//                   Jacobian blocks of Fx / Fi (Filter._predict_error, Filter.py:249-342)
//   warp 2  STAGER  lane = filter: stages the IMU sample stream (dt, om, acc) into a 4-slot shared-memory
//                   ring two steps ahead and adds the Monte-Carlo noise (Philox4x32-10 + single-precision
//                   Box-Muller on the SFU); stages the camera measurement of the epoch
//                   (Imu.eval_expr_single / Filter.propagate_imu, Imu.py:141-196, Filter.py:187-217;
//                   VisualTraj.at_index, VisualTrajectory.py:120-134)
//   warps 4.. COVARIANCE  eight lanes per filter, lane g keeps columns 3g..3g+2 of the 24x24 covariance in
//                   REGISTERS (72 doubles) for the whole launch -- see eskf_cov3.cuh for the algebra:
//                   one propagation = two local sparse products around ONE transposition through shared
//                   memory (72 STS.64 + 36 LDS.128 per lane: all 24 rows, see eskf_cov3.cuh); the camera update (gain, Joseph form,
//                   reset) works on the same register tile and exchanges only S, K, K R, W(:,h) (7-wide
//                   records) between the eight lanes of a filter, with warp-level synchronisation.
// Inside an epoch (the IMU steps between two camera frames) the scalar roles and the covariance warps are
// decoupled: the scalar roles synchronise among themselves (named barrier, 128 threads) and hand the Jacobian
// record of a step to the covariance warps through a two-slot full / empty mbarrier pipeline, so they run up
// to two steps ahead and every covariance warp free-runs at its own pace (their shared-memory and FP64 phases
// drift apart instead of colliding at a CTA barrier per step).  All roles meet at CTA barriers only around
// the camera update.  Records exchanged through shared memory are double buffered:
//   RING[4]  samples (slot (k+1)&3 = new sample of step k, slot k&3 = old sample)       STAGER -> IMU, CAMERA, JACOB
//   RO/RW/V[2] R_WB_old, R_WB and v at the start of step k (slot k&1)                   IMU -> CAMERA, JACOB
//   PK[2]    probe kinematics + notch, notch' at the start of step k (slot k&1)         JACOB -> CAMERA
//   FXB[2]   Jacobian blocks of the step (fx3 layout, [pair][filter] so that the writer's STS.128 and the
//            readers' broadcast LDS.128 are both conflict free)                         JACOB -> COVARIANCE
// Register budget by role (setmaxnreg): scalar warps shrink to REG_S, covariance warps grow to REG_C
// (eskf_launch3.cu).
#pragma once
#include <type_traits>
#include "eskf_cov3.cuh"
#include "eskf_kernel.cuh"

// profiling experiment switches (python -m dvi_ekf_b200.build --exp=...): time one side of the kernel alone
#ifdef ESKF_EXP_NO_SCALAR
#define ESKF3_SCALAR_ON(it) ((it) < 2)  // scalar roles only fill both record slots once per epoch
#else
#define ESKF3_SCALAR_ON(it) true
#endif
#ifdef ESKF_EXP_NO_COV
#define ESKF3_COV_ON false
#else
#define ESKF3_COV_ON true
#endif

// optimisation switches of round 2 (each A/B-timed on the GPU, profiles/r02_*): 0 / 1
#ifndef ESKF_OPT_LATEACQ
#define ESKF_OPT_LATEACQ 0  // producers compute the step first and acquire the record slot only to store
#endif
#ifndef ESKF_OPT_SYNCW
#define ESKF_OPT_SYNCW 1  // full-mask __syncwarp in the step loop of the covariance role
#endif
#ifndef ESKF_OPT_STATS_U0
#define ESKF_OPT_STATS_U0 0  // Filter.calculate_update_mse evaluated during U0 / U1 of the next update instead of step 2
#endif
#ifndef ESKF_OPT_PP
#define ESKF_OPT_PP 1  // per-filter streams from a pre-pass and statistics in a post-pass (KArgs::imu_pf / meas_pf / snap)
#endif
#ifndef ESKF_OPT_JACDUMP
#define ESKF_OPT_JACDUMP 1  // the producers file the Jacobian record of the last step of a launch (KArgs::fx_dump)
#endif
#ifndef ESKF_OPT_TMA
#define ESKF_OPT_TMA 0  // sample stream staged by cp.async.bulk chunks (see CH3_STEPS)
#endif
#ifndef ESKF_OPT_H1S
#define ESKF_OPT_H1S 0  // rows 18:21 of Fx formed by the STAGER role when it is idle (pre-pass noise / noise-free runs)
#endif
#ifndef ESKF_OPT_COLD
#define ESKF_OPT_COLD 0  // covariance role: re-orientation and IMU-noise code outside the step loop
#endif
#ifndef ESKF_OPT_ADDR
#define ESKF_OPT_ADDR 0  // covariance role: buffer offsets kept in (laundered) registers instead of being re-derived every step
#endif
#ifndef ESKF_OPT_STREAM
#define ESKF_OPT_STREAM 1  // pass 2 streams the transposed tile from the buffer (reload fused into the pass)
#endif

namespace eskf {

// ESKF_EXP_TIMING (profiling build): cycles per phase, accumulated by lane 0 of every warp into a global table
// [CTA][warp][16], read back with eskf_debug_timing() (eskf_launch3.cu).  Not part of the product build.
#if defined(ESKF_EXP_TIMING) && defined(ESKF_F)
#define TIMING_SLOTS 16
static __device__ long long g_eskf_timing[256 * 12 * TIMING_SLOTS];  // (one table per CTA-shape translation unit)
struct PhaseTimer {  // (fire-and-forget global reductions: one register pair of state, no accumulators in registers)
  long long t;
  __device__ __forceinline__ PhaseTimer() { t = clock64(); }
  __device__ __forceinline__ void mark(int slot) {
    const long long n = clock64();
    if ((threadIdx.x & 31) == 0 && blockIdx.x < 256)
      atomicAdd(reinterpret_cast<unsigned long long*>(g_eskf_timing) + (blockIdx.x * 12 + (threadIdx.x >> 5)) * TIMING_SLOTS + slot,
                (unsigned long long)(n - t));
    t = n;
  }
  __device__ __forceinline__ void flush() {}
};
#define PT_DECL() PhaseTimer pt_
#define PT_MARK(s) pt_.mark(s)
#define PT_FLUSH() pt_.flush()
#else
#define PT_DECL()
#define PT_MARK(s)
#define PT_FLUSH()
#endif

// ESKF_EXP_JITTER (race-hunting build, tests/test_gpu_jitter.py): every synchronisation point of the role pipelines -- record
// slot acquire / publish / wait / release, the barrier of the scalar roles, the JACOB -> CAMERA hand-over, the CTA barriers
// around the camera update -- is preceded and followed by a pseudo-random, warp-uniform delay (hash of the jitter seed, CTA,
// warp and a per-warp counter; 0 .. g_eskf_jitter_ns nanoseconds), which moves the roles against each other by whole steps.
// A result that depends on the timing of the roles -- a missing ordering -- shows up as a difference against the plain build
// (compute-sanitizer's racecheck is closed on this pool).  Not part of the product build.
#if defined(ESKF_EXP_JITTER) && defined(ESKF_F)
static __device__ unsigned int g_eskf_jitter_seed = 0, g_eskf_jitter_ns = 0;
struct Jitter3 {
  unsigned int n;
  __device__ __forceinline__ void operator()() {
    if (g_eskf_jitter_ns == 0) return;
    unsigned int h = g_eskf_jitter_seed * 0x9E3779B9u ^ (blockIdx.x * 0x85EBCA6Bu) ^ ((threadIdx.x >> 5) * 0xC2B2AE35u) ^ (++n * 0x27D4EB2Fu);
    h ^= h >> 15;
    h *= 0x2C1B3C6Du;
    h ^= h >> 12;
    h *= 0x297A2D39u;
    h ^= h >> 15;
    if (h & 3u) return;  // three of four points pass undisturbed: delays come in bursts, not as a uniform slow-down
    __nanosleep((h >> 2) % g_eskf_jitter_ns);
  }
};
#define JIT() jit_()
#define JIT_DECL() Jitter3 jit_{0}
#else
#define JIT()
#define JIT_DECL()
#endif

// Filter.calculate_update_mse is evaluated by the STAGER role at this step of the NEXT epoch (see role3_stage)
constexpr int STATS_IT3 = 2;

// ESKF_OPT_TMA: the IMU sample stream (dt[T], om_acc[T,6]: shared by the filters of a trajectory) is staged through shared
// memory in chunks of CH3_STEPS samples by bulk-asynchronous copies (cp.async.bulk, completion on an mbarrier), two chunks in
// flight; the STAGER lanes then read the samples of a step from shared memory instead of seven broadcast global loads
constexpr int CH3_STEPS = 16;

constexpr int RS3 = 26;          // row stride of the transposition buffer: even (16-byte rows) and
constexpr int TB3_STRIDE = 632;  // 24*26 + 8; = 8 (mod 16) doubles => conflict-free STS.64 / LDS.128 (DESIGN.md)

// scalar exchange block, element-major: element j of filter f at SX[j * F + f]
constexpr int SX3_RING = 0;     // 4 x 8: om(3) acc(3) dt pad
constexpr int SX3_RO = 32;      // 2 x 9
constexpr int SX3_RW = 50;      // 2 x 9
constexpr int SX3_V = 68;       // 2 x 3
constexpr int PK3 = 20;         // PK slot: p(3) R(9) z6(3) notch notch' dofs[3..5]
constexpr int SX3_PK = 74;      // 2 x PK3
constexpr int SX3_MEAS = 114;   // 8: cam pos(3) quat(4) notch
constexpr int SX3_RES = 122;    // 7: measurement residual            CAMERA -> COVARIANCE
constexpr int SX3_OK = 129;     // residual valid
constexpr int SX3_DELTA = 130;  // 24: error state K res              COVARIANCE -> scalar roles
constexpr int SX3_OK2 = 154;    // update applied
constexpr int SX3_QD = 155;     // 13: diag(Q)
constexpr int SX3_RD = 168;     // 7: diag(R)
constexpr int SX3_ST = 175;     // 12: statistics partials (epilogue)
constexpr int SX3_TR = 187;     // 24: trigonometry cache of the probe kinematics (JACOB writes, CAMERA reads)
constexpr int SX3_SIZE = 212;

template <int F>
struct Lay3 {
  static constexpr int TB = 0;                  // [F][TB3_STRIDE]  (u3 records of a warp's four filters during the update)
  static constexpr int SX = F * TB3_STRIDE;     // [SX3_SIZE][F]
  static constexpr int FXB = SX + SX3_SIZE * F; // [2][FX3_NPAIR][F] d2
  static constexpr int MBAR = FXB + 2 * FX3_NPAIR * 2 * F;   // 4 mbarriers: full[2], empty[2]
#if ESKF_OPT_TMA
  static constexpr int CHBAR = MBAR + 4;                     // 2 mbarriers: chunk[2] of the staged sample stream
  // [2][CHW]: a chunk of the shared stream (om_acc, 6 per step, then dt, 1 per step) or, in pre-pass mode, the block of one
  // step of the per-filter stream (6 per filter)
  static constexpr int CHW = (CH3_STEPS * 7 > F * 6) ? CH3_STEPS * 7 : F * 6;
  static constexpr int CHUNK = CHBAR + 2;
  static constexpr int TOTAL = CHUNK + 2 * CHW;              // doubles
  static_assert((CHUNK % 2) == 0, "16-byte alignment of the bulk-copy destination");
#else
  static constexpr int TOTAL = MBAR + 4;                     // doubles
#endif
  static_assert((SX % 2) == 0 && (FXB % 2) == 0, "16-byte alignment");
  static_assert(4 * U3_SIZE <= 4 * TB3_STRIDE, "update records must fit the transposition buffers of a warp");
};

template <int N>
__device__ __forceinline__ void reg_inc3() {
  if constexpr (N > 0) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;\n" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void reg_dec3() {
  if constexpr (N > 0) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" ::"n"(N));
}

// ---- mbarrier pipeline of the Jacobian records (producers: IMU + JACOB warps, consumers: covariance warps) ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// one arrival for the whole warp: its lanes' shared-memory traffic is ordered by __syncwarp, lane 0 releases it
__device__ __forceinline__ void mbar_arrive_warp(uint64_t* bar) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0)
    asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.shared::cta.b64 st, [%0];\n}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// the same for a warp that is AHEAD of its partner (producers waiting for a free slot): back off between polls
// so that the polling does not take issue slots from the covariance warps of the sub-partition
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
  for (;;) {
    uint32_t done;
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (done) break;
    __nanosleep(64);
  }
}
// bulk-asynchronous copy global -> shared of `bytes` (multiple of 16, both addresses 16-byte aligned), completion counted
// in bytes on the mbarrier (TMA unit: UBLKCP in SASS)
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n}" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
// step kk uses record slot kk & 1; its full barrier completes phase kk >> 1, and the slot is free for step kk
// once the consumers of step kk - 2 have arrived on its empty barrier (phase (kk - 2) >> 1)
__device__ __forceinline__ void fx_slot_acquire(uint64_t* mbar, int64_t kk) {  // producers, before writing
#ifndef ESKF_EXP_NO_PIPE  // (profiling experiment: no coupling between the roles)
  if (kk >= 2) mbar_wait_relaxed(mbar + 2 + (kk & 1), (uint32_t)(((kk - 2) >> 1) & 1));
#endif
}
__device__ __forceinline__ void fx_slot_publish(uint64_t* mbar, int64_t kk) { mbar_arrive_warp(mbar + (kk & 1)); }
__device__ __forceinline__ void fx_slot_wait(uint64_t* mbar, int64_t kk) {  // consumers, before reading
#ifndef ESKF_EXP_NO_PIPE
  mbar_wait(mbar + (kk & 1), (uint32_t)((kk >> 1) & 1));
#endif
}
__device__ __forceinline__ void fx_slot_release(uint64_t* mbar, int64_t kk) { mbar_arrive_warp(mbar + 2 + (kk & 1)); }
// barrier of the four scalar-role warps
__device__ __forceinline__ void scalar_barrier() { asm volatile("bar.sync 1, 128;" ::: "memory"); }
// JACOB -> CAMERA inside a step: the probe kinematics of the step are published (JACOB does not wait)
__device__ __forceinline__ void pk_ready_arrive() { asm volatile("bar.arrive 2, 64;" ::: "memory"); }
__device__ __forceinline__ void pk_ready_wait() { asm volatile("bar.sync 2, 64;" ::: "memory"); }

struct Ctx3;
__device__ __forceinline__ int epoch_steps3(const KArgs& a, const Ctx3& c, int64_t e, int64_t k);

struct Ctx3 {
  double* smem;
  int64_t f0;      // first local filter of the CTA
  int nf;          // filters of this CTA that exist
  int64_t gid0;    // global id of the CTA's first filter
  int64_t traj;
  const int32_t* n_prop;
  const double* dtp;
  uint64_t* mbar;  // full[2], empty[2]
};

// IMU steps of epoch e, k steps into the stream: n_prop[e] clamped to what is left of the stream, so that inconsistent
// DEVICE-resident streams (sum(n_prop) > n_steps; host streams are validated by eskf_run) can never index past the sample
// stream, the ring or the trace rows
__device__ __forceinline__ int epoch_steps3(const KArgs& a, const Ctx3& c, int64_t e, int64_t k) {
  if (!c.n_prop) return (int)a.T;
  const int64_t left = a.T - k;
  const int64_t n = c.n_prop[e];
  return (int)(n < 0 ? 0 : (n > left ? left : n));
}

// the last IMU step the CTA's trajectory executes in this launch (-1: none), where export mode files the Jacobian record:
// the epochs' steps as epoch_steps3 counts them, which may add up to less than n_steps (stacked trajectories share the
// stream length, each has its own n_prop)
__device__ __forceinline__ int64_t last_step3(const KArgs& a, const Ctx3& c) {
  int64_t k = 0;
  for (int64_t e = 0; e < a.E; ++e) k += epoch_steps3(a, c, e, k);
  return k - 1;
}

// ---------------------------------------------------------------------------------------------
// cooperative, coalesced tile store (all threads of the CTA)
template <int F, int NTHR>
__device__ __forceinline__ void store_tiles3(const KArgs& a, const Ctx3& c, int tid) {
  const double* sT = c.smem + Lay3<F>::TB;
  for (int idx = tid; idx < c.nf * 576; idx += NTHR) {
    const int f = idx / 576, r = idx - f * 576;
    const int i = r / 24, j = r - i * 24;
    a.P[(c.f0 + f) * 576 + r] = sT[f * TB3_STRIDE + i * RS3 + j];
  }
}

// statistics rows (Filter.calculate_dof_metric / update_mse) assembled by warp 0 from the partials the
// scalar roles left in SX3_ST: [0] mseA_last [1] mseA_sum [2] mseB_last [3] mseB_sum [4] n_upd [5] status
// [6..11] (dofs - gt)^2
template <int F>
__device__ __forceinline__ void write_stats3(const KArgs& a, const Ctx3& c, int lane) {
  if (!(a.stats_out || a.stats_sum)) return;
  const double* st = c.smem + Lay3<F>::SX + SX3_ST * F + lane;
  double row[ESKF_NSTAT];
#pragma unroll
  for (int i = 0; i < ESKF_NSTAT; ++i) row[i] = 0.0;
  if (lane < c.nf) {
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      row[i] = st[(6 + i) * F];
      acc += row[i];
    }
    row[6] = acc / 6.0;
    row[7] = (st[0] + st[2 * F]) / 12.0;
    row[8] = (st[F] + st[3 * F]) / 12.0;
    row[9] = st[4 * F];
    row[10] = st[5 * F];
    row[11] = 1.0;
    if (a.stats_out) {
#pragma unroll
      for (int i = 0; i < ESKF_NSTAT; ++i) a.stats_out[(c.f0 + lane) * ESKF_NSTAT + i] = row[i];
    }
  }
  if (a.stats_sum) {
#pragma unroll
    for (int i = 0; i < ESKF_NSTAT; ++i) {
      double v = row[i];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) atomicAdd(a.stats_sum + i, v);
    }
  }
}

// trace mode (eskf_streams_t.trace_x): every role files its part of the FilterTraj row
__device__ __forceinline__ void trace_pvq(double* r, const double* p, const double* v, const double* q) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    r[i] = p[i];
    r[3 + i] = v[i];
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) r[6 + i] = q[i];
}
__device__ __forceinline__ void trace_cam(double* r, const double* pc, const double* qc) {
#pragma unroll
  for (int i = 0; i < 3; ++i) r[19 + i] = pc[i];
#pragma unroll
  for (int i = 0; i < 4; ++i) r[22 + i] = qc[i];
}
__device__ __forceinline__ void trace_dofs(double* r, const double* dofs, const double* notch) {
#pragma unroll
  for (int i = 0; i < 6; ++i) r[10 + i] = dofs[i];
#pragma unroll
  for (int i = 0; i < 3; ++i) r[16 + i] = notch[i];
}

// Which scalar role forms rows 18:21 of Fx (Filter._cam_error_jacobian: C1, C2).  The CAMERA warp shares its sub-partition
// with two covariance warps and was the busiest scalar role there (~680 instructions per step against the 2 x ~700 of the
// covariance warps), while the STAGER warp of ITS sub-partition has next to nothing to do once the Monte-Carlo generator runs
// in the pre-pass (or the run is noise free): then it takes this block.  With the generator inside the kernel (batches whose
// pre-pass buffers do not fit) and in export mode the CAMERA warp keeps it.  Same function, same inputs: bit-identical.
template <bool EX>
__device__ __forceinline__ bool h1_by_stager(const KArgs& a) {
#if ESKF_OPT_H1S
  return !EX && (a.imu_pf != nullptr || !a.noise_on);
#else
  return false;
#endif
}

// ---------------------------------------------------------------------------------------------
// role 0: IMU nominal state
template <int F, int NTHR, bool EX>
__device__ __forceinline__ void role3_imu(const KArgs& a, const Ctx3& c, int lane) {
  using L = Lay3<F>;
  const bool act = lane < c.nf;
  double* sx = c.smem + L::SX + lane;
  d2* fxb = reinterpret_cast<d2*>(c.smem + L::FXB) + lane;  // pair j2 of slot s at fxb[(s * FX3_NPAIR + j2) * F]
  double p[3], v[3], q[4], Rwb[9], Rold[9];
  if (act) {
    const double* xg = a.x + (c.f0 + lane) * NX;
    const double* rg = a.Ro + (c.f0 + lane) * 9;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      p[i] = xg[i];
      v[i] = xg[3 + i];
      sx[(SX3_V + i) * F] = v[i];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) q[i] = xg[6 + i];
    quat_to_rot(q, Rwb);  // R_WB of the first step is rot(q); R_WB_old may be stale (quirk Q8)
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      Rold[i] = rg[i];
      sx[(SX3_RO + i) * F] = Rold[i];
      sx[(SX3_RW + i) * F] = Rwb[i];
    }
  }
  __syncthreads();  // prologue
  PT_DECL();
  JIT_DECL();
  const int64_t k_jac = EX ? last_step3(a, c) : -1;  // (export mode: the step whose Jacobian record is filed)
  int64_t k = 0;
  for (int64_t e = 0; e < a.E; ++e) {
    const int n = epoch_steps3(a, c, e, k);
    for (int it = 0; it < n; ++it) {
      const int64_t kk = k + it;
#if !ESKF_OPT_LATEACQ
      PT_MARK(1);
      JIT();
      fx_slot_acquire(c.mbar, kk);  // the covariance warps are done with the record of step kk - 2
      JIT();
      PT_MARK(0);
#endif
#if ESKF_OPT_LATEACQ
      double fx[FX3_SIZE];  // (only the entries of rows 3:9 are ever touched: registers)
#endif
      if (act && ESKF3_SCALAR_ON(it)) {
        const double* uo = sx + (SX3_RING + 8 * (int)(kk & 3)) * F;
        const double* un = sx + (SX3_RING + 8 * (int)((kk + 1) & 3)) * F;
        double om_old[3], acc_old[3], om[3], acc[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          om_old[i] = uo[i * F];
          acc_old[i] = uo[(3 + i) * F];
          om[i] = un[i * F];
          acc[i] = un[(3 + i) * F];
        }
        const double dt = un[6 * F];
#if ESKF_OPT_LATEACQ
        jac_rows_ab(Rold, dt, om_old, acc_old, fx);
#else
        {  // rows 3:9 of Fx (Filter.py:253-255) from the buffered R_WB_old / om_old / acc_old: this role has them
          double fx[FX3_SIZE];
          jac_rows_ab(Rold, dt, om_old, acc_old, fx);
          d2* dst = fxb + ((int)(kk & 1) * FX3_NPAIR) * F;
#pragma unroll
          for (int j = FX3_AB / 2; j < FX3_MAIN / 2; ++j) dst[j * F] = d2{fx[2 * j], fx[2 * j + 1]};
#if ESKF_OPT_JACDUMP
          if (EX && a.fx_dump && kk == k_jac) {  // Filter.Fx / Filter.Fi read-out: the record of the last step of the launch
            double* fd = a.fx_dump + (c.f0 + lane) * FX3_SIZE;
#pragma unroll
            for (int j = FX3_AB; j < FX3_MAIN; ++j) fd[j] = fx[j];
          }
#endif
        }
#endif
        imu_nominal_step(p, v, q, Rwb, dt, om_old, acc_old, om, acc, Rold);
        if (EX && a.trace) trace_pvq(a.trace + ((c.f0 + lane) * a.T + kk) * NX, p, v, q);
        const int s = (int)((kk + 1) & 1);
#pragma unroll
        for (int i = 0; i < 9; ++i) {
          Rwb[i] = Rold[i];
          sx[(SX3_RO + 9 * s + i) * F] = Rold[i];
          sx[(SX3_RW + 9 * s + i) * F] = Rold[i];
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) sx[(SX3_V + 3 * s + i) * F] = v[i];
      }
#if ESKF_OPT_LATEACQ
      // The nominal step never reads the covariance: it is computed while the covariance warps still work on the record
      // that occupies this slot (step kk - 2); only the store of the rows waits for the slot.
      PT_MARK(1);
      JIT();
      fx_slot_acquire(c.mbar, kk);
      JIT();
      PT_MARK(0);
      if (act && ESKF3_SCALAR_ON(it)) {
        d2* dst = fxb + ((int)(kk & 1) * FX3_NPAIR) * F;
#pragma unroll
        for (int j = FX3_AB / 2; j < FX3_MAIN / 2; ++j) dst[j * F] = d2{fx[2 * j], fx[2 * j + 1]};
      }
#endif
      JIT();
      fx_slot_publish(c.mbar, kk);  // rows 3:9 of the record of step kk are in place
      JIT();
      PT_MARK(1);
      JIT();
      scalar_barrier();
      JIT();
      PT_MARK(2);
    }
    k += n;
    if (!a.do_update) continue;
    JIT();
    scalar_barrier();  // (an update-only launch has no step barrier: the measurement must be staged before U0)
    JIT();
    PT_MARK(2);
    PT_MARK(5);
    JIT();
    __syncthreads();  // U0 | U1
    JIT();
    JIT();
    __syncthreads();  // U1 | U2
    JIT();
    PT_MARK(3);
    if (act) {
      if (sx[SX3_OK2 * F] != 0.0) {  // state (+) error state, IMU part (state.py:46-53,116-121)
        const double th[3] = {sx[(SX3_DELTA + 6) * F], sx[(SX3_DELTA + 7) * F], sx[(SX3_DELTA + 8) * F]};
        double dq[4], qn[4];
        quat_about_axis(sqrt(th[0] * th[0] + th[1] * th[1] + th[2] * th[2]), th, dq);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          p[i] += sx[(SX3_DELTA + i) * F];
          v[i] += sx[(SX3_DELTA + 3 + i) * F];
        }
        quat_mul(q, dq, qn);
#pragma unroll
        for (int i = 0; i < 4; ++i) q[i] = qn[i];
        quat_to_rot(q, Rwb);  // R_WB of the next step; R_WB_old keeps the pre-update value (quirk Q8)
        if (EX && a.trace && k > 0) trace_pvq(a.trace + ((c.f0 + lane) * a.T + k - 1) * NX, p, v, q);  // FilterTraj.append_updated_states
        const int s = (int)(k & 1);
#pragma unroll
        for (int i = 0; i < 9; ++i) sx[(SX3_RW + 9 * s + i) * F] = Rwb[i];
#pragma unroll
        for (int i = 0; i < 3; ++i) sx[(SX3_V + 3 * s + i) * F] = v[i];
      }
#if ESKF_OPT_PP
      if (a.snap) {  // statistics in the post-pass (eskf_pp.cuh): snapshot of this update
        double* xs = a.snap + (e * a.N + c.f0 + lane) * 14;
#pragma unroll
        for (int i = 0; i < 3; ++i) xs[i] = v[i];
#pragma unroll
        for (int i = 0; i < 4; ++i) xs[3 + i] = q[i];
      } else
#endif
      if (a.cam_ref && a.imu_ref) {  // statistics of this update are evaluated later, off the critical path
        double* xs = a.x + (c.f0 + lane) * NX;
#pragma unroll
        for (int i = 0; i < 3; ++i) xs[3 + i] = v[i];
#pragma unroll
        for (int i = 0; i < 4; ++i) xs[6 + i] = q[i];
      }
    }
    PT_MARK(6);
    JIT();
    scalar_barrier();  // U2 of the scalar roles done (the covariance warps do not wait: see role3_cov)
    JIT();
    PT_MARK(2);
  }
  // ---- write back ----
  if (act) {
    double* xg = a.x + (c.f0 + lane) * NX;
    double* ug = a.u + (c.f0 + lane) * 6;
    double* rg = a.Ro + (c.f0 + lane) * 9;
    const double* uo = sx + (SX3_RING + 8 * (int)(k & 3)) * F;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      xg[i] = p[i];
      xg[3 + i] = v[i];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) xg[6 + i] = q[i];
#pragma unroll
    for (int i = 0; i < 6; ++i) ug[i] = uo[i * F];
#pragma unroll
    for (int i = 0; i < 9; ++i) rg[i] = Rold[i];
  }
  __syncthreads();  // tiles dumped, statistics partials written
  store_tiles3<F, NTHR>(a, c, threadIdx.x);
  write_stats3<F>(a, c, lane);
}

// ---------------------------------------------------------------------------------------------
// role 1: camera nominal state + measurement residual
template <int F, int NTHR, bool EX>
__device__ __forceinline__ void role3_cam(const KArgs& a, const Ctx3& c, int lane) {
  using L = Lay3<F>;
  const bool act = lane < c.nf;
  double* sx = c.smem + L::SX + lane;
  d2* fxb = reinterpret_cast<d2*>(c.smem + L::FXB) + lane;  // pair j2 of slot s at fxb[(s * FX3_NPAIR + j2) * F]
  const TRView<F> trv{sx + SX3_TR * F};
  double pc[3], qc[4], sig_om[3] = {0, 0, 0};
  double n_upd = 0.0;
  int32_t st = 0;
  if (act) {
    const double* xg = a.x + (c.f0 + lane) * NX;
    const double* pg = a.par + (c.f0 + lane) * PAR_STRIDE;
#pragma unroll
    for (int i = 0; i < 3; ++i) sig_om[i] = pg[PAR_SIGOM + i];
#pragma unroll
    for (int i = 0; i < 3; ++i) pc[i] = xg[19 + i];
#pragma unroll
    for (int i = 0; i < 4; ++i) qc[i] = xg[22 + i];
    st = a.status[c.f0 + lane];
  }
  __syncthreads();  // prologue
  PT_DECL();
  JIT_DECL();
  const bool h1s = h1_by_stager<EX>(a);  // rows 18:21 of Fx are the STAGER's work in this launch (see role3_stage)
  const int64_t k_jac = EX ? last_step3(a, c) : -1;
  int64_t k = 0;
  for (int64_t e = 0; e < a.E; ++e) {
    const int n = epoch_steps3(a, c, e, k);
    for (int it = 0; it < n; ++it) {
      const int64_t kk = k + it;
#if !ESKF_OPT_LATEACQ
      PT_MARK(1);
      JIT();
      if (!h1s) fx_slot_acquire(c.mbar, kk);  // the covariance warps are done with the record of step kk - 2
      JIT();
      PT_MARK(0);
#endif
      if (act && ESKF3_SCALAR_ON(it)) {
        const double* uo = sx + (SX3_RING + 8 * (int)(kk & 3)) * F;
        const double* un = sx + (SX3_RING + 8 * (int)((kk + 1) & 3)) * F;
        const int s = (int)(kk & 1);
        double om_old[3], om[3], vpre[3], Rwb[9], pkp[3], pkR[9], pkz[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          om_old[i] = uo[i * F];
          om[i] = un[i * F];
          vpre[i] = sx[(SX3_V + 3 * s + i) * F];
          pkp[i] = sx[(SX3_PK + PK3 * s + i) * F];
          pkz[i] = sx[(SX3_PK + PK3 * s + 12 + i) * F];
        }
#pragma unroll
        for (int i = 0; i < 9; ++i) {
          Rwb[i] = sx[(SX3_RW + 9 * s + i) * F];
          pkR[i] = sx[(SX3_PK + PK3 * s + 3 + i) * F];
        }
        const double dt = un[6 * F];
        const double notch_d = sx[(SX3_PK + PK3 * s + 16) * F];
        cam_nominal_step(pc, qc, vpre, Rwb, dt, om_old, om, pkp, pkR, pkz, notch_d);
        if (EX && a.trace) trace_cam(a.trace + ((c.f0 + lane) * a.T + kk) * NX, pc, qc);
      }
      PT_MARK(1);
      JIT();
      if (!h1s) pk_ready_wait();
      JIT();
      PT_MARK(4);  // JACOB has published the probe kinematics of the post-predict (dofs, notch): PK slot sn, TR
#if ESKF_OPT_LATEACQ
      double fx[FX3_SIZE];  // (only the entries of rows 18:21 are ever touched: registers)
#endif
      if (!h1s && act && ESKF3_SCALAR_ON(it)) {
        // rows 18:21 of Fx (Filter._cam_error_jacobian, Filter.py:270-342): the half of the Jacobian work that
        // only needs the probe kinematics, R_WB_old and om_old -- taken off JACOB, the longest scalar role
        const double* uo = sx + (SX3_RING + 8 * (int)(kk & 3)) * F;
        const double dt = sx[(SX3_RING + 8 * (int)((kk + 1) & 3) + 6) * F];
        const int s = (int)(kk & 1), sn = s ^ 1;
        const PKView<F> pk{sx + (SX3_PK + PK3 * sn) * F};
        double om_old[3], Ro[9], dofs[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          om_old[i] = uo[i * F];
          dofs[3 + i] = sx[(SX3_PK + PK3 * sn + 17 + i) * F];
        }
#pragma unroll
        for (int i = 0; i < 9; ++i) Ro[i] = sx[(SX3_RO + 9 * s + i) * F];
#if ESKF_OPT_LATEACQ
        jac_rows_h1(a.model, dofs, pk, trv, Ro, dt, om_old, sig_om, fx);
      }
      PT_MARK(1);
      JIT();
      fx_slot_acquire(c.mbar, kk);  // (see role3_imu: only the store waits for the slot)
      JIT();
      PT_MARK(0);
      if (act && ESKF3_SCALAR_ON(it)) {
#else
        double fx[FX3_SIZE];
        jac_rows_h1(a.model, dofs, pk, trv, Ro, dt, om_old, sig_om, fx);
#endif
        d2* dst = fxb + ((int)(kk & 1) * FX3_NPAIR) * F;
#pragma unroll
        for (int j = FX3_H1 / 2; j < FX3_AB / 2; ++j) dst[j * F] = d2{fx[2 * j], fx[2 * j + 1]};
#if ESKF_OPT_JACDUMP
        if (EX && a.fx_dump && kk == k_jac) {
          double* fd = a.fx_dump + (c.f0 + lane) * FX3_SIZE;
#pragma unroll
          for (int j = FX3_H1; j < FX3_AB; ++j) fd[j] = fx[j];
        }
#endif
      }
      JIT();
      if (!h1s) fx_slot_publish(c.mbar, kk);  // rows 18:21 of the record of step kk are in place
      JIT();
      PT_MARK(1);
      JIT();
      scalar_barrier();
      JIT();
      PT_MARK(2);
    }
    k += n;
    if (!a.do_update) continue;
    JIT();
    scalar_barrier();  // (an update-only launch has no step barrier: the measurement must be staged before U0)
    JIT();
    PT_MARK(2);
    // ---- U0: residual (Filter.py:363-375) ----
    if (lane < F) {
      bool ok = false;
      if (act) {
        double cam[7], res[7];
#pragma unroll
        for (int i = 0; i < 7; ++i) cam[i] = sx[(SX3_MEAS + i) * F];
        const double notch_meas = sx[(SX3_MEAS + 7) * F];
        const double notch0 = sx[(SX3_PK + PK3 * (int)(k & 1) + 15) * F];
        Nominal s;  // only pc, qc, notch[0] are read by update_residual
#pragma unroll
        for (int i = 0; i < 3; ++i) s.pc[i] = pc[i];
#pragma unroll
        for (int i = 0; i < 4; ++i) s.qc[i] = qc[i];
        s.notch[0] = notch0;
        ok = update_residual(s, cam, cam + 3, notch_meas, res);
#pragma unroll
        for (int i = 0; i < 7; ++i) sx[(SX3_RES + i) * F] = res[i];
        if (!ok) st |= ESKF_STATUS_ASIN_DOMAIN;
      }
      sx[SX3_OK * F] = ok ? 1.0 : 0.0;
    }
    PT_MARK(5);
    PT_MARK(5);
    JIT();
    __syncthreads();  // U0 | U1
    JIT();
    JIT();
    __syncthreads();  // U1 | U2
    JIT();
    PT_MARK(3);
    PT_MARK(3);
    if (act) {
      if (sx[SX3_OK2 * F] != 0.0) {  // camera part of the injection, incl. the dqc axis slip (quirk Q4, state.py:124)
        const double th[3] = {sx[(SX3_DELTA + 6) * F], sx[(SX3_DELTA + 7) * F], sx[(SX3_DELTA + 8) * F]};
        const double thc[3] = {sx[(SX3_DELTA + 21) * F], sx[(SX3_DELTA + 22) * F], sx[(SX3_DELTA + 23) * F]};
        double dqc[4], qn[4];
        quat_about_axis(sqrt(thc[0] * thc[0] + thc[1] * thc[1] + thc[2] * thc[2]), th, dqc);
#pragma unroll
        for (int i = 0; i < 3; ++i) pc[i] += sx[(SX3_DELTA + 18 + i) * F];
        quat_mul(qc, dqc, qn);
#pragma unroll
        for (int i = 0; i < 4; ++i) qc[i] = qn[i];
        n_upd += 1.0;
        if (EX && a.trace && k > 0) trace_cam(a.trace + ((c.f0 + lane) * a.T + k - 1) * NX, pc, qc);
      } else {
        st |= ESKF_STATUS_UPDATE_SKIPPED;
      }
#if ESKF_OPT_PP
      if (a.snap) {
        double* xs = a.snap + (e * a.N + c.f0 + lane) * 14;
#pragma unroll
        for (int i = 0; i < 3; ++i) xs[7 + i] = pc[i];
#pragma unroll
        for (int i = 0; i < 4; ++i) xs[10 + i] = qc[i];
      } else
#endif
      if (a.cam_ref && a.imu_ref) {  // statistics of this update are evaluated later, off the critical path
        double* xs = a.x + (c.f0 + lane) * NX;
#pragma unroll
        for (int i = 0; i < 3; ++i) xs[19 + i] = pc[i];
#pragma unroll
        for (int i = 0; i < 4; ++i) xs[22 + i] = qc[i];
      }
    }
    PT_MARK(6);
    JIT();
    scalar_barrier();  // U2 of the scalar roles done (the covariance warps do not wait: see role3_cov)
    JIT();
    PT_MARK(2);
  }
  if (act) {
    double* xg = a.x + (c.f0 + lane) * NX;
#pragma unroll
    for (int i = 0; i < 3; ++i) xg[19 + i] = pc[i];
#pragma unroll
    for (int i = 0; i < 4; ++i) xg[22 + i] = qc[i];
    a.status[c.f0 + lane] = st;
    sx[(SX3_ST + 4) * F] = n_upd;
    sx[(SX3_ST + 5) * F] = (double)st;
  }
  __syncthreads();
  store_tiles3<F, NTHR>(a, c, threadIdx.x);
}

// ---------------------------------------------------------------------------------------------
// role 2: dofs / notch, probe kinematics, Jacobian blocks (rows 21:24 and the noise rows; rows 3:9 come from the IMU
// role, rows 18:21 from the CAMERA role).
// The probe kinematics and their trigonometry cache live in shared memory (PK slots, TR), not in registers.
template <int F, int NTHR, bool EX>
__device__ __forceinline__ void role3_jac(const KArgs& a, const Ctx3& c, int lane) {
  using L = Lay3<F>;
  const bool act = lane < c.nf;
  double* sx = c.smem + L::SX + lane;
  d2* fxb = reinterpret_cast<d2*>(c.smem + L::FXB) + lane;  // pair j2 of slot s at fxb[(s * FX3_NPAIR + j2) * F]
  const TRView<F> trv{sx + SX3_TR * F};
  auto pkv = [&](int s) { return PKView<F>{sx + (SX3_PK + PK3 * s) * F}; };
  auto put_notch = [&](int s, const double* notch, const double* dofs) {  // the scalars that go with a PK slot
    sx[(SX3_PK + PK3 * s + 15) * F] = notch[0];
    sx[(SX3_PK + PK3 * s + 16) * F] = notch[1];
#pragma unroll
    for (int i = 3; i < 6; ++i) sx[(SX3_PK + PK3 * s + 14 + i) * F] = dofs[i];
  };
  double dofs[6], notch[3], sig_om[3] = {0, 0, 0};
  bool imu_q = false;
  if (act) {
    const double* xg = a.x + (c.f0 + lane) * NX;
    const double* pg = a.par + (c.f0 + lane) * PAR_STRIDE;
#pragma unroll
    for (int i = 0; i < 6; ++i) dofs[i] = xg[10 + i];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      notch[i] = xg[16 + i];
      sig_om[i] = pg[PAR_SIGOM + i];
    }
    imu_q = (pg[PAR_QD + 3] != 0.0) || (pg[PAR_QD + 4] != 0.0) || (pg[PAR_QD + 5] != 0.0);
#pragma unroll
    for (int j = 0; j < 4; ++j) trv.ang(j) = __longlong_as_double(0x7ff8000000000000LL);  // nothing cached yet
    probe_update_v(a.model, dofs, notch, pkv(0), trv);
    put_notch(0, notch, dofs);
  }
  __syncthreads();  // prologue
  PT_DECL();
  JIT_DECL();
  const int64_t k_jac = EX ? last_step3(a, c) : -1;
  int64_t k = 0;
  for (int64_t e = 0; e < a.E; ++e) {
    const int n = epoch_steps3(a, c, e, k);
    for (int it = 0; it < n; ++it) {
      const int64_t kk = k + it;
#if !ESKF_OPT_LATEACQ
      PT_MARK(1);
      JIT();
      fx_slot_acquire(c.mbar, kk);  // the covariance warps are done with the record of step kk - 2
      JIT();
      PT_MARK(0);
#endif
      if (act && ESKF3_SCALAR_ON(it)) {
        const double dt = sx[(SX3_RING + 8 * (int)((kk + 1) & 3) + 6) * F];
        const int s = (int)(kk & 1), sn = s ^ 1;
        // post-predict (dofs, notch) and their probe kinematics -> PK slot of the next step
        const PKView<F> pk = pkv(sn);
        if (dofs_notch_step(a.model, dofs, notch, dt)) {
          probe_update_v(a.model, dofs, notch, pk, trv);
        } else {
          const PKView<F> po = pkv(s);
#pragma unroll
          for (int i = 0; i < PK_SIZE; ++i) pk.b[i * F] = po.b[i * F];
        }
        put_notch(sn, notch, dofs);
        if (EX && a.trace) trace_dofs(a.trace + ((c.f0 + lane) * a.T + kk) * NX, dofs, notch);
      }
      JIT();
      pk_ready_arrive();  // the CAMERA warp takes rows 18:21 from here
      JIT();
#if ESKF_OPT_LATEACQ
      double fx[FX3_SIZE];  // (rows 21:24 and, with IMU noise in Q, the noise rows: registers)
      if (act && ESKF3_SCALAR_ON(it)) {
        const double* uo = sx + (SX3_RING + 8 * (int)(kk & 3)) * F;
        const double dt = sx[(SX3_RING + 8 * (int)((kk + 1) & 3) + 6) * F];
        const int s = (int)(kk & 1), sn = s ^ 1;
        const PKView<F> pk = pkv(sn);
        double om_old[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) om_old[i] = uo[i * F];
        jac_rows_h2(a.model, notch[1], pk, trv, dt, om_old, sig_om, fx);
        if (imu_q) {
          double Ro[9];
#pragma unroll
          for (int i = 0; i < 9; ++i) Ro[i] = sx[(SX3_RO + 9 * s + i) * F];
          jac_rows_noise(pk, Ro, dt, fx);
        }
      }
      PT_MARK(1);
      JIT();
      fx_slot_acquire(c.mbar, kk);  // (see role3_imu: only the store waits for the slot)
      JIT();
      PT_MARK(0);
      if (act && ESKF3_SCALAR_ON(it)) {
        d2* dst = fxb + ((int)(kk & 1) * FX3_NPAIR) * F;
#pragma unroll
        for (int j = 0; j < FX3_H1 / 2; ++j) dst[j * F] = d2{fx[2 * j], fx[2 * j + 1]};
        if (imu_q) {
#pragma unroll
          for (int j = FX3_NPAIR_MAIN; j < FX3_NPAIR; ++j) dst[j * F] = d2{fx[2 * j], fx[2 * j + 1]};
        }
      }
#else
      if (act && ESKF3_SCALAR_ON(it)) {
        const double* uo = sx + (SX3_RING + 8 * (int)(kk & 3)) * F;
        const double dt = sx[(SX3_RING + 8 * (int)((kk + 1) & 3) + 6) * F];
        const int s = (int)(kk & 1), sn = s ^ 1;
        const PKView<F> pk = pkv(sn);
        double om_old[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) om_old[i] = uo[i * F];
        d2* dst = fxb + ((int)(kk & 1) * FX3_NPAIR) * F;
        double fx[FX3_SIZE];
        jac_rows_h2(a.model, notch[1], pk, trv, dt, om_old, sig_om, fx);
#pragma unroll
        for (int j = 0; j < FX3_H1 / 2; ++j) dst[j * F] = d2{fx[2 * j], fx[2 * j + 1]};
        if (imu_q) {
          double Ro[9];
#pragma unroll
          for (int i = 0; i < 9; ++i) Ro[i] = sx[(SX3_RO + 9 * s + i) * F];
          jac_rows_noise(pk, Ro, dt, fx);
#pragma unroll
          for (int j = FX3_NPAIR_MAIN; j < FX3_NPAIR; ++j) dst[j * F] = d2{fx[2 * j], fx[2 * j + 1]};
        }
#if ESKF_OPT_JACDUMP
        if (EX && a.fx_dump && kk == k_jac) {  // (rows 18:24 of Fi are part of the read-out whether or not Q uses them)
          double* fd = a.fx_dump + (c.f0 + lane) * FX3_SIZE;
          if (!imu_q) {
            double Ro[9];
#pragma unroll
            for (int i = 0; i < 9; ++i) Ro[i] = sx[(SX3_RO + 9 * s + i) * F];
            jac_rows_noise(pk, Ro, dt, fx);
          }
#pragma unroll
          for (int j = 0; j < FX3_H1; ++j) fd[j] = fx[j];
#pragma unroll
          for (int j = FX3_MAIN; j < FX3_SIZE; ++j) fd[j] = fx[j];
        }
#endif
      }
#endif
      JIT();
      fx_slot_publish(c.mbar, kk);  // dt, rows 21:24 (and the noise rows) of the record of step kk are in place
      JIT();
      PT_MARK(1);
      JIT();
      scalar_barrier();
      JIT();
      PT_MARK(2);
    }
    k += n;
    if (!a.do_update) continue;
    JIT();
    scalar_barrier();  // (an update-only launch has no step barrier: the measurement must be staged before U0)
    JIT();
    PT_MARK(2);
    PT_MARK(5);
    JIT();
    __syncthreads();  // U0 | U1
    JIT();
    JIT();
    __syncthreads();  // U1 | U2
    JIT();
    PT_MARK(3);
    if (act) {
      if (sx[SX3_OK2 * F] != 0.0) {
#pragma unroll
        for (int i = 0; i < 6; ++i)
          if (!((a.model.frozen_mask >> i) & 1)) dofs[i] += sx[(SX3_DELTA + 9 + i) * F];  // Filter.py:377-379
#pragma unroll
        for (int i = 0; i < 3; ++i) notch[i] += sx[(SX3_DELTA + 15 + i) * F];
        probe_update_v(a.model, dofs, notch, pkv((int)(k & 1)), trv);
        put_notch((int)(k & 1), notch, dofs);
        if (EX && a.trace && k > 0) trace_dofs(a.trace + ((c.f0 + lane) * a.T + k - 1) * NX, dofs, notch);
      }
    }
    PT_MARK(6);
    JIT();
    scalar_barrier();  // U2 of the scalar roles done (the covariance warps do not wait: see role3_cov)
    JIT();
    PT_MARK(2);
  }
  if (act) {
    double* xg = a.x + (c.f0 + lane) * NX;
#pragma unroll
    for (int i = 0; i < 6; ++i) xg[10 + i] = dofs[i];
#pragma unroll
    for (int i = 0; i < 3; ++i) xg[16 + i] = notch[i];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      const double d = dofs[i] - a.gt_dofs[i];
      sx[(SX3_ST + 6 + i) * F] = d * d;
    }
  }
  __syncthreads();
  store_tiles3<F, NTHR>(a, c, threadIdx.x);
}

// ---------------------------------------------------------------------------------------------
// role 3: sample-stream stager + Monte-Carlo noise
template <int F, int NTHR, bool EX>
__device__ __forceinline__ void role3_stage(const KArgs& a, const Ctx3& c, int lane) {
  using L = Lay3<F>;
  const bool act = lane < c.nf;
  double* sx = c.smem + L::SX + lane;
  const bool h1s = h1_by_stager<EX>(a);
  d2* fxb = reinterpret_cast<d2*>(c.smem + L::FXB) + lane;  // pair j2 of slot s at fxb[(s * FX3_NPAIR + j2) * F]
  const TRView<F> trv{sx + SX3_TR * F};
  double sig_om[3] = {0, 0, 0};
  if (h1s && act) {
    const double* pg = a.par + (c.f0 + lane) * PAR_STRIDE;
#pragma unroll
    for (int i = 0; i < 3; ++i) sig_om[i] = pg[PAR_SIGOM + i];
  }
  // rows 18:21 of the Jacobian record of step kk (what role3_cam does otherwise)
  auto rows_h1 = [&](int64_t kk) {
    const double* uo = sx + (SX3_RING + 8 * (int)(kk & 3)) * F;
    const double dt = sx[(SX3_RING + 8 * (int)((kk + 1) & 3) + 6) * F];
    const int s = (int)(kk & 1), sn = s ^ 1;
    const PKView<F> pk{sx + (SX3_PK + PK3 * sn) * F};
    double om_old[3], Ro[9], dofs[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      om_old[i] = uo[i * F];
      dofs[3 + i] = sx[(SX3_PK + PK3 * sn + 17 + i) * F];
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) Ro[i] = sx[(SX3_RO + 9 * s + i) * F];
    double fx[FX3_SIZE];
    jac_rows_h1(a.model, dofs, pk, trv, Ro, dt, om_old, sig_om, fx);
    d2* dst = fxb + ((int)(kk & 1) * FX3_NPAIR) * F;
#pragma unroll
    for (int j = FX3_H1 / 2; j < FX3_AB / 2; ++j) dst[j * F] = d2{fx[2 * j], fx[2 * j + 1]};
  };
  const int64_t gid = a.noise_mod > 0 ? (c.gid0 + lane) % a.noise_mod : c.gid0 + lane;  // id the noise is keyed by
#if ESKF_OPT_PP
  // pre-pass mode: the (noisy) samples of every filter were prepared by eskf_pp_streams_kernel -- same generator, same sums
  const bool noisy = a.noise_on && !(a.noise_free0 && gid == 0) && !a.imu_pf;
  const double* oap = a.imu_pf ? a.imu_pf + (c.f0 + lane) * 6
                      : a.om_acc ? (a.stream_per_filter ? a.om_acc + (c.f0 + lane) * a.T * 6 : a.om_acc + c.traj * a.T * 6)
                                 : nullptr;
  const int64_t oas = a.imu_pf ? a.N * 6 : 6;  // doubles between consecutive samples of this lane's stream
#else
  const bool noisy = a.noise_on && !(a.noise_free0 && gid == 0);
  const double* oap =
      a.om_acc ? (a.stream_per_filter ? a.om_acc + (c.f0 + lane) * a.T * 6 : a.om_acc + c.traj * a.T * 6) : nullptr;
  const int64_t oas = 6;
#endif
#if ESKF_OPT_TMA
  // Bulk-asynchronous staging (TMA unit, cp.async.bulk completed on an mbarrier), two buffers in flight; lane 0 issues.
  //  * shared stream (one trajectory per CTA, no pre-pass): chunk ch = samples [ch CH3_STEPS, (ch + 1) CH3_STEPS) of om_acc
  //    and dt -> buffer ch & 1; complete chunks only (the tail goes the plain way); needs 16-byte aligned chunk sources.
  //  * pre-pass mode (imu_pf [T][N][6]): the samples of the CTA's filters for ONE step are contiguous (nf x 48 bytes):
  //    one copy per step -> buffer j & 1, issued one step ahead.
  // A buffer is re-filled only after every lane of this warp has passed the scalar barrier that follows its last read.
  uint64_t* chbar = reinterpret_cast<uint64_t*>(c.smem + L::CHBAR);
  double* chunk = c.smem + L::CHUNK;
  const double* oa0 = a.om_acc ? a.om_acc + c.traj * a.T * 6 : nullptr;
  const bool tma_pf = a.imu_pf != nullptr && c.nf > 0;
  const bool tma = !tma_pf && oa0 && c.dtp && !a.stream_per_filter && ((reinterpret_cast<uintptr_t>(oa0) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(c.dtp) & 15) == 0);
  const int64_t n_chunks = tma ? a.T / CH3_STEPS : 0;
  auto issue_chunk = [&](int64_t ch) {
    if (lane == 0 && ch < n_chunks) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      double* buf = chunk + (int)(ch & 1) * L::CHW;
      mbar_expect_tx(chbar + (ch & 1), CH3_STEPS * 56);
      bulk_g2s(buf, oa0 + ch * CH3_STEPS * 6, CH3_STEPS * 48, chbar + (ch & 1));
      bulk_g2s(buf + CH3_STEPS * 6, c.dtp + ch * CH3_STEPS, CH3_STEPS * 8, chbar + (ch & 1));
    }
  };
  auto issue_step = [&](int64_t j) {
    if (lane == 0 && tma_pf && j < a.T) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      const uint32_t bytes = (uint32_t)c.nf * 48u;
      mbar_expect_tx(chbar + (j & 1), bytes);
      bulk_g2s(chunk + (int)(j & 1) * L::CHW, a.imu_pf + (j * a.N + c.f0) * 6, bytes, chbar + (j & 1));
    }
  };
#endif
  auto stage_sample = [&](int64_t j) {  // sample of step j -> ring slot (j + 1) & 3
    double* dst = sx + (SX3_RING + 8 * (int)((j + 1) & 3)) * F;
    double u[6];
#if ESKF_OPT_TMA
    double dtj;
    const int64_t ch = j / CH3_STEPS;
    if (tma_pf) {
      issue_step(j + 1);  // its buffer held step j - 1: every lane is done with it
      mbar_wait(chbar + (j & 1), (uint32_t)((j >> 1) & 1));
      const double* buf = chunk + (int)(j & 1) * L::CHW + lane * 6;
#pragma unroll
      for (int i = 0; i < 6; ++i) u[i] = buf[i];
      dtj = c.dtp[j];
    } else if (ch < n_chunks) {
      const int jj = (int)(j - ch * CH3_STEPS);
      if (jj == 0) issue_chunk(ch + 1);  // its buffer held chunk ch - 1: every lane is done with it
      mbar_wait(chbar + (ch & 1), (uint32_t)((ch >> 1) & 1));
      const double* buf = chunk + (int)(ch & 1) * L::CHW;
#pragma unroll
      for (int i = 0; i < 6; ++i) u[i] = buf[jj * 6 + i];
      dtj = buf[CH3_STEPS * 6 + jj];
    } else {
#pragma unroll
      for (int i = 0; i < 6; ++i) u[i] = oap[j * oas + i];
      dtj = c.dtp[j];
    }
#elif ESKF_OPT_PP
#pragma unroll
    for (int i = 0; i < 6; ++i) u[i] = oap[j * oas + i];
#else
#pragma unroll
    for (int i = 0; i < 6; ++i) u[i] = oap[j * 6 + i];
#endif
    if (noisy) {
      double z[8];
      normal8(a.seed, (uint64_t)gid, (uint64_t)j, RNG_KIND_IMU, z);
#pragma unroll
      for (int i = 0; i < 6; ++i) u[i] += a.imu_noise[i] * z[i];
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) dst[i * F] = u[i];
#if ESKF_OPT_TMA
    dst[6 * F] = dtj;
#else
    dst[6 * F] = c.dtp[j];
#endif
  };
  auto stage_meas = [&](int64_t e) {
#if ESKF_OPT_PP
    if (a.meas_pf) {
      const double* m = a.meas_pf + (e * a.N + c.f0 + lane) * 8;
#pragma unroll
      for (int i = 0; i < 8; ++i) sx[(SX3_MEAS + i) * F] = m[i];
      return;
    }
#endif
    const int64_t mrow = a.meas_per_filter ? (c.f0 + lane) : (c.traj * a.E + e);
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
#pragma unroll
    for (int i = 0; i < 7; ++i) sx[(SX3_MEAS + i) * F] = cam[i];
    sx[(SX3_MEAS + 7) * F] = notch;
  };
  // Filter.calculate_update_mse (Filter.py:397-418) for both halves.  The Euler angles cost two atan2 and an asin per
  // half (~3,500 dependent cycles); evaluated by the IMU / CAMERA roles at the update they delayed the first Jacobian
  // record of the next epoch, for which every covariance warp is waiting (0.32 ms of 5.9 per launch).  Instead those
  // roles park (v, q) / (p_cam, q_cam) in the filter's own row of the state array -- its final destination: the launch
  // read the row in the prologue and rewrites it in the epilogue; ordered by the scalar barrier after U2 -- and this role,
  // which has slack, evaluates the error terms at step STATS_IT3 of the next epoch (or before the next update, whichever
  // comes first).  Same values, same summation order.  (The copies of the LAST update equal the final state the epilogue
  // stores, so the last evaluation may overlap that store.)
  double mseA_last = 0.0, mseA_sum = 0.0, mseB_last = 0.0, mseB_sum = 0.0;
  bool pend = false;
  auto flush_stats = [&](int64_t se) {
    if (!pend) return;
    pend = false;
    const double* xs = a.x + (c.f0 + lane) * NX;
    const double* ir = a.imu_ref + (c.traj * a.E + se) * 6;
    const double* cr = a.cam_ref + (c.traj * a.E + se) * 6;
    double xr[26];
#pragma unroll
    for (int i = 3; i < 10; ++i) xr[i] = __ldcg(xs + i);
#pragma unroll
    for (int i = 19; i < 26; ++i) xr[i] = __ldcg(xs + i);
    double ei[3], ec[3], accA = 0.0, accB = 0.0;
    euler_xyz_deg(xr + 6, ei);
    euler_xyz_deg(xr + 22, ec);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const double d2_ = xr[3 + i] - ir[i], d3 = ei[i] - ir[3 + i];
      accA += d2_ * d2_ + d3 * d3;
      const double d0 = cr[i] - xr[19 + i], d1 = cr[3 + i] - ec[i];
      accB += d0 * d0 + d1 * d1;
    }
    mseA_last = accA;
    mseA_sum += accA;
    mseB_last = accB;
    mseB_sum += accB;
  };
  if (act) {
    const double* ug = a.u + (c.f0 + lane) * 6;
#pragma unroll
    for (int i = 0; i < 6; ++i) sx[(SX3_RING + i) * F] = ug[i];  // slot 0: the buffered previous sample
    sx[(SX3_RING + 6) * F] = 0.0;
  }
#if ESKF_OPT_TMA
  issue_chunk(0);
  issue_step(0);
#endif
  if (act && a.T > 0 && oap) stage_sample(0);
  __syncthreads();  // prologue
  PT_DECL();
  JIT_DECL();
  int64_t k = 0;
  for (int64_t e = 0; e < a.E; ++e) {
    const int n = epoch_steps3(a, c, e, k);
    if (act && a.do_update) stage_meas(e);
    const int fl = n < STATS_IT3 ? n : STATS_IT3;
    for (int it = 0;; ++it) {
#if !ESKF_OPT_STATS_U0
      if (it == fl && act) flush_stats(e - 1);
#endif
      if (it >= n) break;
      if (act && k + it + 1 < a.T && ESKF3_SCALAR_ON(it)) stage_sample(k + it + 1);
      if (h1s) {
        JIT();
        fx_slot_acquire(c.mbar, k + it);  // the covariance warps are done with the record of step kk - 2
        JIT();
        pk_ready_wait();  // JACOB has published the probe kinematics of the post-predict
        JIT();
        if (act && ESKF3_SCALAR_ON(it)) rows_h1(k + it);
        JIT();
        fx_slot_publish(c.mbar, k + it);  // rows 18:21 of the record of step kk are in place
        JIT();
      }
      PT_MARK(1);
      JIT();
      scalar_barrier();
      JIT();
      PT_MARK(2);
    }
    k += n;
    if (!a.do_update) continue;
    JIT();
    scalar_barrier();  // (an update-only launch has no step barrier: the measurement must be staged before U0)
    JIT();
#if ESKF_OPT_STATS_U0
    // error statistics of the PREVIOUS update, evaluated while the covariance warps form S, its inverse and the gain
    // (~9,000 cycles during which every scalar role waits): the parked copies are only overwritten after U1 | U2
    if (act) flush_stats(e - 1);
    (void)fl;
#endif
    PT_MARK(5);
    JIT();
    __syncthreads();  // U0 | U1
    JIT();
    JIT();
    __syncthreads();  // U1 | U2
    JIT();
    PT_MARK(3);
    JIT();
    scalar_barrier();  // U2 of the scalar roles done (the covariance warps do not wait: see role3_cov)
    JIT();
#if ESKF_OPT_PP
    pend = a.cam_ref && a.imu_ref && !a.snap;
#else
    pend = a.cam_ref && a.imu_ref;
#endif
  }
  if (act) {
    flush_stats(a.E - 1);
    sx[(SX3_ST + 0) * F] = mseA_last;
    sx[(SX3_ST + 1) * F] = mseA_sum;
    sx[(SX3_ST + 2) * F] = mseB_last;
    sx[(SX3_ST + 3) * F] = mseB_sum;
  }
  __syncthreads();
  store_tiles3<F, NTHR>(a, c, threadIdx.x);
}

// ---------------------------------------------------------------------------------------------
// covariance role

// 1 / x without the special-case subroutine of the compiler's division (SFU seed + three Newton steps, <= 1 ulp;
// zero / non-finite input gives a non-finite result, which the caller detects)
__device__ __forceinline__ double rcp_nr(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
#pragma unroll
  for (int it = 0; it < 3; ++it) {
    const double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
  }
  return r;
}

// inv(S) (np.linalg.inv, Filter.py:357) by the eight lanes of a filter: in-place Gauss-Jordan elimination with
// partial pivoting, lane r < 7 owning ROW r of S.  The pivot row of column k is chosen among the unused rows by a
// three-stage shuffle reduction (largest |entry|, as LAPACK's partial pivoting does) and is never moved: its lane
// simply plays row k.  Every step is the same code whatever k -- the rows are kept rotated so that the pivot column
// is element 0 and the finished inverse column goes to element 6 -- so the seven steps are a ROLLED loop of ~80
// instructions (the column-owned LU it replaces was 1,500 unrolled instructions and 4.6 k cycles of dependent
// shuffles per update).  Reads S from / writes inv(S) to the u3 record.  False for a singular or non-finite S
// (the reference's LinAlgError branch, Filter.py:358-361).
template <int QS>
__device__ __forceinline__ bool inv7_group3(double* rec, int g, const double* rd, int rds) {
  const unsigned FULL = 0xffffffffu;
  const int r = (g < 7) ? g : 6;  // lane 7 shadows row 6 and never becomes a pivot
  double a[7];
#if ESKF_OPT_UPD
  // row r of the tile's view of S straight from the H P record (upd3_publish_S): entries h_0..h_5 = 18..23 are three
  // 16-byte pairs, h_6 = 15; the measurement noise goes on the diagonal here (the same sum as in the publishing lane)
  {
    const double rr = rd[r * rds];
    double hp[6];
#pragma unroll
    for (int j = 0; j < 6; j += 2) {
      const d2 t = reinterpret_cast<const d2*>(rec)[((U3_HP + 24 * r + 18 + j) >> 1) * QS];
      hp[j] = t.x;
      hp[j + 1] = t.y;
    }
#pragma unroll
    for (int j = 0; j < 6; ++j) a[j] = hp[j] + ((j == r) ? rr : 0.0);
    a[6] = u3_get<QS>(rec, U3_HP + 24 * r + 15) + ((r == 6) ? rr : 0.0);
  }
#else
#pragma unroll
  for (int j = 0; j < 7; ++j) a[j] = u3_get<QS>(rec, U3_S + 7 * r + j);
#endif
  bool used = (g == 7);
  bool ok = true;
  int myk = 0;         // the row of inv(S) this lane ends up holding
  unsigned plist = 0;  // 3 bits per step: lane of the pivot row of column k
#pragma unroll 1
  for (int k = 0; k < 7; ++k) {
    // pivot search over the unused rows
    double best = used ? -1.0 : fabs(a[0]);
    int piv = g;
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
      const double ob = __shfl_xor_sync(FULL, best, o, 8);
      const int op = __shfl_xor_sync(FULL, piv, o, 8);
      if (ob > best || (ob == best && op < piv)) {
        best = ob;
        piv = op;
      }
    }
    ok = ok && (best > 0.0);
    plist |= (unsigned)piv << (3 * k);
    const bool mine = (piv == g);
    if (mine) {
      used = true;
      myk = k;
    }
    // scaled pivot row (column 0 replaced by 1 / pivot), broadcast from its lane
    const double rp = rcp_nr(a[0]);
    double pr[7];
#pragma unroll
    for (int j = 1; j < 7; ++j) pr[j - 1] = __shfl_sync(FULL, a[j] * rp, piv, 8);
    pr[6] = __shfl_sync(FULL, rp, piv, 8);
    const double f = a[0];
    if (mine) {
#pragma unroll
      for (int j = 0; j < 7; ++j) a[j] = pr[j];
    } else {
#pragma unroll
      for (int j = 0; j < 6; ++j) a[j] = a[j + 1] - f * pr[j];
      a[6] = -f * pr[6];
    }
  }
  // lane p_k holds row k of inv(P S) = inv(S) P^T (P: the row permutation of the pivoting): inv(S)(k, p_j) = a[j]
  double chk = 0.0;
#pragma unroll
  for (int j = 0; j < 7; ++j) chk += a[j] * 0.0;  // NaN / inf detector
  ok = ok && (chk == 0.0);
  if (g < 7) {
#pragma unroll
    // (written TRANSPOSED: the record holds the tile's view of S, the transpose of the reference's -- eskf_cov3.cuh)
    for (int j = 0; j < 7; ++j) u3_at<QS>(rec, U3_SINV + 7 * (int)((plist >> (3 * j)) & 7u) + myk) = a[j];
  }
  const unsigned bal = __ballot_sync(FULL, ok);
  const unsigned lane = threadIdx.x & 31u;
  return ((bal >> (lane & 24u)) & 0xffu) == 0xffu;
}

// warp-level synchronisation of the step loop: the eight lanes of a filter exchange their tiles through the filter's
// buffer.  All 32 lanes of a covariance warp run the step loop together (nothing in it depends on the filter), so the
// full-mask form is valid; the per-filter mask compiles into a MATCH / REDUX / BRA.DIV sequence of ~100 cycles.
#if ESKF_OPT_SYNCW
#define COV3_SYNCWARP() __syncwarp()
#else
#define COV3_SYNCWARP() __syncwarp(gmask)
#endif

template <int F, int NTHR>
__device__ __forceinline__ void role3_cov(const KArgs& a, const Ctx3& c, int ct) {
  using L = Lay3<F>;
  const int cf = ct >> 3;  // filter of this lane (padded filters run on an identity tile, never stored)
  const int cg = ct & 7;   // state group owned
  const unsigned gmask = 0xffu << (threadIdx.x & 24);
  double* Tb = c.smem + L::TB + cf * TB3_STRIDE;
  // u3 record of this filter: the transposition buffers of the warp's four filters, pair-interleaved
  double* rec = c.smem + L::TB + (cf & ~3) * TB3_STRIDE + 2 * (cf & 3);
  const double* sxc = c.smem + L::SX + cf;
  double* sxw = c.smem + L::SX + cf;
  const d2* fxb = reinterpret_cast<const d2*>(c.smem + L::FXB) + cf;
  auto qd = [&](int j) { return sxc[(SX3_QD + j) * F]; };
  const bool imu_q = (qd(3) != 0.0) || (qd(4) != 0.0) || (qd(5) != 0.0);
#if ESKF_OPT_COLD
  const bool warp_iq = __any_sync(0xffffffffu, imu_q);  // (warp-uniform: which copy of the step loop this warp runs)
#endif
  double qdv[3];  // diagonal process noise of this lane's three rows
  fx3_noise_diag(cg, qd, qdv);

  // X[i][v] = P[3g+v][i]: rows 3g..3g+2 of P, used as its columns 3g..3g+2 (a covariance is symmetric;
  // the engine never relies on more than that)
  double X[24][3];
  auto dump_rows = [&]() {  // tile -> rows 3g..3g+2 of the buffer (16-byte stores)
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      d2* row = reinterpret_cast<d2*>(Tb + (3 * cg + v) * RS3);
#pragma unroll
      for (int j = 0; j < 12; ++j) row[j] = d2{X[2 * j][v], X[2 * j + 1][v]};
    }
  };
  auto load_rows = [&]() {
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      const d2* row = reinterpret_cast<const d2*>(Tb + (3 * cg + v) * RS3);
#pragma unroll
      for (int j = 0; j < 12; ++j) {
        const d2 t = row[j];
        X[2 * j][v] = t.x;
        X[2 * j + 1][v] = t.y;
      }
    }
  };

  // Orientation of the tile (eskf_cov3.cuh, upd3_publish_S): X is the TRANSPOSE of the reference's matrix after the load
  // (rows used as columns) and every propagation flips it (X' = Fx X^T Fx^T).  The update and the final store want the
  // transposed orientation, so an epoch with an odd number of propagations gets one more pass through the exchange of
  // the step loop -- plain stores instead of pass 1, no pass 2 -- which turns the tile back (never with an even number
  // of IMU samples per frame).  The covariance is symmetric only up to the reference's own rounding, which an
  // ill-conditioned tuning makes large enough to matter.
  load_rows();
#if ESKF_OPT_ADDR
  int o_fx = cf, o_tbw = cf * TB3_STRIDE + 3 * cg, o_tbr = cf * TB3_STRIDE + 3 * cg * RS3;
  asm volatile("" : "+r"(o_fx), "+r"(o_tbw), "+r"(o_tbr));  // (opaque: not re-derived from the thread index inside the loop)
#endif
  __syncthreads();  // prologue
  PT_DECL();
  JIT_DECL();
#ifdef ESKF_EXP_STAGGER  // (profiling experiment: the second covariance warp of every sub-partition starts late)
  if (ct >= 128) {
    const long long t0 = clock64();
    while (clock64() - t0 < ESKF_EXP_STAGGER) {
    }
  }
#endif

  int64_t k = 0;
  for (int64_t e = 0; e < a.E; ++e) {
    const int n = epoch_steps3(a, c, e, k);
    PT_MARK(15);
    JIT();
    if (n > 0) fx_slot_wait(c.mbar, k);  // the Jacobian record of the first step of the epoch is complete
    JIT();
    PT_MARK(0);
#if ESKF_OPT_COLD
    // The step loop holds nothing but the two passes: the re-orientation after an odd number of propagations follows the loop,
    // and the IMU-noise part of Fi Q Fi^T (Q[0:6] != 0: never with config.yaml, where the filter is built with dt = 0) lives in a
    // second copy of the loop that a warp enters only if one of its four filters needs it.  As written before, both sat
    // inside the loop body (82 + 320 instructions between and behind the passes) and were fetched with it on every step: the
    // role loops of this kernel exceed the instruction cache, their code comes from L2 again and again (DESIGN.md section 4).
    auto step_loop = [&](auto IQ) {
      constexpr bool iq = decltype(IQ)::value;
      auto one_step = [&](int it) {
        const int64_t kk = k + it;
        if (ESKF3_COV_ON) {
          const d2* f2 = fxb + ((int)(kk & 1) * FX3_NPAIR) * F;
          fx3_apply_store_il<F, RS3>(X, f2, Tb + 3 * cg);
          COV3_SYNCWARP();
          PT_MARK(1);
          fx3_apply_stream<F, RS3>(X, f2, Tb + 3 * cg * RS3);
          PT_MARK(4);
          JIT();
          if (it + 1 < n) fx_slot_wait(c.mbar, kk + 1);
          JIT();
          COV3_SYNCWARP();  // every lane of the filter is done with the buffer before pass 1 of the next step stores
          PT_MARK(3);
          int gl = cg;
          asm volatile("" : "+r"(gl));
#ifndef ESKF_EXP_NO_QNOISE
          fx3_process_noise<F, iq>(X, gl, f2, qdv, qd, imu_q);
#endif
        }
        JIT();
        fx_slot_release(c.mbar, kk);  // this warp is done with the record
        JIT();
        PT_MARK(4);
      };
#if ESKF_OPT_COLD == 2
      // two steps per trip: the instruction fetch restarts at every taken branch (~115 cycles at the loop head and at the
      // reconvergence before it, and the first ~25 lines of pass 1 arrive late), once per two steps instead of once per step
      int it = 0;
      for (; it + 1 < n; it += 2) {
        one_step(it);
        one_step(it + 1);
      }
      if (it < n) one_step(it);
#else
      for (int it = 0; it < n; ++it) one_step(it);
#endif
    };
    if (warp_iq)
      step_loop(std::true_type{});
    else
      step_loop(std::false_type{});
    if (ESKF3_COV_ON && (n & 1)) {  // (one exchange more after an odd number of propagations: the tile is turned back)
#pragma unroll
      for (int i = 0; i < 24; ++i)
#pragma unroll
        for (int v = 0; v < 3; ++v) Tb[i * RS3 + 3 * cg + v] = X[i][v];
      COV3_SYNCWARP();
      load_rows();
      COV3_SYNCWARP();
    }
#else
    const int n_ex = ESKF3_COV_ON ? n + (n & 1) : n;  // (one exchange more after an odd number of propagations)
    for (int it = 0; it < n_ex; ++it) {
      const int64_t kk = k + it;
      const bool step = it < n;
      if (ESKF3_COV_ON) {
#if ESKF_OPT_ADDR
        const d2* f2 = reinterpret_cast<const d2*>(c.smem + L::FXB) + o_fx + ((int)(kk & 1) * FX3_NPAIR) * F;
        double* const TBW = c.smem + L::TB + o_tbw;
        const double* const TBR = c.smem + L::TB + o_tbr;
#else
        const d2* f2 = fxb + ((int)(kk & 1) * FX3_NPAIR) * F;
        double* const TBW = Tb + 3 * cg;
        const double* const TBR = Tb + 3 * cg * RS3;
#endif
        if (step) {
          // pass 1: T(:, 3g..3g+2) = Fx P(:, 3g..3g+2), rows stored as they are finished
#if ESKF_OPT_ST1
          fx3_apply_store_il<F, RS3>(X, f2, TBW);
#else
          fx3_apply_store<F, RS3>(X, f2, TBW);
#endif
        } else {
#pragma unroll
          for (int i = 0; i < 24; ++i)
#pragma unroll
            for (int v = 0; v < 3; ++v) Tb[i * RS3 + 3 * cg + v] = X[i][v];
        }
        COV3_SYNCWARP();
        PT_MARK(1);
#if ESKF_OPT_STREAM
        if (!step) {
          load_rows();
          COV3_SYNCWARP();
          break;
        }
        // pass 2 fused with the transposed reload: P'(3g+v, :) = Fx T(3g+v, :)^T, T streamed from the buffer
        fx3_apply_stream<F, RS3>(X, f2, TBR);
        PT_MARK(4);
        // the record of the NEXT step: its producers stored it one step ago (ESKF_OPT_LATEACQ) -- normally no wait
        JIT();
        if (it + 1 < n) fx_slot_wait(c.mbar, kk + 1);
        JIT();
        COV3_SYNCWARP();  // every lane of the filter is done with the buffer before pass 1 of the next step stores
        PT_MARK(3);
#else
        load_rows();  // X[k][v] = T(3g+v, k) -- every lane, the identity rows 9:15 included (eskf_cov3.cuh)
        PT_MARK(2);
        // the record of the NEXT step is waited for here, behind the latency of the transposed reload, so that
        // nothing stands between the end of this step and the first coefficient fetch of the next one
        JIT();
        if (it + 1 < n) fx_slot_wait(c.mbar, kk + 1);
        JIT();
        COV3_SYNCWARP();
        PT_MARK(3);
        if (!step) break;
        // pass 2: P'(3g+v, :) = Fx T(3g+v, :)^T
        fx3_apply_inplace<F>(X, f2);
#endif
        // (the lane index is laundered through an empty asm so that the thirteen selected addends of the diagonal
        // are formed here, two selects each, instead of being hoisted out of the loop and spilled)
        int gl = cg;
        asm volatile("" : "+r"(gl));
#ifndef ESKF_EXP_NO_QNOISE
        fx3_process_noise<F, true>(X, gl, f2, qdv, qd, imu_q);
#endif
      }
      JIT();
      fx_slot_release(c.mbar, kk);  // this warp is done with the record
      JIT();
      PT_MARK(4);
    }
#endif
    k += n;
    if (!a.do_update) continue;
    // ---- U0: S and its inverse (the scalar CAMERA role computes the residual meanwhile) ----
#ifdef ESKF_EXP_NO_UPDATE  // (profiling experiment: propagation only)
    __syncthreads();
    if (cg == 0) sxw[SX3_OK2 * F] = 0.0;
    __syncthreads();
    continue;
#endif
    double rd[7];
#pragma unroll
    for (int m = 0; m < 7; ++m) rd[m] = sxc[(SX3_RD + m) * F];
    upd3_publish_S<4>(X, cg, rd, rec);
    __syncwarp(gmask);
    const bool inv_ok = inv7_group3<4>(rec, cg, sxc + SX3_RD * F, F);
    PT_MARK(5);
    JIT();
    __syncthreads();  // U0 | U1
    JIT();
    PT_MARK(6);
    const bool upd_c = inv_ok && (sxc[SX3_OK * F] != 0.0);
    if (upd_c) {
      double K[3][7], res[7], dl[3];
#pragma unroll
      for (int m = 0; m < 7; ++m) res[m] = sxc[(SX3_RES + m) * F];
      upd3_gain<4>(cg, rec, res, K, dl);
#pragma unroll
      for (int v = 0; v < 3; ++v) sxw[(SX3_DELTA + 3 * cg + v) * F] = dl[v];
      if (a.K_out && cf < c.nf) {
#pragma unroll
        for (int v = 0; v < 3; ++v)
#pragma unroll
          for (int m = 0; m < 7; ++m) a.K_out[((c.f0 + cf) * 24 + 3 * cg + v) * 7 + m] = K[v][m];
      }
    }
    if (cg == 0) sxw[SX3_OK2 * F] = upd_c ? 1.0 : 0.0;
    PT_MARK(7);
    JIT();
    __syncthreads();  // U1 | U2  (also orders the K / K R records of the eight lanes)
    JIT();
    PT_MARK(8);
    if (upd_c) {
      upd3_w_pass<4>(X, cg, rec);
      __syncwarp(gmask);
      PT_MARK(9);
#if ESKF_OPT_UPD
      upd3_finish<4, F, F>(X, cg, rec, sxc + SX3_RD * F, sxc + (SX3_DELTA + 6) * F, sxc + (SX3_DELTA + 21) * F);
#else
      const double dth[3] = {sxc[(SX3_DELTA + 6) * F], sxc[(SX3_DELTA + 7) * F], sxc[(SX3_DELTA + 8) * F]};
      const double dthc[3] = {sxc[(SX3_DELTA + 21) * F], sxc[(SX3_DELTA + 22) * F], sxc[(SX3_DELTA + 23) * F]};
      upd3_finish<4, F, 1>(X, cg, rec, sxc + SX3_RD * F, dth, dthc);
#endif
    }
    PT_MARK(10);
    // no CTA barrier here: the scalar roles go on to the first steps of the next epoch while the covariance warps
    // finish the Joseph form (what they exchange next is ordered by the record pipeline and by the next U0 | U1)
  }
  PT_FLUSH();
  dump_rows();
  __syncthreads();
  store_tiles3<F, NTHR>(a, c, threadIdx.x);
}

// ---------------------------------------------------------------------------------------------
// MODE: bit 0 = export mode (FilterTraj rows, Jacobian record of the last step), bit 1 = stacked trajectories.  Separate
// instantiations, so that the production kernel of a single-trajectory batch carries neither (a few integer instructions
// in the prologue are enough to change the register allocation of the whole kernel).
template <int F, int REG_S, int REG_C, int MODE>
__global__ void __launch_bounds__(128 + 8 * F, 1) eskf_kernel3(const __grid_constant__ KArgs a) {
  constexpr bool EX = (MODE & 1) != 0, MT = (MODE & 2) != 0;
  extern __shared__ __align__(16) double smem[];
  using L = Lay3<F>;
  constexpr int NTHR = 128 + 8 * F;
  const int tid = threadIdx.x;
  Ctx3 c;
  c.smem = smem;
  if constexpr (MT) {
    // stacked trajectories: a CTA follows ONE trajectory's epoch structure (stacked_cta, eskf_math.cuh; the grid is
    // stacked_grid) -- fpt need not be a multiple of the CTA shape
    int64_t tl;
    stacked_cta(blockIdx.x, a.N, a.filters_per_traj, F, c.f0, c.nf, tl);
  } else {
    c.f0 = (int64_t)blockIdx.x * F;
    c.nf = (int)((a.N - c.f0) < F ? (a.N - c.f0) : F);
  }
  c.gid0 = a.filter_id0 + c.f0;
  c.traj = (a.n_traj > 1) ? (c.gid0 / a.filters_per_traj) : 0;
  c.n_prop = a.n_prop ? a.n_prop + c.traj * a.E : nullptr;
  c.dtp = a.dt ? a.dt + c.traj * a.T : nullptr;
  c.mbar = reinterpret_cast<uint64_t*>(smem + L::MBAR);
  if (tid == 0) {
    mbar_init(c.mbar + 0, 3);      // full[s]:  the IMU, the CAMERA and the JACOB warp (rows 3:9, 18:21, 21:24)
    mbar_init(c.mbar + 1, 3);
    mbar_init(c.mbar + 2, F / 4);  // empty[s]: the covariance warps
    mbar_init(c.mbar + 3, F / 4);
#if ESKF_OPT_TMA
    mbar_init(reinterpret_cast<uint64_t*>(smem + L::CHBAR), 1);  // chunk[b]: one arrival (expect_tx) + the bytes of the copies
    mbar_init(reinterpret_cast<uint64_t*>(smem + L::CHBAR) + 1, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#endif
  }

  // ---- covariance tiles and parameters (coalesced) ----
  for (int idx = tid; idx < F * 576; idx += NTHR) {
    const int f = idx / 576, r = idx - f * 576;
    const int i = r / 24, j = r - i * 24;
    smem[L::TB + f * TB3_STRIDE + i * RS3 + j] = (f < c.nf) ? a.P[(c.f0 + f) * 576 + r] : ((i == j) ? 1.0 : 0.0);
  }
  for (int idx = tid; idx < F * PAR_STRIDE; idx += NTHR) {
    const int f = idx / PAR_STRIDE, r = idx - f * PAR_STRIDE;
    const int64_t row = (f < c.nf) ? (c.f0 + f) : c.f0;
    if (r < PAR_RD + 7) smem[L::SX + (SX3_QD + r) * F + f] = a.par[row * PAR_STRIDE + r];  // QD(13) then RD(7)
  }
  __syncthreads();

  const int warp = tid >> 5, lane = tid & 31;
  // (setmaxnreg must be executed by all four warps of a warpgroup alike: the scalar roles are warps 0..3, one per SM
  // sub-partition -- a remapping that put two scalar roles on the sub-partition with the single covariance warp hung)
  if (warp >= 4) {
    reg_inc3<REG_C>();
    role3_cov<F, NTHR>(a, c, tid - 128);
  } else {
    // (ptxas 12.9 crashes on kernels with more than one setmaxnreg.dec value, so all four scalar roles
    // share REG_S although the Jacobian warp's sub-partition would have room for more)
    reg_dec3<REG_S>();
    if (warp == 0)
      role3_imu<F, NTHR, EX>(a, c, lane);
    else if (warp == 1)
      role3_cam<F, NTHR, EX>(a, c, lane);
    else if (warp == 2)
      role3_stage<F, NTHR, EX>(a, c, lane);
    else
      role3_jac<F, NTHR, EX>(a, c, lane);
  }
}

template <int F>
cudaError_t launch_eskf_kernel3(const KArgs& a, cudaStream_t stream);

}  // namespace eskf
