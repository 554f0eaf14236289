// One translation unit per CTA shape of the v3 kernel: compiled with -DESKF_F=<filters per CTA>
// (see dvi_ekf_b200/build.py).  Shapes with more than 256 threads split the register file by role
// with setmaxnreg (scalar warps ESKF_REG_S, covariance warps ESKF_REG_C registers per thread).  Registers live in the four SM sub-partitions (16,384 each) and warp w runs on
// sub-partition w % 4, so with F = 28 (11 warps) sub-partitions 0..2 hold one scalar and two covariance
// warps and sub-partition 3 the Jacobian warp and one covariance warp: the kernel launches with 168
// registers per thread (3 x 32 x 168 <= 16,384) and the split must satisfy REG_S + 2 REG_C <= 504, otherwise
// setmaxnreg.inc waits for ever.
#include "eskf_kernel3.cuh"

#ifndef ESKF_F
#error "compile with -DESKF_F=<filters per CTA>"
#endif
#ifndef ESKF_REG_S
#if ESKF_F > 16
#define ESKF_REG_S 104
#define ESKF_REG_C 200
#else
#define ESKF_REG_S 0
#define ESKF_REG_C 0
#endif
#endif

namespace eskf {

template <>
cudaError_t launch_eskf_kernel3<ESKF_F>(const KArgs& a, cudaStream_t stream) {
  constexpr int F = ESKF_F;
  static_assert((8 * F) % 32 == 0, "covariance role must fill whole warps");
  static_assert(F <= 32, "one lane per filter in the scalar roles");
  static_assert(ESKF_REG_S == 0 || ESKF_REG_S + 2 * ESKF_REG_C <= 504, "register split exceeds a sub-partition");
  constexpr size_t smem = (size_t)Lay3<F>::TOTAL * sizeof(double);
  static_assert(smem <= 232448, "shared memory per CTA");
  // export mode (FilterTraj rows, eskf_streams_t.trace_x; Jacobian record of the last step, eskf_keep_jacobians; consistency
  // records, eskf_keep_consistency) and the CTA mapping of stacked trajectories are separate instantiations: the production
  // kernel of a single-trajectory batch carries none of their code (the dump alone cost 10 % through register allocation).
  // A segment of the trajectory (eskf_run_epochs) is a third bit: eskf_run keeps the kernels it had.  Simulated frame loss
  // (eskf_set_meas_dropout) is export code too.
  const int mode = ((a.trace || a.fx_dump || a.cons || a.drop_p) ? 1 : 0) | (a.n_traj > 1 ? 2 : 0) | (a.k_base ? 4 : 0);
  auto kern = mode == 0   ? eskf_kernel3<F, ESKF_REG_S, ESKF_REG_C, 0>
              : mode == 1 ? eskf_kernel3<F, ESKF_REG_S, ESKF_REG_C, 1>
              : mode == 2 ? eskf_kernel3<F, ESKF_REG_S, ESKF_REG_C, 2>
              : mode == 3 ? eskf_kernel3<F, ESKF_REG_S, ESKF_REG_C, 3>
              : mode == 4 ? eskf_kernel3<F, ESKF_REG_S, ESKF_REG_C, 4>
              : mode == 5 ? eskf_kernel3<F, ESKF_REG_S, ESKF_REG_C, 5>
              : mode == 6 ? eskf_kernel3<F, ESKF_REG_S, ESKF_REG_C, 6>
                          : eskf_kernel3<F, ESKF_REG_S, ESKF_REG_C, 7>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  // (stacked trajectories: ceil(fpt / F) CTAs per trajectory, fewer for a partially covered last one: stacked_grid)
  const unsigned grid = a.n_traj > 1 ? (unsigned)stacked_grid(a.N, a.filters_per_traj, F) : (unsigned)((a.N + F - 1) / F);
  kern<<<grid, 128 + 8 * F, smem, stream>>>(a);
  return cudaGetLastError();
}

}  // namespace eskf

#if defined(ESKF_EXP_TIMING) && ESKF_F == 28
// profiling build only: reads (and clears) the phase-cycle table [256 CTAs][12 warps][16 slots]
extern "C" int eskf_debug_timing(long long* out) {
  const size_t bytes = sizeof(long long) * 256 * 12 * TIMING_SLOTS;
  cudaError_t e = cudaMemcpyFromSymbol(out, eskf::g_eskf_timing, bytes);
  if (e != cudaSuccess) return -1;
  void* p = nullptr;
  cudaGetSymbolAddress(&p, eskf::g_eskf_timing);
  cudaMemset(p, 0, bytes);
  return 0;
}
#endif

#if defined(ESKF_EXP_JITTER)
// race-hunting build only (eskf_kernel3.cuh, ESKF_EXP_JITTER): seed and largest delay [ns] of the injected jitter for this CTA
// shape's translation unit; max_ns = 0 switches it off.  One entry point per shape: eskf_debug_set_jitter_<F>.
#define ESKF_JIT_NAME2(f) eskf_debug_set_jitter_##f
#define ESKF_JIT_NAME(f) ESKF_JIT_NAME2(f)
extern "C" int ESKF_JIT_NAME(ESKF_F)(unsigned int seed, unsigned int max_ns) {
  cudaError_t e = cudaMemcpyToSymbol(eskf::g_eskf_jitter_seed, &seed, sizeof(seed));
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(eskf::g_eskf_jitter_ns, &max_ns, sizeof(max_ns));
  return e == cudaSuccess ? 0 : -1;
}
#endif
