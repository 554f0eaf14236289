// Counter-based Gaussian noise for the Monte-Carlo extension of the engine
// (the reference itself is noise free; its only np.random call is dead code in
// dvi_ekf/models/trajectory/ImuTrajectory.py:133).  Philox4x32-10 keyed by the
// run seed, counter = (step, kind*16 + draw, filter id lo, filter id hi), so a
// filter's noise depends only on its GLOBAL id: results are independent of how
// the batch is sharded over CTAs or GPUs.
//
// One Philox block = four 32-bit uniforms = two Box-Muller pairs = four standard
// normals, evaluated in single precision (the construction of curand_normal:
// 32-bit uniforms, r = sqrt(-2 ln u1), angle = 2 pi u2) and widened to FP64.  On
// the device the logarithm / sine / cosine are the SFU approximations (MUFU),
// which is what keeps the generator off the FP64 pipe the filter lives on; the
// noise a run used is therefore defined by the device and can be read back
// with eskf_noise_dump() (include/eskf.h) -- the parity tests feed exactly those
// samples to the oracle.
#pragma once
#include <math.h>
#include <stdint.h>

#ifndef ESKF_HD
#ifdef __CUDACC__
#define ESKF_HD __host__ __device__ __forceinline__
#else
#define ESKF_HD inline
#endif
#endif

namespace eskf {

constexpr uint32_t RNG_KIND_IMU = 1;  // 6 normals per IMU step      (draw 0: om xyz + acc x, draw 1: acc yz)
constexpr uint32_t RNG_KIND_CAM = 2;  // 7 normals per camera update (draw 0: position + theta x, draw 1: theta yz, notch)

ESKF_HD void philox4x32_10(uint32_t* c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c[0];
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c[2];
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0;
    const uint32_t n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
    const uint32_t n3 = (uint32_t)p0;
    c[0] = n0;
    c[1] = n1;
    c[2] = n2;
    c[3] = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
}

// Box-Muller on two 32-bit words: u1 in (0, 1], angle in [-pi, pi)
ESKF_HD void box_muller32(uint32_t a, uint32_t b, double* z) {
  const float u1 = (float)a * 2.3283064365386963e-10f + 1.1641532182693481e-10f;  // a 2^-32 + 2^-33
  const float th = (float)(int32_t)b * 1.4629180792671596e-9f;                     // b pi 2^-31
#ifdef __CUDA_ARCH__
  // (lg2.approx is only accurate to ~2^-22 absolute near 1: for u1 = 1 - 2^-24 the approximate logarithm may come out
  // with the wrong sign; the clamp turns that one-in-2^24 NaN into r = 0 and changes nothing else)
  const float r = sqrtf(fmaxf(0.0f, -2.0f * __logf(u1)));
  const float s = __sinf(th), c = __cosf(th);
#else
  const float r = sqrtf(-2.0f * logf(u1));
  const float s = sinf(th), c = cosf(th);
#endif
  z[0] = (double)(r * c);
  z[1] = (double)(r * s);
}

// four standard normals from one Philox block
ESKF_HD void normal4(uint64_t seed, uint64_t filter, uint64_t step, uint32_t kind, uint32_t draw, double* z) {
  uint32_t c[4] = {(uint32_t)step, kind * 16u + draw + ((uint32_t)(step >> 32) << 8), (uint32_t)filter,
                   (uint32_t)(filter >> 32)};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  box_muller32(c[0], c[1], z);
  box_muller32(c[2], c[3], z + 2);
}

// two Philox blocks side by side (the two draws of normal8: independent chains for the integer pipe).  Kept unrolled:
// a rolled loop over the ten rounds is 100 instructions shorter but lengthens the STAGER role's step and cost 2.5 % of the
// whole kernel (profiles/r01_s4_experiments.md)
ESKF_HD void philox4x32_10_x2(uint32_t* a, uint32_t* b, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t pa0 = (uint64_t)0xD2511F53u * a[0], pa1 = (uint64_t)0xCD9E8D57u * a[2];
    const uint64_t pb0 = (uint64_t)0xD2511F53u * b[0], pb1 = (uint64_t)0xCD9E8D57u * b[2];
    const uint32_t a0 = (uint32_t)(pa1 >> 32) ^ a[1] ^ k0, a2 = (uint32_t)(pa0 >> 32) ^ a[3] ^ k1;
    const uint32_t b0 = (uint32_t)(pb1 >> 32) ^ b[1] ^ k0, b2 = (uint32_t)(pb0 >> 32) ^ b[3] ^ k1;
    a[0] = a0;
    a[1] = (uint32_t)pa1;
    a[2] = a2;
    a[3] = (uint32_t)pa0;
    b[0] = b0;
    b[1] = (uint32_t)pb1;
    b[2] = b2;
    b[3] = (uint32_t)pb0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
}

// z[0..7]: eight normals of (filter, step, kind) = normal4 of draw 0 and draw 1; the IMU stream uses z[0..5], the camera
// stream z[0..6]
ESKF_HD void normal8(uint64_t seed, uint64_t filter, uint64_t step, uint32_t kind, double* z) {
  const uint32_t hi = (uint32_t)(step >> 32) << 8;
  uint32_t a[4] = {(uint32_t)step, kind * 16u + 0u + hi, (uint32_t)filter, (uint32_t)(filter >> 32)};
  uint32_t b[4] = {(uint32_t)step, kind * 16u + 1u + hi, (uint32_t)filter, (uint32_t)(filter >> 32)};
  philox4x32_10_x2(a, b, (uint32_t)seed, (uint32_t)(seed >> 32));
  box_muller32(a[0], a[1], z);
  box_muller32(a[2], a[3], z + 2);
  box_muller32(b[0], b[1], z + 4);
  box_muller32(b[2], b[3], z + 6);
}

// ---- simulated frame loss (eskf_set_meas_dropout, include/eskf.h) ----
// One uniform per (noise id, GLOBAL epoch): word 0 of the Philox block with normal4's counter layout, kind RNG_KIND_DROP and
// draw 0.  u = (x + 1/2) 2^-32 is exact in double precision and lies strictly inside (0, 1): 2^-33 <= u <= 1 - 2^-33.  It
// depends on nothing but (seed, id, epoch), so segments, shards and noise_id_modulus see the draws of one whole-batch run,
// and the other kinds' draws do not move.  eskf_noise_dump(kind = ESKF_NOISE_DROP) reads it back.
constexpr uint32_t RNG_KIND_DROP = 3;

ESKF_HD double unit_open32(uint32_t x) { return ((double)x + 0.5) * 2.3283064365386963e-10; }  // (x + 1/2) 2^-32

ESKF_HD double drop_uniform(uint64_t seed, uint64_t id, uint64_t epoch) {
  uint32_t c[4] = {(uint32_t)epoch, RNG_KIND_DROP * 16u + ((uint32_t)(epoch >> 32) << 8), (uint32_t)id, (uint32_t)(id >> 32)};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  return unit_open32(c[0]);
}

// The measurement of epoch `epoch` is dropped for noise id `id` iff u < p: p = 0 never drops, p = 1 always does.  Within one
// id the masks nest (p1 <= p2: every epoch dropped at p1 is dropped at p2, both compare the same u), which a sweep over p
// relies on.  A noise-free reference filter (nf0: noise_free_filter0 and id 0) makes no random drop: it loses exactly the
// epochs with p == 1.
ESKF_HD bool meas_dropped(double p, uint64_t seed, uint64_t id, uint64_t epoch, bool nf0) {
  if (!(p > 0.0)) return false;
  return nf0 ? p == 1.0 : drop_uniform(seed, id, epoch) < p;
}

// ---- simulated outlier frames (eskf_set_meas_outliers, include/eskf.h) ----
// One uniform and one set of offsets per (noise id, GLOBAL epoch), kind RNG_KIND_OUTLIER: the offsets are normal8 (draws 0
// and 1), u = unit_open32 of word 0 of draw 2 with drop_uniform's counter layout.  Like the dropout draw it depends on
// nothing but (seed, id, epoch): segments, shards and noise_id_modulus see the outliers of one whole-batch run, and no other
// kind's draw moves.  eskf_noise_dump(kind = ESKF_NOISE_OUTLIER) reads u and the offsets back.
constexpr uint32_t RNG_KIND_OUTLIER = 4;

ESKF_HD double outlier_uniform(uint64_t seed, uint64_t id, uint64_t epoch) {
  uint32_t c[4] = {(uint32_t)epoch, RNG_KIND_OUTLIER * 16u + 2u + ((uint32_t)(epoch >> 32) << 8), (uint32_t)id,
                   (uint32_t)(id >> 32)};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  return unit_open32(c[0]);
}

// The measurement of epoch `epoch` is an outlier for noise id `id` iff u < p: p = 0 never, p = 1 always.  The masks nest over
// p and the offsets do not depend on p, so a sweep over p corrupts a superset with the same offsets.  A noise-free reference
// filter (nf0) is never corrupted.
ESKF_HD bool meas_outlier(double p, uint64_t seed, uint64_t id, uint64_t epoch, bool nf0) {
  if (nf0 || !(p > 0.0)) return false;
  return outlier_uniform(seed, id, epoch) < p;
}

}  // namespace eskf
