// CPU harness for the outlier-frame draw (TEST INFRASTRUCTURE): philox4x32_10, outlier_uniform, meas_outlier and the
// kind-4 normals (eskf_rng.cuh), the definitions the persistent kernel and eskf_noise_dump use.  Built by
// tests/test_outlier_host.py.  (The host normals use the C library's logf / sinf / cosf, not the device's SFU approximations:
// only the Philox words and the uniform are bit-exact across the two.)
#include "../../dvi_ekf_b200/csrc/eskf_rng.cuh"

using namespace eskf;

extern "C" {

void hc_philox(const uint32_t* ctr, uint32_t k0, uint32_t k1, uint32_t* out) {
  uint32_t c[4] = {ctr[0], ctr[1], ctr[2], ctr[3]};
  philox4x32_10(c, k0, k1);
  for (int i = 0; i < 4; ++i) out[i] = c[i];
}

// u of noise ids id0 .. id0 + n_ids - 1 and epochs e0 .. e0 + n_epochs - 1: out[n_ids][n_epochs]
void hc_outlier_uniforms(uint64_t seed, uint64_t id0, int64_t n_ids, uint64_t e0, int64_t n_epochs, double* out) {
  for (int64_t i = 0; i < n_ids; ++i)
    for (int64_t k = 0; k < n_epochs; ++k) out[i * n_epochs + k] = outlier_uniform(seed, id0 + i, e0 + k);
}

// the eight kind-4 normals of (seed, id, epoch): out[8]
void hc_outlier_normals(uint64_t seed, uint64_t id, uint64_t epoch, double* out) { normal8(seed, id, epoch, RNG_KIND_OUTLIER, out); }

double hc_unit_open32(uint32_t x) { return unit_open32(x); }

int hc_meas_outlier(double p, uint64_t seed, uint64_t id, uint64_t epoch, int nf0) {
  return meas_outlier(p, seed, id, epoch, nf0 != 0) ? 1 : 0;
}

}  // extern "C"
