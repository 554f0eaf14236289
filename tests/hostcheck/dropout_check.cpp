// CPU harness for the measurement-dropout draw (TEST INFRASTRUCTURE): philox4x32_10, drop_uniform and meas_dropped
// (eskf_rng.cuh), the definitions the persistent kernel and eskf_noise_dump use.  Built by tests/test_dropout_host.py.
#include "../../dvi_ekf_b200/csrc/eskf_rng.cuh"

using namespace eskf;

extern "C" {

// one Philox4x32-10 block: ctr[4] in, out[4] out
void hc_philox(const uint32_t* ctr, uint32_t k0, uint32_t k1, uint32_t* out) {
  uint32_t c[4] = {ctr[0], ctr[1], ctr[2], ctr[3]};
  philox4x32_10(c, k0, k1);
  for (int i = 0; i < 4; ++i) out[i] = c[i];
}

// u of noise ids id0 .. id0 + n_ids - 1 and epochs e0 .. e0 + n_epochs - 1: out[n_ids][n_epochs]
void hc_drop_uniforms(uint64_t seed, uint64_t id0, int64_t n_ids, uint64_t e0, int64_t n_epochs, double* out) {
  for (int64_t i = 0; i < n_ids; ++i)
    for (int64_t k = 0; k < n_epochs; ++k) out[i * n_epochs + k] = drop_uniform(seed, id0 + i, e0 + k);
}

// the map drop_uniform applies to the first Philox word
double hc_unit_open32(uint32_t x) { return unit_open32(x); }

int hc_meas_dropped(double p, uint64_t seed, uint64_t id, uint64_t epoch, int nf0) {
  return meas_dropped(p, seed, id, epoch, nf0 != 0) ? 1 : 0;
}

}  // extern "C"
