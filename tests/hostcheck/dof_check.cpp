// CPU harness for the per-DOF envelope terms of the device (TEST INFRASTRUCTURE): dof_terms (eskf_math.cuh), the
// per-record arithmetic of dof_partial_kernel (eskf_api.cu).  Built by tests/test_dof_envelope_host.py.
#include "../../dvi_ekf_b200/csrc/eskf_math.cuh"

using namespace eskf;

extern "C" {

// the DSUM_USED terms of n records: nis [n], eps [n][6], B [n][36] (row-major), masks [n] -> out [n][DSUM_USED]
void hc_dof_terms(const double* nis, const double* eps, const double* B, const int32_t* mask, int64_t n, double* out) {
  for (int64_t i = 0; i < n; ++i) dof_terms(nis[i], eps + 6 * i, B + 36 * i, 1, mask[i], out + DSUM_USED * i);
}

int hc_dof_used() { return DSUM_USED; }

}  // extern "C"
