// CPU harness for the block map of the grouped reductions (TEST INFRASTRUCTURE): group_blocks / group_block / group_row0
// (eskf_math.cuh), what the reduction kernels of eskf_api.cu and their launches use.  Built by tests/test_groups_host.py.
#include "../../dvi_ekf_b200/csrc/eskf_math.cuh"

using namespace eskf;

extern "C" {

// the blocks of one geometry: rows [nblk][3] = {row0, row1, local group}; returns nblk = group_blocks (-1: cap too small)
int64_t hc_group_map(int64_t N, int64_t id0, int64_t g, int64_t rpb, int64_t* rows, int64_t cap) {
  const int64_t nblk = group_blocks(N, id0, g, rpb);
  if (nblk > cap) return -1;
  for (int64_t b = 0; b < nblk; ++b) group_block(b, N, id0, g, rpb, rows[3 * b], rows[3 * b + 1], rows[3 * b + 2]);
  return nblk;
}

// the first block of local groups 0 .. G (G + 1 values), as the final kernels find a group's blocks
void hc_group_first_blocks(int64_t N, int64_t id0, int64_t g, int64_t rpb, int64_t G, int64_t* out) {
  for (int64_t k = 0; k <= G; ++k) out[k] = group_blocks(group_row0(k, N, id0, g), id0, g, rpb);
}

}  // extern "C"
