// Stable key sort of row indices (cub::DeviceRadixSort on 64-bit keys) shared by the k-means update (sort rows by
// cluster -> segmented sums), the uniqueness loss and the semantic-ID collision digit (sort rows by id tuple -> runs of
// identical tuples); and the in-place 64-bit inclusive sum (cub::DeviceScan) that numbers those runs.
// The library never allocates: the caller provides hv_sort_workspace_bytes(n) bytes.
#pragma once

#include "common.cuh"

namespace hv {

struct SortBuffers {
  uint64_t* keys_in;
  uint64_t* keys_out;
  uint32_t* vals_in;
  uint32_t* vals_out;
  void* temp;
  size_t temp_bytes;
};

size_t sort_workspace_bytes(int64_t n);
// false when the workspace is missing, misaligned or too small for n rows
bool sort_carve(void* workspace, size_t workspace_bytes, int64_t n, SortBuffers* out);
// keys_in / vals_in -> keys_out / vals_out, ascending, stable, bits [0, end_bit) of the key
int sort_pairs(const SortBuffers& b, int64_t n, int end_bit, cudaStream_t stream);

// temporary storage of inclusive_sum_u64 for n words (0 for n <= 0 or n >= 2^31)
size_t scan_temp_bytes(int64_t n);
// data[i] <- data[0] + ... + data[i], in place
int inclusive_sum_u64(void* temp, size_t temp_bytes, uint64_t* data, int64_t n, cudaStream_t stream);

}  // namespace hv
