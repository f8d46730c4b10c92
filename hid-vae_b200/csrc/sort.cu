// cub::DeviceRadixSort and cub::DeviceScan behind sort.cuh (the library's two CUB instantiations: a radix sort of 64-bit keys
// with 32-bit row indices, and an in-place inclusive sum of 64-bit words).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "sort.cuh"

namespace hv {
namespace {

size_t align256(size_t v) { return (v + 255) & ~static_cast<size_t>(255); }

size_t cub_temp_bytes(int64_t n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, static_cast<const uint64_t*>(nullptr), static_cast<uint64_t*>(nullptr),
                                  static_cast<const uint32_t*>(nullptr), static_cast<uint32_t*>(nullptr), static_cast<int>(n), 0, 64);
  return bytes;
}

}  // namespace

size_t sort_workspace_bytes(int64_t n) {
  if (n <= 0 || n >= (1ll << 31)) return 0;
  return 2 * align256(static_cast<size_t>(n) * 8) + 2 * align256(static_cast<size_t>(n) * 4) + align256(cub_temp_bytes(n)) + 256;
}

bool sort_carve(void* workspace, size_t workspace_bytes, int64_t n, SortBuffers* out) {
  const size_t need = sort_workspace_bytes(n);
  if (workspace == nullptr || need == 0 || workspace_bytes < need) return false;
  uint8_t* p = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~static_cast<uintptr_t>(255));
  out->keys_in = reinterpret_cast<uint64_t*>(p);
  p += align256(static_cast<size_t>(n) * 8);
  out->keys_out = reinterpret_cast<uint64_t*>(p);
  p += align256(static_cast<size_t>(n) * 8);
  out->vals_in = reinterpret_cast<uint32_t*>(p);
  p += align256(static_cast<size_t>(n) * 4);
  out->vals_out = reinterpret_cast<uint32_t*>(p);
  p += align256(static_cast<size_t>(n) * 4);
  out->temp = p;
  out->temp_bytes = cub_temp_bytes(n);
  return true;
}

int sort_pairs(const SortBuffers& b, int64_t n, int end_bit, cudaStream_t stream) {
  size_t bytes = b.temp_bytes;
  HV_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(b.temp, bytes, b.keys_in, b.keys_out, b.vals_in, b.vals_out, static_cast<int>(n), 0,
                                                end_bit, stream));
  return HV_OK;
}

size_t scan_temp_bytes(int64_t n) {
  if (n <= 0 || n >= (1ll << 31)) return 0;
  size_t bytes = 0;
  cub::DeviceScan::InclusiveSum(nullptr, bytes, static_cast<uint64_t*>(nullptr), static_cast<int>(n));
  return bytes;
}

int inclusive_sum_u64(void* temp, size_t temp_bytes, uint64_t* data, int64_t n, cudaStream_t stream) {
  size_t bytes = temp_bytes;
  HV_CUDA_CHECK(cub::DeviceScan::InclusiveSum(temp, bytes, data, static_cast<int>(n), stream));
  return HV_OK;
}

}  // namespace hv

extern "C" size_t hv_sort_workspace_bytes(int64_t n) { return hv::sort_workspace_bytes(n); }
