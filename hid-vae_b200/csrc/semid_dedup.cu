// Semantic-ID collision digit (the TIGER-style trailing id position of HSemanticIdTokenizer(use_dedup_dim=True)):
//   digit[r] = prior count of ids[r] + #{ r' < r : ids[r', 0:width] == ids[r, 0:width] }.
// The reference loop compares every 512-row batch with itself and with every row cached before it: O(N^2 / 2 * width).
// Here every row becomes an EXACT key (its ids packed `bits` apart, so equal keys are equal tuples and keys ascend in
// lexicographic tuple order), rows are key-sorted with the stable radix sort of sort.cuh over the key's width*bits bits
// only, and one inclusive sum over the sorted positions numbers the runs of identical tuples and counts the valid rows
// before every position.  A row's digit is its rank inside its run (rows of a run stay in row order: stable sort) plus the
// run's count in a sorted list of tuples seen before this call (the other shards of a catalogue).  O(N) per bit pass, and
// no thread ever walks a run, so a catalogue of one repeated tuple costs the same as one of distinct tuples.
//
// Rows holding an id outside [0, 2^bits) get digit -1, belong to no run, and are counted in stats[2].  They are given the
// largest key of the width*bits bits -- that of the all-(2^bits - 1) tuple, with which they may share a run -- and the scan
// counts valid rows separately from positions, so their presence shifts no valid row's digit.
#include "common.cuh"
#include "sort.cuh"

namespace hv {
namespace {

constexpr int kThreads = 256;
constexpr uint32_t kInvalidRow = 0x80000000u;  // bit of the sorted row index: the row has an id outside [0, 2^bits)

struct Work {
  SortBuffers sort;    // keys_in is reused as the scan's words once the sort has consumed it
  void* scan_temp;
  size_t scan_temp_bytes;
  int64_t* run_start;  // [rows + 1] valid rows before each run; [n_runs] = all valid rows
  int64_t* run_prior;  // [rows] count of the run's tuple in the prior list
};

size_t align256(size_t v) { return (v + 255) & ~static_cast<size_t>(255); }

size_t workspace_bytes(int64_t rows) {
  if (rows <= 0 || rows >= kSemidDedupMaxRows) return 0;
  const size_t n = static_cast<size_t>(rows);
  return sort_workspace_bytes(rows) + align256(scan_temp_bytes(rows)) + align256((n + 1) * 8) + align256(n * 8) + 256;
}

bool carve(void* workspace, size_t bytes, int64_t rows, Work* w) {
  const size_t sort_bytes = sort_workspace_bytes(rows);
  if (workspace == nullptr || bytes < workspace_bytes(rows) || !sort_carve(workspace, sort_bytes, rows, &w->sort)) return false;
  uint8_t* p = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + sort_bytes + 255) & ~static_cast<uintptr_t>(255));
  w->scan_temp = p;
  w->scan_temp_bytes = scan_temp_bytes(rows);
  p += align256(w->scan_temp_bytes);
  w->run_start = reinterpret_cast<int64_t*>(p);
  p += align256((static_cast<size_t>(rows) + 1) * 8);
  w->run_prior = reinterpret_cast<int64_t*>(p);
  return true;
}

struct IdRows {
  const int64_t* ids;
  int64_t rows, width, row_stride, col_stride;
  int bits;
};

// key = sum_c ids[c] << bits * (width - 1 - c); invalid rows get max_key and the kInvalidRow bit, and their digit (-1) here
__global__ void __launch_bounds__(kThreads) dedup_keys_kernel(IdRows a, uint64_t max_key, uint64_t* __restrict__ keys,
                                                              uint32_t* __restrict__ rows_out, int64_t* __restrict__ digits,
                                                              int64_t digit_stride, int64_t* __restrict__ stats) {
  const int64_t r = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x;
  bool bad = false;
  if (r < a.rows) {
    const int64_t* row = a.ids + r * a.row_stride;
    uint64_t key = 0;
    for (int64_t c = 0; c < a.width; ++c) {
      const int64_t v = row[c * a.col_stride];
      bad |= (v >> a.bits) != 0;  // negative, or 2^bits and above
      key = (key << a.bits) | static_cast<uint64_t>(v);
    }
    keys[r] = bad ? max_key : key;
    rows_out[r] = static_cast<uint32_t>(r) | (bad ? kInvalidRow : 0u);
    if (bad) digits[r * digit_stride] = -1;
  }
  const int n_bad = __syncthreads_count(bad);
  if (threadIdx.x == 0 && n_bad) atomicAdd(reinterpret_cast<unsigned long long*>(stats + 2), static_cast<unsigned long long>(n_bad));
}

__device__ __forceinline__ bool is_head(const uint64_t* keys, int64_t p) { return p == 0 || keys[p] != keys[p - 1]; }

// word of sorted position p: (1 if a run starts here) << 32 | (1 if the row is valid).  Their inclusive sum holds the run
// index + 1 in the high half and the valid rows up to p in the low half (< 2^31: no carry into the high half).
__global__ void __launch_bounds__(kThreads) dedup_flags_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ rows,
                                                               int64_t n, uint64_t* __restrict__ words) {
  const int64_t p = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x;
  if (p >= n) return;
  words[p] = (is_head(keys, p) ? (1ull << 32) : 0ull) | ((rows[p] & kInvalidRow) ? 0ull : 1ull);
}

// at every run head: the run's key, the valid rows before it and its count in the prior list (binary search)
__global__ void __launch_bounds__(kThreads) dedup_runs_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ rows,
                                                              const uint64_t* __restrict__ scan, int64_t n,
                                                              const int64_t* __restrict__ prior_keys,
                                                              const int64_t* __restrict__ prior_counts, int64_t n_prior,
                                                              int64_t* __restrict__ run_keys, int64_t* __restrict__ run_start,
                                                              int64_t* __restrict__ run_prior) {
  const int64_t p = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x;
  if (p >= n) return;
  const uint64_t s = scan[p];
  const int64_t run = static_cast<int64_t>(s >> 32) - 1;
  const int64_t valid_incl = static_cast<int64_t>(s & 0xffffffffull);
  if (p == n - 1) run_start[run + 1] = valid_incl;
  if (!is_head(keys, p)) return;
  const int64_t key = static_cast<int64_t>(keys[p]);
  run_keys[run] = key;
  run_start[run] = valid_incl - ((rows[p] & kInvalidRow) ? 0 : 1);
  int64_t lo = 0, hi = n_prior;  // first prior key >= key
  while (lo < hi) {
    const int64_t mid = lo + ((hi - lo) >> 1);
    if (prior_keys[mid] < key) lo = mid + 1;
    else hi = mid;
  }
  run_prior[run] = (lo < n_prior && prior_keys[lo] == key) ? prior_counts[lo] : 0;
}

// digits of the valid rows; run counts, the number of distinct tuples and the largest digit
__global__ void __launch_bounds__(kThreads) dedup_finish_kernel(const uint32_t* __restrict__ rows, const uint64_t* __restrict__ scan,
                                                                int64_t n, const int64_t* __restrict__ run_start,
                                                                const int64_t* __restrict__ run_prior, int64_t* __restrict__ digits,
                                                                int64_t digit_stride, int64_t* __restrict__ run_counts,
                                                                int64_t* __restrict__ stats) {
  __shared__ long long s_max[kThreads / 32];
  const int64_t p = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x;
  long long top = -1;  // largest digit of run p
  if (p < n) {
    const uint64_t s = scan[p];
    const uint32_t row = rows[p];
    if (!(row & kInvalidRow)) {
      const int64_t run = static_cast<int64_t>(s >> 32) - 1;
      digits[static_cast<int64_t>(row) * digit_stride] = static_cast<int64_t>(s & 0xffffffffull) - 1 - run_start[run] + run_prior[run];
    }
    const int64_t n_runs = static_cast<int64_t>(scan[n - 1] >> 32);
    if (p < n_runs) {
      const int64_t count = run_start[p + 1] - run_start[p];  // 0 only for a last run made of invalid rows alone
      run_counts[p] = count;
      if (count > 0) top = run_prior[p] + count - 1;
      if (p == n_runs - 1) stats[0] = count > 0 ? n_runs : n_runs - 1;
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const long long o = __shfl_xor_sync(0xffffffffu, top, off);
    top = o > top ? o : top;
  }
  if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = top;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kThreads / 32; ++w) top = s_max[w] > top ? s_max[w] : top;
    if (top >= 0) atomicMax(reinterpret_cast<long long*>(stats + 1), top);
  }
}

}  // namespace

size_t semid_dedup_workspace_bytes(int64_t rows) { return workspace_bytes(rows); }

int launch_semid_dedup(const SemidDedupArgs& d, void* workspace, size_t workspace_bytes, cudaStream_t s) {
  HV_CUDA_CHECK(cudaMemsetAsync(d.stats, 0, 3 * sizeof(int64_t), s));
  HV_CUDA_CHECK(cudaMemsetAsync(d.stats + 1, 0xff, sizeof(int64_t), s));  // largest digit: -1 until a valid row is seen
  if (d.rows == 0) return HV_OK;
  Work w;
  if (!carve(workspace, workspace_bytes, d.rows, &w)) {
    set_error("hv_semid_dedup: workspace of %zu bytes, %zu needed", workspace ? workspace_bytes : 0, hv::workspace_bytes(d.rows));
    return HV_ERR_WORKSPACE;
  }
  const int end_bit = static_cast<int>(d.width) * d.bits;
  const uint64_t max_key = (1ull << end_bit) - 1;
  const unsigned grid = static_cast<unsigned>((d.rows + kThreads - 1) / kThreads);
  IdRows a{d.ids, d.rows, d.width, d.row_stride, d.col_stride, d.bits};
  dedup_keys_kernel<<<grid, kThreads, 0, s>>>(a, max_key, w.sort.keys_in, w.sort.vals_in, d.digits, d.digit_stride, d.stats);
  HV_CUDA_CHECK(cudaGetLastError());
  if (int st = sort_pairs(w.sort, d.rows, end_bit, s)) return st;
  uint64_t* words = w.sort.keys_in;
  dedup_flags_kernel<<<grid, kThreads, 0, s>>>(w.sort.keys_out, w.sort.vals_out, d.rows, words);
  HV_CUDA_CHECK(cudaGetLastError());
  if (int st = inclusive_sum_u64(w.scan_temp, w.scan_temp_bytes, words, d.rows, s)) return st;
  dedup_runs_kernel<<<grid, kThreads, 0, s>>>(w.sort.keys_out, w.sort.vals_out, words, d.rows, d.prior_keys, d.prior_counts,
                                              d.n_prior, d.run_keys, w.run_start, w.run_prior);
  HV_CUDA_CHECK(cudaGetLastError());
  dedup_finish_kernel<<<grid, kThreads, 0, s>>>(w.sort.vals_out, words, d.rows, w.run_start, w.run_prior, d.digits, d.digit_stride,
                                                d.run_counts, d.stats);
  HV_CUDA_CHECK(cudaGetLastError());
  return HV_OK;
}

}  // namespace hv
