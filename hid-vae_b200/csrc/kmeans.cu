// K-means codebook init, the update half of one Lloyd iteration (init/kmeans.py:52-61) -- HBM/L2-bound.
//
// The assignment half is hv_rq_forward with n_levels = 1 (HV_ALGO_SIMT_DIFF reproduces the reference's
// difference-form table, init/kmeans.py:44-47).  Here:
//   hv_kmeans_accumulate  per-cluster sums / counts of the assigned rows, bit-reproducible from run to run.  That
//                         matters: the reference stops when max ||c_new - c_old|| < 1e-10 (init/kmeans.py:68), i.e.
//                         when the update reproduces the centroids exactly, which an atomics-ordered float sum never does.
//                         Every row chain is a compensated (Kahan) sum in a fixed order: its error stays about two
//                         ulps of sum |x| however many rows a cluster holds (a plain fp32 chain grows with the chain, to
//                         1e-2 relative for 2^20 identical rows), and the order keeps the result bit-reproducible.
//                         Assignments must lie in [0, K).  Two forms, chosen by shape only:
//                           segmented (needs the sort workspace; O(N)): rows are key-sorted by cluster (stable radix
//                             sort, sort.cuh) and ONE WARP PER CLUSTER adds its members in row order -- x is read once,
//                             whatever K is;
//                           scan (small K * N, or no workspace): one CTA per cluster walks the whole assignment vector
//                             (K * N index reads out of L2) and adds its members in a fixed-shape tree.
//   hv_kmeans_finalize    means, empty-cluster reseed, max centroid shift: one warp per cluster.
#include "common.cuh"
#include "ptx.cuh"
#include "sort.cuh"

namespace hv {
namespace {

constexpr int kAccThreads = 256;

// one step of a compensated sum: s - comp is the running total to about twice fp32's precision (comp holds the
// negated low part the last addition lost)
__device__ __forceinline__ void kahan_add(float& s, float& comp, float v) {
  const float y = v - comp;
  const float t = s + y;
  comp = (t - s) - y;
  s = t;
}

template <int D>
__global__ void __launch_bounds__(kAccThreads) kmeans_accumulate_kernel(const float* __restrict__ x, int64_t n,
                                                                        const int64_t* __restrict__ assign,
                                                                        const int64_t* __restrict__ prev_assign, int k,
                                                                        float* __restrict__ sums, float* __restrict__ counts,
                                                                        unsigned long long* __restrict__ n_changed) {
  __shared__ float s_part[kAccThreads / 32][D + 1];
  const int c = blockIdx.x;
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = ptx::warp_index();

  // thread t adds rows t, t + 256, ... of its cluster in one compensated chain per dimension; the assignments of 4 of its
  // rows are loaded ahead (independent loads), then the rows are taken in order
  float acc[D], cmp[D];
#pragma unroll
  for (int i = 0; i < D; ++i) acc[i] = 0.f, cmp[i] = 0.f;
  float cnt = 0.f;
  for (int64_t base = tid; base < n; base += 4 * kAccThreads) {
    int64_t a4[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) a4[u] = base + u * kAccThreads < n ? __ldg(assign + base + u * kAccThreads) : -1;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (a4[u] != c) continue;
      const float4* src = reinterpret_cast<const float4*>(x + (base + u * kAccThreads) * D);
#pragma unroll
      for (int i = 0; i < D / 4; ++i) {
        const float4 v = __ldg(src + i);
        kahan_add(acc[4 * i], cmp[4 * i], v.x);
        kahan_add(acc[4 * i + 1], cmp[4 * i + 1], v.y);
        kahan_add(acc[4 * i + 2], cmp[4 * i + 2], v.z);
        kahan_add(acc[4 * i + 3], cmp[4 * i + 3], v.w);
      }
      cnt += 1.f;
    }
  }
  // fixed-shape reduction of the corrected chains: xor tree inside the warp, then the 8 warp partials in warp order
#pragma unroll
  for (int i = 0; i < D; ++i) {
    float v = acc[i] - cmp[i];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if (lane == 0) s_part[warp][i] = v;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
  if (lane == 0) s_part[warp][D] = cnt;
  __syncthreads();
  for (int i = tid; i <= D; i += kAccThreads) {
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < kAccThreads / 32; ++w) v += s_part[w][i];
    if (i < D)
      sums[static_cast<int64_t>(c) * D + i] = v;
    else
      counts[c] = v;
  }

  if (n_changed != nullptr) {
    // every CTA also counts the changed assignments of its own slice of the rows (integer sum: order-free)
    const int64_t per = (n + k - 1) / k;
    const int64_t lo = static_cast<int64_t>(c) * per;
    const int64_t hi = lo + per < n ? lo + per : n;
    unsigned int changed = 0;
    for (int64_t row = lo + tid; row < hi; row += kAccThreads)
      changed += (prev_assign == nullptr || prev_assign[row] != assign[row]) ? 1u : 0u;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) changed += __shfl_xor_sync(0xffffffffu, changed, off);
    if (lane == 0 && changed) atomicAdd(n_changed, static_cast<unsigned long long>(changed));
  }
}

// ---- segmented form -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) kmeans_keys_kernel(const int64_t* __restrict__ assign, const int64_t* __restrict__ prev_assign,
                                                          int64_t n, uint64_t* __restrict__ keys, uint32_t* __restrict__ vals,
                                                          unsigned long long* __restrict__ n_changed) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  unsigned int changed = 0;
  if (i < n) {
    const int64_t a = assign[i];
    keys[i] = static_cast<uint64_t>(a);
    vals[i] = static_cast<uint32_t>(i);
    changed = (prev_assign == nullptr || prev_assign[i] != a) ? 1u : 0u;
  }
  if (n_changed != nullptr) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) changed += __shfl_xor_sync(0xffffffffu, changed, off);
    if ((threadIdx.x & 31) == 0 && changed) atomicAdd(n_changed, static_cast<unsigned long long>(changed));
  }
}

__device__ __forceinline__ int64_t lower_bound_u64(const uint64_t* __restrict__ a, int64_t n, uint64_t v) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (a[mid] < v) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// one warp per cluster: its members sit in [lo, hi) of the sorted order, in ascending row order (stable sort); lane l owns
// dimensions l, l + 32, ...; 32 row indices are fetched per step and their rows are loaded back to back (independent
// loads), then added in row order to one compensated chain per dimension -- a fixed order whatever the launch shape.
template <int D>
__global__ void __launch_bounds__(256) kmeans_segsum_kernel(const float* __restrict__ x, int64_t n, const uint64_t* __restrict__ keys,
                                                            const uint32_t* __restrict__ rows, int k, float* __restrict__ sums,
                                                            float* __restrict__ counts) {
  constexpr int PER = (D + 31) / 32;
  const int c = ptx::uniform((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= k) return;
  const int64_t lo = lower_bound_u64(keys, n, static_cast<uint64_t>(c));
  const int64_t hi = lower_bound_u64(keys, n, static_cast<uint64_t>(c) + 1);
  float acc[PER], cmp[PER];
#pragma unroll
  for (int p = 0; p < PER; ++p) acc[p] = 0.f, cmp[p] = 0.f;
  for (int64_t base = lo; base < hi; base += 32) {
    const int m = static_cast<int>(hi - base < 32 ? hi - base : 32);
    const uint32_t mine = lane < m ? rows[base + lane] : 0u;
    float v[8][PER];
    for (int t0 = 0; t0 < m; t0 += 8) {
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const uint32_t r = __shfl_sync(0xffffffffu, mine, (t0 + t) & 31);
#pragma unroll
        for (int p = 0; p < PER; ++p)
          v[t][p] = (t0 + t < m && lane + 32 * p < D) ? __ldg(x + static_cast<int64_t>(r) * D + lane + 32 * p) : 0.f;
      }
#pragma unroll
      for (int t = 0; t < 8; ++t)
        if (t0 + t < m)
#pragma unroll
          for (int p = 0; p < PER; ++p) kahan_add(acc[p], cmp[p], v[t][p]);
    }
  }
#pragma unroll
  for (int p = 0; p < PER; ++p)
    if (lane + 32 * p < D) sums[static_cast<int64_t>(c) * D + lane + 32 * p] = acc[p] - cmp[p];
  if (lane == 0) counts[c] = static_cast<float>(hi - lo);
}

template <int D>
int launch_segmented(const float* x, int64_t n, const int64_t* assign, const int64_t* prev, int k, float* sums, float* counts,
                     int64_t* n_changed, const SortBuffers& b, cudaStream_t s) {
  kmeans_keys_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(assign, prev, n, b.keys_in, b.vals_in,
                                                                            reinterpret_cast<unsigned long long*>(n_changed));
  HV_CUDA_CHECK(cudaGetLastError());
  int bits = 1;
  while ((1ll << bits) < k) ++bits;
  if (int st = sort_pairs(b, n, bits, s)) return st;
  kmeans_segsum_kernel<D><<<(k * 32 + 255) / 256, 256, 0, s>>>(x, n, b.keys_out, b.vals_out, k, sums, counts);
  HV_CUDA_CHECK(cudaGetLastError());
  return HV_OK;
}

// one warp per cluster, lanes over the dimensions (coalesced); the two statistics are order-independent reductions (a maximum
// of non-negative floats through their bit pattern, an integer-valued count), so the result does not depend on the schedule
__global__ void __launch_bounds__(256) kmeans_finalize_kernel(const float* __restrict__ sums, const float* __restrict__ counts,
                                                             const float* __restrict__ reseed_rows, int k, int d,
                                                             float* __restrict__ centroids, float* __restrict__ stats) {
  const int c = ptx::uniform((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= k) return;
  const float cnt = counts[c];
  const bool empty = !(cnt > 0.f);
  float shift2 = 0.f;
  for (int i = lane; i < d; i += 32) {
    const int64_t o = static_cast<int64_t>(c) * d + i;
    const float old = centroids[o];
    float nv;
    if (!empty)
      nv = sums[o] / cnt;  // x[members].mean(axis=0), init/kmeans.py:60
    else
      nv = reseed_rows != nullptr ? reseed_rows[o] : old;  // init/kmeans.py:56
    const float df = nv - old;
    shift2 = fmaf(df, df, shift2);
    centroids[o] = nv;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) shift2 += __shfl_xor_sync(0xffffffffu, shift2, off);
  if (lane == 0) {
    atomicMax(reinterpret_cast<int*>(stats), __float_as_int(sqrtf(shift2)));
    if (empty) atomicAdd(stats + 1, 1.0f);
  }
}

template <int D>
int launch_acc(const float* x, int64_t n, const int64_t* assign, const int64_t* prev, int k, float* sums, float* counts,
               int64_t* n_changed, cudaStream_t s) {
  kmeans_accumulate_kernel<D><<<k, kAccThreads, 0, s>>>(x, n, assign, prev, k, sums, counts,
                                                        reinterpret_cast<unsigned long long*>(n_changed));
  HV_CUDA_CHECK(cudaGetLastError());
  return HV_OK;
}

}  // namespace
}  // namespace hv

extern "C" int hv_kmeans_accumulate(const float* x, int64_t n, int d, const int64_t* assign, const int64_t* prev_assign,
                                    int k, float* sums, float* counts, int64_t* n_changed, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  using namespace hv;
  if (n < 0 || d <= 0 || k <= 0) {
    set_error("hv_kmeans_accumulate: bad shape n=%lld d=%d k=%d", (long long)n, d, k);
    return HV_ERR_BAD_SHAPE;
  }
  if (!sums || !counts || (n > 0 && (!x || !assign))) {
    set_error("hv_kmeans_accumulate: null pointer");
    return HV_ERR_NULL;
  }
  if (n > 0 && !aligned16(x)) {
    set_error("hv_kmeans_accumulate: x must be 16-byte aligned");
    return HV_ERR_MISALIGNED;
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (n_changed != nullptr) HV_CUDA_CHECK(cudaMemsetAsync(n_changed, 0, sizeof(int64_t), s));
  // the scan form reads K * N indices: beyond ~2^24 of them (K = 256 x N = 65,536) the segmented form wins
  SortBuffers bufs;
  if (n > 0 && static_cast<int64_t>(k) * n > (1ll << 24) && sort_carve(workspace, workspace_bytes, n, &bufs)) {
    switch (d) {
      case 4: return launch_segmented<4>(x, n, assign, prev_assign, k, sums, counts, n_changed, bufs, s);
      case 8: return launch_segmented<8>(x, n, assign, prev_assign, k, sums, counts, n_changed, bufs, s);
      case 16: return launch_segmented<16>(x, n, assign, prev_assign, k, sums, counts, n_changed, bufs, s);
      case 32: return launch_segmented<32>(x, n, assign, prev_assign, k, sums, counts, n_changed, bufs, s);
      case 64: return launch_segmented<64>(x, n, assign, prev_assign, k, sums, counts, n_changed, bufs, s);
      case 128: return launch_segmented<128>(x, n, assign, prev_assign, k, sums, counts, n_changed, bufs, s);
      default: break;
    }
  }
  switch (d) {
    case 4: return launch_acc<4>(x, n, assign, prev_assign, k, sums, counts, n_changed, s);
    case 8: return launch_acc<8>(x, n, assign, prev_assign, k, sums, counts, n_changed, s);
    case 16: return launch_acc<16>(x, n, assign, prev_assign, k, sums, counts, n_changed, s);
    case 32: return launch_acc<32>(x, n, assign, prev_assign, k, sums, counts, n_changed, s);
    case 64: return launch_acc<64>(x, n, assign, prev_assign, k, sums, counts, n_changed, s);
    case 128: return launch_acc<128>(x, n, assign, prev_assign, k, sums, counts, n_changed, s);
    default:
      set_error("hv_kmeans_accumulate: embed dim %d has no instantiation (supported: 4, 8, 16, 32, 64, 128)", d);
      return HV_ERR_UNSUPPORTED;
  }
}

extern "C" int hv_kmeans_finalize(const float* sums, const float* counts, const float* reseed_rows, int k, int d,
                                  float* centroids, float* stats, void* stream) {
  using namespace hv;
  if (d <= 0 || k <= 0) {
    set_error("hv_kmeans_finalize: bad shape d=%d k=%d", d, k);
    return HV_ERR_BAD_SHAPE;
  }
  if (!sums || !counts || !centroids || !stats) {
    set_error("hv_kmeans_finalize: null pointer");
    return HV_ERR_NULL;
  }
  HV_CUDA_CHECK(cudaMemsetAsync(stats, 0, 2 * sizeof(float), static_cast<cudaStream_t>(stream)));
  kmeans_finalize_kernel<<<(k * 32 + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(sums, counts, reseed_rows, k, d, centroids, stats);
  HV_CUDA_CHECK(cudaGetLastError());
  return HV_OK;
}
