// Semantic-ID uniqueness loss (modules/h_rqvae.py:41-105) and p_unique_ids (:645-648).
//
// The reference materialises a [B, B, L] equality tensor, calls torch.where (a host sync) and gathers pairs.
// Here every row is hashed to a 64-bit key; a tile sweep compares keys of all pairs i < j out of shared memory
// (B^2/2 eight-byte compares, no HBM traffic beyond the ids), and only key-equal pairs -- verified element by
// element, so the hash never decides -- touch the feature rows.  Sums are kept in double, one atomic per CTA.
// No host-side data-dependent control flow: the call is CUDA-graph capturable.
// Beyond a few thousand rows the B^2/2 sweep is replaced by a SORT: rows are key-sorted by the hash of their tuple (stable
// radix sort, sort.cuh), identical tuples then sit in one run in ascending row order, and a thread per sorted position
// walks the rest of its run -- O(B + pairs) instead of O(B^2) (the loss itself is a sum over pairs of identical tuples).
#include "common.cuh"
#include "ptx.cuh"
#include "sort.cuh"

namespace hv {
namespace {

constexpr int kTile = 256;

struct UniqArgs {
  const int64_t* ids;
  int64_t rows, width, row_stride, col_stride;
  const float* feats;
  int d;
  float margin;
};

__device__ __forceinline__ uint64_t mix64(uint64_t h, uint64_t v) {
  h ^= v + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2);
  h *= 0xFF51AFD7ED558CCDull;
  return h ^ (h >> 33);
}

__device__ __forceinline__ uint64_t row_key(const UniqArgs& a, int64_t r) {
  uint64_t h = 0x243F6A8885A308D3ull;
  for (int64_t c = 0; c < a.width; ++c) h = mix64(h, static_cast<uint64_t>(a.ids[r * a.row_stride + c * a.col_stride]));
  return h;
}

__device__ __forceinline__ bool same_tuple(const UniqArgs& a, int64_t i, int64_t j) {
  for (int64_t c = 0; c < a.width; ++c)
    if (a.ids[i * a.row_stride + c * a.col_stride] != a.ids[j * a.row_stride + c * a.col_stride]) return false;
  return true;
}

// cos(f_i, f_j) with F.normalize's eps = 1e-12 clamp on each norm (modules/h_rqvae.py:88-92)
struct PairCos {
  float cs, inv_i, inv_j;
  bool clamped_i, clamped_j;  // the norm is below the clamp: the row is divided by the constant 1e-12
};

__device__ __forceinline__ PairCos pair_cos(const UniqArgs& a, int64_t i, int64_t j) {
  const float* fi = a.feats + i * a.d;
  const float* fj = a.feats + j * a.d;
  float ii = 0.f, jj = 0.f, ij = 0.f;
  for (int c = 0; c < a.d; ++c) {
    const float u = fi[c], v = fj[c];
    ii = fmaf(u, u, ii), jj = fmaf(v, v, jj), ij = fmaf(u, v, ij);
  }
  PairCos p;
  const float ni = sqrtf(ii), nj = sqrtf(jj);
  p.clamped_i = ni < 1e-12f, p.clamped_j = nj < 1e-12f;
  p.inv_i = 1.0f / fmaxf(ni, 1e-12f);
  p.inv_j = 1.0f / fmaxf(nj, 1e-12f);
  p.cs = ij * p.inv_i * p.inv_j;
  return p;
}

// g_feats[i] += coef * d cos / d f_i and g_feats[j] += coef * d cos / d f_j.
// Above the clamp, d cos / d f_i = P_i e / |f_i| with e = fhat_j - fhat_i and P_i = I - fhat_i fhat_i^T (P_i fhat_i = 0):
// the same vector as (fhat_j - cos fhat_i) / |f_i|, without its cancellation.  With s the row of the smaller norm and
// inv_lo the other row's inverse norm, e = (f_j - f_i) inv_lo + f_s (inv_j - inv_i): no term exceeds 2 in size, f_j - f_i
// is exact for near-identical rows, and the rounding of the two norms only moves e along f_s, which P_s removes (and the
// other row's P up to |e|).  So near-identical rows keep fp32's relative precision, and identical rows get exactly 0 (the
// products are kept out of FMA contraction for that).  Below the clamp, the row is divided by the constant 1e-12, whose
// derivative is zero: d cos / d f_i = fhat_j * inv_i, no projection.
__device__ __forceinline__ void pair_grad(const UniqArgs& a, int64_t i, int64_t j, const PairCos& p, float coef,
                                          float* __restrict__ g_feats) {
  const float* fi = a.feats + i * a.d;
  const float* fj = a.feats + j * a.d;
  const bool j_small = p.inv_j >= p.inv_i;
  const float* fs = j_small ? fj : fi;
  const float inv_lo = j_small ? p.inv_i : p.inv_j;
  const float dinv = p.inv_j - p.inv_i;
  float si = 0.f, sj = 0.f;  // fhat_i . e, fhat_j . e
  for (int c = 0; c < a.d; ++c) {
    const float e = fmaf(fj[c] - fi[c], inv_lo, __fmul_rn(fs[c], dinv));
    si = fmaf(__fmul_rn(fi[c], p.inv_i), e, si);
    sj = fmaf(__fmul_rn(fj[c], p.inv_j), e, sj);
  }
  const float ci = coef * p.inv_i, cj = coef * p.inv_j;
  for (int c = 0; c < a.d; ++c) {
    const float hi = __fmul_rn(fi[c], p.inv_i), hj = __fmul_rn(fj[c], p.inv_j);
    const float e = fmaf(fj[c] - fi[c], inv_lo, __fmul_rn(fs[c], dinv));
    atomicAdd(g_feats + i * a.d + c, ci * (p.clamped_i ? hj : fmaf(-si, hi, e)));
    atomicAdd(g_feats + j * a.d + c, cj * (p.clamped_j ? hi : fmaf(sj, hj, -e)));
  }
}

// one pair i < j of identical tuples, in both kernels: its forward statistics, or its share of the gradient
template <bool BACKWARD>
__device__ __forceinline__ void visit_pair(const UniqArgs& a, int64_t i, int64_t j, float coef, float* __restrict__ g_feats,
                                           double& hinge_sum, double& pair_count, double& has_later) {
  const PairCos p = pair_cos(a, i, j);
  const float hinge = p.cs - a.margin;
  if (!BACKWARD) {
    has_later = 1.0;
    pair_count += 1.0;
    if (hinge > 0.f) hinge_sum += static_cast<double>(hinge);
  } else if (hinge > 0.f && coef != 0.f) {
    pair_grad(a, i, j, p, coef, g_feats);
  }
}

// Keys of rows [row0, row0 + kTile) into s_keys (every thread of the CTA calls it; rows past the end get 0).  Narrow rows:
// a thread per row.  Wide rows (the as-wired transposed call of the reference hands over [L, B]: 3 rows of B ids): a warp
// per row, lanes striding the columns, lane hashes combined order-independently -- a row of 8,192 ids is 256 loads per lane
// instead of a serial chain of 8,192.  Any deterministic function of the row's content serves as a key: equal keys are
// always confirmed element by element.
__device__ __forceinline__ void tile_keys(const UniqArgs& a, int64_t row0, uint64_t* s_keys) {
  if (a.width <= 64) {
    const int64_t r = row0 + threadIdx.x;
    s_keys[threadIdx.x] = r < a.rows ? row_key(a, r) : 0ull;
    return;
  }
  const int lane = threadIdx.x & 31, warp = ptx::warp_index();
  for (int t = warp; t < kTile; t += kTile / 32) {
    const int64_t r = row0 + t;
    uint64_t h = 0ull;
    if (r < a.rows) {
      h = 0x243F6A8885A308D3ull + static_cast<uint64_t>(lane);
      for (int64_t c = lane; c < a.width; c += 32) h = mix64(h, static_cast<uint64_t>(a.ids[r * a.row_stride + c * a.col_stride]));
      h = mix64(h, static_cast<uint64_t>(lane) + 1ull);
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) h ^= __shfl_xor_sync(0xffffffffu, h, off);
    }
    if (lane == 0) s_keys[t] = h;
  }
}

template <typename T>
__device__ __forceinline__ T block_sum(T v, T* scratch) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  const int lane = threadIdx.x & 31, warp = ptx::warp_index();
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  T total = 0;
  if (threadIdx.x == 0)
    for (int w = 0; w < kTile / 32; ++w) total += scratch[w];
  return total;  // valid in thread 0
}

// BACKWARD = false: stats[0] += sum of hinges, stats[1] += pairs, stats[2] += rows with a later identical row
// BACKWARD = true : g_feats += coef * d(sum of hinges)/d feats, coef = g_out * weight / stats[1]
template <bool BACKWARD>
__global__ void __launch_bounds__(kTile) uniq_kernel(UniqArgs a, double* __restrict__ stats_out, const double* __restrict__ stats_in,
                                                     float weight, const float* __restrict__ g_out, float* __restrict__ g_feats) {
  __shared__ uint64_t s_keys[kTile];
  __shared__ double s_scratch[kTile / 32];

  const int64_t i = static_cast<int64_t>(blockIdx.x) * kTile + threadIdx.x;
  const bool valid_i = i < a.rows;
  const int64_t n_tiles = (a.rows + kTile - 1) / kTile;

  float coef = 0.f;
  if (BACKWARD) {
    const double pairs = stats_in[1];
    if (!(pairs > 0.0)) return;  // no identical pair in the batch (uniform across the grid): the gradient is zero
    coef = static_cast<float>(static_cast<double>(g_out[0]) * weight / pairs);
  }
  tile_keys(a, static_cast<int64_t>(blockIdx.x) * kTile, s_keys);
  __syncthreads();
  const uint64_t my_key = s_keys[threadIdx.x];

  double hinge_sum = 0.0, pair_count = 0.0, has_later = 0.0;
  for (int64_t jt = blockIdx.x; jt < n_tiles; ++jt) {
    if (jt > blockIdx.x) {  // (the first tile of the sweep is the CTA's own: its keys are in place)
      __syncthreads();
      tile_keys(a, jt * kTile, s_keys);
      __syncthreads();
    }
    if (!valid_i) continue;
    const int64_t j0 = jt * kTile;
    const int j_end = static_cast<int>(a.rows - j0 < kTile ? a.rows - j0 : kTile);
    for (int jj = 0; jj < j_end; ++jj) {
      if (s_keys[jj] != my_key) continue;
      const int64_t j = j0 + jj;
      if (j <= i || !same_tuple(a, i, j)) continue;
      visit_pair<BACKWARD>(a, i, j, coef, g_feats, hinge_sum, pair_count, has_later);
    }
  }
  if (!BACKWARD) {
    const double t0 = block_sum<double>(hinge_sum, s_scratch);
    const double t1 = block_sum<double>(pair_count, s_scratch);
    const double t2 = block_sum<double>(has_later, s_scratch);
    if (threadIdx.x == 0) {
      if (t0 != 0.0) atomicAdd(stats_out + 0, t0);
      if (t1 != 0.0) atomicAdd(stats_out + 1, t1);
      if (t2 != 0.0) atomicAdd(stats_out + 2, t2);
    }
  }
}

// ---- sorted form ----------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kTile) uniq_keys_kernel(UniqArgs a, uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * kTile + threadIdx.x;
  if (i < a.rows) {
    keys[i] = row_key(a, i);
    vals[i] = static_cast<uint32_t>(i);
  }
}

template <bool BACKWARD>
__global__ void __launch_bounds__(kTile) uniq_sorted_kernel(UniqArgs a, const uint64_t* __restrict__ keys, const uint32_t* __restrict__ order,
                                                            double* __restrict__ stats_out, const double* __restrict__ stats_in, float weight,
                                                            const float* __restrict__ g_out, float* __restrict__ g_feats) {
  __shared__ double s_scratch[kTile / 32];
  const int64_t p = static_cast<int64_t>(blockIdx.x) * kTile + threadIdx.x;
  float coef = 0.f;
  if (BACKWARD) {
    const double pairs = stats_in[1];
    if (!(pairs > 0.0)) return;  // no identical pair: zero gradient
    coef = static_cast<float>(static_cast<double>(g_out[0]) * weight / pairs);
  }
  double hinge_sum = 0.0, pair_count = 0.0, has_later = 0.0;
  if (p < a.rows) {
    const uint64_t my_key = keys[p];
    const int64_t i = order[p];
    for (int64_t q = p + 1; q < a.rows && keys[q] == my_key; ++q) {
      const int64_t j = order[q];  // (stable sort: j > i)
      if (!same_tuple(a, i, j)) continue;
      visit_pair<BACKWARD>(a, i, j, coef, g_feats, hinge_sum, pair_count, has_later);
    }
  }
  if (!BACKWARD) {
    const double t0 = block_sum<double>(hinge_sum, s_scratch);
    const double t1 = block_sum<double>(pair_count, s_scratch);
    const double t2 = block_sum<double>(has_later, s_scratch);
    if (threadIdx.x == 0) {
      if (t0 != 0.0) atomicAdd(stats_out + 0, t0);
      if (t1 != 0.0) atomicAdd(stats_out + 1, t1);
      if (t2 != 0.0) atomicAdd(stats_out + 2, t2);
    }
  }
}

constexpr int64_t kSortFromRows = 4096;  // below: the pairwise sweep is one small launch and wins

template <bool BACKWARD>
int launch_sorted(const UniqArgs& a, const SortBuffers& b, double* stats_out, const double* stats_in, float weight, const float* g_out,
                  float* g_feats, cudaStream_t s) {
  const unsigned grid = static_cast<unsigned>((a.rows + kTile - 1) / kTile);
  uniq_keys_kernel<<<grid, kTile, 0, s>>>(a, b.keys_in, b.vals_in);
  HV_CUDA_CHECK(cudaGetLastError());
  if (int st = sort_pairs(b, a.rows, 64, s)) return st;
  uniq_sorted_kernel<BACKWARD><<<grid, kTile, 0, s>>>(a, b.keys_out, b.vals_out, stats_out, stats_in, weight, g_out, g_feats);
  HV_CUDA_CHECK(cudaGetLastError());
  return HV_OK;
}

int check(const int64_t* ids, int64_t rows, int64_t width, const float* feats, int d, const char* who) {
  if (rows < 0 || width <= 0 || d < 0) {
    set_error("%s: bad shape rows=%lld width=%lld d=%d", who, (long long)rows, (long long)width, d);
    return HV_ERR_BAD_SHAPE;
  }
  if (rows > 0 && (!ids || (d > 0 && !feats))) {
    set_error("%s: null pointer", who);
    return HV_ERR_NULL;
  }
  return HV_OK;
}

}  // namespace
}  // namespace hv

extern "C" int hv_uniq_forward(const int64_t* ids, int64_t rows, int64_t width, int64_t row_stride, int64_t col_stride,
                               const float* feats, int d, float margin, double* stats, void* workspace, size_t workspace_bytes,
                               void* stream) {
  using namespace hv;
  if (int st = check(ids, rows, width, feats, d, "hv_uniq_forward")) return st;
  if (!stats) {
    set_error("hv_uniq_forward: stats is null");
    return HV_ERR_NULL;
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  HV_CUDA_CHECK(cudaMemsetAsync(stats, 0, 3 * sizeof(double), s));
  if (rows == 0) return HV_OK;
  UniqArgs a{ids, rows, width, row_stride, col_stride, feats, d, margin};
  SortBuffers bufs;
  if (rows >= kSortFromRows && sort_carve(workspace, workspace_bytes, rows, &bufs))
    return launch_sorted<false>(a, bufs, stats, nullptr, 0.f, nullptr, nullptr, s);
  const unsigned grid = static_cast<unsigned>((rows + kTile - 1) / kTile);
  uniq_kernel<false><<<grid, kTile, 0, s>>>(a, stats, nullptr, 0.f, nullptr, nullptr);
  HV_CUDA_CHECK(cudaGetLastError());
  return HV_OK;
}

extern "C" int hv_uniq_backward(const int64_t* ids, int64_t rows, int64_t width, int64_t row_stride, int64_t col_stride,
                                const float* feats, int d, float margin, float weight, const double* stats,
                                const float* g_out, float* g_feats, void* workspace, size_t workspace_bytes, void* stream) {
  using namespace hv;
  if (int st = check(ids, rows, width, feats, d, "hv_uniq_backward")) return st;
  if (!stats || !g_out || (rows > 0 && d > 0 && !g_feats)) {
    set_error("hv_uniq_backward: null pointer");
    return HV_ERR_NULL;
  }
  if (rows == 0) return HV_OK;
  UniqArgs a{ids, rows, width, row_stride, col_stride, feats, d, margin};
  SortBuffers bufs;
  if (rows >= kSortFromRows && sort_carve(workspace, workspace_bytes, rows, &bufs))
    return launch_sorted<true>(a, bufs, nullptr, stats, weight, g_out, g_feats, static_cast<cudaStream_t>(stream));
  const unsigned grid = static_cast<unsigned>((rows + kTile - 1) / kTile);
  uniq_kernel<true><<<grid, kTile, 0, static_cast<cudaStream_t>(stream)>>>(a, nullptr, stats, weight, g_out, g_feats);
  HV_CUDA_CHECK(cudaGetLastError());
  return HV_OK;
}
