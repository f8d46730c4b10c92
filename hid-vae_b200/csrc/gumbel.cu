// Gumbel-softmax quantiser level (SURVEY.md section 8 a5 / f3), training mode of modules/quantize.py:108-130,144 with
// distributions/gumbel.py:8-18:
//     dist_k = |x|^2 + |c_k|^2 - 2 x.c_k          ids = argmin_k dist_k (first index)
//     g_k    = -log(-log(u_k + 1e-20) + 1e-20)    w = softmax((-dist + g) / T)        emb = w @ codebook  (= emb_out)
//     loss   = |sg(x) - emb|^2 + beta |x - sg(emb)|^2
// The reference materialises dist, u, g, y and w as [N, K] tensors (five of them, plus their autograd copies); here the
// [N, K] quantities only ever exist in registers / shared memory.
//
//   FORWARD   one WARP per row, lane l owns codes l, l + 32, ...; the fp32 codebook sits in shared memory with a row stride
//             of D + 4 floats (one code per lane: conflict-free LDS.128).  Online softmax per lane (running maximum, sum and
//             weighted code sum), lanes merged once per row.  Also writes lse = log sum_k exp(y_k) per row for the backward.
//   BACKWARD  recomputes y_k from (x, codebook, noise) and w_k = exp(y_k - lse).  With ge = g_emb + 2 g_loss (emb - x):
//                 a_k  = dL/d dist_k = -w_k (ge.c_k - ge.emb) / T                  (sum_k a_k = 0)
//                 g_x  = 2 beta g_loss (x - emb) - 2 sum_k a_k c_k
//                 g_ck = sum_rows [ w_k ge - 2 a_k x ] + 2 c_k sum_rows a_k
//             phase A (warp per row) leaves w, a of a 16-row tile in shared memory; phase B (thread per code) folds the tile
//             into a register accumulator of its code's gradient row -- no atomics inside the loop, K * D atomics per CTA
//             at the very end.
//   NOISE     `uniforms` [N, K] (the reference's torch.rand draw: parity tests) or, when NULL, counter-based Philox4x32-10:
//             element (n, k) is output (k >> 5) & 3 of the block with key = seed and counter = offset +
//             (n * 32 + (k & 31)) * ceil(K / 128) + (k >> 7)  -- the lane that owns the code generates it, four codes per
//             call, and the backward regenerates exactly the same draw from (seed, offset).  (seed, offset) are host scalars
//             or, for the *_devrng entries, the pair {seed, offset} in device memory: a seed drawn on the device (by a CUDA
//             graph, afresh at every replay) gives the same draw as the host seed of the same value.
// Served: D in {16, 32, 64}, K <= 256 (HiD-VAE: D = 32, K = 256); other shapes report HV_ERR_UNSUPPORTED.
#include <math.h>

#include "common.cuh"
#include "ptx.cuh"

namespace hv {
namespace {

constexpr int kWarps = 8;
constexpr int kThreads = kWarps * 32;
constexpr int kMaxK = 256;
constexpr int kTile = 16;  // rows per backward tile
constexpr float kEps = 1e-20f;

struct GumbelArgs {
  const float* x;         // [N, D]
  const float* codebook;  // [K, D] effective
  int64_t n;
  int k;
  float temperature;
  float beta;
  const float* uniforms;  // [N, K] or null
  uint64_t seed, offset;
  const uint64_t* rng;    // device {seed, offset}, or null: then seed and offset above
  // forward outputs / backward inputs
  float* emb_out;   // [N, D]
  int64_t* ids;     // [N] (forward) or null
  float* loss;      // [N] or null
  float* lse;       // [N]
  // backward
  const float* g_emb;   // [N, D] or null
  const float* g_loss;  // [N] or null
  float* g_x;           // [N, D]
  float* g_codebook;    // [K, D], accumulated into
};

__device__ __forceinline__ uint32_t mulhilo(uint32_t a, uint32_t b, uint32_t* hi) {
  const uint64_t p = static_cast<uint64_t>(a) * b;
  *hi = static_cast<uint32_t>(p >> 32);
  return static_cast<uint32_t>(p);
}

// Philox4x32-10 (Salmon et al., SC'11): 10 rounds, key schedule by the Weyl constants
__device__ __forceinline__ uint4 philox4x32_10(uint2 key, uint4 c) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, hi1;
    const uint32_t lo0 = mulhilo(0xD2511F53u, c.x, &hi0);
    const uint32_t lo1 = mulhilo(0xCD9E8D57u, c.z, &hi1);
    c = make_uint4(hi1 ^ c.y ^ key.x, lo1, hi0 ^ c.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return c;
}

// the Philox stream of a call: key = seed, counters from offset
struct Stream {
  uint2 key;
  uint64_t offset;
};

// read once per thread (the backward: once per CTA, into shared memory), before the row loop
__device__ __forceinline__ Stream stream_of(const GumbelArgs& a) {
  uint64_t seed = a.seed, offset = a.offset;
  if (a.rng != nullptr) seed = a.rng[0], offset = a.rng[1];
  return {make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)), offset};
}

// the uniforms of codes k = lane + 32 j, j in [4 jq, 4 jq + 4), of row n
__device__ __forceinline__ void draw4(const Stream& st, int64_t n, int lane, int jq, int blocks_per_lane, float (&u)[4]) {
  const uint64_t ctr = st.offset + (static_cast<uint64_t>(n) * 32u + static_cast<uint64_t>(lane)) * static_cast<uint64_t>(blocks_per_lane) +
                       static_cast<uint64_t>(jq);
  const uint4 r = philox4x32_10(st.key, make_uint4(static_cast<uint32_t>(ctr), static_cast<uint32_t>(ctr >> 32), 0u, 0u));
  constexpr float kScale = 5.9604644775390625e-08f;  // 2^-24: 24-bit uniforms in [0, 1) like torch.rand
  u[0] = static_cast<float>(r.x >> 8) * kScale;
  u[1] = static_cast<float>(r.y >> 8) * kScale;
  u[2] = static_cast<float>(r.z >> 8) * kScale;
  u[3] = static_cast<float>(r.w >> 8) * kScale;
}

__device__ __forceinline__ float gumbel_of(float u) { return -logf(-logf(u + kEps) + kEps); }  // distributions/gumbel.py:10-11

template <int D>
__device__ __forceinline__ void load_codebook(const GumbelArgs& a, float* s_cb, float* s_cn) {
  constexpr int RS = D + 4;
  for (int i = threadIdx.x; i < a.k * (D / 4); i += kThreads) {
    const int k = i / (D / 4), c = i % (D / 4);
    *reinterpret_cast<float4*>(s_cb + k * RS + 4 * c) = __ldg(reinterpret_cast<const float4*>(a.codebook + static_cast<int64_t>(k) * D) + c);
  }
  __syncthreads();
  for (int k = threadIdx.x; k < a.k; k += kThreads) {
    float s = 0.f;
#pragma unroll
    for (int d = 0; d < D; ++d) s = fmaf(s_cb[k * RS + d], s_cb[k * RS + d], s);
    s_cn[k] = s;
  }
  __syncthreads();
}

template <int D>
__device__ __forceinline__ void lds_row(const float* s_row, float (&c)[D]) {
#pragma unroll
  for (int i = 0; i < D; i += 4) {
    const float4 v = *reinterpret_cast<const float4*>(s_row + i);
    c[i] = v.x, c[i + 1] = v.y, c[i + 2] = v.z, c[i + 3] = v.w;
  }
}

template <int D>
__device__ __forceinline__ float dot_row(const float (&p)[D], const float (&q)[D]) {
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
  for (int i = 0; i < D; i += 4) {
    s0 = fmaf(p[i], q[i], s0);
    s1 = fmaf(p[i + 1], q[i + 1], s1);
    s2 = fmaf(p[i + 2], q[i + 2], s2);
    s3 = fmaf(p[i + 3], q[i + 3], s3);
  }
  return (s0 + s1) + (s2 + s3);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, off));
  return v;
}

// column sums of the warp's 32 lane-partial D-vectors: lane writes its vector into s_red[lane][.] (stride D + 1), then
// lane dd adds column dd over the lanes in lane order (a fixed order: results do not depend on the schedule)
template <int D>
__device__ __forceinline__ void lanes_to_columns(float* s_red, const float (&v)[D], int lane, float (&col)[(D + 31) / 32]) {
  __syncwarp();
#pragma unroll
  for (int d = 0; d < D; ++d) s_red[lane * (D + 1) + d] = v[d];
  __syncwarp();
#pragma unroll
  for (int p = 0; p < (D + 31) / 32; ++p) {
    const int dd = lane + 32 * p;
    float s = 0.f;
    if (dd < D) {
#pragma unroll 8
      for (int l = 0; l < 32; ++l) s += s_red[l * (D + 1) + dd];
    }
    col[p] = s;
  }
}

template <int D>
__global__ void __launch_bounds__(kThreads) gumbel_fwd_kernel(GumbelArgs a) {
  constexpr int RS = D + 4;
  constexpr int PER = (D + 31) / 32;
  extern __shared__ __align__(16) float smem[];
  float* s_cb = smem;                  // [kMaxK][RS]
  float* s_cn = s_cb + kMaxK * RS;     // [kMaxK]
  float* s_red = s_cn + kMaxK + (threadIdx.x >> 5) * 32 * (D + 1);
  load_codebook<D>(a, s_cb, s_cn);

  const int warp = ptx::warp_index(), lane = threadIdx.x & 31;
  const int blocks_per_lane = (a.k + 127) / 128;
  const Stream st = stream_of(a);
  for (int64_t row = static_cast<int64_t>(blockIdx.x) * kWarps + warp; row < a.n; row += static_cast<int64_t>(gridDim.x) * kWarps) {
    float x[D];
    load_row<D>(x, a.x + row * D);
    const float xx = dot_row<D>(x, x);
    float m = -INFINITY, s = 0.f, best = INFINITY;
    int best_k = 0;
    float e[D];
#pragma unroll
    for (int d = 0; d < D; ++d) e[d] = 0.f;
    float u4[4];
#pragma unroll 1
    for (int k = lane, j = 0; k < a.k; k += 32, ++j) {
      float c[D];
      lds_row<D>(s_cb + k * RS, c);
      const float dist = (xx + s_cn[k]) - 2.0f * dot_row<D>(x, c);  // modules/quantize.py:109-113
      if (dist < best) best = dist, best_k = k;                      // k ascends within the lane: the first minimum stays
      float u;
      if (a.uniforms != nullptr) {
        u = __ldg(a.uniforms + row * a.k + k);
      } else {
        if ((j & 3) == 0) draw4(st, row, lane, j >> 2, blocks_per_lane, u4);
        u = u4[j & 3];
      }
      const float y = __fdiv_rn(gumbel_of(u) - dist, a.temperature);  // (logits + G) / T, logits = -dist
      const float m_new = fmaxf(m, y);
      const float sc = __expf(m - m_new), p = __expf(y - m_new);
      s = fmaf(s, sc, p);
#pragma unroll
      for (int d = 0; d < D; ++d) e[d] = fmaf(e[d], sc, p * c[d]);
      m = m_new;
    }
    // ---- merge the lanes ----
    const float m_row = warp_max(m);
    const float scl = m == -INFINITY ? 0.f : __expf(m - m_row);
    const float s_row = warp_sum(s * scl);
#pragma unroll
    for (int d = 0; d < D; ++d) e[d] *= scl;
    float col[PER];
    lanes_to_columns<D>(s_red, e, lane, col);
    const float inv_s = 1.0f / s_row;
    float a2 = 0.f;
#pragma unroll
    for (int p = 0; p < PER; ++p) {
      const int dd = lane + 32 * p;
      if (dd < D) {
        const float emb = col[p] * inv_s;
        a.emb_out[row * D + dd] = emb;
        const float df = __ldg(a.x + row * D + dd) - emb;
        a2 = fmaf(df, df, a2);
      }
    }
    a2 = warp_sum(a2);
    // argmin over the lanes: smallest distance, lowest code index on exact ties (torch.min)
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, off);
      const int ok = __shfl_xor_sync(0xffffffffu, best_k, off);
      if (ob < best || (ob == best && ok < best_k)) best = ob, best_k = ok;
    }
    if (lane == 0) {
      if (a.ids != nullptr) a.ids[row] = best_k;
      if (a.loss != nullptr) a.loss[row] = a2 + a.beta * a2;  // modules/loss.py:41-44
      a.lse[row] = m_row + logf(s_row);
    }
  }
}

template <int D>
__global__ void __launch_bounds__(kThreads) gumbel_bwd_kernel(GumbelArgs a) {
  constexpr int RS = D + 4;
  constexpr int PER = (D + 31) / 32;
  extern __shared__ __align__(16) float smem[];
  float* s_cb = smem;                                   // [kMaxK][RS]
  float* s_cn = s_cb + kMaxK * RS;                      // [kMaxK]
  float* s_w = s_cn + kMaxK;                            // [kTile][kMaxK]  softmax weights of the tile
  float* s_a = s_w + kTile * kMaxK;                     // [kTile][kMaxK]  dL/d dist
  float* s_x = s_a + kTile * kMaxK;                     // [kTile][D]
  float* s_ge = s_x + kTile * D;                        // [kTile][D]
  float* s_red = s_ge + kTile * D + (threadIdx.x >> 5) * 32 * (D + 1);
  // the stream stays in shared memory: at D = 64 the row loop already spills, and four more live registers would add spills
  __shared__ Stream s_st;
  if (threadIdx.x == 0) s_st = stream_of(a);  // (made visible by load_codebook's barrier)
  load_codebook<D>(a, s_cb, s_cn);

  const int warp = ptx::warp_index(), lane = threadIdx.x & 31;
  const int blocks_per_lane = (a.k + 127) / 128;
  const Stream& st = s_st;
  const float inv_t = 1.0f / a.temperature;
  float acc[D];
#pragma unroll
  for (int d = 0; d < D; ++d) acc[d] = 0.f;
  float asum = 0.f;

  const int64_t n_tiles = (a.n + kTile - 1) / kTile;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    // ---------------- phase A: a warp per row ----------------
#pragma unroll 1
    for (int rr = warp; rr < kTile; rr += kWarps) {
      const int64_t row = tile * kTile + rr;
      if (row >= a.n) {  // padding rows contribute nothing
        for (int k = lane; k < a.k; k += 32) s_w[rr * kMaxK + k] = 0.f, s_a[rr * kMaxK + k] = 0.f;
        for (int d = lane; d < D; d += 32) s_x[rr * D + d] = 0.f, s_ge[rr * D + d] = 0.f;
        continue;
      }
      const float gl = a.g_loss != nullptr ? __ldg(a.g_loss + row) : 0.f;
      float x[D], ge[D];
      load_row<D>(x, a.x + row * D);
      float gee;
      {
        float eo[D];
        load_row<D>(eo, a.emb_out + row * D);
        if (a.g_emb != nullptr) {
          load_row<D>(ge, a.g_emb + row * D);
        } else {
#pragma unroll
          for (int d = 0; d < D; ++d) ge[d] = 0.f;
        }
#pragma unroll
        for (int d = 0; d < D; ++d) ge[d] = fmaf(2.0f * gl, eo[d] - x[d], ge[d]);  // + d emb_loss / d emb (modules/loss.py:42)
        // in the summation order of ge.c_k below: where emb equals a code bit for bit (K = 1, or a softmax that underflowed to
        // one-hot at low T) its a_k is then exactly 0, as in exact arithmetic, instead of fp32 noise amplified by 1 / T
        gee = dot_row<D>(ge, eo);
      }
      const float xx = dot_row<D>(x, x);
      const float lse = __ldg(a.lse + row);
      float v[D];
#pragma unroll
      for (int d = 0; d < D; ++d) v[d] = 0.f;
      float u4[4];
#pragma unroll 1
      for (int k = lane, j = 0; k < a.k; k += 32, ++j) {
        float c[D];
        lds_row<D>(s_cb + k * RS, c);
        const float dist = (xx + s_cn[k]) - 2.0f * dot_row<D>(x, c);
        float u;
        if (a.uniforms != nullptr) {
          u = __ldg(a.uniforms + row * a.k + k);
        } else {
          if ((j & 3) == 0) draw4(st, row, lane, j >> 2, blocks_per_lane, u4);
          u = u4[j & 3];
        }
        const float y = __fdiv_rn(gumbel_of(u) - dist, a.temperature);
        const float w = __expf(y - lse);
        const float aa = -w * (dot_row<D>(ge, c) - gee) * inv_t;
#pragma unroll
        for (int d = 0; d < D; ++d) v[d] = fmaf(aa, c[d], v[d]);
        s_w[rr * kMaxK + k] = w;
        s_a[rr * kMaxK + k] = aa;
      }
      float col[PER];
      lanes_to_columns<D>(s_red, v, lane, col);
#pragma unroll
      for (int p = 0; p < PER; ++p) {
        const int dd = lane + 32 * p;
        if (dd < D) {
          const float xd = __ldg(a.x + row * D + dd), ed = __ldg(a.emb_out + row * D + dd);
          const float gd = (a.g_emb != nullptr ? __ldg(a.g_emb + row * D + dd) : 0.f) + 2.0f * gl * (ed - xd);
          a.g_x[row * D + dd] = fmaf(2.0f * a.beta * gl, xd - ed, -2.0f * col[p]);  // query loss + the path through dist
          s_x[rr * D + dd] = xd;
          s_ge[rr * D + dd] = gd;
        }
      }
    }
    __syncthreads();
    // ---------------- phase B: a thread per code ----------------
    if (static_cast<int>(threadIdx.x) < a.k) {
#pragma unroll 1
      for (int rr = 0; rr < kTile; ++rr) {
        const float w = s_w[rr * kMaxK + threadIdx.x], aa = s_a[rr * kMaxK + threadIdx.x];
        asum += aa;
        const float m2a = -2.0f * aa;
#pragma unroll
        for (int i = 0; i < D; i += 4) {
          const float4 g4 = *reinterpret_cast<const float4*>(s_ge + rr * D + i);
          const float4 x4 = *reinterpret_cast<const float4*>(s_x + rr * D + i);
          acc[i] = fmaf(m2a, x4.x, fmaf(w, g4.x, acc[i]));
          acc[i + 1] = fmaf(m2a, x4.y, fmaf(w, g4.y, acc[i + 1]));
          acc[i + 2] = fmaf(m2a, x4.z, fmaf(w, g4.z, acc[i + 2]));
          acc[i + 3] = fmaf(m2a, x4.w, fmaf(w, g4.w, acc[i + 3]));
        }
      }
    }
    __syncthreads();
  }
  if (static_cast<int>(threadIdx.x) < a.k) {
    const int k = threadIdx.x;
    float* out = a.g_codebook + static_cast<int64_t>(k) * D;
#pragma unroll
    for (int d = 0; d < D; ++d) atomicAdd(out + d, fmaf(2.0f * asum, s_cb[k * RS + d], acc[d]));
  }
}

// the draw itself, [N, K]: what the two kernels above generate for (seed, offset) -- for recording / reproducing a step
__global__ void __launch_bounds__(kThreads) gumbel_uniforms_kernel(GumbelArgs a, float* __restrict__ out) {
  const int blocks_per_lane = (a.k + 127) / 128;
  const int64_t total = a.n * 32 * blocks_per_lane;  // one Philox block per thread
  const Stream st = stream_of(a);
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x; i < total; i += static_cast<int64_t>(gridDim.x) * kThreads) {
    const int jq = static_cast<int>(i % blocks_per_lane);
    const int lane = static_cast<int>((i / blocks_per_lane) % 32);
    const int64_t row = i / (static_cast<int64_t>(blocks_per_lane) * 32);
    float u4[4];
    draw4(st, row, lane, jq, blocks_per_lane, u4);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int k = lane + 32 * (4 * jq + t);
      if (k < a.k) out[row * a.k + k] = u4[t];
    }
  }
}

template <int D>
constexpr int fwd_smem() { return (kMaxK * (D + 4) + kMaxK + kWarps * 32 * (D + 1)) * 4; }
template <int D>
constexpr int bwd_smem() { return (kMaxK * (D + 4) + kMaxK + 2 * kTile * kMaxK + 2 * kTile * D + kWarps * 32 * (D + 1)) * 4; }

template <int D>
int launch_fwd(const GumbelArgs& a, int sm_count, cudaStream_t s) {
  const int64_t groups = (a.n + kWarps - 1) / kWarps;
  const unsigned grid = static_cast<unsigned>(groups < 2ll * sm_count ? groups : 2ll * sm_count);
  if (int st = prepare_kernel(gumbel_fwd_kernel<D>, 0, fwd_smem<D>())) return st;
  gumbel_fwd_kernel<D><<<grid, kThreads, fwd_smem<D>(), s>>>(a);
  HV_CUDA_CHECK(cudaGetLastError());
  return HV_OK;
}
template <int D>
int launch_bwd(const GumbelArgs& a, int sm_count, cudaStream_t s) {
  const int64_t tiles = (a.n + kTile - 1) / kTile;
  const int per_sm = D <= 32 ? 2 : 1;
  const unsigned grid = static_cast<unsigned>(tiles < static_cast<int64_t>(per_sm) * sm_count ? tiles : static_cast<int64_t>(per_sm) * sm_count);
  if (int st = prepare_kernel(gumbel_bwd_kernel<D>, 0, bwd_smem<D>())) return st;
  gumbel_bwd_kernel<D><<<grid, kThreads, bwd_smem<D>(), s>>>(a);
  HV_CUDA_CHECK(cudaGetLastError());
  return HV_OK;
}

int check_common(const char* who, const float* x, int64_t n, int d, const float* codebook, int k, float temperature) {
  if (n < 0 || d <= 0 || k <= 0) {
    set_error("%s: bad shape n=%lld d=%d k=%d", who, static_cast<long long>(n), d, k);
    return HV_ERR_BAD_SHAPE;
  }
  if (!(temperature > 0.f)) {
    set_error("%s: temperature must be positive (got %g)", who, static_cast<double>(temperature));
    return HV_ERR_BAD_SHAPE;
  }
  if ((d != 16 && d != 32 && d != 64) || k > kMaxK) {
    set_error("%s: no fused Gumbel-softmax instantiation for D=%d K=%d (served: D in {16, 32, 64}, K <= %d)", who, d, k, kMaxK);
    return HV_ERR_UNSUPPORTED;
  }
  if (n > 0 && (!x || !codebook)) {
    set_error("%s: null pointer", who);
    return HV_ERR_NULL;
  }
  if (!aligned16(x) || !aligned16(codebook)) {
    set_error("%s: x and codebook must be 16-byte aligned", who);
    return HV_ERR_MISALIGNED;
  }
  return HV_OK;
}

// The host-seed entries pass (seed, offset) and rng = null; the *_devrng entries pass rng, which must be non-null when n > 0.
int uniforms_impl(const char* who, int64_t n, int k, uint64_t seed, uint64_t offset, const uint64_t* rng, bool devrng,
                  float* uniforms, void* stream) {
  if (n < 0 || k <= 0) {
    set_error("%s: bad shape n=%lld k=%d", who, static_cast<long long>(n), k);
    return HV_ERR_BAD_SHAPE;
  }
  if (n == 0) return HV_OK;
  if (!uniforms || (devrng && !rng)) {
    set_error("%s: null pointer", who);
    return HV_ERR_NULL;
  }
  GumbelArgs a{};
  a.n = n, a.k = k, a.seed = seed, a.offset = offset, a.rng = rng;
  const int64_t total = n * 32 * ((k + 127) / 128);
  const int64_t blocks = (total + kThreads - 1) / kThreads;
  gumbel_uniforms_kernel<<<static_cast<unsigned>(blocks < 65535 ? blocks : 65535), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(a, uniforms);
  HV_CUDA_CHECK(cudaGetLastError());
  return HV_OK;
}

int forward_impl(const char* who, const float* x, int64_t n, int d, const float* codebook, int k, float temperature, float beta,
                 const float* uniforms, uint64_t seed, uint64_t offset, const uint64_t* rng, bool devrng, float* emb_out,
                 int64_t* ids, float* loss, float* lse, void* stream) {
  if (int st = check_common(who, x, n, d, codebook, k, temperature)) return st;
  if (n == 0) return HV_OK;
  if (!emb_out || !lse) {
    set_error("%s: emb_out and lse are required", who);
    return HV_ERR_NULL;
  }
  if (devrng && !rng) {
    set_error("%s: rng (the device pair {seed, offset}) is required", who);
    return HV_ERR_NULL;
  }
  DeviceProps props;
  if (int st = device_props(&props)) return st;
  GumbelArgs a{};
  a.x = x, a.codebook = codebook, a.n = n, a.k = k, a.temperature = temperature, a.beta = beta;
  a.uniforms = uniforms, a.seed = seed, a.offset = offset, a.rng = rng;
  a.emb_out = emb_out, a.ids = ids, a.loss = loss, a.lse = lse;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  switch (d) {
    case 16: return launch_fwd<16>(a, props.sm_count, s);
    case 32: return launch_fwd<32>(a, props.sm_count, s);
    default: return launch_fwd<64>(a, props.sm_count, s);
  }
}

int backward_impl(const char* who, const float* x, int64_t n, int d, const float* codebook, int k, float temperature, float beta,
                  const float* uniforms, uint64_t seed, uint64_t offset, const uint64_t* rng, bool devrng, const float* emb_out,
                  const float* lse, const float* g_emb, const float* g_loss, float* g_x, float* g_codebook, void* stream) {
  if (int st = check_common(who, x, n, d, codebook, k, temperature)) return st;
  if (n == 0) return HV_OK;
  if (!emb_out || !lse || !g_x || !g_codebook) {
    set_error("%s: emb_out, lse, g_x and g_codebook are required", who);
    return HV_ERR_NULL;
  }
  if (devrng && !rng) {
    set_error("%s: rng (the device pair {seed, offset}) is required", who);
    return HV_ERR_NULL;
  }
  if (!aligned16(emb_out) || !aligned16(g_emb)) {
    set_error("%s: emb_out and g_emb must be 16-byte aligned", who);
    return HV_ERR_MISALIGNED;
  }
  DeviceProps props;
  if (int st = device_props(&props)) return st;
  GumbelArgs a{};
  a.x = x, a.codebook = codebook, a.n = n, a.k = k, a.temperature = temperature, a.beta = beta;
  a.uniforms = uniforms, a.seed = seed, a.offset = offset, a.rng = rng;
  a.emb_out = const_cast<float*>(emb_out), a.lse = const_cast<float*>(lse);
  a.g_emb = g_emb, a.g_loss = g_loss, a.g_x = g_x, a.g_codebook = g_codebook;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  switch (d) {
    case 16: return launch_bwd<16>(a, props.sm_count, s);
    case 32: return launch_bwd<32>(a, props.sm_count, s);
    default: return launch_bwd<64>(a, props.sm_count, s);
  }
}

}  // namespace
}  // namespace hv

extern "C" int hv_gumbel_supported(int d, int k) { return (d == 16 || d == 32 || d == 64) && k >= 1 && k <= hv::kMaxK; }

extern "C" int hv_gumbel_uniforms(int64_t n, int k, uint64_t seed, uint64_t offset, float* uniforms, void* stream) {
  return hv::uniforms_impl("hv_gumbel_uniforms", n, k, seed, offset, nullptr, false, uniforms, stream);
}

extern "C" int hv_gumbel_uniforms_devrng(int64_t n, int k, const uint64_t* rng, float* uniforms, void* stream) {
  return hv::uniforms_impl("hv_gumbel_uniforms_devrng", n, k, 0, 0, rng, true, uniforms, stream);
}

extern "C" int hv_gumbel_forward(const float* x, int64_t n, int d, const float* codebook, int k, float temperature, float beta,
                                 const float* uniforms, uint64_t seed, uint64_t offset, float* emb_out, int64_t* ids, float* loss,
                                 float* lse, void* stream) {
  return hv::forward_impl("hv_gumbel_forward", x, n, d, codebook, k, temperature, beta, uniforms, seed, offset, nullptr, false,
                          emb_out, ids, loss, lse, stream);
}

extern "C" int hv_gumbel_forward_devrng(const float* x, int64_t n, int d, const float* codebook, int k, float temperature,
                                        float beta, const float* uniforms, const uint64_t* rng, float* emb_out, int64_t* ids,
                                        float* loss, float* lse, void* stream) {
  return hv::forward_impl("hv_gumbel_forward_devrng", x, n, d, codebook, k, temperature, beta, uniforms, 0, 0, rng, true,
                          emb_out, ids, loss, lse, stream);
}

extern "C" int hv_gumbel_backward(const float* x, int64_t n, int d, const float* codebook, int k, float temperature, float beta,
                                  const float* uniforms, uint64_t seed, uint64_t offset, const float* emb_out, const float* lse,
                                  const float* g_emb, const float* g_loss, float* g_x, float* g_codebook, void* stream) {
  return hv::backward_impl("hv_gumbel_backward", x, n, d, codebook, k, temperature, beta, uniforms, seed, offset, nullptr, false,
                           emb_out, lse, g_emb, g_loss, g_x, g_codebook, stream);
}

extern "C" int hv_gumbel_backward_devrng(const float* x, int64_t n, int d, const float* codebook, int k, float temperature,
                                         float beta, const float* uniforms, const uint64_t* rng, const float* emb_out,
                                         const float* lse, const float* g_emb, const float* g_loss, float* g_x,
                                         float* g_codebook, void* stream) {
  return hv::backward_impl("hv_gumbel_backward_devrng", x, n, d, codebook, k, temperature, beta, uniforms, 0, 0, rng, true,
                           emb_out, lse, g_emb, g_loss, g_x, g_codebook, stream);
}
