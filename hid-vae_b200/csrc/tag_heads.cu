// Eval-mode tag heads (TagPredictor, modules/h_rqvae.py:69-99; reference h_rqvae.py:108-227, called by predict_tags at
// :674-738) for sm_100a.  Per level i, per row:
//     x = concat(emb_0 .. emb_i)                      E = D (i+1)
//     g = x * sigmoid(W3 gelu(W2 relu(W1 x)))         the attention gate, fp32 on CUDA cores      (tag_gate_kernel)
//     g = normalize(g) if i > 0
//     h = relu(LN(Wf g));  h += LN(relu(Wb relu(LN(Wa h))))  twice;  c = relu(Wc2 relu(LN(Wc1 h)));  logit = Wc3 c
//     pred = argmax(logit) (first index on ties), conf = 1 / sum_j exp(logit_j - max)
// Every Linear after the gate is one launch of tag_gemm_kernel<KIND> over a sub-chunk of kChunkRows rows:
//
//   PRECISION  operands are rounded to fp16 (the encoder's numerics: TF32's significand), products accumulate in fp32 in
//              tensor memory, LayerNorm statistics, the gate, the softmax and the argmax are fp32.  Every activation that
//              feeds a GEMM is stored as fp16; a LayerNorm input is stored as fp16 too and normalised in a second sweep.
//   LAYOUT     activations live in a workspace as 128-row tiles of 64-column chunks, each chunk a 16 KB block in the UMMA
//              K-major core-matrix layout ([K group of 8][row 128][8 fp16]); weights live in the image as blocks of
//              (<= 256 outputs) x 64 inputs in the same layout.  One 1-D bulk copy lands each block MMA-ready.  Widths are
//              zero-padded to multiples of 64 (zero weights and biases: exact for Linear and ReLU); LayerNorm divides by
//              the true width and leaves the padded columns out of its statistics.
//   CTA        one 128-row tile over the full output width, in N-chunks of <= 256 columns double-buffered in tensor
//              memory (512 columns).  Warp 0 streams (activation, weight) block pairs, warp 1 issues the MMAs, warps 4-7
//              run the epilogue with TMEM lane = row, so a row's LayerNorm sums live in one thread's registers.
//   EPILOGUES  LN_RELU      bias -> LN -> ReLU                      (feature extractor, block inner, classifier 1)
//              RELU_LN_RES  bias -> ReLU -> LN -> + residual        (block outer)
//              RELU         bias -> ReLU                            (classifier 2; LN_RELU without LayerNorm)
//              RES_RELU     bias -> ReLU -> + residual              (block outer without LayerNorm)
//              ARGMAX       bias -> argmax / confidence, written through strides into the caller's int64 table
// The sub-chunk keeps the live activations of one level (two residual buffers and the inner one) in L2.
#include <cuda_fp16.h>

#include <algorithm>

#include "common.cuh"
#include "ptx.cuh"

namespace hv {
namespace {

constexpr int kTileRows = 128;
constexpr int kChunkRows = 148 * kTileRows;  // one tile per SM of a B200 per launch
constexpr int kThreads = 256;                // warp 0 loader, 1 MMA issuer, 2 TMEM allocator, 4..7 epilogue
constexpr int kEpiWarp0 = 4;
constexpr int kNChunk = 256;
constexpr int kABlockBytes = kTileRows * 64 * 2;    // 16 KB: 128 rows x 64 fp16
constexpr int kBBlockBytes = kNChunk * 64 * 2;      // 32 KB: 256 outputs x 64 fp16
constexpr int kStages = 4;
constexpr int kStageBytes = kABlockBytes + kBBlockBytes;
constexpr int kSmemBytes = kStages * kStageBytes + 128;
constexpr int kMaxLevels = 8;
constexpr int kMaxGateWidth = 128;   // E = D (i+1) of the gate kernel's shared-memory plan
constexpr int kMaxWidth = 4096;
constexpr float kLnEps = 1e-5f;      // nn.LayerNorm default
static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");

enum Kind : int { LN_RELU = 0, RELU_LN_RES = 1, RELU = 2, RES_RELU = 3, ARGMAX = 4 };

__host__ __device__ constexpr int pad64(int v) { return (v + 63) / 64 * 64; }
__host__ __device__ constexpr uint32_t idesc_f16(uint32_t m, uint32_t n) { return (1u << 4) | ((n >> 3) << 17) | ((m >> 4) << 24); }

// ---------------------------------------------------------------------------------------------------------------------
// host plan: widths and image offsets of every level
// ---------------------------------------------------------------------------------------------------------------------
struct Lin {
  int n, k, np, kp;
  size_t w, b, g, be;  // byte offsets in the image: fp16 weight blocks, fp32 bias, LayerNorm gamma / beta (0 = none)
};
struct Level {
  int e, h, i, i2, c;
  size_t gw[3], gb[3];  // the gate's three Linear layers, fp32 row-major as nn.Linear stores them
  Lin f, a[2], b[2], c1, c2, c3;
};
struct Plan {
  int n_levels = 0;
  bool norm = false;
  Level lv[kMaxLevels];
  size_t image_bytes = 0;
  int res_width = 0, inner_width = 0;  // padded widths of the residual buffers and of the inner buffer
};

bool make_plan(int n_levels, int d, int first_hidden, const int* class_counts, int use_norm, Plan* p) {
  if (n_levels < 1 || n_levels > kMaxLevels || d < 4 || first_hidden < 2 || !class_counts) return false;
  p->n_levels = n_levels;
  p->norm = use_norm != 0;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t at = off;
    off += (bytes + 255) / 256 * 256;
    return at;
  };
  auto lin = [&](int n, int k) {
    Lin l{n, k, pad64(n), pad64(k), 0, 0, 0, 0};
    l.w = take(static_cast<size_t>(l.np) * l.kp * 2);
    return l;
  };
  for (int i = 0; i < n_levels; ++i) {
    Level& L = p->lv[i];
    L.e = d * (i + 1);
    L.h = first_hidden / 2 * (i + 1);
    L.i = static_cast<int>(L.h * 0.9);  // int(hidden_dim * 0.9), modules/h_rqvae.py:78
    L.i2 = L.i / 2;
    L.c = class_counts[i];
    if (L.e > kMaxGateWidth || L.e / 4 < 1 || L.h < 1 || L.i2 < 1 || L.c < 1 || pad64(L.h) > kMaxWidth ||
        pad64(L.i) > kMaxWidth || pad64(L.c) > kMaxWidth)
      return false;
    const int ge[4] = {L.e, L.e / 4, L.e / 2, L.e};
    for (int j = 0; j < 3; ++j) {
      L.gw[j] = take(static_cast<size_t>(ge[j + 1]) * ge[j] * 4);
      L.gb[j] = take(static_cast<size_t>(ge[j + 1]) * 4);
    }
    L.f = lin(L.h, L.e);
    for (int r = 0; r < 2; ++r) {
      L.a[r] = lin(L.i, L.h);
      L.b[r] = lin(L.h, L.i);
    }
    L.c1 = lin(L.i, L.h);
    L.c2 = lin(L.i2, L.i);
    L.c3 = lin(L.c, L.i2);
    Lin* with_ln[6] = {&L.f, &L.a[0], &L.b[0], &L.a[1], &L.b[1], &L.c1};
    for (Lin* l : {&L.f, &L.a[0], &L.b[0], &L.a[1], &L.b[1], &L.c1, &L.c2, &L.c3}) l->b = take(static_cast<size_t>(l->np) * 4);
    if (p->norm)
      for (Lin* l : with_ln) {
        l->g = take(static_cast<size_t>(l->np) * 4);
        l->be = take(static_cast<size_t>(l->np) * 4);
      }
    p->res_width = std::max({p->res_width, pad64(L.h), pad64(L.i2), pad64(L.e)});
    p->inner_width = std::max(p->inner_width, pad64(L.i));
  }
  p->image_bytes = off;
  return true;
}

size_t scratch_bytes(const Plan& p, int64_t rows) {
  const int64_t r = std::min<int64_t>(std::max<int64_t>(rows, 1), kChunkRows);
  const int64_t tiles = (r + kTileRows - 1) / kTileRows;
  return static_cast<size_t>(tiles) * kTileRows * (2 * p.res_width + p.inner_width) * 2;
}

// ---------------------------------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ float2 unpack_f16(uint32_t v) { return __half22float2(*reinterpret_cast<const __half2*>(&v)); }

// byte offset of (row r, column n) of a tile-blocked activation buffer whose width is `wp` (a multiple of 64)
__device__ __forceinline__ size_t act_off(int64_t tile, int wp, int r, int n) {
  return static_cast<size_t>(tile) * wp * (kTileRows * 2) + static_cast<size_t>(n >> 6) * kABlockBytes + ((n & 63) >> 3) * 2048 +
         r * 16 + (n & 7) * 2;
}
// 32 fp32 values -> fp16 -> columns [n0, n0 + 32) of row r (four 16-byte stores; a warp's 32 rows are 512 contiguous bytes)
__device__ __forceinline__ void store32(uint8_t* buf, int64_t tile, int wp, int r, int n0, const float (&x)[32]) {
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const uint4 v = make_uint4(pack_f16(x[8 * u], x[8 * u + 1]), pack_f16(x[8 * u + 2], x[8 * u + 3]),
                               pack_f16(x[8 * u + 4], x[8 * u + 5]), pack_f16(x[8 * u + 6], x[8 * u + 7]));
    *reinterpret_cast<uint4*>(buf + act_off(tile, wp, r, n0 + 8 * u)) = v;
  }
}
__device__ __forceinline__ void load32(const uint8_t* buf, int64_t tile, int wp, int r, int n0, float (&x)[32]) {
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const uint4 v = *reinterpret_cast<const uint4*>(buf + act_off(tile, wp, r, n0 + 8 * u));
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = unpack_f16(w[j]);
      x[8 * u + 2 * j] = f.x;
      x[8 * u + 2 * j + 1] = f.y;
    }
  }
}
// 32 consecutive fp32 of a vector every thread of the warp reads at the same address (broadcast)
__device__ __forceinline__ void vec32(const float* p, float (&x)[32]) {
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p) + u);
    x[4 * u] = v.x, x[4 * u + 1] = v.y, x[4 * u + 2] = v.z, x[4 * u + 3] = v.w;
  }
}

struct GemmArgs {
  const uint8_t* a;      // input activations, width kp
  const uint8_t* w;      // weight blocks
  const float* bias;     // [np]
  const float* gamma;    // [np] (LayerNorm kinds)
  const float* beta;
  uint8_t* out;          // output activations, width np
  const uint8_t* res;    // residual activations, width np (RELU_LN_RES, RES_RELU)
  int kp, np, n_true;
  int64_t rows;          // valid rows of this sub-chunk
  int64_t* pred;         // ARGMAX: pred[row * pred_stride], row counted from the sub-chunk's first row
  int64_t pred_stride;
  float* conf;           // nullable
  int64_t conf_stride;
  float* logits;         // nullable: [rows, n_true] fp32
};

template <int KIND>
__global__ void __launch_bounds__(kThreads, 1) tag_gemm_kernel(GemmArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  uint64_t* full = s_bar;                 // [kStages]  both blocks of a stage landed
  uint64_t* empty = full + kStages;       // [kStages]  the MMAs that read the stage completed
  uint64_t* acc_full = empty + kStages;   // [2]        an N-chunk's accumulator is complete
  uint64_t* acc_empty = acc_full + 2;     // [2]        the 4 epilogue warps drained it
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = ptx::warp_index();
  const int lane = threadIdx.x & 31;
  const int64_t tile = blockIdx.x;
  const int n_chunks = (a.np + kNChunk - 1) / kNChunk;
  const int k_chunks = a.kp / 64;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kStages; ++i) {
      ptx::mbar_init(ptx::smem_u32(&full[i]), 1);
      ptx::mbar_init(ptx::smem_u32(&empty[i]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(ptx::smem_u32(&acc_full[i]), 1);
      ptx::mbar_init(ptx::smem_u32(&acc_empty[i]), 4);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(ptx::smem_u32(s_tmem), 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem = *s_tmem;

  if (warp == 0) {
    // ============================================ block loader ===================================================
    if (ptx::elect_one()) {
      const uint8_t* a_tile = a.a + static_cast<size_t>(tile) * a.kp * (kTileRows * 2);
      uint32_t seq = 0;
      for (int j = 0; j < n_chunks; ++j) {
        const int nc = min(kNChunk, a.np - j * kNChunk);
        const uint8_t* w_chunk = a.w + static_cast<size_t>(j) * kNChunk * a.kp * 2;
        for (int c = 0; c < k_chunks; ++c, ++seq) {
          const uint32_t s = seq % kStages, use = seq / kStages;
          if (use > 0) ptx::mbar_wait(ptx::smem_u32(&empty[s]), (use - 1) & 1u);
          const uint32_t bar = ptx::smem_u32(&full[s]);
          const uint32_t dst = ptx::smem_u32(smem + s * kStageBytes);
          ptx::mbar_arrive_expect_tx(bar, kABlockBytes + nc * 128);
          ptx::bulk_g2s(dst, a_tile + static_cast<size_t>(c) * kABlockBytes, kABlockBytes, bar);
          ptx::bulk_g2s(dst + kABlockBytes, w_chunk + static_cast<size_t>(c) * nc * 128, nc * 128, bar);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ============================================= MMA issuer ====================================================
    if (ptx::elect_one()) {
      const uint32_t sbo_hi = ptx::umma_desc_hi(128);
      uint32_t seq = 0;
      for (int j = 0; j < n_chunks; ++j) {
        const int nc = min(kNChunk, a.np - j * kNChunk);
        const uint32_t buf = j & 1;
        if (j >= 2) {
          ptx::mbar_wait(ptx::smem_u32(&acc_empty[buf]), ((j >> 1) - 1) & 1u);
          ptx::tc_fence_after_sync();
        }
        const uint32_t idesc = idesc_f16(128, nc);
        for (int c = 0; c < k_chunks; ++c, ++seq) {
          const uint32_t s = seq % kStages;
          ptx::mbar_wait(ptx::smem_u32(&full[s]), (seq / kStages) & 1u);
          ptx::tc_fence_after_sync();
          const uint32_t a_base = ptx::smem_u32(smem + s * kStageBytes), b_base = a_base + kABlockBytes;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint64_t ad = ptx::umma_desc(ptx::umma_desc_lo(a_base + ks * 2 * 2048, 2048), sbo_hi);
            const uint64_t bd = ptx::umma_desc(ptx::umma_desc_lo(b_base + ks * 2 * nc * 16, nc * 16), sbo_hi);
            ptx::umma_bf16(tmem + buf * kNChunk, ad, bd, idesc, (c | ks) > 0 ? 1u : 0u);
          }
          ptx::umma_commit(ptx::smem_u32(&empty[s]));
        }
        ptx::umma_commit(ptx::smem_u32(&acc_full[buf]));
      }
    }
    __syncwarp();
  } else if (warp >= kEpiWarp0) {
    // ============================================== epilogue =====================================================
    const int q = warp - kEpiWarp0;  // TMEM lane quarter (== warp % 4)
    const int r = q * 32 + lane;     // the row this thread owns
    const uint32_t tl = tmem + (static_cast<uint32_t>(q * 32) << 16);
    constexpr bool kStats = KIND == LN_RELU || KIND == RELU_LN_RES;
    float shift = 0.f, s1 = 0.f, s2 = 0.f;          // LayerNorm sums of (x - shift), shift = the row's first value
    float m = -INFINITY, se = 0.f;                  // ARGMAX: running max and sum of exp(x - m)
    int best = 0;
    const int64_t grow = tile * kTileRows + r;      // row inside the sub-chunk
    for (int j = 0; j < n_chunks; ++j) {
      const int nc = min(kNChunk, a.np - j * kNChunk);
      const uint32_t buf = j & 1;
      ptx::mbar_wait(ptx::smem_u32(&acc_full[buf]), (j >> 1) & 1u);
      ptx::tc_fence_after_sync();
#pragma unroll 1
      for (int g = 0; g < nc / 32; ++g) {
        const int n0 = j * kNChunk + 32 * g;
        uint32_t v[32];
        ptx::tmem_ld_32x32(tl + buf * kNChunk + 32 * g, v);
        float b[32], x[32];
        vec32(a.bias + n0, b);
        ptx::tmem_wait_ld(v);
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          x[e] = __uint_as_float(v[e]) + b[e];
          if constexpr (KIND != LN_RELU && KIND != ARGMAX) x[e] = fmaxf(x[e], 0.f);
        }
        if constexpr (kStats) {
          if (n0 == 0) shift = x[0];
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if (n0 + e < a.n_true) {
              const float t = x[e] - shift;
              s1 += t;
              s2 = fmaf(t, t, s2);
            }
        }
        if constexpr (KIND == ARGMAX) {
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if (n0 + e < a.n_true) {
              if (x[e] > m) {
                se = fmaf(se, expf(m - x[e]), 1.f);
                m = x[e];
                best = n0 + e;
              } else {
                se += expf(x[e] - m);
              }
            }
          if (a.logits && grow < a.rows) {
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (n0 + e < a.n_true) a.logits[grow * a.n_true + n0 + e] = x[e];
          }
        } else {
          if constexpr (KIND == RES_RELU) {
            float h[32];
            load32(a.res, tile, a.np, r, n0, h);
#pragma unroll
            for (int e = 0; e < 32; ++e) x[e] += h[e];
          }
          store32(a.out, tile, a.np, r, n0, x);
        }
      }
      ptx::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&acc_empty[buf]));
    }
    if constexpr (kStats) {
      // second sweep over the row this thread has just written: normalise (+ ReLU | + residual)
      const float inv_n = 1.f / static_cast<float>(a.n_true);
      const float mu = s1 * inv_n;
      const float var = fmaxf(s2 * inv_n - mu * mu, 0.f);
      const float mean = shift + mu, rstd = rsqrtf(var + kLnEps);
#pragma unroll 1
      for (int n0 = 0; n0 < a.np; n0 += 32) {
        float x[32], gm[32], bt[32];
        load32(a.out, tile, a.np, r, n0, x);
        vec32(a.gamma + n0, gm);
        vec32(a.beta + n0, bt);
#pragma unroll
        for (int e = 0; e < 32; ++e) x[e] = fmaf((x[e] - mean) * rstd, gm[e], bt[e]);
        if constexpr (KIND == LN_RELU) {
#pragma unroll
          for (int e = 0; e < 32; ++e) x[e] = fmaxf(x[e], 0.f);
        } else {
          float h[32];
          load32(a.res, tile, a.np, r, n0, h);
#pragma unroll
          for (int e = 0; e < 32; ++e) x[e] += h[e];
        }
        store32(a.out, tile, a.np, r, n0, x);
      }
    }
    if constexpr (KIND == ARGMAX) {
      if (grow < a.rows) {
        a.pred[grow * a.pred_stride] = best;
        if (a.conf) a.conf[grow * a.conf_stride] = 1.f / se;
      }
    }
  }

  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc(tmem, 512);
  }
}

// The attention gate of one level on CUDA cores (0.875 E^2 MACs a row), fp32: kGateParts threads per row, each computing
// every kGateParts-th output of a layer, the rows of the tile transposed in shared memory so that every access is conflict
// free, the weights read as broadcasts (a warp holds 32 rows of one part).  Writes g as fp16 into the first GEMM's operand
// layout, zeros in the padded columns and in the rows past the end.
constexpr int kGateParts = 4;

struct GateArgs {
  const float* emb;      // [L, N, D] fp32 (last dimension contiguous), already offset to the sub-chunk's first row
  int64_t level_stride, row_stride;
  int d, e, normalize;
  int64_t rows;
  const float *w0, *b0, *w1, *b1, *w2, *b2;
  uint8_t* out;          // width pad64(e)
};

int gate_smem_bytes(int e) { return (e + e / 4 + e / 2 + kGateParts) * kTileRows * 4; }

__global__ void __launch_bounds__(kTileRows * kGateParts) tag_gate_kernel(GateArgs a) {
  extern __shared__ float gsm[];
  const int e = a.e, e4 = e / 4, e2 = e / 2;
  const int r = threadIdx.x % kTileRows, part = threadIdx.x / kTileRows;
  float* sx = gsm;                     // [e][128]
  float* s1 = sx + e * kTileRows;      // [e4][128]
  float* s2 = s1 + e4 * kTileRows;     // [e2][128]
  float* sss = s2 + e2 * kTileRows;    // [kGateParts][128] partial sums of g^2
  const int64_t tile = blockIdx.x, row = tile * kTileRows + r;
  const bool live = row < a.rows;
  for (int k = part; k < e; k += kGateParts) {
    const int lvl = k / a.d, c = k % a.d;
    sx[k * kTileRows + r] = live ? __ldg(a.emb + lvl * a.level_stride + row * a.row_stride + c) : 0.f;
  }
  __syncthreads();
  for (int o = part; o < e4; o += kGateParts) {
    float s = __ldg(a.b0 + o);
    for (int k = 0; k < e; ++k) s = fmaf(__ldg(a.w0 + o * e + k), sx[k * kTileRows + r], s);
    s1[o * kTileRows + r] = fmaxf(s, 0.f);
  }
  __syncthreads();
  for (int o = part; o < e2; o += kGateParts) {
    float s = __ldg(a.b1 + o);
    for (int k = 0; k < e4; ++k) s = fmaf(__ldg(a.w1 + o * e4 + k), s1[k * kTileRows + r], s);
    s2[o * kTileRows + r] = 0.5f * s * (1.f + erff(s * 0.70710678118654752f));  // nn.GELU(): the exact erf form
  }
  __syncthreads();
  float ss = 0.f;
  for (int o = part; o < e; o += kGateParts) {
    float s = __ldg(a.b2 + o);
    for (int k = 0; k < e2; ++k) s = fmaf(__ldg(a.w2 + o * e2 + k), s2[k * kTileRows + r], s);
    const float g = sx[o * kTileRows + r] / (1.f + expf(-s));
    sx[o * kTileRows + r] = g;   // only this thread reads or writes column o from here on
    ss = fmaf(g, g, ss);
  }
  sss[part * kTileRows + r] = ss;
  __syncthreads();
  ss = 0.f;
#pragma unroll
  for (int p = 0; p < kGateParts; ++p) ss += sss[p * kTileRows + r];
  const float inv = a.normalize ? 1.f / fmaxf(sqrtf(ss), 1e-12f) : 1.f;  // F.normalize(p=2, eps=1e-12)
  const int ep = pad64(e);
  for (int n0 = 32 * part; n0 < ep; n0 += 32 * kGateParts) {
    float x[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) x[j] = (live && n0 + j < e) ? sx[(n0 + j) * kTileRows + r] * inv : 0.f;
    store32(a.out, tile, ep, r, n0, x);
  }
}

// One parameter of a TagPredictor -> the image: a Linear weight [n, k] as fp16 blocks (block (j, c) = outputs
// [256 j, 256 j + nc) x inputs [64 c, 64 c + 64), inside [K group][output][8 fp16]), or a vector / gate matrix as fp32
// zero-padded to `np` entries.
__global__ void tag_pack_kernel(const float* __restrict__ src, int n, int k, int np, int kp, int as_blocks, uint8_t* __restrict__ dst) {
  const int64_t u = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (!as_blocks) {
    if (u < np) reinterpret_cast<float*>(dst)[u] = u < static_cast<int64_t>(n) * k ? src[u] : 0.f;
    return;
  }
  if (u >= static_cast<int64_t>(np) * kp / 8) return;  // one 16-byte unit (8 fp16) per thread
  const int64_t off = u * 8;                             // fp16 element offset inside the matrix's blocks
  const int j = static_cast<int>(off / (static_cast<int64_t>(kNChunk) * kp));
  const int nc = min(kNChunk, np - j * kNChunk);
  const int64_t in_chunk = off - static_cast<int64_t>(j) * kNChunk * kp;
  const int c = static_cast<int>(in_chunk / (nc * 64));
  const int in_block = static_cast<int>(in_chunk % (nc * 64));
  const int kg = in_block / (nc * 8), o = (in_block % (nc * 8)) / 8;
  const int row = j * kNChunk + o, col0 = c * 64 + kg * 8;
  float v[8];
#pragma unroll
  for (int t = 0; t < 8; ++t) v[t] = (row < n && col0 + t < k) ? src[static_cast<int64_t>(row) * k + col0 + t] : 0.f;
  *reinterpret_cast<uint4*>(dst + off * 2) = make_uint4(pack_f16(v[0], v[1]), pack_f16(v[2], v[3]), pack_f16(v[4], v[5]), pack_f16(v[6], v[7]));
}

int pack_one(const float* src, int n, int k, int np, int kp, bool blocks, uint8_t* dst, cudaStream_t st) {
  const int64_t units = blocks ? static_cast<int64_t>(np) * kp / 8 : np;
  tag_pack_kernel<<<static_cast<unsigned>((units + 255) / 256), 256, 0, st>>>(src, n, k, np, kp, blocks ? 1 : 0, dst);
  HV_CUDA_CHECK(cudaGetLastError());
  return HV_OK;
}

int params_per_level(bool norm) { return norm ? 34 : 22; }

int launch_gemm(int kind, const GemmArgs& g, int64_t tiles, cudaStream_t st) {
  auto go = [&](auto kernel) -> int {
    if (int s = prepare_kernel(kernel, 0, kSmemBytes)) return s;
    kernel<<<static_cast<unsigned>(tiles), kThreads, kSmemBytes, st>>>(g);
    HV_CUDA_CHECK(cudaGetLastError());
    return HV_OK;
  };
  switch (kind) {
    case LN_RELU: return go(tag_gemm_kernel<LN_RELU>);
    case RELU_LN_RES: return go(tag_gemm_kernel<RELU_LN_RES>);
    case RELU: return go(tag_gemm_kernel<RELU>);
    case RES_RELU: return go(tag_gemm_kernel<RES_RELU>);
    default: return go(tag_gemm_kernel<ARGMAX>);
  }
}

}  // namespace
}  // namespace hv

extern "C" {

size_t hv_tag_heads_workspace_bytes(int n_levels, int d, int first_hidden, const int* class_counts, int use_norm, int64_t rows,
                                    size_t* image_bytes) {
  hv::Plan p;
  if (!hv::make_plan(n_levels, d, first_hidden, class_counts, use_norm, &p)) {
    if (image_bytes) *image_bytes = 0;
    return 0;
  }
  if (image_bytes) *image_bytes = p.image_bytes;
  return hv::scratch_bytes(p, rows);
}

int hv_tag_heads_pack(const float* const* params, int n_params, int n_levels, int d, int first_hidden, const int* class_counts,
                      int use_norm, void* image, size_t image_bytes, void* stream) {
  using namespace hv;
  Plan p;
  if (!make_plan(n_levels, d, first_hidden, class_counts, use_norm, &p)) {
    set_error("hv_tag_heads_pack: no tag-head instantiation for this shape");
    return HV_ERR_UNSUPPORTED;
  }
  if (n_params != n_levels * params_per_level(p.norm)) {
    set_error("hv_tag_heads_pack: expected %d parameters (%d per level), got %d", n_levels * params_per_level(p.norm),
              params_per_level(p.norm), n_params);
    return HV_ERR_BAD_SHAPE;
  }
  if (!params || !image) {
    set_error("hv_tag_heads_pack: null pointer");
    return HV_ERR_NULL;
  }
  for (int i = 0; i < n_params; ++i)
    if (!params[i]) {
      set_error("hv_tag_heads_pack: parameter %d is null", i);
      return HV_ERR_NULL;
    }
  if (!aligned16(image)) {
    set_error("hv_tag_heads_pack: the image must be 16-byte aligned");
    return HV_ERR_MISALIGNED;
  }
  if (image_bytes < p.image_bytes) {
    set_error("hv_tag_heads_pack: the image is %zu bytes (got %zu)", p.image_bytes, image_bytes);
    return HV_ERR_WORKSPACE;
  }
  auto st = static_cast<cudaStream_t>(stream);
  uint8_t* img = static_cast<uint8_t*>(image);
  const float* const* q = params;
  for (int i = 0; i < n_levels; ++i) {
    const Level& L = p.lv[i];
    const int ge[4] = {L.e, L.e / 4, L.e / 2, L.e};
    for (int j = 0; j < 3; ++j) {  // attention.{0,2,4}.weight / .bias
      const int nw = ge[j + 1] * ge[j];
      if (int s = pack_one(*q++, nw, 1, nw, 0, false, img + L.gw[j], st)) return s;
      if (int s = pack_one(*q++, ge[j + 1], 1, ge[j + 1], 0, false, img + L.gb[j], st)) return s;
    }
    // TagPredictor parameter order: Linear weight, bias, then the LayerNorm's weight, bias where there is one
    auto linear = [&](const Lin& l, bool ln) -> int {
      if (int s = pack_one(*q++, l.n, l.k, l.np, l.kp, true, img + l.w, st)) return s;
      if (int s = pack_one(*q++, l.n, 1, l.np, 0, false, img + l.b, st)) return s;
      if (ln && p.norm) {
        if (int s = pack_one(*q++, l.n, 1, l.np, 0, false, img + l.g, st)) return s;
        if (int s = pack_one(*q++, l.n, 1, l.np, 0, false, img + l.be, st)) return s;
      }
      return HV_OK;
    };
    const Lin* order[8] = {&L.f, &L.a[0], &L.b[0], &L.a[1], &L.b[1], &L.c1, &L.c2, &L.c3};
    const bool ln[8] = {true, true, true, true, true, true, false, false};
    for (int k = 0; k < 8; ++k)
      if (int s = linear(*order[k], ln[k])) return s;
  }
  return HV_OK;
}

int hv_tag_heads_forward(const float* emb, int64_t emb_level_stride, int64_t emb_row_stride, int64_t n, int n_levels, int d,
                         int first_hidden, const int* class_counts, int use_norm, const void* image, size_t image_bytes,
                         int64_t* pred_out, int64_t pred_row_stride, int64_t pred_level_stride, float* conf_out,
                         int64_t conf_row_stride, int64_t conf_level_stride, float* const* logits_out, void* workspace,
                         size_t workspace_bytes, void* stream) {
  using namespace hv;
  if (n < 0) {
    set_error("hv_tag_heads_forward: bad row count %lld", static_cast<long long>(n));
    return HV_ERR_BAD_SHAPE;
  }
  Plan p;
  if (!make_plan(n_levels, d, first_hidden, class_counts, use_norm, &p)) {
    set_error("hv_tag_heads_forward: no tag-head instantiation for this shape");
    return HV_ERR_UNSUPPORTED;
  }
  if (n == 0) return HV_OK;
  if (!emb || !image || !pred_out || !workspace) {
    set_error("hv_tag_heads_forward: null pointer");
    return HV_ERR_NULL;
  }
  if (!aligned16(image) || !aligned16(workspace)) {
    set_error("hv_tag_heads_forward: the image and the workspace must be 16-byte aligned");
    return HV_ERR_MISALIGNED;
  }
  if (image_bytes < p.image_bytes || workspace_bytes < scratch_bytes(p, n)) {
    set_error("hv_tag_heads_forward: needs an image of %zu bytes and a workspace of %zu bytes (got %zu, %zu)", p.image_bytes,
              scratch_bytes(p, n), image_bytes, workspace_bytes);
    return HV_ERR_WORKSPACE;
  }
  DeviceProps props;
  if (int st = device_props(&props)) return st;
  if (props.cc_major != 10) {
    set_error("hv_tag_heads_forward: built for sm_100a, current device is sm_%d%d", props.cc_major, props.cc_minor);
    return HV_ERR_UNSUPPORTED;
  }
  auto st = static_cast<cudaStream_t>(stream);
  const uint8_t* img = static_cast<const uint8_t*>(image);
  const int64_t chunk_rows = std::min<int64_t>(n, kChunkRows);
  const size_t buf_rows = static_cast<size_t>((chunk_rows + kTileRows - 1) / kTileRows) * kTileRows;
  uint8_t* h0 = static_cast<uint8_t*>(workspace);
  uint8_t* h1 = h0 + buf_rows * p.res_width * 2;
  uint8_t* t = h1 + buf_rows * p.res_width * 2;
  auto f32 = [&](size_t off) { return reinterpret_cast<const float*>(img + off); };
  for (int64_t r0 = 0; r0 < n; r0 += kChunkRows) {
    const int64_t rows = std::min<int64_t>(kChunkRows, n - r0);
    const int64_t tiles = (rows + kTileRows - 1) / kTileRows;
    for (int i = 0; i < n_levels; ++i) {
      const Level& L = p.lv[i];
      GateArgs ga{emb + r0 * emb_row_stride, emb_level_stride, emb_row_stride, d, L.e, i > 0 ? 1 : 0, rows,
                  f32(L.gw[0]), f32(L.gb[0]), f32(L.gw[1]), f32(L.gb[1]), f32(L.gw[2]), f32(L.gb[2]), h1};
      const int gate_smem = gate_smem_bytes(L.e);
      if (int s = prepare_kernel(tag_gate_kernel, 0, gate_smem)) return s;
      tag_gate_kernel<<<static_cast<unsigned>(tiles), kTileRows * kGateParts, gate_smem, st>>>(ga);
      HV_CUDA_CHECK(cudaGetLastError());
      auto gemm = [&](int kind, const Lin& l, const uint8_t* in, uint8_t* out, const uint8_t* res) -> int {
        GemmArgs g{};
        g.a = in, g.w = img + l.w, g.bias = f32(l.b), g.out = out, g.res = res;
        g.gamma = l.g ? f32(l.g) : nullptr, g.beta = l.be ? f32(l.be) : nullptr;
        g.kp = l.kp, g.np = l.np, g.n_true = l.n, g.rows = rows;
        if (kind == ARGMAX) {
          g.pred = pred_out + r0 * pred_row_stride + i * pred_level_stride, g.pred_stride = pred_row_stride;
          g.conf = conf_out ? conf_out + r0 * conf_row_stride + i * conf_level_stride : nullptr, g.conf_stride = conf_row_stride;
          g.logits = logits_out && logits_out[i] ? logits_out[i] + r0 * l.n : nullptr;
        }
        return launch_gemm(kind, g, tiles, st);
      };
      const int ln_relu = p.norm ? LN_RELU : RELU, outer = p.norm ? RELU_LN_RES : RES_RELU;
      if (int s = gemm(ln_relu, L.f, h1, h0, nullptr)) return s;                   // feature extractor
      if (int s = gemm(ln_relu, L.a[0], h0, t, nullptr)) return s;                 // residual_block1
      if (int s = gemm(outer, L.b[0], t, h1, h0)) return s;
      if (int s = gemm(ln_relu, L.a[1], h1, t, nullptr)) return s;                 // residual_block2
      if (int s = gemm(outer, L.b[1], t, h0, h1)) return s;
      if (int s = gemm(ln_relu, L.c1, h0, t, nullptr)) return s;                   // classifier
      if (int s = gemm(RELU, L.c2, t, h1, nullptr)) return s;
      if (int s = gemm(ARGMAX, L.c3, h1, nullptr, nullptr)) return s;
    }
  }
  return HV_OK;
}

}  // extern "C"
