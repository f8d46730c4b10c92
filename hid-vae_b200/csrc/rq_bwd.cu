// Fused backward of the L-level residual quantiser (STE / rotation trick / eval) -- HBM-bound, no GEMM.
//
// One pass over the rows.  A row is spread over D/W lanes (W = 4 or 8 floats each, Frag) so every global access of a warp
// is a run of contiguous 16-byte pieces; dot products are reduced with xor-shuffles inside the lane group.
// The forward chain r_l, e_l is recomputed from x, ids and the codebooks (nothing was saved by the forward; level_forward),
// then the recursion of SURVEY.md section 8a runs from the last level to the first (level_backward):
//     h   = g_emb_l - G                      (G = dLoss/d r_{l+1})
//     Jh  = h                                (STE)      | h - 2 (h.w) w + 2 (h.q) u   (rotation trick)
//     G   = G + Jh + 2 beta (r_l - e_l) g_loss          | eval: G = G + 2 beta (r_l - e_l) g_loss
//     gC_l[id_l] += 2 (e_l - r_l) g_loss                | eval: += h + 2 (e_l - r_l) g_loss
// The codebook gradient is a scatter-add by id (the embedding_dense_backward of modules/quantize.py:97-98): one
// red.global.add.v4.f32 per 16-byte piece, spread over zeroed replicas of [L, K, D] for large N (folded by a second tiny kernel).
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"
#include "ptx.cuh"

namespace hv {
namespace {

constexpr int kMaxLevels = 8;
constexpr int kBwdThreads = 256;
constexpr int kBwdMinBlocks = 3;  // CTAs per SM the exact-level row-kernel instantiations are compiled for (register cap 80)

struct RqBwdArgs {
  const float* x;
  const float* codebooks;
  int64_t n;
  int n_levels;
  int k;
  float beta;
  int training;
  const int64_t* ids;
  int64_t ids_row_stride;
  int64_t ids_level_stride;
  const float* g_emb;
  int64_t g_emb_level_stride;
  int64_t g_emb_row_stride;
  const float* g_loss;
  int64_t g_loss_stride;
  const float* g_level_loss;
  float* g_x;
  float* g_codebooks;
  float* replicas;    // [n_replicas, L, K, D] zeroed scratch or null: CTAs spread their reductions over the copies
  int n_replicas;
};

template <int LPR>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int off = LPR / 2; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

// A lane's W floats of a row.  W = 4: one 16-byte piece, dims [4 sub, 4 sub + 4).  W = 8: two pieces HALF A ROW apart (those
// dims and D/2 + the same), so that the lanes of a row cover whole 32-byte sectors with each instruction.  The helpers below
// take the row's first element and the lane's index in the row's lane group.
template <int W>
struct Frag {
  static_assert(W == 4 || W == 8, "four or eight floats per lane");
  float v[W];
};

// piece j of the lane: float4 number sub + j D/8 of the row
template <int D, int W>
__device__ __forceinline__ Frag<W> ldg_frag(const float* row, int sub) {
  Frag<W> f;
  const float4 t = __ldg(reinterpret_cast<const float4*>(row) + sub);
  f.v[0] = t.x, f.v[1] = t.y, f.v[2] = t.z, f.v[3] = t.w;
  if constexpr (W == 8) {
    const float4 u = __ldg(reinterpret_cast<const float4*>(row) + sub + D / 8);
    f.v[4] = u.x, f.v[5] = u.y, f.v[6] = u.z, f.v[7] = u.w;
  }
  return f;
}
template <int D, int W>
__device__ __forceinline__ Frag<W> lds_frag(const float* row, int sub) {
  Frag<W> f;
  const float4 t = reinterpret_cast<const float4*>(row)[sub];
  f.v[0] = t.x, f.v[1] = t.y, f.v[2] = t.z, f.v[3] = t.w;
  if constexpr (W == 8) {
    const float4 u = reinterpret_cast<const float4*>(row)[sub + D / 8];
    f.v[4] = u.x, f.v[5] = u.y, f.v[6] = u.z, f.v[7] = u.w;
  }
  return f;
}
template <int D, int W>
__device__ __forceinline__ void store_frag(float* row, int sub, const Frag<W>& f) {
  reinterpret_cast<float4*>(row)[sub] = make_float4(f.v[0], f.v[1], f.v[2], f.v[3]);
  if constexpr (W == 8) reinterpret_cast<float4*>(row)[sub + D / 8] = make_float4(f.v[4], f.v[5], f.v[6], f.v[7]);
}
// one 16-byte reduction per piece instead of four scalar atomics (sm_90+: red.global.add.v4.f32)
__device__ __forceinline__ void red_add_v4(float* addr, float x, float y, float z, float w) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
template <int D, int W>
__device__ __forceinline__ void red_add_frag(float* base, int64_t row_off, int sub, const Frag<W>& f) {  // row = base + row_off
  float* p = base + (row_off + sub * 4);
  red_add_v4(p, f.v[0], f.v[1], f.v[2], f.v[3]);
  if constexpr (W == 8) red_add_v4(p + D / 2, f.v[4], f.v[5], f.v[6], f.v[7]);
}
// the lane's part of a dot product: one fmaf chain at W = 4, two accumulators at W = 8
template <int W>
__device__ __forceinline__ float dot(const Frag<W>& a, const Frag<W>& b) {
  if constexpr (W == 4) {
    return fmaf(a.v[0], b.v[0], fmaf(a.v[1], b.v[1], fmaf(a.v[2], b.v[2], a.v[3] * b.v[3])));
  } else {
    float s0 = a.v[0] * b.v[0], s1 = a.v[1] * b.v[1];
#pragma unroll
    for (int i = 2; i < W; i += 2) s0 = fmaf(a.v[i], b.v[i], s0), s1 = fmaf(a.v[i + 1], b.v[i + 1], s1);
    return s0 + s1;
  }
}

// One level of the recomputed forward chain: r_l -> r_{l+1} = r_l - o_l with o = e (STE, eval) or o = cr r + ce e (rotation
// trick, modules/quantize.py:34-45), whose scalars are kept in `c` for the backward.  r.r, e.e and r.e are the only row sums
// (3 shuffle reductions instead of 5).
template <int LPR, int W, bool ROT>
__device__ __forceinline__ void level_forward(Frag<W>& r, const Frag<W>& e, RotCoeffs& c) {
  Frag<W> o = e;
  if constexpr (ROT) {
    const float rr = group_sum<LPR>(dot(r, r));
    const float ee = group_sum<LPR>(dot(e, e));
    const float re = group_sum<LPR>(dot(r, e));
    c = rot_coeffs(rr, ee, re);
#pragma unroll
    for (int i = 0; i < W; ++i) o.v[i] = fmaf(c.cr, r.v[i], c.ce * e.v[i]);
  }
#pragma unroll
  for (int i = 0; i < W; ++i) r.v[i] -= o.v[i];
}

// One step of the recursion at level l (rl = r_l, el = e_l, ge = g_emb_l, gl = the level's loss gradient): G becomes
// dLoss/d r_l; returns the lane's piece of the gradient of the code row e_l.
template <int LPR, int W, bool ROT, bool TRAIN>
__device__ __forceinline__ Frag<W> level_backward(Frag<W>& G, const Frag<W>& ge, const Frag<W>& rl, const Frag<W>& el,
                                                  const RotCoeffs& c, float gl, float beta) {
  Frag<W> h, diff, ge_code;
#pragma unroll
  for (int i = 0; i < W; ++i) h.v[i] = ge.v[i] - G.v[i];
#pragma unroll
  for (int i = 0; i < W; ++i) diff.v[i] = rl.v[i] - el.v[i];
  const float c2 = 2.0f * gl;
#pragma unroll
  for (int i = 0; i < W; ++i) ge_code.v[i] = -c2 * diff.v[i];
  const float cb2 = beta * c2;
  if constexpr (TRAIN) {
    if constexpr (ROT) {  // Jh with u = r ir, q = e ie, w = (u + q) is
      Frag<W> u, q, w;
#pragma unroll
      for (int i = 0; i < W; ++i) u.v[i] = rl.v[i] * c.ir;
#pragma unroll
      for (int i = 0; i < W; ++i) q.v[i] = el.v[i] * c.ie;
#pragma unroll
      for (int i = 0; i < W; ++i) w.v[i] = (u.v[i] + q.v[i]) * c.is;
      const float hw2 = 2.0f * group_sum<LPR>(dot(h, w));
      const float hq2 = 2.0f * group_sum<LPR>(dot(h, q));
#pragma unroll
      for (int i = 0; i < W; ++i) h.v[i] = h.v[i] - hw2 * w.v[i] + hq2 * u.v[i];
    }
#pragma unroll
    for (int i = 0; i < W; ++i) G.v[i] += h.v[i] + cb2 * diff.v[i];
  } else {
#pragma unroll
    for (int i = 0; i < W; ++i) G.v[i] += cb2 * diff.v[i];
#pragma unroll
    for (int i = 0; i < W; ++i) ge_code.v[i] += h.v[i];
  }
  return ge_code;
}

// Row kernel: four floats per lane, code rows gathered from global memory.
// NL > 0: exactly NL levels, known at compile time (no per-level branches, register arrays of that size; 1..4 cover
// every shipped config and keep the kernel at 3+ CTAs per SM); NL == 0: runtime level count up to kMaxLevels.
// ROT / TRAIN: rotation-trick Jacobian / training semantics (eval: emb_out = e for every mode, quantize.py:146-147).
template <int D, bool ROT, bool TRAIN, int NL>
__global__ void __launch_bounds__(kBwdThreads, NL > 0 ? kBwdMinBlocks : 1) rq_bwd_kernel(RqBwdArgs a) {
  static_assert(TRAIN || !ROT, "eval has no rotation");
  constexpr int LMAX = NL > 0 ? NL : kMaxLevels;
  constexpr int LPR = D / 4;  // lanes per row
  constexpr int ROWS_PER_WARP = 32 / LPR;

  const int64_t lkd = static_cast<int64_t>(a.n_levels) * a.k * D;
  const int lane = threadIdx.x & 31;
  const int sub = lane % LPR;
  const int warp_global = ptx::uniform((blockIdx.x * kBwdThreads + threadIdx.x) >> 5);  // (see ptx::warp_index)
  const int n_warps = (gridDim.x * kBwdThreads) >> 5;
  const int64_t n_groups = (a.n + ROWS_PER_WARP - 1) / ROWS_PER_WARP;
  float* gc_base = a.n_replicas > 0 ? a.replicas + static_cast<int64_t>(blockIdx.x % a.n_replicas) * lkd : a.g_codebooks;

  for (int64_t g = warp_global; g < n_groups; g += n_warps) {
    const int64_t row = g * ROWS_PER_WARP + lane / LPR;
    const bool valid = row < a.n;
    const int64_t rrow = valid ? row : 0;  // keep every lane in the shuffles; mask the stores

    Frag<4> R[LMAX], E[LMAX];
    RotCoeffs rc[LMAX];
    int id[LMAX];
    Frag<4> r = ldg_frag<D, 4>(a.x + rrow * D, sub);
#pragma unroll
    for (int l = 0; l < LMAX; ++l) {
      if (NL > 0 || l < a.n_levels) {
        int64_t code = a.ids[rrow * a.ids_row_stride + l * a.ids_level_stride];
        code = code < 0 ? 0 : (code >= a.k ? a.k - 1 : code);
        id[l] = static_cast<int>(code);
        E[l] = ldg_frag<D, 4>(a.codebooks + (static_cast<int64_t>(l) * a.k + code) * D, sub);
        R[l] = r;
        level_forward<LPR, 4, ROT>(r, E[l], rc[l]);
      }
    }

    // every load of the row is issued before the recursion (the red.add below orders memory, so nothing can be
    // hoisted across it by the compiler): one latency exposure per row instead of one per level
    const float gl_all = a.g_loss != nullptr ? a.g_loss[rrow * a.g_loss_stride] : 0.f;
    Frag<4> GE[LMAX];
    float GL[LMAX];
#pragma unroll
    for (int l = 0; l < LMAX; ++l) {
      GE[l] = Frag<4>{};
      GL[l] = gl_all;
      if (NL > 0 || l < a.n_levels) {
        if (a.g_emb != nullptr) GE[l] = ldg_frag<D, 4>(a.g_emb + l * a.g_emb_level_stride + rrow * a.g_emb_row_stride, sub);
        if (a.g_level_loss != nullptr) GL[l] += a.g_level_loss[static_cast<int64_t>(l) * a.n + rrow];
      }
    }
    Frag<4> G{};
#pragma unroll
    for (int l = LMAX - 1; l >= 0; --l) {
      if (NL > 0 || l < a.n_levels) {
        const Frag<4> ge_code = level_backward<LPR, 4, ROT, TRAIN>(G, GE[l], R[l], E[l], rc[l], GL[l], a.beta);
        if (valid) red_add_frag<D>(gc_base, (static_cast<int64_t>(l) * a.k + id[l]) * D, sub, ge_code);
      }
    }
    if (valid) store_frag<D>(a.g_x + row * D, sub, G);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Large-N kernel for codebooks that fit in shared memory (L K D 4 <= 96 KB: every HiD-VAE config).  Same arithmetic as the
// row kernel, without the memory latency that kernel exposes per row (ncu: stall_long_scoreboard 39 % of warp time):
//   * the fp32 codebooks are staged in shared memory once per persistent CTA: the id -> code row gather
//     is an LDS.128 instead of a dependent round trip to L2 (and 4 L D bytes per row less L2 traffic), and the backward
//     sweep reads the chosen code rows from there a second time instead of keeping them in registers;
//   * the row's inputs (x, ids, g_emb, g_loss) are loaded ONE ITERATION AHEAD into registers, so no load of the current
//     row is ever waited for.
// W = 8 serves the rotation trick in training.  At W = 4 that chain is bound by issue slots (ncu: 70 % issue utilisation,
// 554 instructions per 4 rows), and about half of them are the per-row scalars -- shuffle reductions, three reciprocal norms,
// the rotation coefficients -- that every lane of a row repeats.  With half as many lanes per row each of those warp
// instructions serves twice as many rows and a reduction is one shuffle shorter.
// ---------------------------------------------------------------------------------------------------------------------
// One CTA per SM, of
//   W = 4: 512 threads.  STE training backward at 4 Mi rows: 0.674 ms at 2 x 320 threads, 0.642 at 1 x 384, 0.600 at 1 x 512;
//          the W = 8 kernel measures 0.708 on this chain -- it pays off where the per-row scalars dominate.
//   W = 8: 384 threads, i.e. 168 registers per thread: nothing spills and the compiler keeps more of the chain in registers.
//          Measured at 4 Mi rows (D = 32, L = 3): 2 x 256 threads (128 registers, 56 B of spills) 0.708 ms, 1 x 320 0.687,
//          1 x 352 0.637, 1 x 384 0.600, 1 x 416 / 448 (152 / 144 registers) 0.84, 1 x 512 0.696, 2 x 320 1.19, 3 x 192 1.89.
template <int W>
constexpr int kSmemThreads = W == 8 ? 384 : 512;
constexpr int kSmemLimit = 96 * 1024;
// Below this many rows the row kernel runs: staging the codebooks does not pay off (a threshold of 4,096 rows measured
// slower at 12 k and 32 k rows).
constexpr int64_t kSmemMinRows = 65536;

template <int D, int W, bool ROT, bool TRAIN, int NL>
__global__ void __launch_bounds__(kSmemThreads<W>, 1) rq_bwd_smem_kernel(RqBwdArgs a) {
  static_assert(TRAIN || !ROT, "eval has no rotation");
  constexpr int kThreads = kSmemThreads<W>;
  constexpr int LPR = D / W;
  constexpr int ROWS_PER_WARP = 32 / LPR;
  extern __shared__ __align__(16) float s_cb[];  // [NL][K][D]
  {
    const int total4 = NL * a.k * (D / 4);
    for (int i = threadIdx.x; i < total4; i += kThreads)
      reinterpret_cast<float4*>(s_cb)[i] = __ldg(reinterpret_cast<const float4*>(a.codebooks) + i);
  }
  __syncthreads();

  const int64_t lkd = static_cast<int64_t>(NL) * a.k * D;
  const int lane = threadIdx.x & 31;
  const int sub = lane % LPR;
  // (the broadcast tells the compiler that the value -- and with it the trip count of the row loop -- is warp-uniform: without it
  // every shuffle of the loop carries a WARPSYNC.COLLECTIVE / ENDCOLLECTIVE pair and register moves)
  const int warp_global = ptx::uniform((blockIdx.x * kThreads + threadIdx.x) >> 5);
  const int n_warps = (gridDim.x * kThreads) >> 5;
  const int64_t n_groups = (a.n + ROWS_PER_WARP - 1) / ROWS_PER_WARP;
  float* gc_base = a.n_replicas > 0 ? a.replicas + static_cast<int64_t>(blockIdx.x % a.n_replicas) * lkd : a.g_codebooks;

  // the next iteration's inputs
  Frag<W> nx, nge[NL];
  int nid[NL];
  float ngl;
  auto fetch = [&](int64_t g) {
    const int64_t row = g * ROWS_PER_WARP + lane / LPR;
    const int64_t rrow = row < a.n ? row : 0;  // keep every lane in the shuffles; the stores are masked
    nx = ldg_frag<D, W>(a.x + rrow * D, sub);
    ngl = a.g_loss != nullptr ? __ldg(a.g_loss + rrow * a.g_loss_stride) : 0.f;
#pragma unroll
    for (int l = 0; l < NL; ++l) {
      int64_t code = __ldg(a.ids + rrow * a.ids_row_stride + l * a.ids_level_stride);
      code = code < 0 ? 0 : (code >= a.k ? a.k - 1 : code);
      nid[l] = static_cast<int>(code);
      nge[l] = a.g_emb != nullptr ? ldg_frag<D, W>(a.g_emb + l * a.g_emb_level_stride + rrow * a.g_emb_row_stride, sub) : Frag<W>{};
    }
  };
  if (warp_global < n_groups) fetch(warp_global);

  for (int64_t g = warp_global; g < n_groups; g += n_warps) {
    const int64_t row = g * ROWS_PER_WARP + lane / LPR;
    const bool valid = row < a.n;
    Frag<W> r = nx;
    const float gl = ngl;
    Frag<W> GE[NL];
    int id[NL];
#pragma unroll
    for (int l = 0; l < NL; ++l) GE[l] = nge[l], id[l] = nid[l];
    if (g + n_warps < n_groups) fetch(g + n_warps);
    auto code_row = [&](int l) { return s_cb + (static_cast<int64_t>(l) * a.k + id[l]) * D; };

    Frag<W> R[NL];
    RotCoeffs rc[NL];
#pragma unroll
    for (int l = 0; l < NL; ++l) {
      R[l] = r;
      level_forward<LPR, W, ROT>(r, lds_frag<D, W>(code_row(l), sub), rc[l]);
    }
    Frag<W> G{};
#pragma unroll
    for (int l = NL - 1; l >= 0; --l) {
      const Frag<W> ge_code = level_backward<LPR, W, ROT, TRAIN>(G, GE[l], R[l], lds_frag<D, W>(code_row(l), sub), rc[l], gl, a.beta);
      if (valid) red_add_frag<D>(gc_base, (static_cast<int64_t>(l) * a.k + id[l]) * D, sub, ge_code);
    }
    if (valid) store_frag<D>(a.g_x + row * D, sub, G);
  }
}

// shapes the shared-memory kernel serves: exact-level instantiation, codebooks within 96 KB, no per-level loss gradient,
// and enough rows to amortise staging the codebooks
template <int D>
bool bwd_smem_ok(const RqBwdArgs& a) {
  return (D == 16 || D == 32 || D == 64) && a.n_levels >= 1 && a.n_levels <= 4 && a.g_level_loss == nullptr && a.n >= kSmemMinRows &&
         static_cast<int64_t>(a.n_levels) * a.k * D * 4 <= kSmemLimit;
}

template <int D>
int launch_d(const RqBwdArgs& a, bool rot, cudaStream_t stream) {
  DeviceProps props;
  if (int st = device_props(&props)) return st;
  constexpr int LPR = D / 4;
  constexpr int rows_per_cta = (kBwdThreads / 32) * (32 / LPR);
  int64_t ctas = (a.n + rows_per_cta - 1) / rows_per_cta;
  const int64_t cap = static_cast<int64_t>(props.sm_count) * 16;
  if (ctas > cap) ctas = cap;
  using Kernel = void (*)(RqBwdArgs);
  auto go = [&](Kernel kernel, int64_t grid, int threads, int smem_bytes) -> int {
    if (smem_bytes > 0) {
      if (int st = prepare_kernel(kernel, 0, smem_bytes)) return st;
    }
    kernel<<<static_cast<unsigned>(grid), threads, smem_bytes, stream>>>(a);
    HV_CUDA_CHECK(cudaGetLastError());
    return HV_OK;
  };
  const bool train = a.training != 0;
  const bool r = rot && train;  // eval: the rotation plays no part
  auto pick = [&](auto nl) -> int {
    constexpr int NLc = decltype(nl)::value;
    if constexpr (NLc > 0 && (D == 16 || D == 32 || D == 64)) {
      if (bwd_smem_ok<D>(a)) {  // eight floats per lane for the rotation trick in training, four for STE and eval
        const Kernel k = r ? rq_bwd_smem_kernel<D, 8, true, true, NLc>
                           : train ? rq_bwd_smem_kernel<D, 4, false, true, NLc> : rq_bwd_smem_kernel<D, 4, false, false, NLc>;
        return go(k, props.sm_count, r ? kSmemThreads<8> : kSmemThreads<4>, a.n_levels * a.k * D * 4);
      }
    }
    const Kernel k = r ? rq_bwd_kernel<D, true, true, NLc> : train ? rq_bwd_kernel<D, false, true, NLc> : rq_bwd_kernel<D, false, false, NLc>;
    return go(k, ctas, kBwdThreads, 0);
  };
  if constexpr (D == 16 || D == 32 || D == 64) {  // the shipped shapes get exact-level instantiations
    switch (a.n_levels) {
      case 1: return pick(std::integral_constant<int, 1>{});
      case 2: return pick(std::integral_constant<int, 2>{});
      case 3: return pick(std::integral_constant<int, 3>{});
      case 4: return pick(std::integral_constant<int, 4>{});
      default: break;
    }
  }
  return pick(std::integral_constant<int, 0>{});
}

}  // namespace

namespace {
// g_codebooks += sum over the replicas (they were zeroed before the main kernel ran)
__global__ void rq_bwd_fold_replicas_kernel(const float* __restrict__ replicas, int n_replicas, int64_t lkd4,
                                            float* __restrict__ g_codebooks) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= lkd4) return;
  float4 acc = reinterpret_cast<float4*>(g_codebooks)[i];
  for (int r = 0; r < n_replicas; ++r) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(replicas) + r * lkd4 + i);
    acc.x += v.x, acc.y += v.y, acc.z += v.z, acc.w += v.w;
  }
  reinterpret_cast<float4*>(g_codebooks)[i] = acc;
}

}  // namespace

// Replicas of the [L, K, D] gradient the CTAs spread their red.add over: the L2 atomic units serialise per address,
// and with 768 hot lines (K = 256, D = 32, L = 3) that serialisation was 40 % of the kernel (profiles/README.md).
int rq_bwd_replicas(int64_t n, int d, int k, int n_levels) {
  const int64_t lkd_bytes = static_cast<int64_t>(n_levels) * k * d * 4;
  if (n < 32768 || lkd_bytes <= 0) return 0;
  int64_t r = (32ll << 20) / lkd_bytes;  // at most 32 MiB of scratch
  r = r > 32 ? 32 : r;
  return r < 2 ? 0 : static_cast<int>(r);
}
size_t rq_bwd_workspace_bytes(int64_t n, int d, int k, int n_levels) {
  return static_cast<size_t>(rq_bwd_replicas(n, d, k, n_levels)) * n_levels * k * d * 4;
}
}  // namespace hv

extern "C" int hv_rq_backward(const float* x, int64_t n, int d, const float* codebooks, int n_levels, int k, int mode,
                              int training, float beta, const int64_t* ids, int64_t ids_row_stride,
                              int64_t ids_level_stride, const float* g_emb, int64_t g_emb_level_stride,
                              int64_t g_emb_row_stride, const float* g_loss, int64_t g_loss_stride,
                              const float* g_level_loss, float* g_x, float* g_codebooks, void* workspace,
                              size_t workspace_bytes, void* stream) {
  using namespace hv;
  if (n < 0 || d <= 0 || k <= 0 || n_levels <= 0) {
    set_error("hv_rq_backward: bad shape n=%lld d=%d k=%d L=%d", (long long)n, d, k, n_levels);
    return HV_ERR_BAD_SHAPE;
  }
  if (n_levels > kMaxLevels) {
    set_error("hv_rq_backward: at most %d levels are supported (got %d)", kMaxLevels, n_levels);
    return HV_ERR_UNSUPPORTED;
  }
  if (mode != HV_MODE_STE && mode != HV_MODE_ROTATION_TRICK) {
    set_error("hv_rq_backward: forward mode %d has no fused kernel (STE=2, ROTATION_TRICK=3)", mode);
    return HV_ERR_UNSUPPORTED;
  }
  if (n == 0) return HV_OK;
  if (!x || !codebooks || !ids || !g_x || !g_codebooks) {
    set_error("hv_rq_backward: null pointer");
    return HV_ERR_NULL;
  }
  if (!aligned16(x) || !aligned16(codebooks) || !aligned16(g_x) || !aligned16(g_codebooks) || (g_emb && !aligned16(g_emb)) ||
      (g_emb && ((g_emb_level_stride % 4) || (g_emb_row_stride % 4)))) {
    set_error("hv_rq_backward: x, codebooks, g_x, g_emb must be 16-byte aligned with strides that are multiples of 4");
    return HV_ERR_MISALIGNED;
  }
  RqBwdArgs a{x, codebooks, n, n_levels, k, beta, training ? 1 : 0, ids, ids_row_stride, ids_level_stride,
              g_emb, g_emb_level_stride, g_emb_row_stride, g_loss, g_loss_stride, g_level_loss, g_x, g_codebooks, nullptr, 0};
  const bool rot = mode == HV_MODE_ROTATION_TRICK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int n_rep = rq_bwd_replicas(n, d, k, n_levels);
  const size_t rep_bytes = rq_bwd_workspace_bytes(n, d, k, n_levels);
  const bool use_rep = n_rep > 0 && workspace != nullptr && workspace_bytes >= rep_bytes && aligned16(workspace);
  if (use_rep) {
    HV_CUDA_CHECK(cudaMemsetAsync(workspace, 0, rep_bytes, s));
    a.replicas = static_cast<float*>(workspace);
    a.n_replicas = n_rep;
  }
  int st;
  switch (d) {
    case 4: st = launch_d<4>(a, rot, s); break;
    case 8: st = launch_d<8>(a, rot, s); break;
    case 16: st = launch_d<16>(a, rot, s); break;
    case 32: st = launch_d<32>(a, rot, s); break;
    case 64: st = launch_d<64>(a, rot, s); break;
    case 128: st = launch_d<128>(a, rot, s); break;
    default:
      set_error("hv_rq_backward: embed dim %d has no instantiation (supported: 4, 8, 16, 32, 64, 128)", d);
      return HV_ERR_UNSUPPORTED;
  }
  if (st != HV_OK || !use_rep) return st;
  const int64_t lkd4 = static_cast<int64_t>(n_levels) * k * d / 4;
  rq_bwd_fold_replicas_kernel<<<static_cast<unsigned>((lkd4 + 255) / 256), 256, 0, s>>>(a.replicas, n_rep, lkd4, g_codebooks);
  HV_CUDA_CHECK(cudaGetLastError());
  return HV_OK;
}
