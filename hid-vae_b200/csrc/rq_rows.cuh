// Building blocks of the row-owner kernel of the fused quantiser forward (rq_fwd_tc_v11.cu): D = 32, K <= 256, one 256-code
// operand image per level resident in shared memory, a level = two units of 128 codes on 128-column accumulators in tensor
// memory, A operand (the residual's bf16 hi | lo halves) in tensor memory: the argmax scan, the MMA issue of one unit and the
// bf16 split.  The streamed generation (rq_fwd_tc_v4.cu) scans its 256-column units with the same fold.
//
// Measured on B200 (tools/micro/tmem_ld_shapes.cu): max.f32 with two inputs issues at 3.9 warp-instructions / cycle / SM,
// with three inputs at 1.95 -- a 3-input maximum costs the ALU pipe as much as two 2-input ones and only saves the issue
// slot; tcgen05.ld 32x32b.x16 + wait takes 40 cycles alone on the SM and delivers 374 B / cycle / SM with >= 12 warps
// (.x8: 308).
#pragma once

#include "common.cuh"
#include "ptx.cuh"

namespace hv {
namespace rows {

constexpr int D = 32;
constexpr int kTileRows = 128;
constexpr int kNTile = 256;   // codes per operand image
constexpr int kUnitCols = 128;
constexpr int kAccs = 3;
constexpr int kMaxLevels = 3;
constexpr int kQueue = 8;     // staged (warpgroup, level) requests waiting for the issuer
constexpr int kOnesBytes = 2 * kTileRows * 16;
constexpr int kBarBytes = 1024;
constexpr int kImageBytes = kNTile * (4 * D + 32);  // packed bf16 image of one level (rq_pack.cu)
constexpr int kCbBytes = kNTile * D * 4;            // swizzled fp32 codebook of one level
constexpr int kSmemLimit = 227 * 1024;

__device__ __forceinline__ float max3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));  // FMNMX3
  return d;
}
__device__ __forceinline__ float f(uint32_t v) { return __uint_as_float(v); }
__device__ __forceinline__ float max8(const uint32_t (&v)[8]) {
  return max3(max3(f(v[0]), f(v[1]), f(v[2])), max3(f(v[3]), f(v[4]), f(v[5])), fmaxf(f(v[6]), f(v[7])));
}
constexpr float kBig = 1.329227995784916e36f;  // 2^120

// Exact first-index (max, argmax) of one chunk of W columns against the running pair (slow path).
template <int W>
__device__ __forceinline__ void scan_chunk_exact(const uint32_t (&v)[W], int base, float& best, int& best_col) {
  float m = f(v[0]);
#pragma unroll
  for (int j = 1; j < W; ++j) m = fmaxf(m, f(v[j]));
  if (m > best) {  // strict: an earlier chunk keeps exact ties
    float t = -INFINITY;
#pragma unroll
    for (int j = 0; j < W; ++j) t = fmaxf(t, fmaf(f(v[j]) - m, kBig, static_cast<float>(W - j)));
    best = m;
    best_col = base + W - static_cast<int>(t);
  }
}

// Every scan below returns the maximum of this thread's row over the 128 columns of one accumulator at TMEM address `t0`
// and its FIRST column.  Fast path: a 2-D fold -- maxima per column class (column mod W) and per chunk (column / W) --
// locates the maximiser when exactly one class and one chunk attain it; otherwise the warp re-reads the unit and takes the
// exact first-index path.

// Location of the maximiser from the fold over 8 classes x NC chunks (shared by the 8-column scans).
template <int NC>
__device__ __forceinline__ void locate_8(uint32_t t0, const float (&g)[8], const float (&cm)[NC], float& m_out, int& col_out) {
  static_assert(NC == 8 || NC == 16 || NC == 32, "64, 128 or 256 columns");
  float m8[NC / 8];
#pragma unroll
  for (int i = 0; i < NC / 8; ++i)
    m8[i] = max3(max3(cm[8 * i], cm[8 * i + 1], cm[8 * i + 2]), max3(cm[8 * i + 3], cm[8 * i + 4], cm[8 * i + 5]), fmaxf(cm[8 * i + 6], cm[8 * i + 7]));
  float m = m8[0];
#pragma unroll
  for (int i = 1; i < NC / 8; ++i) m = fmaxf(m, m8[i]);
  // class of the maximiser: sum_j [g_j == m] * (16 + j);  chunk: sum_c [cm_c == m] * (NC + c)   (FMA pipe)
  float s2[2] = {0.f, 0.f};
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float e = __saturatef(fmaf(g[j] - m, kBig, 1.0f));
    s2[j & 1] = fmaf(e, static_cast<float>(16 + j), s2[j & 1]);
  }
  float c4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const float e = __saturatef(fmaf(cm[c] - m, kBig, 1.0f));
    c4[c & 3] = fmaf(e, static_cast<float>(NC + c), c4[c & 3]);
  }
  const float cls = s2[0] + s2[1];
  const float chk = (c4[0] + c4[1]) + (c4[2] + c4[3]);
  // one class: 16..23, two or more: >= 33; one chunk: NC..2 NC - 1, two or more: >= 2 NC + 1
  const bool unique = (cls < 32.f && chk < static_cast<float>(2 * NC)) || m < -1e29f;
  float best = m;
  int col = 8 * (static_cast<int>(chk) - NC) + static_cast<int>(cls) - 16;
  if (__any_sync(0xffffffffu, !unique)) {
    best = -INFINITY;
    col = 0;
    uint32_t v[8];
#pragma unroll 1
    for (int c = 0; c < NC; ++c) {
      ptx::tmem_ld_32x8(t0 + 8 * c, v);
      ptx::tmem_wait_ld8(v);
      scan_chunk_exact<8>(v, 8 * c, best, col);
    }
  }
  m_out = best;
  col_out = col;
}

// 8-column loads over 8 NC columns from `t0`, software-pipelined: while one pair of loads is processed (3-input maxima,
// 1.0 ALU instruction per score) the next pair is in flight.  It takes the same 32 load registers as an unpipelined scan of
// two 16-column loads per step and spills nothing beside the 32-float row (that scan spilled 20 bytes and exposed the load
// latency four times per unit): 4 Mi-row encode 0.609 -> 0.587 ms, training forward 0.927 -> 0.852 ms.
template <int NC>
__device__ __forceinline__ void scan_x8_pairs(uint32_t t0, float& m_out, int& col_out) {
  float g[8], cm[NC];
  uint32_t a[2][8], b[2][8];
  ptx::tmem_ld_32x8(t0, a[0]);
  ptx::tmem_ld_32x8(t0 + 8, b[0]);
  ptx::tmem_wait_ld8(a[0], b[0]);
#pragma unroll
  for (int p = 0; p < NC / 2; ++p) {
    if (p + 1 < NC / 2) {
      ptx::tmem_ld_32x8(t0 + 16 * (p + 1), a[(p + 1) & 1]);
      ptx::tmem_ld_32x8(t0 + 16 * (p + 1) + 8, b[(p + 1) & 1]);
    }
    cm[2 * p] = max8(a[p & 1]);
    cm[2 * p + 1] = max8(b[p & 1]);
#pragma unroll
    for (int j = 0; j < 8; ++j)
      g[j] = p == 0 ? fmaxf(f(a[0][j]), f(b[0][j])) : max3(g[j], f(a[p & 1][j]), f(b[p & 1][j]));
    if (p + 1 < NC / 2) ptx::tmem_wait_ld8(a[(p + 1) & 1], b[(p + 1) & 1]);
  }
  locate_8<NC>(t0, g, cm, m_out, col_out);
}

__device__ __forceinline__ void scan_unit_x8_pairs(uint32_t t0, float& m_out, int& col_out) { scan_x8_pairs<16>(t0, m_out, col_out); }

// One unit (128 codes starting at code `col0` of the level's image): 3*D/16 MMAs with A from tensor memory, the norm
// MMA with the constant ones block from shared memory, one commit.  Called by ONE elected thread.
__device__ __forceinline__ void issue_unit(uint32_t acc, uint32_t a_tmem, uint32_t ones, uint32_t b_tile, int col0,
                                           uint32_t bar_done) {
  constexpr uint32_t idesc = ptx::umma_idesc_bf16(kTileRows, kUnitCols);
  const uint32_t hi = ptx::umma_desc_hi(128);
  constexpr uint32_t chunk_b = kNTile * 16;  // bytes between K chunks of the B image
  constexpr uint32_t b_step = 2 * kNTile;    // one K=16 step = two chunks, in 16-byte units
  const uint32_t b_hi = b_tile + col0 * 16;
  const uint32_t d_bhi = ptx::umma_desc_lo(b_hi, chunk_b);
  const uint32_t d_blo = ptx::umma_desc_lo(b_hi + (D / 8) * chunk_b, chunk_b);
  const uint32_t d_bnrm = ptx::umma_desc_lo(b_hi + 2 * (D / 8) * chunk_b, chunk_b);
  const uint32_t d_one = ptx::umma_desc_lo(ones, kTileRows * 16);
  const uint32_t a_hi = a_tmem, a_lo = a_tmem + D / 2;  // D/2 columns each: two bf16 per column
#pragma unroll
  for (int j = 0; j < D / 16; ++j)  // r_hi . c_hi
    ptx::umma_bf16_ts(acc, a_hi + 8 * j, ptx::umma_desc(d_bhi + j * b_step, hi), idesc, j > 0 ? 1u : 0u);
#pragma unroll
  for (int j = 0; j < D / 16; ++j)  // r_lo . c_hi
    ptx::umma_bf16_ts(acc, a_lo + 8 * j, ptx::umma_desc(d_bhi + j * b_step, hi), idesc, 1u);
#pragma unroll
  for (int j = 0; j < D / 16; ++j)  // r_hi . c_lo
    ptx::umma_bf16_ts(acc, a_hi + 8 * j, ptx::umma_desc(d_blo + j * b_step, hi), idesc, 1u);
  ptx::umma_bf16(acc, ptx::umma_desc(d_one, hi), ptx::umma_desc(d_bnrm, hi), idesc, 1u);  // 1 * (-|c|^2 / 2)
  ptx::umma_commit(bar_done);
}

// constant A block that multiplies the norm pieces: row -> [1, 1, 1, 0, 0, 0, 0, 0 | 0 x 8]; called by 128 threads (i = row)
__device__ __forceinline__ void write_ones_block(uint8_t* s_ones, int i) {
  *reinterpret_cast<uint4*>(s_ones + i * 16) = make_uint4(0x3F803F80u, 0x00003F80u, 0u, 0u);
  *reinterpret_cast<uint4*>(s_ones + kTileRows * 16 + i * 16) = make_uint4(0u, 0u, 0u, 0u);
  ptx::fence_proxy_async_smem();
}

// bf16 hi | lo split of a pair of values: hi = RN_bf16(x), lo = RN_bf16(x - hi), two values per 32-bit word
__device__ __forceinline__ void split_pair(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat162 hh = __floats2bfloat162_rn(x0, x1);
  const uint32_t hw = *reinterpret_cast<const uint32_t*>(&hh);
  const float h0 = __uint_as_float(hw << 16), h1 = __uint_as_float(hw & 0xFFFF0000u);
  const __nv_bfloat162 ll = __floats2bfloat162_rn(x0 - h0, x1 - h1);
  hi = hw;
  lo = *reinterpret_cast<const uint32_t*>(&ll);
}

}  // namespace rows
}  // namespace hv
