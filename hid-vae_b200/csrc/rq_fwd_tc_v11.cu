// tcgen05 kernel of the fused L-level residual quantiser for sm_100a -- generation 11 ("row owners").
// D = 32, K <= 256 (one operand image per level), everything resident in shared memory.
//
// What the measurements of generations 7-10 showed (profiles/README.md): a (128-row tile, level) costs ~900 tensor
// cycles and ~1050 cycles of accumulator read-out, but took 2700-3100 cycles because a level of a tile is a chain of
// hand-overs -- A operand through shared memory + proxy fence, row group -> MMA -> scan group -> row group through
// mbarriers, the code gather through L2 -- with only 3-4 tiles in flight.  This generation removes the hand-overs
// instead of speeding them up:
//
//   OWNERSHIP  three warpgroups, each owns one row tile for its L levels; thread t of the warpgroup owns row t (= TMEM
//              lane t) in registers from the x load to the last id.  There is no row group / scan group split, no
//              candidate table, no second layout.
//   A IN TMEM  the residual's bf16 hi / lo halves are written by their owner with tcgen05.st into 32 TMEM columns of
//              the warpgroup (lane = row, two bf16 per column) and the MMAs read A from tensor memory
//              (tcgen05.mma [d], [a], b-desc): no shared-memory A buffers, no generic->async proxy fence.
//   GATHER     the fp32 codebooks sit in shared memory beside the bf16 operand images (216 KB for L = 3: possible
//              because A no longer lives there), rows XOR-swizzled by 16-byte chunk, so the chosen code row is eight
//              LDS.128 instead of a round trip to L2.
//   ISSUER     a level is two units of 128 codes (3*D/16 tcgen05.mma from TMEM + 1 from the constant ones block, one
//              commit each).  tcgen05.mma blocks its thread while the MMA queue is full, so a thirteenth warp does
//              nothing else: warpgroups queue "level staged" requests, the issuer serves them first come first served,
//              giving every unit the next of three 128-column accumulators (unit number % 3) as soon as its previous
//              user has been scanned.  The scan of unit 0 overlaps the MMAs of unit 1 and of other tiles, and no
//              scanning warp ever waits inside an issue loop (which, with the owners issuing for themselves, held
//              accumulators hostage: measured 9000 cycles per level).
//   WAITS      every wait is a hardware-parked mbarrier wait (a completion barrier per (warpgroup, unit), a "scanned"
//              barrier per accumulator, a doorbell for the request queue).  The first builds polled shared-memory
//              counters: the poll loops were 15 % of all issued instructions and took issue slots from the scanning
//              warps (4 Mi-row encode 0.725 -> 0.61 ms when they went).
//   SCAN       by the row's owner: 2-D fold (maxima per column class and per chunk, 3-input maxima) over pipelined
//              8-column loads (rq_rows.cuh), exact first-index path when a row has more than one maximiser; the id
//              stays in a register.
//   score[row, k] = r.c_k - |c_k|^2 / 2 with the bf16 3-way split exactly as in the other generations
//   (modules/quantize.py:108-122); only ids (and emb_out / loss in training) leave the SM.
#include <stdlib.h>

#include "rq_rows.cuh"

namespace hv {
namespace {

using namespace rows;

constexpr int kWGs = 3;  // row tiles in flight per CTA (owner warpgroups); measured: three owners at 128 registers beat four at 112 (spills)
constexpr int kIssuerWarp = kWGs * 4;   // the warp after the owners issues every tcgen05.mma
constexpr int kThreads = (kWGs + 1) * 128;  // (register allocation is per warpgroup: the issuer's three siblings idle)
constexpr int kLaunchRegs = (65536 / kThreads) / 8 * 8;
constexpr int kOwnerRegs = 128, kIssuerRegs = 128;  // three owners: 128 for everybody
static_assert(kWGs * 128 * kOwnerRegs + 128 * kIssuerRegs <= kThreads * kLaunchRegs, "register hand-over must stay inside the launch allocation");
constexpr int kTmemCols = 512;  // 3 x 128 accumulator columns + 4 x 32 A columns
#ifdef HV_TC_INSTRUMENT
constexpr bool kInstr = true;
#else
constexpr bool kInstr = false;
#endif

struct V11Params {
  const uint8_t* images;  // [L] packed bf16 images
  const uint8_t* cb32;    // [L] swizzled fp32 codebooks
  int debug;
};

// OUT = false: ids only (bulk assignment / eval encode without outputs) -- the value / loss / output code is compiled out
template <bool ROT, bool OUT>
__global__ void __launch_bounds__(kThreads, 1) rq_fwd_tc_v11_kernel(RqFwdArgs a, V11Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  // [ones | barriers + counters | operand images (L) | fp32 codebooks (L)]
  uint8_t* s_ones = smem;
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + kOnesBytes);
  uint8_t* s_img = smem + kOnesBytes + kBarBytes;
  uint8_t* s_cb = s_img + a.n_levels * kImageBytes;

  uint64_t* bar_b_full = s_bar;                      // [kMaxLevels]  TMA -> everybody (images + codebooks of a level)
  // Every wait of an owner is a hardware-parked mbarrier wait (polled progress counters were 15 % of the issued
  // instructions).  A (warpgroup, unit) barrier completes once per level of the warpgroup, in order, so its parity is
  // exact; an accumulator's "scanned" barrier has one waiter (the issuer) that never skips a phase.
  uint64_t* bar_done = bar_b_full + kMaxLevels;      // [kWGs][2]  unit of the warpgroup's level committed (issuer + MMA completion)
  uint64_t* bar_free = bar_done + 2 * kWGs;          // [kAccs]  the four warps of the owner have scanned the accumulator
  uint64_t* bar_req = bar_free + kAccs;              // doorbell: one arrival (= one phase) per queued request
  uint32_t* s_qtail = reinterpret_cast<uint32_t*>(bar_req + 1);  // requests pushed so far
  uint32_t* s_q = s_qtail + 1;                       // [kQueue] (sequence + 1) << 8 | level << 4 | warpgroup
  uint32_t* s_tk = s_q + kQueue;                     // [kWGs][2]  accumulator of the warpgroup's unit (published by the issuer's arrive)
  uint32_t* s_tmem = s_tk + 2 * kWGs;
  uint32_t* s_ts = s_tmem + 1;                       // [192] timestamps of block 0, warpgroup 0 (instrumented builds)

  const int warp = ptx::warp_index();
  const int lane = threadIdx.x & 31;
  const int wg = warp >> 2;
  const int q = warp & 3;        // TMEM lane quarter of this warp
  const int t = q * 32 + lane;   // the thread's row of the tile == its TMEM lane
  const int n_levels = a.n_levels;
  int ts_n = 0;
  const bool ts_on = kInstr && (p.debug & 64) && blockIdx.x == 0 && threadIdx.x == 0;
  auto stamp = [&](int code) {
    if (ts_on && ts_n < 90) {
      s_ts[2 * ts_n] = code;
      s_ts[2 * ts_n + 1] = static_cast<uint32_t>(clock64());
      ++ts_n;
    }
  };

  if (threadIdx.x == 0) {
    for (int i = 0; i < kMaxLevels; ++i) ptx::mbar_init(ptx::smem_u32(&bar_b_full[i]), 1);
    for (int i = 0; i < 2 * kWGs; ++i) ptx::mbar_init(ptx::smem_u32(&bar_done[i]), 2);
    for (int i = 0; i < kAccs; ++i) ptx::mbar_init(ptx::smem_u32(&bar_free[i]), 4);
    ptx::mbar_init(ptx::smem_u32(bar_req), 1);
    for (int i = 0; i < kQueue; ++i) s_q[i] = 0;
    *s_qtail = 0;
    ptx::fence_mbar_init();
    for (int l = 0; l < n_levels; ++l) {  // resident for the whole kernel
      const uint32_t bar = ptx::smem_u32(&bar_b_full[l]);
      ptx::mbar_arrive_expect_tx(bar, kImageBytes + kCbBytes);
      ptx::bulk_g2s(ptx::smem_u32(s_img + l * kImageBytes), p.images + static_cast<size_t>(l) * kImageBytes, kImageBytes, bar);
      ptx::bulk_g2s(ptx::smem_u32(s_cb + l * kCbBytes), p.cb32 + static_cast<size_t>(l) * kCbBytes, kCbBytes, bar);
    }
  }
  if (warp == 1) {
    ptx::tmem_alloc(ptx::smem_u32(s_tmem), kTmemCols);
    ptx::tmem_relinquish();
  }
  if (threadIdx.x >= 128 && threadIdx.x < 128 + kTileRows) {
    write_ones_block(s_ones, threadIdx.x - 128);
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *s_tmem;
  const uint32_t lane_bits = static_cast<uint32_t>(q * 32) << 16;
  const uint32_t a_tmem = tmem_base + kAccs * kUnitCols + wg * D;  // the warpgroup's A operand: hi (16 columns) | lo (16)
  const uint32_t ones = ptx::smem_u32(s_ones);
  const uint32_t bar_wg = 1 + wg;

  const int64_t n_row_tiles = (a.n + kTileRows - 1) / kTileRows;
  const int my_tiles = static_cast<int>((n_row_tiles - 1 - blockIdx.x) / gridDim.x + 1);  // grid <= n_row_tiles
  auto tile_row0 = [&](int i) -> int64_t { return (static_cast<int64_t>(blockIdx.x) + static_cast<int64_t>(i) * gridDim.x) * kTileRows; };
  const bool want_loss = OUT && (a.loss != nullptr || a.level_loss != nullptr);
  // the last level's code row is only needed when something other than ids is asked for
  const bool tail_last = OUT && (a.emb_out != nullptr || want_loss || a.final_residual != nullptr);

  if (warp >= kIssuerWarp) {
    // =========================================== MMA issuer ===================================================
    if constexpr (kIssuerRegs < kLaunchRegs) ptx::setmaxnreg_dec<kIssuerRegs>();
    if (warp == kIssuerWarp && ptx::elect_one()) {
      // One request per staged level.  Unit 0 of a request goes out at once; its unit 1 follows -- after unit 0 of the
      // NEXT request if one is already queued, so that a waiting tile starts half a level earlier and unit 1's
      // accumulator is parked full for a shorter time (it cannot be scanned before unit 0 anyway).
      const uint32_t n_req = static_cast<uint32_t>(my_tiles) * static_cast<uint32_t>(n_levels);
      uint32_t unit = 0;  // units issued so far: accumulator = unit % 3, its use number = unit / 3
      auto issue = [&](uint32_t rwg, uint32_t l, uint32_t u) {
        const uint32_t acc = unit % kAccs, use = unit / kAccs;
        if (use > 0) ptx::mbar_wait(ptx::smem_u32(&bar_free[acc]), (use - 1u) & 1u);  // every earlier use of the accumulator is scanned
        ptx::tc_fence_after_sync();
        s_tk[2 * rwg + u] = acc;
        const uint32_t bar = ptx::smem_u32(&bar_done[2 * rwg + u]);
        issue_unit(tmem_base + acc * kUnitCols, tmem_base + kAccs * kUnitCols + rwg * D, ones, ptx::smem_u32(s_img + l * kImageBytes),
                   u * kUnitCols, bar);
        ptx::mbar_arrive(bar);  // (release: publishes s_tk; the phase completes with the MMAs' own arrival)
        ++unit;
      };
      bool have_pending = false;
      uint32_t pend_wg = 0, pend_l = 0;
      for (uint32_t s = 0; s < n_req; ++s) {
        const uint32_t q_addr = ptx::smem_u32(&s_q[s % kQueue]);
        uint32_t qv = ptx::counter_ld_acquire(q_addr);
        if ((qv >> 8) != s + 1u) {
          if (have_pending) {  // nothing queued: the deferred unit 1 goes now
            issue(pend_wg, pend_l, 1u);
            have_pending = false;
          }
          // Park on the doorbell instead of polling the queue slot (measured equal to polling, 0.573 vs 0.580 ms: one polling
          // warp does not matter; kept so that no warp of the kernel spins).  Request s rings phase s; a wake-up while an
          // earlier request's arrival is still in flight is harmless: the slot is checked again.
          const long long t_start = clock64();
          while (((qv = ptx::counter_ld_acquire(q_addr)) >> 8) != s + 1u) {
            ptx::mbar_try_wait_parked(ptx::smem_u32(bar_req), s & 1u, 100000u);
            if (clock64() - t_start > 4000000000LL) {
              printf("hidvae_b200: issuer request wait timed out (block %d request %u)\n", blockIdx.x, s);
              __trap();
            }
          }
        }
        const uint32_t rwg = qv & 0xFu, l = (qv >> 4) & 0xFu;
        if (s < static_cast<uint32_t>(kWGs * n_levels)) ptx::mbar_wait(ptx::smem_u32(&bar_b_full[l]), 0u);  // images are loaded once
        issue(rwg, l, 0u);
        if (have_pending) issue(pend_wg, pend_l, 1u);
        have_pending = true, pend_wg = rwg, pend_l = l;
      }
      if (have_pending) issue(pend_wg, pend_l, 1u);
    }
    __syncwarp();
  } else {
  if constexpr (kOwnerRegs > kLaunchRegs) ptx::setmaxnreg_inc<kOwnerRegs>();
  float r[D];
  auto load_x = [&](int i) {  // the thread's row of this CTA's i-th tile (rows beyond n read as zero)
    const int64_t grow = tile_row0(i) + t;
    if (grow < a.n) {
      load_row<D>(r, a.x + grow * D);
    } else {
#pragma unroll
      for (int d = 0; d < D; ++d) r[d] = 0.f;
    }
  };

  bool have_x = false;
  uint32_t lvl = 0;  // levels done by this warpgroup (parity of its unit barriers)
  for (int i = wg; i < my_tiles; i += kWGs) {
    const int64_t grow = tile_row0(i) + t;
    const bool valid = grow < a.n;
    if (q == 0 && lane == 0 && i + kWGs < my_tiles) {  // pull the warpgroup's next tile into L2
      const int64_t next0 = tile_row0(i + kWGs);
      const int64_t rows = a.n - next0 < kTileRows ? a.n - next0 : kTileRows;
      ptx::bulk_prefetch_l2(a.x + next0 * D, static_cast<uint32_t>(rows * D * 4));
    }
    stamp(1);
    if (!have_x) load_x(i);
    have_x = false;
    float loss = 0.f;

    for (int l = 0; l < n_levels; ++l, ++lvl) {
      const bool last = l + 1 == n_levels;
      const bool tail = !last || tail_last;
      stamp(2);
      if (OUT && a.residuals != nullptr && valid) store_row<D>(a.residuals + (static_cast<int64_t>(l) * a.n + grow) * D, r);
      // ---- the residual's bf16 hi | lo halves -> the warpgroup's A columns in tensor memory ----
      {
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) split_pair(r[2 * j], r[2 * j + 1], hi[j], lo[j]);
        ptx::tmem_st_32x16(a_tmem + lane_bits, hi);
        ptx::tmem_st_32x16(a_tmem + lane_bits + 16, lo);
        ptx::tmem_wait_st();
      }
      ptx::tc_fence_before_sync();
      ptx::named_bar_sync(bar_wg, 128);
      if (q == 0 && lane == 0) {  // the level is staged: queue it for the issuer
        const uint32_t sq = atomicAdd(s_qtail, 1u);
        asm volatile("st.release.cta.shared::cta.u32 [%0], %1;" ::"r"(ptx::smem_u32(&s_q[sq % kQueue])),
                     "r"(((sq + 1u) << 8) | (static_cast<uint32_t>(l) << 4) | static_cast<uint32_t>(wg))
                     : "memory");
        ptx::mbar_arrive(ptx::smem_u32(bar_req));
      }
      stamp(3);
      stamp(4);
      if (last && !tail && i + kWGs < my_tiles) {  // encode: the row is dead now -- the next tile's travels behind the MMAs
        load_x(i + kWGs);
        have_x = true;
      }
      if (i < kWGs) ptx::mbar_wait(ptx::smem_u32(&bar_b_full[l]), 0u);  // (the gather reads the level's codebook)

      // ---- the owner scans its row in both units ----
      float best = -INFINITY;
      int col = 0;
#pragma unroll
      for (uint32_t u = 0; u < 2; ++u) {
        ptx::mbar_wait(ptx::smem_u32(&bar_done[2 * wg + u]), lvl & 1u);
        const uint32_t acc = *reinterpret_cast<volatile uint32_t*>(&s_tk[2 * wg + u]);
        ptx::tc_fence_after_sync();
        stamp(u == 0 ? 5 : 9);
        float m;
        int c;
        scan_unit_x8_pairs(tmem_base + acc * kUnitCols + lane_bits, m, c);
        if (u == 0) stamp(8);
        ptx::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(&bar_free[acc]));
        if (m > best) {  // strict: the lower unit keeps exact ties
          best = m;
          col = c + static_cast<int>(u) * kUnitCols;
        }
      }
      stamp(6);
      const uint32_t k_sel = static_cast<uint32_t>(col) < static_cast<uint32_t>(a.k) ? static_cast<uint32_t>(col)
                                                                                    : static_cast<uint32_t>(a.k - 1);
      if (valid) a.ids[grow * a.ids_row_stride + l * a.ids_level_stride] = k_sel;
      if (tail) {
        // ---- the chosen fp32 code row from shared memory (chunk c of code k sits at chunk c ^ (k & 7)) ----
        float e[D];
        // (rows are 128-byte aligned: (c ^ sw) << 4 == (c << 4) ^ (sw << 4), one LOP3 with an immediate per chunk)
        const uint32_t row_sw = (ptx::smem_u32(s_cb + l * kCbBytes) + k_sel * (D * 4)) | ((k_sel & 7u) << 4);
#pragma unroll
        for (uint32_t c = 0; c < 8; ++c) {
          const float4 v = ptx::lds128(row_sw ^ (c << 4));
          e[4 * c] = v.x, e[4 * c + 1] = v.y, e[4 * c + 2] = v.z, e[4 * c + 3] = v.w;
        }
        if (OUT && tail_last) {  // something besides ids is wanted: value / loss / outputs (modules/quantize.py:131-148)
          // emb_out through the warpgroup's A columns (idle between the level's last MMA and the next staging): written in
          // the row-owner layout (32x32b), read back in the accumulator-fragment layout (16x256b), so that a quad of lanes
          // stores one full 32-byte sector of a row; thread-per-row 16-byte stores touch 32 lines per instruction
          // (measured 1.25 -> 1.16 ms on the 4 Mi-row training forward).  Warp-collective: every lane takes part.
          stamp(10);
          float o[D];
          const float ll = rq_level_tail_o<D, ROT>(r, e, a.beta, o);
          stamp(11);
          if (a.emb_out != nullptr) {
            uint32_t ob[32];
#pragma unroll
            for (int d = 0; d < D; ++d) ob[d] = __float_as_uint(o[d]);
            ptx::tmem_st_32x32(a_tmem + lane_bits, ob);
            ptx::tmem_wait_st();
            __syncwarp();
            stamp(12);
            float* out_l = a.emb_out + (static_cast<int64_t>(l) * a.n + tile_row0(i) + q * 32) * D + 2 * (lane & 3);
            const int64_t rows_left = a.n - (tile_row0(i) + q * 32);
#pragma unroll
            for (int half = 0; half < 2; ++half) {
              uint32_t v[16];
              ptx::tmem_ld_16x256_x4(a_tmem + lane_bits + (static_cast<uint32_t>(16 * half) << 16), v);
              ptx::tmem_wait_ld16(v);
              const int r0 = 16 * half + (lane >> 2), r1 = r0 + 8;
#pragma unroll
              for (int rep = 0; rep < 4; ++rep) {
                if (r0 < rows_left) *reinterpret_cast<float2*>(out_l + r0 * D + 8 * rep) = make_float2(__uint_as_float(v[4 * rep]), __uint_as_float(v[4 * rep + 1]));
                if (r1 < rows_left) *reinterpret_cast<float2*>(out_l + r1 * D + 8 * rep) = make_float2(__uint_as_float(v[4 * rep + 2]), __uint_as_float(v[4 * rep + 3]));
              }
            }
            __syncwarp();  // every lane's read-back is done before the next level's A operand overwrites the columns
          }
          loss += ll;
          if (valid) {
            if (a.level_loss != nullptr) a.level_loss[static_cast<int64_t>(l) * a.n + grow] = ll;
            if (last && a.loss != nullptr) a.loss[grow] = loss;
            if (last && a.final_residual != nullptr) store_row<D>(a.final_residual + grow * D, r);
          }
        } else {
#pragma unroll
          for (int d = 0; d < D; ++d) r[d] = r[d] - e[d];
        }
      }
      stamp(7);
    }
  }

  if (ts_on) s_ts[190] = ts_n;
  }  // row owners
  ptx::tc_fence_before_sync();
  __syncthreads();
#ifdef HV_TC_INSTRUMENT
  if ((p.debug & 64) && blockIdx.x == 0 && threadIdx.x == 0) {
    const int n = s_ts[190];
    for (int i = 0; i < n; ++i) printf("TS 0 %u %u\n", s_ts[2 * i], s_ts[2 * i + 1]);
  }
#endif
  if (warp == 1) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

int smem_bytes(int n_levels) { return kOnesBytes + kBarBytes + n_levels * (kImageBytes + kCbBytes); }

}  // namespace

bool rq_fwd_tc_v11_supported(int d, int k, int n_levels) {
  return d == D && k >= 1 && k <= kNTile && n_levels >= 1 && n_levels <= kMaxLevels && smem_bytes(n_levels) <= kSmemLimit;
}

// bytes of the swizzled fp32 codebook copy that follows the operand images in the workspace (0: shape not served)
size_t rq_fwd_tc_v11_extra_bytes(int d, int k, int n_levels) {
  return rq_fwd_tc_v11_supported(d, k, n_levels) ? static_cast<size_t>(n_levels) * kCbBytes : 0;
}

// `images` = operand images, `cb32` = swizzled fp32 copy of the codebooks (chunk c of code k at chunk c ^ (k & 7)), both
// written by launch_rq_pack
int launch_rq_fwd_tc_v11(const RqFwdArgs& a, bool rot, const void* images, const void* cb32, cudaStream_t stream) {
  if (!rq_fwd_tc_v11_supported(D, a.k, a.n_levels)) {
    set_error("hv_rq_forward: no generation-11 tcgen05 instantiation for K=%d L=%d", a.k, a.n_levels);
    return HV_ERR_UNSUPPORTED;
  }
  if (a.n == 0) return HV_OK;
  DeviceProps props;
  if (int st = device_props(&props)) return st;
  const int64_t n_row_tiles = (a.n + kTileRows - 1) / kTileRows;
  const unsigned grid = static_cast<unsigned>(n_row_tiles < props.sm_count ? n_row_tiles : props.sm_count);
#ifdef HV_TC_INSTRUMENT
  static const int debug = [] {  // instrumented builds only: bit 64 prints block 0's timeline
    const char* e = getenv("HIDVAE_TC_DEBUG");
    return e != nullptr ? atoi(e) : 0;
  }();
#else
  constexpr int debug = 0;
#endif
  V11Params p{static_cast<const uint8_t*>(images), static_cast<const uint8_t*>(cb32), debug};
  const int smem = smem_bytes(a.n_levels);
  auto go = [&](auto kernel) -> int {
    if (int st = prepare_kernel(kernel, kOwnerRegs > kLaunchRegs ? kLaunchRegs : 0, smem)) return st;  // (the check guards a setmaxnreg.inc)
    kernel<<<grid, kThreads, smem, stream>>>(a, p);
    HV_CUDA_CHECK(cudaGetLastError());
    return HV_OK;
  };
  const bool out = a.emb_out != nullptr || a.loss != nullptr || a.level_loss != nullptr || a.final_residual != nullptr || a.residuals != nullptr;
  if (!out) return go(rq_fwd_tc_v11_kernel<false, false>);
  return rot ? go(rq_fwd_tc_v11_kernel<true, true>) : go(rq_fwd_tc_v11_kernel<false, true>);
}

}  // namespace hv
