// Shared host/device helpers for the hidvae_b200 kernels (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/hidvae_b200.h"

namespace hv {

// thread-local error text behind hv_last_error()
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define HV_CUDA_CHECK(expr)                                       \
  do {                                                            \
    cudaError_t _e = (expr);                                      \
    if (_e != cudaSuccess) return ::hv::cuda_fail(_e, #expr);     \
  } while (0)

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

struct DeviceProps {
  int sm_count = 0;
  int cc_major = 0;
  int cc_minor = 0;
  int max_smem_optin = 0;
};
// cached per device; returns non-zero status on failure
int device_props(DeviceProps* out);

// One-time (per kernel and device) launch preparation: checks that the kernel was built with at least `min_regs`
// registers per thread (0 = no check; a setmaxnreg.inc hand-over would otherwise wait forever) and raises its dynamic
// shared-memory limit to at least `smem_bytes`.  Later calls with the same or a smaller size cost one table lookup.
int prepare_kernel_impl(const void* kernel, int min_regs, int smem_bytes);
template <typename K>
int prepare_kernel(K kernel, int min_regs, int smem_bytes) {
  return prepare_kernel_impl(reinterpret_cast<const void*>(kernel), min_regs, smem_bytes);
}

// Arguments of the fused forward, shared by the SIMT and tcgen05 variants.
struct RqFwdArgs {
  const float* x;
  const float* codebooks;  // [L, K, D] fp32, effective
  int64_t n;
  int n_levels;
  int k;
  float beta;
  int64_t* ids;
  int64_t ids_row_stride;
  int64_t ids_level_stride;
  float* emb_out;         // [L, N, D] or null
  float* residuals;       // [L, N, D] or null
  float* loss;            // [N] or null
  float* level_loss;      // [L, N] or null
  float* final_residual;  // [N, D] or null
};

int launch_rq_fwd_simt(const RqFwdArgs& a, int d, bool rot, bool diff_form, cudaStream_t stream);
// returns HV_ERR_UNSUPPORTED when the shape has no tcgen05 instantiation
int launch_rq_fwd_tc(const RqFwdArgs& a, int d, bool rot, void* workspace, size_t workspace_bytes, bool prepacked,
                     cudaStream_t stream);
int launch_rq_pack(const float* codebooks, int n_levels, int k, int d, void* workspace, size_t workspace_bytes,
                   cudaStream_t stream);
// streamed operand images (generation 4): D = 16 / 32 / 64, any K; `packed` = image written by launch_rq_pack
int launch_rq_fwd_tc_v4(const RqFwdArgs& a, int d, bool rot, void* packed, cudaStream_t stream);
bool rq_fwd_tc_v4_supported(int d, int k, int n_levels);
// generation 11 (row owners): D = 32, K <= 256, A operand in tensor memory, fp32 codebooks in shared memory
int launch_rq_fwd_tc_v11(const RqFwdArgs& a, bool rot, const void* images, const void* cb32, cudaStream_t stream);
bool rq_fwd_tc_v11_supported(int d, int k, int n_levels);
size_t rq_fwd_tc_v11_extra_bytes(int d, int k, int n_levels);
bool rq_fwd_tc_supported(int d, int k, int n_levels);
size_t rq_fwd_tc_workspace_bytes(int d, int k, int n_levels);
size_t rq_bwd_workspace_bytes(int64_t n, int d, int k, int n_levels);

// Collision digit of semantic-ID tuples (semid_dedup.cu); arguments are those of hv_semid_dedup, validated by it.
struct SemidDedupArgs {
  const int64_t* ids;
  int64_t rows, width, row_stride, col_stride;
  int bits;
  const int64_t* prior_keys;
  const int64_t* prior_counts;
  int64_t n_prior;
  int64_t* digits;
  int64_t digit_stride;
  int64_t* run_keys;
  int64_t* run_counts;
  int64_t* stats;
};
constexpr int64_t kSemidDedupMaxRows = 1ll << 31;  // row indices travel as uint32 with a flag bit; cub takes an int count
size_t semid_dedup_workspace_bytes(int64_t rows);
int launch_semid_dedup(const SemidDedupArgs& a, void* workspace, size_t workspace_bytes, cudaStream_t stream);

// 1 / (sqrt(v) + eps) and 1 / max(sqrt(v), floor) on the special-function unit: sqrt.approx (max relative error 2^-23) and
// rcp.approx followed by one Newton step (the reciprocal is then correctly rounded up to the last bit of its argument).
// 6 instructions instead of the ~16 + slow-path branches of an IEEE sqrt and division; three of these per row and level.
// The .ftz forms drop the denormal pre-/post-scaling (4 more instructions per call) and give the same results here: the
// reciprocals' arguments are >= 1e-8, and a denormal sum of squares (|v| < 1e-19) vanishes against the 1e-8 / 1e-6 it is
// added to or clamped at.
__device__ __forceinline__ float fast_rcp(float d) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d));
  return fmaf(fmaf(-d, r, 1.0f), r, r);
}
__device__ __forceinline__ float fast_inv_norm_eps(float v, float eps) {
  float s;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(s) : "f"(v));
  return fast_rcp(s + eps);
}
__device__ __forceinline__ float fast_inv_norm_floor(float v, float floor) {
  float s;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(s) : "f"(v));
  return fast_rcp(fmaxf(s, floor));
}

// Scalars of one rotation-trick level (modules/quantize.py:34-45) from the three row sums rr = r.r, ee = e.e, re = r.e.
// o = r - 2 (r.w) w + 2 (r.u) q with u = r ir, q = e ie, w = (u + q) is collapses to  o = cr r + ce e:
//   r.u = rr ir,  r.q = re ie,  |u + q|^2 = rr ir^2 + ee ie^2 + 2 re ir ie,
//   a2 = 2 (r.u + r.q) is^2,  cr = 1 - a2 ir,  ce = (2 r.u - a2) ie.
// Two passes over the row instead of five.  |u + q|^2 from the row sums already at hand has an absolute error of ~4e-7 on a
// value in [0, 4], i.e. 1e-7 relative on 1/|s| away from r = -e.  The forward and the backward's recomputation of the
// chain both call this, so they agree to the bit.
struct RotCoeffs {
  float ir, ie, is, cr, ce;
};
__device__ __forceinline__ RotCoeffs rot_coeffs(float rr, float ee, float re) {
  RotCoeffs c;
  c.ir = fast_inv_norm_eps(rr, 1e-8f);  // u = r / (|r| + 1e-8)
  c.ie = fast_inv_norm_eps(ee, 1e-8f);  // q = e / (|e| + 1e-8)
  const float ru = rr * c.ir, rq = re * c.ie;
  const float ss = fmaf(2.0f * rq, c.ir, fmaf(ru, c.ir, ee * c.ie * c.ie));
  c.is = fast_inv_norm_floor(ss, 1e-6f);  // w = (u + q) / max(|u + q|, 1e-6)
  const float a2 = 2.0f * (ru + rq) * c.is * c.is;
  c.cr = 1.0f - a2 * c.ir;
  c.ce = (2.0f * ru - a2) * c.ie;
  return c;
}

// ---------------------------------------------------------------------------------------------------------
// Per-row "tail" of one quantiser level: everything after the argmin.  One thread owns one row in registers.
//   r      in : residual entering the level (r_l)            out: r_{l+1} = r_l - o_l
//   e         : the chosen code row C_l[id] (fp32)
//   returns the level loss a + beta*a with a = |r - e|^2      (modules/loss.py:41-44)
//   o (emb_out) is written to `o_out` when non-null.
// ROT implements modules/quantize.py:34-45,134-140:  o = r - 2 (r.w) w + 2 (r.u) q  (collapsed to two row passes, rot_coeffs)
// ---------------------------------------------------------------------------------------------------------
template <int D, bool ROT>
__device__ __forceinline__ float rq_level_tail_o(float (&r)[D], const float (&e)[D], float beta, float (&o)[D]) {
  float a = 0.f;
#pragma unroll
  for (int i = 0; i < D; ++i) {
    const float df = r[i] - e[i];
    a = fmaf(df, df, a);
  }
  const float level_loss = a + beta * a;
  if constexpr (!ROT) {
#pragma unroll
    for (int i = 0; i < D; ++i) o[i] = e[i];
  } else {
    float rr = 0.f, ee = 0.f;
#pragma unroll
    for (int i = 0; i < D; ++i) {
      rr = fmaf(r[i], r[i], rr);
      ee = fmaf(e[i], e[i], ee);
    }
    const RotCoeffs c = rot_coeffs(rr, ee, 0.5f * ((rr + ee) - a));  // r.e from the loss sum: |r - e|^2 = r.r + e.e - 2 r.e
#pragma unroll
    for (int i = 0; i < D; ++i) o[i] = fmaf(c.cr, r[i], c.ce * e[i]);
  }
#pragma unroll
  for (int i = 0; i < D; ++i) r[i] = r[i] - o[i];
  return level_loss;
}

// same, with emb_out written straight from the owning thread (one 128-bit store per 4 floats) when o_out != null
template <int D, bool ROT>
__device__ __forceinline__ float rq_level_tail(float (&r)[D], const float (&e)[D], float beta, float* o_out) {
  float o[D];
  const float level_loss = rq_level_tail_o<D, ROT>(r, e, beta, o);
  if (o_out != nullptr) {
#pragma unroll
    for (int i = 0; i < D; i += 4)
      *reinterpret_cast<float4*>(o_out + i) = make_float4(o[i], o[i + 1], o[i + 2], o[i + 3]);
  }
  return level_loss;
}

template <int D>
__device__ __forceinline__ void load_row(float (&dst)[D], const float* __restrict__ src) {
#pragma unroll
  for (int i = 0; i < D; i += 4) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(src + i));
    dst[i] = v.x, dst[i + 1] = v.y, dst[i + 2] = v.z, dst[i + 3] = v.w;
  }
}

template <int D>
__device__ __forceinline__ void store_row(float* __restrict__ dst, const float (&src)[D]) {
#pragma unroll
  for (int i = 0; i < D; i += 4)
    *reinterpret_cast<float4*>(dst + i) = make_float4(src[i], src[i + 1], src[i + 2], src[i + 3]);
}

}  // namespace hv
