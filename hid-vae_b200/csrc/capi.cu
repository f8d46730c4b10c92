// C-ABI front door of libhidvae_b200.so: error text, device query, workspace sizing and the dispatcher of
// hv_rq_forward (include/hidvae_b200.h).  No torch types, no allocation, no CPU fallback.
#include <stdarg.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "common.cuh"

namespace hv {

namespace {
thread_local char g_error[512] = "";
std::mutex g_props_mutex;
DeviceProps g_props[64];
bool g_props_known[64] = {};
}  // namespace

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) in %s", static_cast<int>(e), cudaGetErrorString(e), what);
  return HV_ERR_CUDA;
}

int device_props(DeviceProps* out) {
  int dev = -1;
  HV_CUDA_CHECK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) {
    set_error("device ordinal %d out of range", dev);
    return HV_ERR_CUDA;
  }
  std::lock_guard<std::mutex> lock(g_props_mutex);
  if (!g_props_known[dev]) {
    DeviceProps p;
    HV_CUDA_CHECK(cudaDeviceGetAttribute(&p.sm_count, cudaDevAttrMultiProcessorCount, dev));
    HV_CUDA_CHECK(cudaDeviceGetAttribute(&p.cc_major, cudaDevAttrComputeCapabilityMajor, dev));
    HV_CUDA_CHECK(cudaDeviceGetAttribute(&p.cc_minor, cudaDevAttrComputeCapabilityMinor, dev));
    HV_CUDA_CHECK(cudaDeviceGetAttribute(&p.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    g_props[dev] = p;
    g_props_known[dev] = true;
  }
  *out = g_props[dev];
  return HV_OK;
}

int prepare_kernel_impl(const void* kernel, int min_regs, int smem_bytes) {
  struct Entry { const void* kernel; int dev; int smem; };
  static std::mutex mu;
  static std::vector<Entry> done;
  int dev = -1;
  HV_CUDA_CHECK(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  for (Entry& e : done)
    if (e.kernel == kernel && e.dev == dev) {
      if (e.smem >= smem_bytes) return HV_OK;
      HV_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
      e.smem = smem_bytes;
      return HV_OK;
    }
  if (min_regs > 0) {
    cudaFuncAttributes attr;
    HV_CUDA_CHECK(cudaFuncGetAttributes(&attr, kernel));
    if (attr.numRegs < min_regs) {
      set_error("kernel was built with %d registers/thread, its register hand-over needs %d", attr.numRegs, min_regs);
      return HV_ERR_UNSUPPORTED;
    }
  }
  HV_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  done.push_back({kernel, dev, smem_bytes});
  return HV_OK;
}

}  // namespace hv

extern "C" {

int hv_version(void) { return 100; }  // major*10000 + minor*100 + patch

const char* hv_last_error(void) { return hv::g_error; }

int hv_device_info(int* sm_count, int* cc_major, int* cc_minor) {
  hv::DeviceProps p;
  if (int st = hv::device_props(&p)) return st;
  if (sm_count) *sm_count = p.sm_count;
  if (cc_major) *cc_major = p.cc_major;
  if (cc_minor) *cc_minor = p.cc_minor;
  return HV_OK;
}

size_t hv_workspace_bytes(int op, int64_t n, int d, int k, int n_levels) {
  if (op == HV_OP_RQ_FORWARD) return hv::rq_fwd_tc_workspace_bytes(d, k, n_levels);
  if (op == HV_OP_RQ_BACKWARD && n > 0 && d > 0 && k > 0 && n_levels > 0) return hv::rq_bwd_workspace_bytes(n, d, k, n_levels);
  return 0;
}

int hv_rq_pack_codebooks(const float* codebooks, int n_levels, int k, int d, void* workspace, size_t workspace_bytes,
                         void* stream) {
  if (n_levels <= 0 || k <= 0 || d <= 0) {
    hv::set_error("hv_rq_pack_codebooks: bad shape d=%d k=%d L=%d", d, k, n_levels);
    return HV_ERR_BAD_SHAPE;
  }
  if (!codebooks) {
    hv::set_error("hv_rq_pack_codebooks: codebooks is null");
    return HV_ERR_NULL;
  }
  return hv::launch_rq_pack(codebooks, n_levels, k, d, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

int hv_rq_forward(const float* x, int64_t n, int d, const float* codebooks, int n_levels, int k, int mode,
                  int training, float beta, int64_t* ids, int64_t ids_row_stride, int64_t ids_level_stride,
                  float* emb_out, float* residuals, float* loss, float* level_loss, float* final_residual, int algo,
                  void* workspace, size_t workspace_bytes, void* stream) {
  using namespace hv;
  if (n < 0 || d <= 0 || k <= 0 || n_levels <= 0) {
    set_error("hv_rq_forward: bad shape n=%lld d=%d k=%d L=%d", (long long)n, d, k, n_levels);
    return HV_ERR_BAD_SHAPE;
  }
  if (mode == HV_MODE_GUMBEL_SOFTMAX) {
    set_error("hv_rq_forward: GUMBEL_SOFTMAX takes a temperature and a noise source: call hv_gumbel_forward / hv_gumbel_backward (one level per call); this entry point serves STE=2 and ROTATION_TRICK=3");
    return HV_ERR_UNSUPPORTED;
  }
  if (mode != HV_MODE_STE && mode != HV_MODE_ROTATION_TRICK) {
    set_error("hv_rq_forward: unknown forward mode %d", mode);
    return HV_ERR_UNSUPPORTED;
  }
  if (n == 0) return HV_OK;
  if (!x || !codebooks || !ids) {
    set_error("hv_rq_forward: x, codebooks and ids must be non-null");
    return HV_ERR_NULL;
  }
  if (d % 4 != 0) {
    set_error("hv_rq_forward: embed dim %d must be a multiple of 4 (rows are moved as 16-byte vectors)", d);
    return HV_ERR_UNSUPPORTED;
  }
  if (!aligned16(x) || !aligned16(codebooks) || (emb_out && !aligned16(emb_out)) || (residuals && !aligned16(residuals)) ||
      (final_residual && !aligned16(final_residual))) {
    set_error("hv_rq_forward: x, codebooks, emb_out, residuals, final_residual must be 16-byte aligned");
    return HV_ERR_MISALIGNED;
  }
  DeviceProps props;
  if (int st = device_props(&props)) return st;
  if (props.cc_major != 10) {
    set_error("hv_rq_forward: built for sm_100a, current device is sm_%d%d", props.cc_major, props.cc_minor);
    return HV_ERR_UNSUPPORTED;
  }

  RqFwdArgs a{x, codebooks, n, n_levels, k, beta, ids, ids_row_stride, ids_level_stride,
              emb_out, residuals, loss, level_loss, final_residual};
  // eval semantics (modules/quantize.py:146-148): emb_out = e whatever the forward mode
  const bool rot = mode == HV_MODE_ROTATION_TRICK && training != 0;
  cudaStream_t s = static_cast<cudaStream_t>(stream);

  if (algo == HV_ALGO_AUTO) {
    const size_t need = rq_fwd_tc_workspace_bytes(d, k, n_levels);
    algo = (need > 0 && workspace != nullptr && workspace_bytes >= need && aligned16(workspace)) ? HV_ALGO_TCGEN05
                                                                                               : HV_ALGO_SIMT;
  }
  switch (algo) {
    case HV_ALGO_TCGEN05: return launch_rq_fwd_tc(a, d, rot, workspace, workspace_bytes, false, s);
    case HV_ALGO_TCGEN05_PREPACKED: return launch_rq_fwd_tc(a, d, rot, workspace, workspace_bytes, true, s);
    case HV_ALGO_SIMT: return launch_rq_fwd_simt(a, d, rot, false, s);
    case HV_ALGO_SIMT_DIFF: return launch_rq_fwd_simt(a, d, rot, true, s);
    default:
      set_error("hv_rq_forward: unknown algo %d", algo);
      return HV_ERR_UNSUPPORTED;
  }
}

size_t hv_semid_dedup_workspace_bytes(int64_t rows) { return hv::semid_dedup_workspace_bytes(rows); }

int hv_semid_dedup(const int64_t* ids, int64_t rows, int64_t width, int64_t row_stride, int64_t col_stride, int bits,
                   const int64_t* prior_keys, const int64_t* prior_counts, int64_t n_prior, int64_t* digits, int64_t digit_stride,
                   int64_t* run_keys, int64_t* run_counts, int64_t* stats, void* workspace, size_t workspace_bytes, void* stream) {
  using namespace hv;
  if (rows < 0 || width <= 0 || bits <= 0 || n_prior < 0) {
    set_error("hv_semid_dedup: bad shape rows=%lld width=%lld bits=%d n_prior=%lld", (long long)rows, (long long)width, bits,
              (long long)n_prior);
    return HV_ERR_BAD_SHAPE;
  }
  if (width > 63 || bits > 63 || width * bits > 63) {
    set_error("hv_semid_dedup: width * bits = %lld exceeds the 63 bits of an exact key", (long long)width * bits);
    return HV_ERR_UNSUPPORTED;
  }
  if (rows >= kSemidDedupMaxRows) {
    set_error("hv_semid_dedup: %lld rows, at most 2^31 - 1 per call", (long long)rows);
    return HV_ERR_UNSUPPORTED;
  }
  if (!stats || (rows > 0 && (!ids || !digits || !run_keys || !run_counts)) || (n_prior > 0 && (!prior_keys || !prior_counts))) {
    set_error("hv_semid_dedup: ids, digits, run_keys, run_counts, stats (and prior_keys / prior_counts when n_prior > 0) must be non-null");
    return HV_ERR_NULL;
  }
  if (rows > 0 && (workspace == nullptr || workspace_bytes < semid_dedup_workspace_bytes(rows))) {
    set_error("hv_semid_dedup: workspace of %zu bytes, hv_semid_dedup_workspace_bytes(%lld) = %zu needed", workspace ? workspace_bytes : 0,
              (long long)rows, semid_dedup_workspace_bytes(rows));
    return HV_ERR_WORKSPACE;
  }
  SemidDedupArgs a{ids, rows, width, row_stride, col_stride, bits, prior_keys, prior_counts, n_prior, digits, digit_stride,
                   run_keys, run_counts, stats};
  return launch_semid_dedup(a, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
