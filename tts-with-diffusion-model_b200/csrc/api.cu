// Error plumbing, device queries and TMA tensor-map encoding shared by all entry points.
#include <stdarg.h>
#include <stdio.h>
#include <string.h>


#include <cstdlib>

#include "common.cuh"

namespace vb200 {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", static_cast<int>(e), cudaGetErrorString(e), what);
  return VB200_ERR_CUDA;
}

int num_sms() {
  static thread_local int cached_dev = -1, cached_sms = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev != cached_dev) {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
      sms = 148;
    cached_dev = dev;
    cached_sms = sms;
  }
  return cached_sms;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess || !p) {
    return nullptr;
  }
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

int make_tmap_2d(CUtensorMap* out, vb200_dtype dtype, const void* gptr, uint64_t inner,
                 uint64_t outer, uint64_t row_stride_bytes, uint32_t box_inner, uint32_t box_outer) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled driver entry point unavailable");
    return VB200_ERR_CUDA;
  }
  if ((reinterpret_cast<uintptr_t>(gptr) & 15) || (row_stride_bytes & 15)) {
    set_error("TMA operand must be 16-byte aligned (ptr=%p, row stride=%llu B)", gptr,
              static_cast<unsigned long long>(row_stride_bytes));
    return VB200_ERR_INVALID;
  }
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {row_stride_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t elem[2] = {1, 1};
  const CUtensorMapDataType dt = dtype == VB200_F32   ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                 : dtype == VB200_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                                      : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  CUresult r = fn(out, dt, 2, const_cast<void*>(gptr), dims, strides,
                  box, elem, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (inner=%llu outer=%llu stride=%llu box=%ux%u)",
              static_cast<int>(r), static_cast<unsigned long long>(inner),
              static_cast<unsigned long long>(outer),
              static_cast<unsigned long long>(row_stride_bytes), box_inner, box_outer);
    return VB200_ERR_CUDA;
  }
  return VB200_OK;
}

// Tensor maps are pure functions of (pointer, dtype, shape, box), so they are memoised — per host THREAD:
// a launch touches no lock and no shared state (the eager / first-batch / denoise_logits path makes up to
// three look-ups per launch; graph replays make none).  Open addressing over a fixed table; a full
// table is simply wiped (sessions reuse a few dozen buffers, so that does not happen in practice).
struct TmapSlot {
  const void* ptr; uint64_t inner, outer, stride; uint32_t box_inner, box_outer; int dtype; bool used;
  CUtensorMap map;
};
constexpr int kTmapSlots = 1024;      // power of two

int cached_tmap(CUtensorMap* out, vb200_dtype dtype, const void* ptr, uint64_t inner,
                uint64_t outer, uint64_t stride_bytes, uint32_t box_inner, uint32_t box_outer) {
  static thread_local TmapSlot* slots = nullptr;
  static thread_local int n_used = 0;
  if (!slots) slots = static_cast<TmapSlot*>(calloc(kTmapSlots, sizeof(TmapSlot)));
  if (!slots) return make_tmap_2d(out, dtype, ptr, inner, outer, stride_bytes, box_inner, box_outer);
  uint64_t h = reinterpret_cast<uintptr_t>(ptr) * 0x9E3779B97F4A7C15ull;
  h ^= (inner * 0xC2B2AE3D27D4EB4Full) ^ (outer * 0x165667B19E3779F9ull) ^ (static_cast<uint64_t>(box_inner) << 40) ^
       (static_cast<uint64_t>(box_outer) << 20) ^ static_cast<uint64_t>(dtype);
  int i = static_cast<int>((h >> 32) & (kTmapSlots - 1));
  for (int probe = 0; probe < kTmapSlots; ++probe, i = (i + 1) & (kTmapSlots - 1)) {
    TmapSlot& s = slots[i];
    if (!s.used) break;
    if (s.ptr == ptr && s.inner == inner && s.outer == outer && s.stride == stride_bytes && s.box_inner == box_inner &&
        s.box_outer == box_outer && s.dtype == static_cast<int>(dtype)) {
      *out = s.map;
      return VB200_OK;
    }
  }
  const int rc = make_tmap_2d(out, dtype, ptr, inner, outer, stride_bytes, box_inner, box_outer);
  if (rc != VB200_OK) return rc;
  if (n_used >= kTmapSlots / 2) {                // keep probes short
    memset(slots, 0, kTmapSlots * sizeof(TmapSlot));
    n_used = 0;
    i = static_cast<int>((h >> 32) & (kTmapSlots - 1));
  }
  while (slots[i].used) i = (i + 1) & (kTmapSlots - 1);
  slots[i] = TmapSlot{ptr, inner, outer, stride_bytes, box_inner, box_outer, static_cast<int>(dtype), true, *out};
  ++n_used;
  return VB200_OK;
}

}  // namespace vb200

namespace vb200 {
thread_local int g_pdl_tag = 0;
int pdl_mask() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("VB200_PDL");
    v = e ? atoi(e) : (2 | 4 | 8 | 16 | 32);      // default: every launch that lands one CTA per SM (see common.cuh)
  }
  return v;
}
bool pdl_enabled() { return (pdl_mask() & 1) != 0; }
}  // namespace vb200

extern "C" const char* vb200_last_error(void) { return vb200::g_err; }
extern "C" int vb200_version(void) { return 100; }
extern "C" int vb200_device_sms(void) {
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return VB200_ERR_CUDA;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
    return VB200_ERR_CUDA;
  return sms;
}

extern "C" int64_t vb200_workspace_bytes(int64_t M, int64_t M_resp, int32_t d, int32_t n_out,
                                         vb200_dtype logits_dtype, int64_t* sizes) {
  using namespace vb200;
  if (M < 0 || M_resp < 0 || M_resp > M || d <= 0 || n_out <= 0 || !sizes) {
    set_error("workspace_bytes: bad sizes M=%lld M_resp=%lld d=%d n_out=%d", static_cast<long long>(M),
              static_cast<long long>(M_resp), d, n_out);
    return VB200_ERR_INVALID;
  }
  const int64_t lsz = logits_dtype == VB200_F32 ? 4 : 2;
  const int64_t raw[7] = {M * d * 4, M * d * 2, M * 3 * d * 2, M * d * 2, M * 4 * d * 2,
                          M_resp * d * 2, M_resp * n_out * lsz};
  int64_t total = 0;
  for (int i = 0; i < 7; ++i) {
    sizes[i] = (raw[i] + 255) & ~static_cast<int64_t>(255);
    total += sizes[i];
  }
  return total;
}

extern "C" int vb200_head_posterior_sample_known(int32_t* x_out, void* logits, vb200_dtype logits_dtype,
                                                 const void* head_in_bf16, vb200_dtype head_in_dtype,
                                                 const void* W_bf16, const float* bias,
                                                 int32_t n_rows, int32_t d, int32_t n_levels, int32_t K,
                                                 const int32_t* x_t, const int32_t* row_utt, const int32_t* t_utt,
                                                 const int32_t* utt, const float* table, int32_t S,
                                                 vb200_transition tr, vb200_noise noise, const float* uniforms,
                                                 uint64_t seed, const int32_t* known, vb200_stream_t stream) {
  if (head_in_dtype != VB200_BF16 && head_in_dtype != VB200_F16) {
    vb200::set_error("head_posterior_sample: head_in must be bf16 or f16");
    return VB200_ERR_INVALID;
  }
  // fused form: the reverse step runs as the GEMM's epilogue and `logits` stays untouched
  if (n_rows > 0 && vb200_head_fused(d, K, noise)) {
    if (!(x_out && head_in_bf16 && W_bf16 && bias && x_t && row_utt && t_utt && utt && table)) {
      vb200::set_error("head_posterior_sample: null pointer");
      return VB200_ERR_INVALID;
    }
    if (reinterpret_cast<uintptr_t>(bias) & 15) {                // the epilogue reads bias as float4
      vb200::set_error("head_posterior_sample: bias must be 16-byte aligned");
      return VB200_ERR_INVALID;
    }
    return vb200::head_sample_fused(x_out, head_in_bf16, W_bf16, bias, x_t, row_utt, t_utt, utt, table, n_rows, d,
                             n_levels, K, S, static_cast<int>(tr), static_cast<int>(noise), seed,
                             head_in_dtype == VB200_F16, known, static_cast<cudaStream_t>(stream));
  }
  const int rc = vb200_gemm_bf16(logits, logits_dtype, head_in_bf16, head_in_dtype, W_bf16, bias, nullptr, n_rows,
                                 n_levels * K, d, VB200_EPI_BIAS, stream);
  if (rc != VB200_OK) return rc;
  return vb200_posterior_sample_from_logits_known(x_out, nullptr, logits, logits_dtype,
                                                  static_cast<int64_t>(n_levels) * K, x_t, row_utt, t_utt, utt,
                                                  table, n_rows, n_levels, K, S, tr, noise, uniforms, seed, known,
                                                  stream);
}

extern "C" int vb200_head_posterior_sample(int32_t* x_out, void* logits, vb200_dtype logits_dtype,
                                           const void* head_in_bf16, vb200_dtype head_in_dtype,
                                           const void* W_bf16, const float* bias,
                                           int32_t n_rows, int32_t d, int32_t n_levels, int32_t K,
                                           const int32_t* x_t, const int32_t* row_utt, const int32_t* t_utt,
                                           const int32_t* utt, const float* table, int32_t S,
                                           vb200_transition tr, vb200_noise noise, const float* uniforms,
                                           uint64_t seed, vb200_stream_t stream) {
  return vb200_head_posterior_sample_known(x_out, logits, logits_dtype, head_in_bf16, head_in_dtype, W_bf16, bias,
                                           n_rows, d, n_levels, K, x_t, row_utt, t_utt, utt, table, S, tr, noise,
                                           uniforms, seed, nullptr, stream);
}

extern "C" int vb200_head_ce_loss(float* loss, const void* head_in_bf16, vb200_dtype head_in_dtype,
                                  const void* W_bf16, const float* bias,
                                  const int32_t* targets, int32_t n_rows, int32_t d, int32_t n_levels, int32_t K,
                                  vb200_stream_t stream) {
  if (n_rows == 0) return VB200_OK;
  if (!(loss && head_in_bf16 && W_bf16 && bias && targets)) {
    vb200::set_error("head_ce_loss: null pointer");
    return VB200_ERR_INVALID;
  }
  if (reinterpret_cast<uintptr_t>(bias) & 15) {                  // the epilogue reads bias as float4
    vb200::set_error("head_ce_loss: bias must be 16-byte aligned");
    return VB200_ERR_INVALID;
  }
  if (n_rows < 0 || n_levels < 1 || d <= 0 || d % 8 != 0 || K < 256 || K % 256 != 0) {
    vb200::set_error("head_ce_loss: needs d %% 8 == 0 and K a multiple of 256 (n_rows=%d d=%d n_levels=%d K=%d)",
                     n_rows, d, n_levels, K);
    return VB200_ERR_UNSUPPORTED;
  }
  if (head_in_dtype != VB200_BF16 && head_in_dtype != VB200_F16) {
    vb200::set_error("head_ce_loss: head_in must be bf16 or f16");
    return VB200_ERR_INVALID;
  }
  return vb200::head_ce_fused(loss, head_in_bf16, W_bf16, bias, targets, n_rows, d, n_levels, K,
                              head_in_dtype == VB200_F16, static_cast<cudaStream_t>(stream));
}
