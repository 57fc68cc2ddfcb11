// C-ABI glue: error state, version, mode dispatch of the convolution entry points.
#include <stdarg.h>
#include <stdlib.h>

#include "common.cuh"

static thread_local char g_err[512] = "";

void mm3d_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

#include <atomic>
static std::atomic<long long> g_launches{0};
void mm3d_count_launches(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
extern "C" long long mm3d_kernel_launches(void) { return g_launches.load(std::memory_order_relaxed); }

bool mm3d_pdl_enabled() {
  static int on = -1;
  if (on < 0) on = getenv("MM3D_NO_PDL") ? 0 : 1;
  return on != 0;
}

extern "C" const char* mm3d_last_error(void) { return g_err; }
extern "C" int mm3d_abi_version(void) { return MM3D_ABI_VERSION; }

extern "C" int mm3d_device_supports_tc(void) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return -1;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return -1;
  return major == 10 ? 1 : 0;
}

// conv_simt.cu
struct ConvEpi;
size_t mm3d_conv_simt_workspace_bytes(int c_in, int c_out, int K);
int mm3d_conv_fwd_simt(const float* in, int64_t n_in, int c_in, float* out, int64_t n_out, int c_out,
                       const float* weight, int K, const int32_t* tbl, int64_t tbl_stride,
                       const uint8_t* onehot_off, int flags, void* ws, size_t ws_bytes, cudaStream_t stream,
                       const float* add = nullptr, const ConvEpi* epi = nullptr);
int mm3d_conv_wgrad_simt(const float* in, int64_t n_in, int c_in, const float* d_out, int64_t n_out, int c_out,
                         float* d_weight, int K, const int32_t* tbl, int64_t tbl_stride,
                         const uint8_t* onehot_off, int accumulate, cudaStream_t stream);

// conv_tc.cu
size_t mm3d_conv_tc_workspace_bytes(int c_in, int c_out, int K);
int mm3d_conv_tc_supported(int c_in, int c_out, int K);
// conv_tc_wgrad.cu
int mm3d_conv_wgrad_tc_supported(int c_in, int c_out, int K);
int mm3d_conv_wgrad_tc(const float* in, int64_t n_in, int c_in, const float* d_out, int64_t n_out, int c_out,
                       float* d_weight, int K, const void* plan, int64_t plan_cap, int accumulate,
                       cudaStream_t stream, int bf16 = 0, void* slab = nullptr, size_t slab_bytes = 0);
size_t mm3d_conv_wgrad_tc_slab_bytes(int c_in, int c_out, int K);
int mm3d_conv_fwd_tc(const float* in, int64_t n_in, int c_in, float* out, int64_t n_out, int c_out,
                     const float* weight, int K, const void* plan, int64_t plan_cap, int flags, void* ws,
                     size_t ws_bytes, cudaStream_t stream);

extern "C" size_t mm3d_conv_workspace_bytes(int64_t n_in, int64_t n_out, int c_in, int c_out, int K, int mode) {
  (void)n_in; (void)n_out;
  // one size for every use of a layer's scratch (forward, dgrad with c_in/c_out swapped, wgrad)
  size_t a = mm3d_conv_simt_workspace_bytes(c_in, c_out, K);
  size_t b = mm3d_conv_tc_workspace_bytes(c_in, c_out, K), c = mm3d_conv_tc_workspace_bytes(c_out, c_in, K);
  if (b > a) a = b;
  if (c > a) a = c;
  return mode == MM3D_MODE_TF32X3 ? 2 * a : a;  // two weight images
}

static int check_conv_args(const void* in, const void* out, const void* w, const int32_t* tbl, int64_t n_in,
                           int64_t n_out, int c_in, int c_out, int K, int64_t tbl_stride, const uint8_t* onehot) {
  MM3D_REQUIRE(n_in >= 0 && n_out >= 0 && c_in > 0 && c_out > 0 && K > 0, MM3D_ERR_INVALID, "bad conv sizes");
  MM3D_REQUIRE(n_out == 0 || (in && out && w && tbl), MM3D_ERR_INVALID, "null conv pointer");
  MM3D_REQUIRE(onehot || tbl_stride >= n_out, MM3D_ERR_INVALID, "tbl_stride %lld < n_out %lld",
               (long long)tbl_stride, (long long)n_out);
  return MM3D_OK;
}

extern "C" int mm3d_conv_fwd(const float* in, int64_t n_in, int c_in, float* out, int64_t n_out, int c_out,
                             const float* weight, int K, const int32_t* tbl, int64_t tbl_stride,
                             const uint8_t* onehot_off, const void* plan, int64_t plan_cap, int flags, int mode,
                             void* ws, size_t ws_bytes, mm3d_stream_t stream) {
  int rc = check_conv_args(in, out, weight, tbl, n_in, n_out, c_in, c_out, K, tbl_stride, onehot_off);
  if (rc) return rc;
  switch (mode) {
    case MM3D_MODE_FP32:
      return mm3d_conv_fwd_simt(in, n_in, c_in, out, n_out, c_out, weight, K, tbl, tbl_stride, onehot_off, flags,
                                ws, ws_bytes, (cudaStream_t)stream);
    case MM3D_MODE_TF32:
      // rows that are not whole 64-byte pieces (an unpadded 3-channel stem) stay on the FP32 SIMT kernel
      if (!mm3d_conv_tc_supported(c_in, c_out, K))
        return mm3d_conv_fwd_simt(in, n_in, c_in, out, n_out, c_out, weight, K, tbl, tbl_stride, onehot_off, flags,
                                  ws, ws_bytes, (cudaStream_t)stream);
      MM3D_REQUIRE(plan, MM3D_ERR_INVALID, "mm3d_conv_fwd: tf32 mode needs the table's row plan (mm3d_build_plan)");
      return mm3d_conv_fwd_tc(in, n_in, c_in, out, n_out, c_out, weight, K, plan, plan_cap, flags, ws, ws_bytes,
                              (cudaStream_t)stream);
    case MM3D_MODE_BF16:
      // `in`: an FP32 plane and the BF16 plane behind it (mm3d_split_bf16); the BF16 plane is what is gathered
      MM3D_REQUIRE(mm3d_conv_tc_supported(c_in, c_out, K), MM3D_ERR_UNSUPPORTED,
                   "bf16 conv: c_in %d must be a multiple of 16 (pad the channels)", c_in);
      MM3D_REQUIRE(plan, MM3D_ERR_INVALID, "mm3d_conv_fwd: bf16 mode needs the table's row plan (mm3d_build_plan)");
      return mm3d_conv_fwd_tc(in, n_in, c_in, out, n_out, c_out, weight, K, plan, plan_cap, flags | MM3D_CONV_BF16, ws, ws_bytes,
                              (cudaStream_t)stream);
    case MM3D_MODE_TF32X3:
      MM3D_REQUIRE(mm3d_conv_tc_supported(c_in, c_out, K), MM3D_ERR_UNSUPPORTED,
                   "tf32x3 conv: c_in %d must be a multiple of 16 (pad the channels)", c_in);
      MM3D_REQUIRE(plan, MM3D_ERR_INVALID, "mm3d_conv_fwd: tf32x3 mode needs the table's row plan (mm3d_build_plan)");
      return mm3d_conv_fwd_tc(in, n_in, c_in, out, n_out, c_out, weight, K, plan, plan_cap, flags | MM3D_CONV_X3, ws, ws_bytes,
                              (cudaStream_t)stream);
    default:
      MM3D_REQUIRE(false, MM3D_ERR_UNSUPPORTED, "conv mode %d not implemented in this build", mode);
  }
}

extern "C" size_t mm3d_conv_wgrad_workspace_bytes(int64_t n_out, int c_in, int c_out, int K, int mode, int flags) {
  (void)n_out;
  if (!(flags & MM3D_DETERMINISTIC) || mode == MM3D_MODE_FP32) return 0;
  return mm3d_conv_wgrad_tc_slab_bytes(c_in, c_out, K);  // (0 for the shapes only the SIMT kernel takes)
}

extern "C" int mm3d_conv_wgrad_ex(const float* in, int64_t n_in, int c_in, const float* d_out, int64_t n_out,
                                  int c_out, float* d_weight, int K, const int32_t* tbl, int64_t tbl_stride,
                                  const uint8_t* onehot_off, const void* plan, int64_t plan_cap, int accumulate, int mode,
                                  void* ws, size_t ws_bytes, mm3d_stream_t stream, int flags) {
  MM3D_REQUIRE((flags & ~MM3D_DETERMINISTIC) == 0, MM3D_ERR_INVALID, "conv_wgrad: unknown flags %#x", flags);
  const bool det = flags & MM3D_DETERMINISTIC;
  int rc = check_conv_args(in, d_out, d_weight, tbl, n_in, n_out, c_in, c_out, K, tbl_stride, onehot_off);
  if (rc) return rc;
  // deterministic: the tcgen05 kernels with per-CTA slabs in `ws`; the SIMT kernel has no such form
  MM3D_REQUIRE(!det || (mode != MM3D_MODE_FP32 && mm3d_conv_wgrad_tc_supported(c_in, c_out, K)), MM3D_ERR_UNSUPPORTED,
               "conv_wgrad: no deterministic form for %s (c_in %d c_out %d K %d): only the tensor-core modes on shapes "
               "the tcgen05 kernel takes (pad the channels to a multiple of 16)",
               mode == MM3D_MODE_FP32 ? "the fp32 mode" : "this shape", c_in, c_out, K);
  void* slab = det ? ws : nullptr;
  const size_t slab_bytes = det ? ws_bytes : 0;
  switch (mode) {
    case MM3D_MODE_TF32X3: {
      // d_weight = in_hi^T d_out_hi + in_lo^T d_out_hi + in_hi^T d_out_lo: three launches of the TF32 kernel that
      // accumulate into d_weight (both operands carry a hi and a lo plane)
      MM3D_REQUIRE(mm3d_conv_wgrad_tc_supported(c_in, c_out, K), MM3D_ERR_UNSUPPORTED,
                   "tf32x3 wgrad: unsupported shape c_in %d c_out %d K %d", c_in, c_out, K);
      MM3D_REQUIRE(plan, MM3D_ERR_INVALID, "mm3d_conv_wgrad: tf32x3 mode needs the table's row plan (mm3d_build_plan)");
      const float* in_lo = in + n_in * (int64_t)c_in;
      const float* dout_lo = d_out + n_out * (int64_t)c_out;
      rc = mm3d_conv_wgrad_tc(in, n_in, c_in, d_out, n_out, c_out, d_weight, K, plan, plan_cap, accumulate, (cudaStream_t)stream,
                              0, slab, slab_bytes);
      if (!rc) rc = mm3d_conv_wgrad_tc(in_lo, n_in, c_in, d_out, n_out, c_out, d_weight, K, plan, plan_cap, 1, (cudaStream_t)stream,
                                       0, slab, slab_bytes);
      if (!rc) rc = mm3d_conv_wgrad_tc(in, n_in, c_in, dout_lo, n_out, c_out, d_weight, K, plan, plan_cap, 1, (cudaStream_t)stream,
                                       0, slab, slab_bytes);
      return rc;
    }
    case MM3D_MODE_BF16:
      // BF16 planes of both operands (behind the FP32 ones) where the two-ring kernel takes the shape (c_in <= 128);
      // otherwise the TF32 kernel on the FP32 planes
      if (plan && mm3d_conv_wgrad_tc_supported(c_in, c_out, K) && n_out > 0) {
        rc = mm3d_conv_wgrad_tc(in + n_in * (int64_t)c_in, n_in, c_in, d_out + n_out * (int64_t)c_out, n_out, c_out, d_weight, K,
                                plan, plan_cap, accumulate, (cudaStream_t)stream, 1, slab, slab_bytes);
        if (rc != MM3D_ERR_UNSUPPORTED) return rc;
      }
      // fall through
    case MM3D_MODE_TF32:
      if (mm3d_conv_wgrad_tc_supported(c_in, c_out, K)) {
        MM3D_REQUIRE(plan, MM3D_ERR_INVALID, "mm3d_conv_wgrad: tf32 mode needs the table's row plan (mm3d_build_plan)");
        return mm3d_conv_wgrad_tc(in, n_in, c_in, d_out, n_out, c_out, d_weight, K, plan, plan_cap, accumulate,
                                  (cudaStream_t)stream, 0, slab, slab_bytes);
      }
      // fall through: shapes the tcgen05 kernel does not take (the 3-channel stem) use the FP32 kernel
    case MM3D_MODE_FP32:
      return mm3d_conv_wgrad_simt(in, n_in, c_in, d_out, n_out, c_out, d_weight, K, tbl, tbl_stride, onehot_off,
                                  accumulate, (cudaStream_t)stream);
    default:
      MM3D_REQUIRE(false, MM3D_ERR_UNSUPPORTED, "wgrad mode %d not implemented in this build", mode);
  }
}

extern "C" int mm3d_conv_wgrad(const float* in, int64_t n_in, int c_in, const float* d_out, int64_t n_out,
                               int c_out, float* d_weight, int K, const int32_t* tbl, int64_t tbl_stride,
                               const uint8_t* onehot_off, const void* plan, int64_t plan_cap, int accumulate, int mode,
                               void* ws, size_t ws_bytes, mm3d_stream_t stream) {
  return mm3d_conv_wgrad_ex(in, n_in, c_in, d_out, n_out, c_out, d_weight, K, tbl, tbl_stride, onehot_off, plan, plan_cap,
                            accumulate, mode, ws, ws_bytes, stream, 0);
}
