// Shared helpers of libmm3d: error reporting, key packing, hashing, launch geometry.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/mm3d.h"

// internal convolution flags (next to the public MM3D_CONV_TRANSPOSE_W / MM3D_CONV_MIRROR_K of mm3d.h)
#define MM3D_CONV_WEIGHT_LO 4  // weight image of tf32(w - tf32(w)) instead of tf32(w)
#define MM3D_CONV_X3 8         // error-compensated products: `in` carries hi and lo planes, two weight images
#define MM3D_CONV_BF16 16      // BF16 operands: `in` carries an FP32 plane and, behind it, a BF16 plane (the one gathered)

#define MM3D_NUM_SMS 148  // B200: 2 dies x 74 SMs; persistent / grid-stride kernels size to this

// SM count of the current device (cached per device); kernels that wait on each other size their grids from this
// and from the occupancy API, not from the constant above
int mm3d_sm_count();

void mm3d_set_error(const char* fmt, ...);
void mm3d_count_launches(int n);  // bookkeeping for mm3d_kernel_launches()

// groupby.cu: CSR lists start[n_keys + 1] / list[] of the entries of every key in ascending entry index (key < 0 = no
// key); `counts` = the per-key counts when the caller has them (NULL: counted here)
size_t mm3d_group_by_workspace_bytes(int64_t n_keys);
int mm3d_group_by(const int32_t* key, const int32_t* counts, int64_t n, int64_t n_keys, int32_t* start, int32_t* list,
                  void* ws, size_t ws_bytes, cudaStream_t stream);

#define MM3D_REQUIRE(cond, code, ...)     \
  do {                                    \
    if (!(cond)) {                        \
      mm3d_set_error(__VA_ARGS__);        \
      return (code);                      \
    }                                     \
  } while (0)

#define MM3D_CHECK_LAUNCH(name)                                                      \
  do {                                                                               \
    cudaError_t e__ = cudaGetLastError();                                            \
    if (e__ != cudaSuccess) {                                                        \
      mm3d_set_error("%s: launch failed: %s", (name), cudaGetErrorString(e__));      \
      return MM3D_ERR_CUDA;                                                          \
    }                                                                                \
  } while (0)

#define MM3D_CUDA(call)                                                              \
  do {                                                                               \
    cudaError_t e__ = (call);                                                        \
    if (e__ != cudaSuccess) {                                                        \
      mm3d_set_error("%s failed: %s", #call, cudaGetErrorString(e__));               \
      return MM3D_ERR_CUDA;                                                          \
    }                                                                                \
  } while (0)

// index of the current device for per-device one-time setup (function attributes are per device)
static inline int mm3d_device_slot() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
  return dev;
}

static inline int64_t mm3d_cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline size_t mm3d_align(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }
// Layers wider than a kernel takes run as slices of shapes it does: `c` channels cut into ceil(c / max) near-equal
// slices whose starts are multiples of q (max a multiple of q).  The width of every slice but the last; one slice
// of the whole width when c <= max.
static inline int mm3d_slice_step(int c, int max, int q) {
  const int n = (int)mm3d_cdiv(c, max);
  return (int)mm3d_cdiv(mm3d_cdiv(c, n), q) * q;
}

// grid for a grid-stride kernel over n items: enough CTAs to cover n once, capped at a few
// waves of the 148 SMs so tiny levels do not launch thousands of empty CTAs.
static inline int mm3d_grid(int64_t n, int block, int ctas_per_sm = 8) {
  int64_t g = mm3d_cdiv(n > 0 ? n : 1, block);
  int64_t cap = (int64_t)MM3D_NUM_SMS * ctas_per_sm;
  return (int)(g < cap ? g : cap);
}

// ---- programmatic dependent launch: a kernel launched with mm3d_launch_pdl may start (block scheduling, its
// prologue up to mm3d_griddep_wait()) while the previous kernel of the stream is still draining; everything
// that reads or writes global memory comes after mm3d_griddep_wait(), which returns once the previous kernel
// has completed and its writes are visible.  Kernels call mm3d_griddep_launch() early so that their own
// successor can be scheduled as soon as SM resources free up.  MM3D_NO_PDL=1 launches plainly.
#ifdef __CUDACC__
// Sticky device-error words live in mapped pinned host memory (mm3d_device_err_flag): word 0 = a bounded wait of a
// kernel pipeline / grid barrier timed out, word 1 = a lift index outside the image.  A plain store + system fence
// is enough (the words only ever go 0 -> 1) and the host can poll them without any CUDA call.
__device__ __forceinline__ void mm3d_raise(int* err, int word = 0) {
  if (err) {
    *reinterpret_cast<volatile int*>(err + word) = 1;
    __threadfence_system();
  }
}
// round-to-nearest (ties away) to TF32: what a producer stores when its consumer is a kind::tf32 tcgen05.mma, which
// would otherwise TRUNCATE the low 13 mantissa bits of a raw FP32 operand
__device__ __forceinline__ float mm3d_rna_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
__device__ __forceinline__ void mm3d_griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void mm3d_griddep_launch() {
#ifdef MM3D_PDL_EARLY_TRIGGER
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
}

bool mm3d_pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t mm3d_launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                   Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = mm3d_pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
#endif

#define MM3D_KEY_EMPTY 0xFFFFFFFFFFFFFFFFull

__host__ __device__ __forceinline__ uint64_t mm3d_pack_key(uint64_t x, uint64_t y, uint64_t z, uint64_t b) {
  return (b << 48) | (x << 32) | (y << 16) | z;
}
__host__ __device__ __forceinline__ int mm3d_key_x(uint64_t k) { return (int)((k >> 32) & 0xFFFF); }
__host__ __device__ __forceinline__ int mm3d_key_y(uint64_t k) { return (int)((k >> 16) & 0xFFFF); }
__host__ __device__ __forceinline__ int mm3d_key_z(uint64_t k) { return (int)(k & 0xFFFF); }
__host__ __device__ __forceinline__ uint64_t mm3d_key_b(uint64_t k) { return k >> 48; }

// murmur3 finaliser: spreads the structured (mostly low-entropy) voxel keys over the table
__device__ __forceinline__ uint32_t mm3d_hash(uint64_t k) {
  k ^= k >> 33;
  k *= 0xff51afd7ed558ccdULL;
  k ^= k >> 33;
  k *= 0xc4ceb9fe1a85ec53ULL;
  k ^= k >> 33;
  return (uint32_t)k;
}

// read-only lookup in an open-addressing table (linear probing); -1 when absent
__device__ __forceinline__ int mm3d_hash_find(const uint64_t* __restrict__ keys,
                                              const int32_t* __restrict__ vals, uint32_t mask,
                                              uint64_t key) {
  uint32_t s = mm3d_hash(key) & mask;
  while (true) {
    uint64_t k = __ldg(keys + s);
    if (k == key) return __ldg(vals + s);
    if (k == MM3D_KEY_EMPTY) return -1;
    s = (s + 1) & mask;
  }
}
