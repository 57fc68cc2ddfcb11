// InputLayer / OutputLayer feature kernels and the 2D->3D lift: HBM-bound gathers/scatters.
//
// InputLayer (mode 4): voxel row = mean of its points' features  (SURVEY A.2);
// OutputLayer: point row = copy of its voxel's row, backward = sum over the voxel's points (A.7);
// lift: out[n,:] = fmap[b(n), :, row(n), col(n)] on an NCHW map (2d_net/model.py:131-137).
// One thread per (row, channel-vector); consecutive threads walk a row, so the row side of
// every gather/scatter is fully coalesced and the indexed side moves whole 16/32-byte pieces.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

int* mm3d_device_err_flag();  // conv_tc.cu
int mm3d_det_sum_parts(const double* part, int nparts, int words, float* dst, cudaStream_t stream);  // heads.cu

namespace {

// ------------------------------------------------------------------ InputLayer
// One thread per point, 4 points per thread in flight: the point's C features are read as one contiguous piece and
// written to its voxel's row -- a plain store when the point is alone in its voxel (88 % of the points), atomics
// otherwise (the row was zeroed by the launch's memset).  No per-element index division.
template <int C>
__global__ void __launch_bounds__(256)
k_input_fwd(const float* __restrict__ feats, const int32_t* __restrict__ p2v, const int32_t* __restrict__ npts,
            int64_t n_points, int c_rt, int mode, float* __restrict__ out) {
  mm3d_griddep_wait();
  const int c = C > 0 ? C : c_rt;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_points; p += stride) {
    const int32_t v = __ldg(p2v + p);
    const int32_t cnt = __ldg(npts + v);
    const float* src = feats + p * c;
    float* dst = out + (int64_t)v * c;
    if (C > 0) {
      float f[C > 0 ? C : 1];
#pragma unroll
      for (int j = 0; j < C; ++j) f[j] = __ldg(src + j);
      if (cnt == 1) {
#pragma unroll
        for (int j = 0; j < C; ++j) dst[j] = f[j];
      } else {
#pragma unroll
        for (int j = 0; j < C; ++j) atomicAdd(dst + j, mode == 4 ? f[j] / (float)cnt : f[j]);
      }
    } else {
      for (int j = 0; j < c; ++j) {
        const float f = __ldg(src + j);
        if (cnt == 1) dst[j] = f;
        else atomicAdd(dst + j, mode == 4 ? f / (float)cnt : f);
      }
    }
  }
}

template <int C>
__global__ void __launch_bounds__(256)
k_input_bwd(const float* __restrict__ d_vox, const int32_t* __restrict__ p2v, const int32_t* __restrict__ npts,
            int64_t n_points, int c_rt, int mode, float* __restrict__ d_feats) {
  mm3d_griddep_wait();
  const int c = C > 0 ? C : c_rt;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_points; p += stride) {
    const int32_t v = __ldg(p2v + p);
    const float* src = d_vox + (int64_t)v * c;
    float* dst = d_feats + p * c;
    const int32_t cnt = mode == 4 ? __ldg(npts + v) : 1;
    if (C > 0) {
#pragma unroll
      for (int j = 0; j < C; ++j) dst[j] = cnt > 1 ? __ldg(src + j) / (float)cnt : __ldg(src + j);
    } else {
      for (int j = 0; j < c; ++j) dst[j] = cnt > 1 ? __ldg(src + j) / (float)cnt : __ldg(src + j);
    }
  }
}


// InputLayer with the RGB-mask prologue of Net3DSeg.forward (3d_net/model.py:46-48) folded in: the point's features
// are scaled by s = sigmoid(x . w + b) on their way into the voxel row -- the masked [N, C] tensor of the reference
// (and its three element-wise kernels) never exists.  wb = [w_0 .. w_{C-1}, b]; s_out keeps the gate for the backward.
template <int C>
__global__ void __launch_bounds__(256)
k_input_masked_fwd(const float* __restrict__ feats, const int32_t* __restrict__ p2v, const int32_t* __restrict__ npts,
                   int64_t n_points, int mode, const float* __restrict__ wb, float* __restrict__ out, float* __restrict__ s_out) {
  mm3d_griddep_wait();
  float w[C + 1];
#pragma unroll
  for (int j = 0; j <= C; ++j) w[j] = __ldg(wb + j);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_points; p += stride) {
    const int32_t v = __ldg(p2v + p);
    const int32_t cnt = __ldg(npts + v);
    float f[C], acc = w[C];
#pragma unroll
    for (int j = 0; j < C; ++j) {
      f[j] = __ldg(feats + p * C + j);
      acc = fmaf(f[j], w[j], acc);
    }
    const float sg = 1.f / (1.f + expf(-acc));
    s_out[p] = sg;
    float* dst = out + (int64_t)v * C;
#pragma unroll
    for (int j = 0; j < C; ++j) {
      const float y = f[j] * sg;
      if (cnt == 1) dst[j] = y;
      else atomicAdd(dst + j, mode == 4 ? y / (float)cnt : y);
    }
  }
}

// backward of the above: g = d_vox[voxel] (/ count); t = (g . x) s (1 - s); d_feats = g s + t w; d_w += t x; d_b += t
// (FP64 totals, one atomic per CTA and value, as in heads.cu).  DET: no atomics -- the CTA's totals, its warps summed
// in warp order, go to its own row dwb[blockIdx.x][C + 1], which mm3d_det_sum_parts (heads.cu) sums in CTA order.
template <int C, bool DET>
__global__ void __launch_bounds__(256)
k_input_masked_bwd(const float* __restrict__ d_vox, const float* __restrict__ feats, const float* __restrict__ s_in,
                   const int32_t* __restrict__ p2v, const int32_t* __restrict__ npts, int64_t n_points, int mode,
                   const float* __restrict__ wb, float* __restrict__ d_feats, double* __restrict__ dwb) {
  mm3d_griddep_wait();
  __shared__ double red[C + 1];
  __shared__ double wred[DET ? 8 : 1][C + 1];
  if (threadIdx.x <= C) red[threadIdx.x] = 0.0;
  __syncthreads();
  float w[C];
#pragma unroll
  for (int j = 0; j < C; ++j) w[j] = __ldg(wb + j);
  double loc[C + 1];
#pragma unroll
  for (int j = 0; j <= C; ++j) loc[j] = 0.0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_points; p += stride) {
    const int32_t v = __ldg(p2v + p);
    const int32_t cnt = mode == 4 ? __ldg(npts + v) : 1;
    const float sg = __ldg(s_in + p);
    float g[C], x[C], dot = 0.f;
#pragma unroll
    for (int j = 0; j < C; ++j) {
      g[j] = __ldg(d_vox + (int64_t)v * C + j);
      if (cnt > 1) g[j] /= (float)cnt;
      x[j] = __ldg(feats + p * C + j);
      dot = fmaf(g[j], x[j], dot);
    }
    const float t = dot * sg * (1.f - sg);
#pragma unroll
    for (int j = 0; j < C; ++j) {
      if (d_feats) d_feats[p * C + j] = fmaf(t, w[j], g[j] * sg);
      loc[j] += (double)(t * x[j]);
    }
    loc[C] += (double)t;
  }
#pragma unroll
  for (int j = 0; j <= C; ++j) {
    double vv = loc[j];
    for (int o = 16; o; o >>= 1) vv += __shfl_xor_sync(0xffffffffu, vv, o);
    if ((threadIdx.x & 31) == 0) {
      if (DET) wred[threadIdx.x >> 5][j] = vv;
      else atomicAdd(&red[j], vv);
    }
  }
  __syncthreads();
  if (threadIdx.x <= C) {
    if (DET) {  // 256 threads = 8 warps
      double t = 0.0;
      for (int w = 0; w < 8; ++w) t += wred[w][threadIdx.x];
      dwb[(int64_t)blockIdx.x * (C + 1) + threadIdx.x] = t;
    } else {
      atomicAdd(dwb + threadIdx.x, red[threadIdx.x]);
    }
  }
}

__global__ void k_f64_to_f32_io(const double* __restrict__ src, float* __restrict__ dst, int n) {
  mm3d_griddep_wait();
  for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = (float)src[i];
}

// ------------------------------------------------------------------ OutputLayer
// cv float4 per row (cv a power of two <= 32 in the vector path): cv consecutive lanes copy one point's row, a warp
// moves 32 / cv points per pass and every thread keeps 4 passes in flight.  32-bit index arithmetic.
template <int VEC>
__global__ void __launch_bounds__(256)
k_output_fwd(const float* __restrict__ vox, const int32_t* __restrict__ p2v, int64_t n_points, int cv, int cv_shift,
             float* __restrict__ out) {
  mm3d_griddep_wait();
  const int64_t total = n_points * cv;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (VEC == 4) {
    const int ch = (int)(i & (cv - 1));  // stride is a multiple of cv: the lane keeps its channel vector
    for (; i + 3 * stride < total; i += 4 * stride) {
      int32_t v[4];
      float4 t[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = __ldg(p2v + ((i + u * stride) >> cv_shift));
#pragma unroll
      for (int u = 0; u < 4; ++u) t[u] = __ldg(reinterpret_cast<const float4*>(vox) + ((int64_t)v[u] << cv_shift) + ch);
#pragma unroll
      for (int u = 0; u < 4; ++u) reinterpret_cast<float4*>(out)[i + u * stride] = t[u];
    }
    for (; i < total; i += stride)
      reinterpret_cast<float4*>(out)[i] = __ldg(reinterpret_cast<const float4*>(vox) + ((int64_t)__ldg(p2v + (i >> cv_shift)) << cv_shift) + ch);
  } else {
    for (; i < total; i += stride) {
      const int64_t p = i / cv;
      out[i] = __ldg(vox + (int64_t)__ldg(p2v + p) * cv + (int)(i - p * cv));
    }
  }
}

// backward: voxel gradient = sum over its points.  Vector path: one red.global.add.v4.f32 per float4 (a quarter of
// the atomics of the scalar form); d_vox was zeroed by the launch's memset.
template <int VEC>
__global__ void __launch_bounds__(256)
k_output_bwd(const float* __restrict__ d_out, const int32_t* __restrict__ p2v, int64_t n_points, int cv, int cv_shift,
             float* __restrict__ d_vox) {
  mm3d_griddep_wait();
  const int64_t total = n_points * cv;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (VEC == 4) {
    const int ch = (int)(i & (cv - 1));
    for (; i < total; i += stride) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(d_out) + i);
      float* dst = d_vox + ((((int64_t)__ldg(p2v + (i >> cv_shift)) << cv_shift) + ch) << 2);
      asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(g.x), "f"(g.y), "f"(g.z), "f"(g.w) : "memory");
    }
  } else {
    for (; i < total; i += stride) {
      const int64_t p = i / cv;
      atomicAdd(d_vox + (int64_t)__ldg(p2v + p) * cv + (int)(i - p * cv), __ldg(d_out + i));
    }
  }
}

// ------------------------------------------------------------------ lift
__device__ __forceinline__ int find_sample(const int64_t* __restrict__ offs, int B, int64_t n) {
  int lo = 0, hi = B;  // offs[lo] <= n < offs[hi]
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (__ldg(offs + mid) <= n) lo = mid; else hi = mid;
  }
  return lo;
}

// One thread per (point, group of G channels), group fastest: the point's pixel index (one 16-byte load) and its
// sample (binary search over the B + 1 offsets) are resolved once per G values, and the [N, C] side is coalesced.  The
// map is addressed through its element strides (sb, sc, sh, sw): for a channels-last map (sc == 1, what cuDNN produces
// for the 2D network) the C values of a pixel are one contiguous piece and a point costs one or two sectors; for a
// channel-major map (NCHW) every value sits in its own plane -- 32 bytes moved per 4 used, inherent to that layout.
template <class T, int G>
__global__ void __launch_bounds__(256)
k_lift_fwd(const T* __restrict__ fmap, int B, int C, int H, int W, int64_t sb, int64_t sc, int64_t sh, int64_t sw,
           const int64_t* __restrict__ idx, const int64_t* __restrict__ offs, int64_t n, T* __restrict__ out, int* err) {
  const int groups = C / G;
  const int64_t total = n * groups;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = total < (1ll << 31) ? (int64_t)((uint32_t)i / (uint32_t)groups) : i / groups;
    const int ch0 = (int)(i - p * groups) * G;
    const longlong2 rc = __ldg(reinterpret_cast<const longlong2*>(idx) + p);
    int64_t r = rc.x, col = rc.y;
    if (r < 0) r += H;      // torch advanced indexing wraps negative indices
    if (col < 0) col += W;
    T* dst = out + p * C + ch0;
    if ((uint64_t)r >= (uint64_t)H || (uint64_t)col >= (uint64_t)W) {
      // torch raises IndexError here (2d_net/model.py:131-137); a kernel cannot: zero row + sticky error word 1
#pragma unroll
      for (int j = 0; j < G; ++j) dst[j] = T(0.f);
      if (ch0 == 0) mm3d_raise(err, 1);
      continue;
    }
    const T* src = fmap + find_sample(offs, B, p) * sb + ch0 * sc + r * sh + col * sw;
    T v[G];
#pragma unroll
    for (int j = 0; j < G; ++j) v[j] = src[j * sc];
#pragma unroll
    for (int j = 0; j < G; ++j) dst[j] = v[j];
  }
}

__device__ __forceinline__ void lift_atomic_add(float* p, float v) { atomicAdd(p, v); }
__device__ __forceinline__ void lift_atomic_add(__half* p, __half v) { atomicAdd(p, v); }
__device__ __forceinline__ void lift_atomic_add(__nv_bfloat16* p, __nv_bfloat16 v) { atomicAdd(p, v); }

// backward: scatter-add into the (zero-filled) map gradient; several points may share a pixel
template <class T, int G>
__global__ void __launch_bounds__(256)
k_lift_bwd(const T* __restrict__ d_out, int B, int C, int H, int W, int64_t sb, int64_t sc, int64_t sh, int64_t sw,
           const int64_t* __restrict__ idx, const int64_t* __restrict__ offs, int64_t n, T* __restrict__ d_fmap, int* err) {
  const int groups = C / G;
  const int64_t total = n * groups;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = total < (1ll << 31) ? (int64_t)((uint32_t)i / (uint32_t)groups) : i / groups;
    const int ch0 = (int)(i - p * groups) * G;
    const longlong2 rc = __ldg(reinterpret_cast<const longlong2*>(idx) + p);
    int64_t r = rc.x, col = rc.y;
    if (r < 0) r += H;
    if (col < 0) col += W;
    if ((uint64_t)r >= (uint64_t)H || (uint64_t)col >= (uint64_t)W) {  // skipped + sticky error word 1
      if (ch0 == 0) mm3d_raise(err, 1);
      continue;
    }
    const T* src = d_out + p * C + ch0;
    T* dst = d_fmap + find_sample(offs, B, p) * sb + ch0 * sc + r * sh + col * sw;
    T v[G];
#pragma unroll
    for (int j = 0; j < G; ++j) v[j] = src[j];
#pragma unroll
    for (int j = 0; j < G; ++j) lift_atomic_add(dst + j * sc, v[j]);
  }
}

// ---- bilinear variant (an extension: the reference only ever gathers at integer pixels).  uv = float32 (row, col) in
// pixel units, pixel centres at the integers; the four neighbouring pixels are blended with the usual weights and a
// neighbour outside the map contributes zero -- F.grid_sample(mode="bilinear", padding_mode="zeros",
// align_corners=True) on the normalised coordinates.  Same thread layout as the integer gather; arithmetic in FP32.
template <class T> __device__ __forceinline__ float lift_to_f32(T v) { return (float)v; }

struct BilinearTaps {
  int64_t off[4];  // element offset of the tap inside the sample's map (without the channel term)
  float w[4];      // 0 for a tap outside the map
  int rr[4], cc[4];  // the tap's pixel (valid where w != 0)
};

__device__ __forceinline__ BilinearTaps bilinear_taps(float r, float c, int H, int W, int64_t sh, int64_t sw) {
  BilinearTaps t;
  const float r0f = floorf(r), c0f = floorf(c);
  const float fr = r - r0f, fc = c - c0f;
  // (coordinates far outside the map: every tap is outside; clamp before the integer conversion)
  const int r0 = (int)fminf(fmaxf(r0f, -2.f), (float)H), c0 = (int)fminf(fmaxf(c0f, -2.f), (float)W);
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int rr = r0 + (q >> 1), cc = c0 + (q & 1);
    const bool in = (unsigned)rr < (unsigned)H && (unsigned)cc < (unsigned)W;
    const float w = ((q >> 1) ? fr : 1.f - fr) * ((q & 1) ? fc : 1.f - fc);
    t.w[q] = in ? w : 0.f;
    t.off[q] = in ? rr * sh + cc * sw : 0;
    t.rr[q] = rr;
    t.cc[q] = cc;
  }
  return t;
}

template <class T, int G>
__global__ void __launch_bounds__(256)
k_lift_bilinear_fwd(const T* __restrict__ fmap, int B, int C, int H, int W, int64_t sb, int64_t sc, int64_t sh, int64_t sw,
                    const float* __restrict__ uv, const int64_t* __restrict__ offs, int64_t n, T* __restrict__ out, int* err) {
  (void)err;
  const int groups = C / G;
  const int64_t total = n * groups;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = total < (1ll << 31) ? (int64_t)((uint32_t)i / (uint32_t)groups) : i / groups;
    const int ch0 = (int)(i - p * groups) * G;
    const float2 rc = __ldg(reinterpret_cast<const float2*>(uv) + p);
    const BilinearTaps t = bilinear_taps(rc.x, rc.y, H, W, sh, sw);
    const T* base = fmap + find_sample(offs, B, p) * sb + ch0 * sc;
    float acc[G];
#pragma unroll
    for (int j = 0; j < G; ++j) acc[j] = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (t.w[q] != 0.f) {
#pragma unroll
        for (int j = 0; j < G; ++j) acc[j] = fmaf(t.w[q], lift_to_f32(base[t.off[q] + j * sc]), acc[j]);
      }
    }
    T* dst = out + p * C + ch0;
#pragma unroll
    for (int j = 0; j < G; ++j) dst[j] = T(acc[j]);
  }
}

// backward with respect to the map (the projected coordinates are data: no gradient for uv)
template <class T, int G>
__global__ void __launch_bounds__(256)
k_lift_bilinear_bwd(const T* __restrict__ d_out, int B, int C, int H, int W, int64_t sb, int64_t sc, int64_t sh, int64_t sw,
                    const float* __restrict__ uv, const int64_t* __restrict__ offs, int64_t n, T* __restrict__ d_fmap, int* err) {
  (void)err;
  const int groups = C / G;
  const int64_t total = n * groups;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = total < (1ll << 31) ? (int64_t)((uint32_t)i / (uint32_t)groups) : i / groups;
    const int ch0 = (int)(i - p * groups) * G;
    const float2 rc = __ldg(reinterpret_cast<const float2*>(uv) + p);
    const BilinearTaps t = bilinear_taps(rc.x, rc.y, H, W, sh, sw);
    T* base = d_fmap + find_sample(offs, B, p) * sb + ch0 * sc;
    float g[G];
#pragma unroll
    for (int j = 0; j < G; ++j) g[j] = lift_to_f32(d_out[p * C + ch0 + j]);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (t.w[q] != 0.f) {
#pragma unroll
        for (int j = 0; j < G; ++j) lift_atomic_add(base + t.off[q] + j * sc, T(t.w[q] * g[j]));
      }
    }
  }
}

// ------------------------------------------------------------------ deterministic forms: segmented sums
// Each output row (voxel) or pixel is written ONCE by the thread that owns it, summing its entries in the ascending
// entry order of the group-by-key lists (groupby.cu): no memset, no atomics, the same bits on every run.

// InputLayer forward.  Mode 4 sums f / cnt in point order -- the terms of k_input_fwd -- so a voxel of one point gets
// exactly the bits of the default path.
__global__ void __launch_bounds__(256)
k_input_fwd_csr(const float* __restrict__ feats, const int32_t* __restrict__ vstart, const int32_t* __restrict__ vpts,
                int64_t n_vox, int c, int mode, float* __restrict__ out) {
  mm3d_griddep_wait();
  const int64_t total = n_vox * c;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t v = i / c;
    const int j = (int)(i - v * c);
    const int32_t b = __ldg(vstart + v), e = __ldg(vstart + v + 1), cnt = e - b;
    float acc;
    if (cnt == 1) {
      acc = __ldg(feats + (int64_t)__ldg(vpts + b) * c + j);
    } else {
      acc = 0.f;
      for (int32_t q = b; q < e; ++q) {
        const float f = __ldg(feats + (int64_t)__ldg(vpts + q) * c + j);
        acc += mode == 4 ? f / (float)cnt : f;
      }
    }
    out[i] = acc;
  }
}

// InputLayer forward with the RGB mask folded in (k_input_masked_fwd): one thread per voxel writes its row and the gates
// of its points (every point is in exactly one list).  The gate and the terms y / cnt are computed as there and summed in
// point order, so a voxel of one point gets exactly the bits of the default path.
template <int C>
__global__ void __launch_bounds__(256)
k_input_masked_fwd_csr(const float* __restrict__ feats, const int32_t* __restrict__ vstart, const int32_t* __restrict__ vpts,
                       int64_t n_vox, int mode, const float* __restrict__ wb, float* __restrict__ out,
                       float* __restrict__ s_out) {
  mm3d_griddep_wait();
  float w[C + 1];
#pragma unroll
  for (int j = 0; j <= C; ++j) w[j] = __ldg(wb + j);
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n_vox; v += (int64_t)gridDim.x * blockDim.x) {
    const int32_t b = __ldg(vstart + v), e = __ldg(vstart + v + 1), cnt = e - b;
    float acc[C];
#pragma unroll
    for (int j = 0; j < C; ++j) acc[j] = 0.f;
    for (int32_t q = b; q < e; ++q) {
      const int64_t p = __ldg(vpts + q);
      float f[C], a = w[C];
#pragma unroll
      for (int j = 0; j < C; ++j) {
        f[j] = __ldg(feats + p * C + j);
        a = fmaf(f[j], w[j], a);
      }
      const float sg = 1.f / (1.f + expf(-a));
      s_out[p] = sg;
#pragma unroll
      for (int j = 0; j < C; ++j) {
        const float y = f[j] * sg;
        if (cnt == 1) acc[j] = y;
        else acc[j] += mode == 4 ? y / (float)cnt : y;
      }
    }
#pragma unroll
    for (int j = 0; j < C; ++j) out[v * C + j] = acc[j];
  }
}

// OutputLayer backward: a voxel's gradient = the sum of its points' gradients, in point order
__global__ void __launch_bounds__(256)
k_output_bwd_csr(const float* __restrict__ d_out, const int32_t* __restrict__ vstart, const int32_t* __restrict__ vpts,
                 int64_t n_vox, int c, float* __restrict__ d_vox) {
  mm3d_griddep_wait();
  const int64_t total = n_vox * c;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t v = i / c;
    const int j = (int)(i - v * c);
    const int32_t b = __ldg(vstart + v), e = __ldg(vstart + v + 1);
    float acc = 0.f;
    for (int32_t q = b; q < e; ++q) acc += __ldg(d_out + (int64_t)__ldg(vpts + q) * c + j);
    d_vox[i] = acc;
  }
}

// Keys of the lift's pixel lists: pixel (b H + r) W + c of every point (integer lift, negative indices wrapped as
// k_lift_bwd does; an index outside the map gets no key and raises error word 1 like there), or of every (point, tap)
// entry 4 p + q of the bilinear lift (a tap outside the map, or of weight zero, gets no key: k_lift_bilinear_bwd
// skips it too)
__global__ void k_lift_keys(const int64_t* __restrict__ idx, const float* __restrict__ uv, const int64_t* __restrict__ offs,
                            int B, int H, int W, int64_t n, int32_t* __restrict__ key, int* err) {
  mm3d_griddep_wait();
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t base = (int64_t)find_sample(offs, B, p) * H;
    if (idx) {
      const longlong2 rc = __ldg(reinterpret_cast<const longlong2*>(idx) + p);
      int64_t r = rc.x, col = rc.y;
      if (r < 0) r += H;
      if (col < 0) col += W;
      if ((uint64_t)r >= (uint64_t)H || (uint64_t)col >= (uint64_t)W) {
        key[p] = -1;
        mm3d_raise(err, 1);
      } else {
        key[p] = (int32_t)((base + r) * W + col);
      }
    } else {
      const float2 rc = __ldg(reinterpret_cast<const float2*>(uv) + p);
      const BilinearTaps t = bilinear_taps(rc.x, rc.y, H, W, 0, 0);
#pragma unroll
      for (int q = 0; q < 4; ++q) key[4 * p + q] = t.w[q] != 0.f ? (int32_t)((base + t.rr[q]) * W + t.cc[q]) : -1;
    }
  }
}

// Lift backward over the pixel lists: one thread per (pixel, channel), channel fastest; FP32 accumulation in entry
// order, rounded once to T and stored into the caller's zero-filled map.  BIL: entries are (point, tap) pairs 4 p + q
// and a term is w_q * g as in k_lift_bilinear_bwd.
template <class T, bool BIL>
__global__ void __launch_bounds__(256)
k_lift_bwd_csr(const T* __restrict__ d_out, int C, int H, int W, int64_t sb, int64_t sc, int64_t sh, int64_t sw,
               const float* __restrict__ uv, const int32_t* __restrict__ pstart, const int32_t* __restrict__ pent,
               int64_t n_pix, T* __restrict__ d_fmap) {
  mm3d_griddep_wait();
  const int64_t total = n_pix * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t pix = i / C;
    const int ch = (int)(i - pix * C);
    const int32_t b0 = __ldg(pstart + pix), e0 = __ldg(pstart + pix + 1);
    if (b0 == e0) continue;
    float acc = 0.f;
    for (int32_t q = b0; q < e0; ++q) {
      const int32_t ent = __ldg(pent + q);
      if (BIL) {
        const int64_t p = ent >> 2;
        const float2 rc = __ldg(reinterpret_cast<const float2*>(uv) + p);
        const BilinearTaps t = bilinear_taps(rc.x, rc.y, H, W, 0, 0);
        acc += t.w[ent & 3] * lift_to_f32(d_out[p * C + ch]);
      } else {
        acc += lift_to_f32(d_out[(int64_t)ent * C + ch]);
      }
    }
    const int64_t hw = (int64_t)H * W;
    const int64_t b = pix / hw, rem = pix - b * hw, r = rem / W, col = rem - r * W;
    d_fmap[b * sb + ch * sc + r * sh + col * sw] = T(acc);
  }
}

// channels per thread: contiguous channels (sc == 1, channels-last) in groups of 4 or 2; one per thread for a
// channel-major map, where neighbouring threads should walk neighbouring planes of one pixel
#define LIFT_DISPATCH(KERNEL, T, ...)                                                                               \
  do {                                                                                                              \
    if (sc == 1 && C % 4 == 0) KERNEL<T, 4><<<mm3d_grid(n * (C / 4), 256, 16), 256, 0, stream>>>(__VA_ARGS__);      \
    else if (sc == 1 && C % 2 == 0) KERNEL<T, 2><<<mm3d_grid(n * (C / 2), 256, 16), 256, 0, stream>>>(__VA_ARGS__); \
    else KERNEL<T, 1><<<mm3d_grid(n * C, 256, 16), 256, 0, stream>>>(__VA_ARGS__);                                  \
  } while (0)

}  // namespace

static int pow2_shift(int v) {  // log2 of a power of two <= 32, else -1
  for (int sft = 0; sft <= 5; ++sft)
    if ((1 << sft) == v) return sft;
  return -1;
}

extern "C" int mm3d_input_fwd(const float* feats, const int32_t* p2v, const int32_t* npts, int64_t n_points,
                              int64_t n_vox, int c, int mode, float* out_vox, mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(mode == 3 || mode == 4, MM3D_ERR_UNSUPPORTED, "InputLayer mode %d not implemented (3=sum, 4=mean)", mode);
  MM3D_REQUIRE(c > 0 && n_points >= 0 && n_vox >= 0, MM3D_ERR_INVALID, "bad sizes");
  if (n_vox > 0) MM3D_CUDA(cudaMemsetAsync(out_vox, 0, sizeof(float) * (size_t)n_vox * c, stream));
  if (n_points > 0) {
    const dim3 grid(mm3d_grid(n_points, 256, 16)), block(256);
    if (c == 3) MM3D_CUDA(mm3d_launch_pdl(k_input_fwd<3>, grid, block, 0, stream, feats, p2v, npts, n_points, c, mode, out_vox));
    else if (c == 1) MM3D_CUDA(mm3d_launch_pdl(k_input_fwd<1>, grid, block, 0, stream, feats, p2v, npts, n_points, c, mode, out_vox));
    else MM3D_CUDA(mm3d_launch_pdl(k_input_fwd<0>, grid, block, 0, stream, feats, p2v, npts, n_points, c, mode, out_vox));
  }
  mm3d_count_launches(n_points > 0 ? 1 : 0);
  MM3D_CHECK_LAUNCH("mm3d_input_fwd");
  return MM3D_OK;
}

extern "C" int mm3d_input_bwd(const float* d_vox, const int32_t* p2v, const int32_t* npts, int64_t n_points,
                              int c, int mode, float* d_feats, mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(mode == 3 || mode == 4, MM3D_ERR_UNSUPPORTED, "InputLayer mode %d not implemented", mode);
  if (n_points > 0) {
    const dim3 grid(mm3d_grid(n_points, 256, 16)), block(256);
    if (c == 3) MM3D_CUDA(mm3d_launch_pdl(k_input_bwd<3>, grid, block, 0, stream, d_vox, p2v, npts, n_points, c, mode, d_feats));
    else if (c == 1) MM3D_CUDA(mm3d_launch_pdl(k_input_bwd<1>, grid, block, 0, stream, d_vox, p2v, npts, n_points, c, mode, d_feats));
    else MM3D_CUDA(mm3d_launch_pdl(k_input_bwd<0>, grid, block, 0, stream, d_vox, p2v, npts, n_points, c, mode, d_feats));
  }
  mm3d_count_launches(n_points > 0 ? 1 : 0);
  MM3D_CHECK_LAUNCH("mm3d_input_bwd");
  return MM3D_OK;
}

// InputLayer forward with the RGB mask folded in (3 feature channels: the reference's rgb features): out_vox as
// mm3d_input_fwd of feats * sigmoid(feats . w + b); wb = [w_0, w_1, w_2, b] on the device, s_out [n_points] = the gates.
extern "C" int mm3d_input_masked_fwd(const float* feats, const int32_t* p2v, const int32_t* npts, int64_t n_points,
                                     int64_t n_vox, int c, int mode, const float* wb, float* out_vox, float* s_out,
                                     mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(mode == 3 || mode == 4, MM3D_ERR_UNSUPPORTED, "InputLayer mode %d not implemented (3=sum, 4=mean)", mode);
  MM3D_REQUIRE(c == 3, MM3D_ERR_UNSUPPORTED, "masked InputLayer: 3 feature channels supported, got %d", c);
  MM3D_REQUIRE(n_points >= 0 && n_vox >= 0 && wb && (n_points == 0 || (feats && s_out)), MM3D_ERR_INVALID, "masked InputLayer: bad arguments");
  if (n_vox > 0) MM3D_CUDA(cudaMemsetAsync(out_vox, 0, sizeof(float) * (size_t)n_vox * c, stream));
  if (n_points > 0) {
    MM3D_CUDA(mm3d_launch_pdl(k_input_masked_fwd<3>, dim3(mm3d_grid(n_points, 256, 16)), dim3(256), 0, stream, feats, p2v, npts, n_points,
                              mode, wb, out_vox, s_out));
    mm3d_count_launches(1);
  }
  MM3D_CHECK_LAUNCH("mm3d_input_masked_fwd");
  return MM3D_OK;
}

// ... and its backward: d_feats [n_points, c] (may be NULL: the features are data), d_wb [c + 1] = d_w, d_b
// (overwritten); feats = the UNMASKED features, s = the gates of the forward; ws: (c + 1) doubles
// (flags MM3D_DETERMINISTIC: MM3D_DET_CTAS * (c + 1) doubles, one row per CTA, summed in CTA order by a second launch)
extern "C" int mm3d_input_masked_bwd_ex(const float* d_vox, const float* feats, const float* s, const int32_t* p2v,
                                        const int32_t* npts, int64_t n_points, int c, int mode, const float* wb, float* d_feats,
                                        float* d_wb, void* ws, size_t ws_bytes, mm3d_stream_t stream_, int flags) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(mode == 3 || mode == 4, MM3D_ERR_UNSUPPORTED, "InputLayer mode %d not implemented", mode);
  MM3D_REQUIRE(c == 3, MM3D_ERR_UNSUPPORTED, "masked InputLayer: 3 feature channels supported, got %d", c);
  MM3D_REQUIRE((flags & ~MM3D_DETERMINISTIC) == 0, MM3D_ERR_INVALID, "masked InputLayer: unknown flags %#x", flags);
  const bool det = flags & MM3D_DETERMINISTIC;
  MM3D_REQUIRE(d_wb && wb && ws && ws_bytes >= sizeof(double) * (size_t)(c + 1) * (det ? MM3D_DET_CTAS : 1), MM3D_ERR_WORKSPACE,
               "masked InputLayer: workspace too small");
  if (det) {
    const int64_t g = mm3d_grid(n_points, 256, 8);
    const int grid = n_points > 0 ? (int)(g < MM3D_DET_CTAS ? g : MM3D_DET_CTAS) : 0;
    if (n_points > 0) {
      MM3D_REQUIRE(d_vox && feats && s, MM3D_ERR_INVALID, "masked InputLayer: null pointer");
      MM3D_CUDA(mm3d_launch_pdl(k_input_masked_bwd<3, true>, dim3(grid), dim3(256), 0, stream, d_vox, feats, s, p2v, npts,
                                n_points, mode, wb, d_feats, (double*)ws));
      mm3d_count_launches(1);
    }
    const int rc = mm3d_det_sum_parts((const double*)ws, grid, c + 1, d_wb, stream);
    if (rc) return rc;
    MM3D_CHECK_LAUNCH("mm3d_input_masked_bwd_ex");
    return MM3D_OK;
  }
  MM3D_CUDA(cudaMemsetAsync(ws, 0, sizeof(double) * (size_t)(c + 1), stream));
  if (n_points > 0) {
    MM3D_REQUIRE(d_vox && feats && s, MM3D_ERR_INVALID, "masked InputLayer: null pointer");
    MM3D_CUDA(mm3d_launch_pdl(k_input_masked_bwd<3, false>, dim3(mm3d_grid(n_points, 256, 8)), dim3(256), 0, stream, d_vox, feats, s, p2v, npts,
                              n_points, mode, wb, d_feats, (double*)ws));
    mm3d_count_launches(1);
  }
  MM3D_CUDA(mm3d_launch_pdl(k_f64_to_f32_io, dim3(1), dim3(32), 0, stream, (const double*)ws, d_wb, c + 1));
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_input_masked_bwd");
  return MM3D_OK;
}

extern "C" int mm3d_input_masked_bwd(const float* d_vox, const float* feats, const float* s, const int32_t* p2v,
                                     const int32_t* npts, int64_t n_points, int c, int mode, const float* wb, float* d_feats,
                                     float* d_wb, void* ws, size_t ws_bytes, mm3d_stream_t stream) {
  return mm3d_input_masked_bwd_ex(d_vox, feats, s, p2v, npts, n_points, c, mode, wb, d_feats, d_wb, ws, ws_bytes, stream, 0);
}

extern "C" int mm3d_output_fwd(const float* vox, const int32_t* p2v, int64_t n_points, int c, float* out,
                               mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (n_points > 0) {
    const int sft = (c % 4 == 0) ? pow2_shift(c / 4) : -1;
    const bool vec = sft >= 0 && (((uintptr_t)vox | (uintptr_t)out) & 15) == 0;
    if (vec)  // a quarter of the threads of one-float4-per-thread: every thread keeps 4 float4 in flight
      MM3D_CUDA(mm3d_launch_pdl(k_output_fwd<4>, dim3(mm3d_grid(n_points * (c / 4) / 4 + 1, 256, 16)), dim3(256), 0, stream, vox, p2v,
                                n_points, c / 4, sft, out));
    else
      MM3D_CUDA(mm3d_launch_pdl(k_output_fwd<1>, dim3(mm3d_grid(n_points * c, 256)), dim3(256), 0, stream, vox, p2v, n_points, c, 0, out));
  }
  mm3d_count_launches(n_points > 0 ? 1 : 0);
  MM3D_CHECK_LAUNCH("mm3d_output_fwd");
  return MM3D_OK;
}

extern "C" int mm3d_output_bwd(const float* d_out, const int32_t* p2v, int64_t n_points, int64_t n_vox, int c,
                               float* d_vox, mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (n_vox > 0) MM3D_CUDA(cudaMemsetAsync(d_vox, 0, sizeof(float) * (size_t)n_vox * c, stream));
  if (n_points > 0) {
    const int sft = (c % 4 == 0) ? pow2_shift(c / 4) : -1;
    const bool vec = sft >= 0 && (((uintptr_t)d_vox | (uintptr_t)d_out) & 15) == 0;
    if (vec)
      MM3D_CUDA(mm3d_launch_pdl(k_output_bwd<4>, dim3(mm3d_grid(n_points * (c / 4), 256, 16)), dim3(256), 0, stream, d_out, p2v, n_points,
                                c / 4, sft, d_vox));
    else
      MM3D_CUDA(mm3d_launch_pdl(k_output_bwd<1>, dim3(mm3d_grid(n_points * c, 256)), dim3(256), 0, stream, d_out, p2v, n_points, c, 0, d_vox));
  }
  mm3d_count_launches(n_points > 0 ? 1 : 0);
  MM3D_CHECK_LAUNCH("mm3d_output_bwd");
  return MM3D_OK;
}

// strides in ELEMENTS of the [B, C, H, W] map (a contiguous NCHW map: C*H*W, H*W, W, 1; channels-last: H*W*C, 1, W*C, C)
extern "C" int mm3d_lift2d_fwd(const void* fmap, int dtype, int B, int C, int H, int W, int64_t sb, int64_t sc, int64_t sh,
                               int64_t sw, const int64_t* idx, const int64_t* sample_offsets, int64_t n, void* out,
                               mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && n >= 0, MM3D_ERR_INVALID, "bad lift sizes");
  MM3D_REQUIRE(sb > 0 && sc > 0 && sh > 0 && sw > 0, MM3D_ERR_INVALID, "bad lift strides");
  if (n == 0) return MM3D_OK;
  int* err = mm3d_device_err_flag();
  MM3D_REQUIRE((((uintptr_t)idx) & 15) == 0, MM3D_ERR_INVALID, "lift: the index array must be 16-byte aligned");
  switch (dtype) {
    case 0: LIFT_DISPATCH(k_lift_fwd, float, (const float*)fmap, B, C, H, W, sb, sc, sh, sw, idx, sample_offsets, n, (float*)out, err); break;
    case 1: LIFT_DISPATCH(k_lift_fwd, __half, (const __half*)fmap, B, C, H, W, sb, sc, sh, sw, idx, sample_offsets, n, (__half*)out, err); break;
    case 2: LIFT_DISPATCH(k_lift_fwd, __nv_bfloat16, (const __nv_bfloat16*)fmap, B, C, H, W, sb, sc, sh, sw, idx, sample_offsets, n, (__nv_bfloat16*)out, err); break;
    default: MM3D_REQUIRE(false, MM3D_ERR_UNSUPPORTED, "lift dtype %d (0=f32,1=f16,2=bf16)", dtype);
  }
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_lift2d_fwd");
  return MM3D_OK;
}

extern "C" int mm3d_lift2d_bwd(const void* d_out, int dtype, int B, int C, int H, int W, int64_t sb, int64_t sc, int64_t sh,
                               int64_t sw, const int64_t* idx, const int64_t* sample_offsets, int64_t n, void* d_fmap,
                               mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && n >= 0, MM3D_ERR_INVALID, "bad lift sizes");
  MM3D_REQUIRE(sb > 0 && sc > 0 && sh > 0 && sw > 0, MM3D_ERR_INVALID, "bad lift strides");
  if (n == 0) return MM3D_OK;
  int* err = mm3d_device_err_flag();
  MM3D_REQUIRE((((uintptr_t)idx) & 15) == 0, MM3D_ERR_INVALID, "lift: the index array must be 16-byte aligned");
  switch (dtype) {
    case 0: LIFT_DISPATCH(k_lift_bwd, float, (const float*)d_out, B, C, H, W, sb, sc, sh, sw, idx, sample_offsets, n, (float*)d_fmap, err); break;
    case 1: LIFT_DISPATCH(k_lift_bwd, __half, (const __half*)d_out, B, C, H, W, sb, sc, sh, sw, idx, sample_offsets, n, (__half*)d_fmap, err); break;
    case 2: LIFT_DISPATCH(k_lift_bwd, __nv_bfloat16, (const __nv_bfloat16*)d_out, B, C, H, W, sb, sc, sh, sw, idx, sample_offsets, n, (__nv_bfloat16*)d_fmap, err); break;
    default: MM3D_REQUIRE(false, MM3D_ERR_UNSUPPORTED, "lift dtype %d (0=f32,1=f16,2=bf16)", dtype);
  }
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_lift2d_bwd");
  return MM3D_OK;
}

extern "C" int mm3d_lift2d_bilinear_fwd(const void* fmap, int dtype, int B, int C, int H, int W, int64_t sb, int64_t sc,
                                        int64_t sh, int64_t sw, const float* uv, const int64_t* sample_offsets, int64_t n,
                                        void* out, mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && n >= 0, MM3D_ERR_INVALID, "bad lift sizes");
  MM3D_REQUIRE(sb > 0 && sc > 0 && sh > 0 && sw > 0, MM3D_ERR_INVALID, "bad lift strides");
  if (n == 0) return MM3D_OK;
  int* err = nullptr;
  MM3D_REQUIRE(uv && (((uintptr_t)uv) & 7) == 0, MM3D_ERR_INVALID, "lift: the coordinate array must be 8-byte aligned");
  switch (dtype) {
    case 0: LIFT_DISPATCH(k_lift_bilinear_fwd, float, (const float*)fmap, B, C, H, W, sb, sc, sh, sw, uv, sample_offsets, n, (float*)out, err); break;
    case 1: LIFT_DISPATCH(k_lift_bilinear_fwd, __half, (const __half*)fmap, B, C, H, W, sb, sc, sh, sw, uv, sample_offsets, n, (__half*)out, err); break;
    case 2: LIFT_DISPATCH(k_lift_bilinear_fwd, __nv_bfloat16, (const __nv_bfloat16*)fmap, B, C, H, W, sb, sc, sh, sw, uv, sample_offsets, n, (__nv_bfloat16*)out, err); break;
    default: MM3D_REQUIRE(false, MM3D_ERR_UNSUPPORTED, "lift dtype %d (0=f32,1=f16,2=bf16)", dtype);
  }
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_lift2d_bilinear_fwd");
  return MM3D_OK;
}

extern "C" int mm3d_lift2d_bilinear_bwd(const void* d_out, int dtype, int B, int C, int H, int W, int64_t sb, int64_t sc,
                                        int64_t sh, int64_t sw, const float* uv, const int64_t* sample_offsets, int64_t n,
                                        void* d_fmap, mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && n >= 0, MM3D_ERR_INVALID, "bad lift sizes");
  MM3D_REQUIRE(sb > 0 && sc > 0 && sh > 0 && sw > 0, MM3D_ERR_INVALID, "bad lift strides");
  if (n == 0) return MM3D_OK;
  int* err = nullptr;
  MM3D_REQUIRE(uv && (((uintptr_t)uv) & 7) == 0, MM3D_ERR_INVALID, "lift: the coordinate array must be 8-byte aligned");
  switch (dtype) {
    case 0: LIFT_DISPATCH(k_lift_bilinear_bwd, float, (const float*)d_out, B, C, H, W, sb, sc, sh, sw, uv, sample_offsets, n, (float*)d_fmap, err); break;
    case 1: LIFT_DISPATCH(k_lift_bilinear_bwd, __half, (const __half*)d_out, B, C, H, W, sb, sc, sh, sw, uv, sample_offsets, n, (__half*)d_fmap, err); break;
    case 2: LIFT_DISPATCH(k_lift_bilinear_bwd, __nv_bfloat16, (const __nv_bfloat16*)d_out, B, C, H, W, sb, sc, sh, sw, uv, sample_offsets, n, (__nv_bfloat16*)d_fmap, err); break;
    default: MM3D_REQUIRE(false, MM3D_ERR_UNSUPPORTED, "lift dtype %d (0=f32,1=f16,2=bf16)", dtype);
  }
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_lift2d_bilinear_bwd");
  return MM3D_OK;
}

// ------------------------------------------------------------------------------------------------
// Deterministic forms (MM3D_DETERMINISTIC): segmented sums over the group-by-key lists of groupby.cu
// ------------------------------------------------------------------------------------------------
extern "C" int mm3d_input_fwd_csr(const float* feats, const int32_t* vox_start, const int32_t* vox_pts, int64_t n_vox, int c,
                                  int mode, float* out_vox, mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(mode == 3 || mode == 4, MM3D_ERR_UNSUPPORTED, "InputLayer mode %d not implemented (3=sum, 4=mean)", mode);
  MM3D_REQUIRE(c > 0 && n_vox >= 0, MM3D_ERR_INVALID, "bad sizes");
  if (n_vox == 0) return MM3D_OK;
  MM3D_REQUIRE(feats && vox_start && vox_pts && out_vox, MM3D_ERR_INVALID, "input_fwd_csr: null pointer");
  MM3D_CUDA(mm3d_launch_pdl(k_input_fwd_csr, dim3(mm3d_grid(n_vox * c, 256, 16)), dim3(256), 0, stream, feats, vox_start,
                            vox_pts, n_vox, c, mode, out_vox));
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_input_fwd_csr");
  return MM3D_OK;
}

// mm3d_input_masked_fwd over the voxel point lists: one thread per voxel row, no memset, no atomics
extern "C" int mm3d_input_masked_fwd_csr(const float* feats, const int32_t* vox_start, const int32_t* vox_pts, int64_t n_vox,
                                         int c, int mode, const float* wb, float* out_vox, float* s_out, mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(mode == 3 || mode == 4, MM3D_ERR_UNSUPPORTED, "InputLayer mode %d not implemented (3=sum, 4=mean)", mode);
  MM3D_REQUIRE(c == 3, MM3D_ERR_UNSUPPORTED, "masked InputLayer: 3 feature channels supported, got %d", c);
  MM3D_REQUIRE(n_vox >= 0 && wb, MM3D_ERR_INVALID, "masked input_fwd_csr: bad arguments");
  if (n_vox == 0) return MM3D_OK;
  MM3D_REQUIRE(feats && vox_start && vox_pts && out_vox && s_out, MM3D_ERR_INVALID, "masked input_fwd_csr: null pointer");
  MM3D_CUDA(mm3d_launch_pdl(k_input_masked_fwd_csr<3>, dim3(mm3d_grid(n_vox, 256, 16)), dim3(256), 0, stream, feats, vox_start,
                            vox_pts, n_vox, mode, wb, out_vox, s_out));
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_input_masked_fwd_csr");
  return MM3D_OK;
}

extern "C" int mm3d_output_bwd_csr(const float* d_out, const int32_t* vox_start, const int32_t* vox_pts, int64_t n_vox, int c,
                                   float* d_vox, mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(c > 0 && n_vox >= 0, MM3D_ERR_INVALID, "bad sizes");
  if (n_vox == 0) return MM3D_OK;
  MM3D_REQUIRE(d_out && vox_start && vox_pts && d_vox, MM3D_ERR_INVALID, "output_bwd_csr: null pointer");
  MM3D_CUDA(mm3d_launch_pdl(k_output_bwd_csr, dim3(mm3d_grid(n_vox * c, 256, 16)), dim3(256), 0, stream, d_out, vox_start,
                            vox_pts, n_vox, c, d_vox));
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_output_bwd_csr");
  return MM3D_OK;
}

extern "C" size_t mm3d_lift_csr_workspace_bytes(int B, int H, int W, int64_t n, int bilinear) {
  const int64_t n_ent = (bilinear ? 4 : 1) * (n > 0 ? n : 1);
  return mm3d_align(sizeof(int32_t) * (size_t)n_ent) + mm3d_group_by_workspace_bytes((int64_t)B * H * W);
}

extern "C" int mm3d_lift_csr(const int64_t* idx, const float* uv, const int64_t* sample_offsets, int B, int H, int W, int64_t n,
                             int32_t* pix_start, int32_t* pix_ent, void* ws, size_t ws_bytes, mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(B > 0 && H > 0 && W > 0 && n >= 0, MM3D_ERR_INVALID, "lift_csr: bad sizes");
  MM3D_REQUIRE((idx == nullptr) != (uv == nullptr), MM3D_ERR_INVALID, "lift_csr: give exactly one of idx and uv");
  const int64_t n_pix = (int64_t)B * H * W, n_ent = (uv ? 4 : 1) * n;
  MM3D_REQUIRE(n_pix < (1ll << 31) && n_ent < (1ll << 31), MM3D_ERR_INVALID, "lift_csr: more than 2^31 pixels or entries");
  MM3D_REQUIRE(ws && ws_bytes >= mm3d_lift_csr_workspace_bytes(B, H, W, n, uv != nullptr), MM3D_ERR_WORKSPACE,
               "lift_csr: workspace too small");
  MM3D_REQUIRE(((uintptr_t)idx & 15) == 0 && ((uintptr_t)uv & 7) == 0, MM3D_ERR_INVALID, "lift_csr: misaligned idx / uv");
  int32_t* key = (int32_t*)ws;
  const size_t key_bytes = mm3d_align(sizeof(int32_t) * (size_t)(n_ent > 0 ? n_ent : 1));
  if (n > 0) {
    MM3D_REQUIRE(sample_offsets, MM3D_ERR_INVALID, "lift_csr: null sample_offsets");
    MM3D_CUDA(mm3d_launch_pdl(k_lift_keys, dim3(mm3d_grid(n, 256, 16)), dim3(256), 0, stream, idx, uv, sample_offsets, B, H, W, n,
                              key, mm3d_device_err_flag()));
    mm3d_count_launches(1);
  }
  return mm3d_group_by(key, nullptr, n_ent, n_pix, pix_start, pix_ent, (char*)ws + key_bytes, ws_bytes - key_bytes, stream);
}

#define LIFT_CSR_LAUNCH(T, BIL)                                                                                          \
  MM3D_CUDA(mm3d_launch_pdl(k_lift_bwd_csr<T, BIL>, dim3(mm3d_grid(n_pix * C, 256, 16)), dim3(256), 0, stream,           \
                            (const T*)d_out, C, H, W, sb, sc, sh, sw, uv, pix_start, pix_ent, n_pix, (T*)d_fmap))

static int lift_bwd_csr(const void* d_out, int dtype, int B, int C, int H, int W, int64_t sb, int64_t sc, int64_t sh, int64_t sw,
                        const float* uv, const int32_t* pix_start, const int32_t* pix_ent, void* d_fmap, cudaStream_t stream,
                        const char* name) {
  MM3D_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, MM3D_ERR_INVALID, "bad lift sizes");
  MM3D_REQUIRE(sb > 0 && sc > 0 && sh > 0 && sw > 0, MM3D_ERR_INVALID, "bad lift strides");
  MM3D_REQUIRE(d_out && pix_start && pix_ent && d_fmap, MM3D_ERR_INVALID, "%s: null pointer", name);
  const int64_t n_pix = (int64_t)B * H * W;
  const bool bil = uv != nullptr;
  switch (dtype) {
    case 0: if (bil) LIFT_CSR_LAUNCH(float, true); else LIFT_CSR_LAUNCH(float, false); break;
    case 1: if (bil) LIFT_CSR_LAUNCH(__half, true); else LIFT_CSR_LAUNCH(__half, false); break;
    case 2: if (bil) LIFT_CSR_LAUNCH(__nv_bfloat16, true); else LIFT_CSR_LAUNCH(__nv_bfloat16, false); break;
    default: MM3D_REQUIRE(false, MM3D_ERR_UNSUPPORTED, "lift dtype %d (0=f32,1=f16,2=bf16)", dtype);
  }
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH(name);
  return MM3D_OK;
}

extern "C" int mm3d_lift2d_bwd_csr(const void* d_out, int dtype, int B, int C, int H, int W, int64_t sb, int64_t sc, int64_t sh,
                                   int64_t sw, const int32_t* pix_start, const int32_t* pix_ent, void* d_fmap,
                                   mm3d_stream_t stream) {
  return lift_bwd_csr(d_out, dtype, B, C, H, W, sb, sc, sh, sw, nullptr, pix_start, pix_ent, d_fmap, (cudaStream_t)stream,
                      "mm3d_lift2d_bwd_csr");
}

extern "C" int mm3d_lift2d_bilinear_bwd_csr(const void* d_out, int dtype, int B, int C, int H, int W, int64_t sb, int64_t sc,
                                            int64_t sh, int64_t sw, const float* uv, const int32_t* pix_start,
                                            const int32_t* pix_ent, void* d_fmap, mm3d_stream_t stream) {
  MM3D_REQUIRE(uv && (((uintptr_t)uv) & 7) == 0, MM3D_ERR_INVALID, "lift: the coordinate array must be 8-byte aligned");
  return lift_bwd_csr(d_out, dtype, B, C, H, W, sb, sc, sh, sw, uv, pix_start, pix_ent, d_fmap, (cudaStream_t)stream,
                      "mm3d_lift2d_bilinear_bwd_csr");
}

// ------------------------------------------------------------------------------------------------
// Point values -> image: the loaders' sparse depth / 2D label maps
//     depth = zeros(H, W); depth[idx[:,0], idx[:,1]] = z            (lib/dataset/nuscenes_dataloader.py:275-278)
// numpy assigns repeated indices in order, so the LAST point of a pixel wins: pass 1 records the largest
// point index per pixel (atomicMax), pass 2 writes that point's value -- deterministic, same result.
// ------------------------------------------------------------------------------------------------
namespace {

__global__ void k_raster_fill(float* __restrict__ out, int32_t* __restrict__ winner, int64_t total, float fill) {
  mm3d_griddep_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    out[i] = fill;
    winner[i] = -1;
  }
}

__device__ __forceinline__ int64_t raster_pixel(const int64_t* __restrict__ idx, const int64_t* __restrict__ offs, int B,
                                                int H, int W, int64_t i) {
  int lo = 0, hi = B - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(offs + mid) <= i) lo = mid; else hi = mid - 1;
  }
  const int64_t r = __ldg(idx + 2 * i), c = __ldg(idx + 2 * i + 1);
  if ((uint64_t)r >= (uint64_t)H || (uint64_t)c >= (uint64_t)W) return -1;
  return ((int64_t)lo * H + r) * W + c;
}

__global__ void k_raster_winner(const int64_t* __restrict__ idx, const int64_t* __restrict__ offs, int B, int H, int W,
                                int64_t n, int32_t* __restrict__ winner) {
  mm3d_griddep_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t px = raster_pixel(idx, offs, B, H, W, i);
    if (px >= 0) atomicMax(winner + px, (int32_t)i);
  }
}

__global__ void k_raster_write(const int64_t* __restrict__ idx, const int64_t* __restrict__ offs, int B, int H, int W,
                               int64_t n, const float* __restrict__ vals, const int32_t* __restrict__ winner,
                               float* __restrict__ out) {
  mm3d_griddep_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t px = raster_pixel(idx, offs, B, H, W, i);
    if (px >= 0 && winner[px] == (int32_t)i) out[px] = __ldg(vals + i);
  }
}

}  // namespace

extern "C" size_t mm3d_raster2d_workspace_bytes(int B, int H, int W) { return mm3d_align(sizeof(int32_t) * (size_t)B * H * W); }

extern "C" int mm3d_raster2d(const int64_t* idx, const int64_t* sample_offsets, int B, int H, int W, int64_t n,
                             const float* vals, float fill, float* out, void* ws, size_t ws_bytes, mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(B > 0 && H > 0 && W > 0 && n >= 0 && n < (1ll << 31), MM3D_ERR_INVALID, "raster2d: bad sizes");
  MM3D_REQUIRE(out && ws && ws_bytes >= mm3d_raster2d_workspace_bytes(B, H, W), MM3D_ERR_WORKSPACE, "raster2d: workspace too small");
  const int64_t total = (int64_t)B * H * W;
  int32_t* winner = (int32_t*)ws;
  MM3D_CUDA(mm3d_launch_pdl(k_raster_fill, dim3(mm3d_grid(total, 256)), dim3(256), 0, stream, out, winner, total, fill));
  if (n > 0) {
    MM3D_REQUIRE(idx && sample_offsets && vals, MM3D_ERR_INVALID, "raster2d: null pointer");
    MM3D_CUDA(mm3d_launch_pdl(k_raster_winner, dim3(mm3d_grid(n, 256)), dim3(256), 0, stream, idx, sample_offsets, B, H, W, n, winner));
    MM3D_CUDA(mm3d_launch_pdl(k_raster_write, dim3(mm3d_grid(n, 256)), dim3(256), 0, stream, idx, sample_offsets, B, H, W, n, vals,
                              (const int32_t*)winner, out));
  }
  mm3d_count_launches(n > 0 ? 3 : 1);
  MM3D_CHECK_LAUNCH("mm3d_raster2d");
  return MM3D_OK;
}
