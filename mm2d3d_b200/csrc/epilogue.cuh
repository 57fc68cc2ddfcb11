// Convolution epilogue destinations of the inference forward (unet_exec.cu mm3d_unet_topo_infer).
//
// The epilogue value of a convolution is v = acc (+ add).  Instead of one plain store of v, an inference-form kernel
// writes it to up to kEpiDsts destinations, each one column block of a row-major tensor:
//   raw: v;   bn: o = fmaf(v - mean, scale, beta), o > 0 ? o : o * 0.f  (eval-mode BatchNorm + ReLU, scale =
//   rsqrtf(running_var + eps) * gamma) -- the float operations of bnrelu.cu k_bn_apply, so the stored bits are the ones
// a plain store followed by that kernel gives;
// stored in one of the store_planes forms of bnrelu.cu (0 as is, 1 TF32-rounded, 2 TF32x3 hi / lo planes, 3 TF32 FP32
// plane + BF16 plane), or 4: the BF16 plane only (the inference forward gathers nothing else in the BF16 mode).
#pragma once

#include <cuda_bf16.h>

#include "common.cuh"

constexpr int kEpiDsts = 3;

struct EpiDst {
  float* p;          // FP32 (hi) plane at the block's first column, rows `ld` floats apart (unused in store mode 4)
  void* p2;          // lo plane (store 2) or BF16 plane (3, 4) at the block's first column, indexed like `p`
  const float* mean;  // bn: running mean, scale and beta of the block's channels; NULL = raw
  const float* scale;
  const float* beta;
  int ld;
  int store;
};

struct ConvEpi {
  EpiDst d[kEpiDsts];
  int n;  // destinations in use
};

// one destination
template <int VEC>
__device__ __forceinline__ void epi_store_one(const EpiDst& d, int64_t row, int c, const float (&v)[VEC]) {
  {
    float o[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) o[j] = v[j];
    if (d.mean) {
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const float t = fmaf(o[j] - __ldg(d.mean + c + j), __ldg(d.scale + c + j), __ldg(d.beta + c + j));
        o[j] = t > 0.f ? t : t * 0.f;
      }
    }
    const int64_t at = row * d.ld + c;
    if (d.store >= 3) {
      __nv_bfloat16* b = reinterpret_cast<__nv_bfloat16*>(d.p2) + at;
      if (VEC == 4) {
        const __nv_bfloat162 b01 = __floats2bfloat162_rn(o[0], o[1 % VEC]), b23 = __floats2bfloat162_rn(o[2 % VEC], o[3 % VEC]);
        uint2 u;
        u.x = *reinterpret_cast<const unsigned int*>(&b01);
        u.y = *reinterpret_cast<const unsigned int*>(&b23);
        *reinterpret_cast<uint2*>(b) = u;
      } else {
#pragma unroll
        for (int j = 0; j < VEC; ++j) b[j] = __float2bfloat16_rn(o[j]);
      }
      if (d.store == 4) return;
    }
    float lo[VEC];
    if (d.store >= 1) {
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const float hi = mm3d_rna_tf32(o[j]);
        lo[j] = mm3d_rna_tf32(o[j] - hi);
        o[j] = hi;
      }
    }
    if (VEC == 4) {
      *reinterpret_cast<float4*>(d.p + at) = make_float4(o[0], o[1 % VEC], o[2 % VEC], o[3 % VEC]);
      if (d.store == 2) *reinterpret_cast<float4*>(reinterpret_cast<float*>(d.p2) + at) = make_float4(lo[0], lo[1 % VEC], lo[2 % VEC], lo[3 % VEC]);
    } else {
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        d.p[at + j] = o[j];
        if (d.store == 2) reinterpret_cast<float*>(d.p2)[at + j] = lo[j];
      }
    }
  }
}

// v: VEC consecutive channels c.. of row `row`, to every destination of e
template <int VEC>
__device__ __forceinline__ void epi_store(const ConvEpi& e, int64_t row, int c, const float (&v)[VEC]) {
#pragma unroll
  for (int i = 0; i < kEpiDsts; ++i)
    if (i < e.n) epi_store_one<VEC>(e.d[i], row, c, v);
}

// the destinations of e from column c0 on: the epilogue of a column slice (the wide layers' slicing) indexes its own
// columns from 0
inline ConvEpi epi_columns(const ConvEpi& e, int c0) {
  ConvEpi r = e;
  for (int i = 0; i < r.n; ++i) {
    EpiDst& d = r.d[i];
    if (d.p) d.p += c0;
    if (d.store == 2) d.p2 = reinterpret_cast<float*>(d.p2) + c0;
    if (d.store >= 3) d.p2 = reinterpret_cast<__nv_bfloat16*>(d.p2) + c0;
    if (d.mean) { d.mean += c0; d.scale += c0; d.beta += c0; }
  }
  return r;
}
