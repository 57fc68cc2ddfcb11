// FP32 SIMT rule-table convolution: the parity mode (1e-4) of the sparse convolutions.
//
//   forward / dgrad :  out[j,:] = sum_k in[tbl(j,k),:] . W'[k]        (output stationary)
//   wgrad           :  dW[k]    = sum_j in[tbl(j,k),:]^T . dout[j,:]   (pair-list reduction)
//
// Output-stationary means every output row is produced by exactly one warp, accumulated in
// registers over all K offsets and written once: no atomics, no read-modify-write of `out`
// (SparseConvNet's kernels re-read and re-write the output rows once per offset), and the
// result is bit-reproducible.  The tcgen05 kernels in conv_tc.cu share this contract.
#include "common.cuh"
#include "epilogue.cuh"

namespace {

constexpr int kRows = 8;        // output rows per warp
constexpr int kWarps = 4;       // warps per CTA
constexpr int kFwdThreads = kWarps * 32;

__device__ __forceinline__ int table_lookup(const int32_t* __restrict__ tbl, int64_t tbl_stride,
                                            const uint8_t* __restrict__ onehot_off, int64_t j, int k) {
  if (onehot_off) return (int)__ldg(onehot_off + j) == k ? __ldg(tbl + j) : -1;
  return __ldg(tbl + (int64_t)k * tbl_stride + j);
}

// W' = per-offset transpose (and optional offset mirror) of the forward layer's weight:
// wt[k][ci][co] = w[ksel][co][ci], ci < c_in, co < c_out, ksel = mirror ? K-1-k : k
__global__ void k_weight_transpose(const float* __restrict__ w, float* __restrict__ wt, int K, int c_in,
                                   int c_out, int mirror) {
  const int64_t total = (int64_t)K * c_in * c_out;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int co = (int)(i % c_out);
    const int ci = (int)((i / c_out) % c_in);
    const int k = (int)(i / ((int64_t)c_out * c_in));
    const int ks = mirror ? K - 1 - k : k;
    wt[i] = __ldg(w + ((int64_t)ks * c_out + co) * c_in + ci);
  }
}

// Epi: empty (the default kernel) or one ConvEpi (the inference form: the value goes to its destinations, not to `out`)
template <int CPL, class... Epi>
__global__ void __launch_bounds__(kFwdThreads)
k_conv_fwd_simt(const float* __restrict__ in, float* __restrict__ out, const float* __restrict__ W,
                const int32_t* __restrict__ tbl, int64_t tbl_stride, const uint8_t* __restrict__ onehot_off,
                int64_t n_out, int c_in, int c_out, int K, const float* add, const __grid_constant__ Epi... epi) {
  extern __shared__ __align__(16) float s_rows[];  // [kWarps][kRows][c_in]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* a = s_rows + (size_t)warp * kRows * c_in;
  const bool vec = (c_in & 3) == 0;

  for (int64_t j0 = ((int64_t)blockIdx.x * kWarps + warp) * kRows; j0 < n_out;
       j0 += (int64_t)gridDim.x * kWarps * kRows) {
    float acc[kRows][CPL];
#pragma unroll
    for (int r = 0; r < kRows; ++r)
#pragma unroll
      for (int j = 0; j < CPL; ++j) acc[r][j] = 0.f;

    for (int k = 0; k < K; ++k) {
      int nb = -1;
      if (lane < kRows && j0 + lane < n_out) nb = table_lookup(tbl, tbl_stride, onehot_off, j0 + lane, k);
      const unsigned mask = __ballot_sync(0xffffffffu, nb >= 0);
      if (mask == 0) continue;
      // stage the present input rows of this offset (coalesced row copies)
#pragma unroll
      for (int r = 0; r < kRows; ++r) {
        const int src = __shfl_sync(0xffffffffu, nb, r);
        if (mask & (1u << r)) {
          const float* p = in + (int64_t)src * c_in;
          if (vec) {
            for (int c = lane; c < (c_in >> 2); c += 32)
              reinterpret_cast<float4*>(a + r * c_in)[c] = __ldg(reinterpret_cast<const float4*>(p) + c);
          } else {
            for (int c = lane; c < c_in; c += 32) a[r * c_in + c] = __ldg(p + c);
          }
        }
      }
      __syncwarp();
      const float* Wk = W + (int64_t)k * c_in * c_out;
      if (vec) {
        for (int ci = 0; ci < c_in; ci += 4) {
          float w[4][CPL];
#pragma unroll
          for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int j = 0; j < CPL; ++j) {
              const int co = lane + 32 * j;
              w[q][j] = co < c_out ? __ldg(Wk + (int64_t)(ci + q) * c_out + co) : 0.f;
            }
#pragma unroll
          for (int r = 0; r < kRows; ++r) {
            if (mask & (1u << r)) {
              const float4 av = *reinterpret_cast<const float4*>(a + r * c_in + ci);
#pragma unroll
              for (int j = 0; j < CPL; ++j) {
                acc[r][j] = fmaf(av.x, w[0][j], acc[r][j]);
                acc[r][j] = fmaf(av.y, w[1][j], acc[r][j]);
                acc[r][j] = fmaf(av.z, w[2][j], acc[r][j]);
                acc[r][j] = fmaf(av.w, w[3][j], acc[r][j]);
              }
            }
          }
        }
      } else {
        for (int ci = 0; ci < c_in; ++ci) {
          float w[CPL];
#pragma unroll
          for (int j = 0; j < CPL; ++j) {
            const int co = lane + 32 * j;
            w[j] = co < c_out ? __ldg(Wk + (int64_t)ci * c_out + co) : 0.f;
          }
#pragma unroll
          for (int r = 0; r < kRows; ++r) {
            if (mask & (1u << r)) {
              const float av = a[r * c_in + ci];
#pragma unroll
              for (int j = 0; j < CPL; ++j) acc[r][j] = fmaf(av, w[j], acc[r][j]);
            }
          }
        }
      }
      __syncwarp();
    }
#pragma unroll
    for (int r = 0; r < kRows; ++r) {
      if (j0 + r < n_out) {
#pragma unroll
        for (int j = 0; j < CPL; ++j) {
          const int co = lane + 32 * j;
          if (co < c_out) {
            const int64_t o = (j0 + r) * c_out + co;
            if constexpr (sizeof...(Epi) > 0) {
              const float v[1] = {add ? add[o] + acc[r][j] : acc[r][j]};
              (epi_store<1>(epi, j0 + r, co, v), ...);
            } else {
              out[o] = add ? add[o] + acc[r][j] : acc[r][j];  // (add may be `out`: each element is read, then written once)
            }
          }
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------ wgrad
constexpr int kWgThreads = 256;  // 16 (ci groups) x 16 (co groups)
constexpr int kPairBatch = 32;
constexpr int kMaxTI = 12;       // c_in  <= 192
constexpr int kMaxTJ = 8;        // c_out <= 128

template <int TI, int TJ>
__global__ void __launch_bounds__(kWgThreads)
k_conv_wgrad_simt(const float* __restrict__ in, const float* __restrict__ dout, float* __restrict__ dW,
                  const int32_t* __restrict__ tbl, int64_t tbl_stride, const uint8_t* __restrict__ onehot_off,
                  int64_t n_out, int c_in, int c_out, int rows_per_chunk) {
  extern __shared__ __align__(16) float s_wg[];  // A[kPairBatch][c_in] | D[kPairBatch][c_out]
  __shared__ int s_pair_in[kWgThreads], s_pair_out[kWgThreads];
  __shared__ int s_warp_cnt[kWgThreads / 32];
  float* sA = s_wg;
  float* sD = s_wg + kPairBatch * c_in;
  const int k = blockIdx.y;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t row_begin = (int64_t)blockIdx.x * rows_per_chunk;
  const int64_t row_end = row_begin + rows_per_chunk < n_out ? row_begin + rows_per_chunk : n_out;

  float acc[TI][TJ];
#pragma unroll
  for (int i = 0; i < TI; ++i)
#pragma unroll
    for (int j = 0; j < TJ; ++j) acc[i][j] = 0.f;

  for (int64_t base = row_begin; base < row_end; base += kWgThreads) {
    // compact the present pairs of this offset among 256 consecutive output rows
    const int64_t j = base + threadIdx.x;
    const int nb = j < row_end ? table_lookup(tbl, tbl_stride, onehot_off, j, k) : -1;
    const unsigned bal = __ballot_sync(0xffffffffu, nb >= 0);
    if (lane == 0) s_warp_cnt[warp] = __popc(bal);
    __syncthreads();
    int woff = 0, total = 0;
#pragma unroll
    for (int w = 0; w < kWgThreads / 32; ++w) {
      const int cnt = s_warp_cnt[w];
      if (w < warp) woff += cnt;
      total += cnt;
    }
    if (nb >= 0) {
      const int pos = woff + __popc(bal & ((1u << lane) - 1));
      s_pair_in[pos] = nb;
      s_pair_out[pos] = (int)(j - base);
    }
    __syncthreads();
    for (int b0 = 0; b0 < total; b0 += kPairBatch) {
      const int nb_pairs = total - b0 < kPairBatch ? total - b0 : kPairBatch;
      // stage the batch: pair p is copied by 8 lanes, 16-byte pieces of the input row and then of
      // the d_out row interleaved over the lanes, four loads in flight per thread
      if (((c_in | c_out) & 3) == 0) {
        const int p = threadIdx.x >> 3, l8 = threadIdx.x & 7;
        if (p < nb_pairs) {
          const float4* src_a = reinterpret_cast<const float4*>(in + (int64_t)s_pair_in[b0 + p] * c_in);
          const float4* src_d = reinterpret_cast<const float4*>(dout + (base + s_pair_out[b0 + p]) * c_out);
          float4* dst_a = reinterpret_cast<float4*>(sA + p * c_in);
          float4* dst_d = reinterpret_cast<float4*>(sD + p * c_out);
          const int qa = c_in >> 2, qt = (c_in + c_out) >> 2;
          for (int c0 = l8; c0 < qt; c0 += 32) {
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int c = c0 + 8 * u;
              if (c < qt) v[u] = c < qa ? __ldg(src_a + c) : __ldg(src_d + (c - qa));
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int c = c0 + 8 * u;
              if (c < qt) {
                if (c < qa) dst_a[c] = v[u]; else dst_d[c - qa] = v[u];
              }
            }
          }
        }
      } else {
        for (int p = warp; p < nb_pairs; p += kWgThreads / 32) {
          const float* src_a = in + (int64_t)s_pair_in[b0 + p] * c_in;
          const float* src_d = dout + (base + s_pair_out[b0 + p]) * c_out;
          for (int c = lane; c < c_in; c += 32) sA[p * c_in + c] = __ldg(src_a + c);
          for (int c = lane; c < c_out; c += 32) sD[p * c_out + c] = __ldg(src_d + c);
        }
      }
      __syncthreads();
      for (int p = 0; p < nb_pairs; ++p) {
        float av[TI], dv[TJ];
#pragma unroll
        for (int i = 0; i < TI; ++i) { const int ci = ty + 16 * i; av[i] = ci < c_in ? sA[p * c_in + ci] : 0.f; }
#pragma unroll
        for (int jj = 0; jj < TJ; ++jj) { const int co = tx + 16 * jj; dv[jj] = co < c_out ? sD[p * c_out + co] : 0.f; }
#pragma unroll
        for (int i = 0; i < TI; ++i)
#pragma unroll
          for (int jj = 0; jj < TJ; ++jj) acc[i][jj] = fmaf(av[i], dv[jj], acc[i][jj]);
      }
      __syncthreads();
    }
  }
  float* dWk = dW + (int64_t)k * c_in * c_out;
#pragma unroll
  for (int i = 0; i < TI; ++i) {
    const int ci = ty + 16 * i;
    if (ci < c_in) {
#pragma unroll
      for (int jj = 0; jj < TJ; ++jj) {
        const int co = tx + 16 * jj;
        if (co < c_out && acc[i][jj] != 0.f) atomicAdd(dWk + (int64_t)ci * c_out + co, acc[i][jj]);
      }
    }
  }
}

template <int TI>
int launch_wgrad_tj(int tj, dim3 grid, size_t smem, cudaStream_t stream, const float* in, const float* dout,
                    float* dW, const int32_t* tbl, int64_t tbl_stride, const uint8_t* onehot_off, int64_t n_out,
                    int c_in, int c_out, int rows_per_chunk) {
#define WG_CASE(TJ)                                                                                          \
  case TJ:                                                                                                   \
    k_conv_wgrad_simt<TI, TJ><<<grid, kWgThreads, smem, stream>>>(in, dout, dW, tbl, tbl_stride, onehot_off,   \
                                                                 n_out, c_in, c_out, rows_per_chunk);        \
    return 0;
  switch (tj) {
    WG_CASE(1) WG_CASE(2) WG_CASE(3) WG_CASE(4) WG_CASE(5) WG_CASE(6) WG_CASE(7) WG_CASE(8)
  }
#undef WG_CASE
  return 1;
}

}  // namespace

// ---- host entry points used by capi.cu -------------------------------------------------------

size_t mm3d_conv_simt_workspace_bytes(int c_in, int c_out, int K) {
  return mm3d_align(sizeof(float) * (size_t)K * c_in * c_out);  // transposed weights for dgrad
}

int mm3d_conv_fwd_simt(const float* in, int64_t n_in, int c_in, float* out, int64_t n_out, int c_out,
                       const float* weight, int K, const int32_t* tbl, int64_t tbl_stride,
                       const uint8_t* onehot_off, int flags, void* ws, size_t ws_bytes, cudaStream_t stream,
                       const float* add, const ConvEpi* epi) {
  (void)n_in;
  MM3D_REQUIRE(c_out <= 32 * 8, MM3D_ERR_UNSUPPORTED, "SIMT conv: c_out %d > 256", c_out);
  MM3D_REQUIRE(c_in <= 384, MM3D_ERR_UNSUPPORTED, "SIMT conv: c_in %d > 384", c_in);
  if (n_out == 0) return MM3D_OK;
  const float* W = weight;
  if (flags & (MM3D_CONV_TRANSPOSE_W | MM3D_CONV_MIRROR_K)) {
    MM3D_REQUIRE(flags & MM3D_CONV_TRANSPOSE_W, MM3D_ERR_UNSUPPORTED, "MIRROR_K without TRANSPOSE_W not implemented");
    MM3D_REQUIRE(ws && ws_bytes >= mm3d_conv_simt_workspace_bytes(c_in, c_out, K), MM3D_ERR_WORKSPACE,
                 "conv workspace too small");
    float* wt = (float*)ws;
    k_weight_transpose<<<mm3d_grid((int64_t)K * c_in * c_out, 256), 256, 0, stream>>>(
        weight, wt, K, c_in, c_out, (flags & MM3D_CONV_MIRROR_K) ? 1 : 0);
    W = wt;
  }
  const int cpl = (c_out + 31) / 32;
  const size_t smem = sizeof(float) * kWarps * kRows * (size_t)c_in;
  const int grid = mm3d_grid(mm3d_cdiv(n_out, kRows) * 32, kFwdThreads, 16);
#define FWD_CASE(CPL)                                                                                       \
  case CPL:                                                                                                 \
    if (epi)                                                                                                \
      k_conv_fwd_simt<CPL, ConvEpi><<<grid, kFwdThreads, smem, stream>>>(in, out, W, tbl, tbl_stride, onehot_off, \
                                                                        n_out, c_in, c_out, K, add, *epi);       \
    else                                                                                                    \
      k_conv_fwd_simt<CPL><<<grid, kFwdThreads, smem, stream>>>(in, out, W, tbl, tbl_stride, onehot_off, n_out, \
                                                               c_in, c_out, K, add);                             \
    break;
  switch (cpl) {
    FWD_CASE(1) FWD_CASE(2) FWD_CASE(3) FWD_CASE(4) FWD_CASE(5) FWD_CASE(6) FWD_CASE(7) FWD_CASE(8)
    default: MM3D_REQUIRE(false, MM3D_ERR_UNSUPPORTED, "SIMT conv: c_out %d", c_out);
  }
#undef FWD_CASE
  mm3d_count_launches(W == weight ? 1 : 2);
  MM3D_CHECK_LAUNCH("mm3d_conv_fwd_simt");
  return MM3D_OK;
}

int mm3d_conv_wgrad_simt(const float* in, int64_t n_in, int c_in, const float* d_out, int64_t n_out, int c_out,
                         float* d_weight, int K, const int32_t* tbl, int64_t tbl_stride,
                         const uint8_t* onehot_off, int accumulate, cudaStream_t stream) {
  (void)n_in;
  MM3D_REQUIRE(c_in <= 16 * kMaxTI && c_out <= 16 * kMaxTJ, MM3D_ERR_UNSUPPORTED,
               "SIMT wgrad: channels (%d,%d) beyond (192,128)", c_in, c_out);
  if (!accumulate) MM3D_CUDA(cudaMemsetAsync(d_weight, 0, sizeof(float) * (size_t)K * c_in * c_out, stream));
  if (n_out == 0) return MM3D_OK;
  int ti = (c_in + 15) / 16, tj = (c_out + 15) / 16;
  if (ti == 9 || ti == 11) ++ti;  // only even tile heights are instantiated above 8
  // Row chunks of 2048: the pairs of a 3^3 table are very unevenly spread over the offsets (the
  // centre offset alone holds every row), so many small (chunk, offset) CTAs balance far better
  // than a few big ones; CTAs whose offset has no pair in the chunk exit without touching d_weight.
  int rows_per_chunk = 2048;
  while (rows_per_chunk > kWgThreads && mm3d_cdiv(n_out, rows_per_chunk) * K < 4 * MM3D_NUM_SMS) rows_per_chunk >>= 1;
  const int64_t chunks = mm3d_cdiv(n_out, rows_per_chunk);
  dim3 grid((unsigned)chunks, (unsigned)K);
  const size_t smem = sizeof(float) * kPairBatch * (size_t)(c_in + c_out);
  int miss = 1;
#define WG_TI(TI)                                                                                           \
  case TI:                                                                                                  \
    miss = launch_wgrad_tj<TI>(tj, grid, smem, stream, in, d_out, d_weight, tbl, tbl_stride, onehot_off,     \
                               n_out, c_in, c_out, rows_per_chunk);                                         \
    break;
  switch (ti) {
    WG_TI(1) WG_TI(2) WG_TI(3) WG_TI(4) WG_TI(5) WG_TI(6) WG_TI(7) WG_TI(8) WG_TI(10) WG_TI(12)
  }
#undef WG_TI
  MM3D_REQUIRE(miss == 0, MM3D_ERR_UNSUPPORTED, "SIMT wgrad: no kernel for channels (%d,%d)", c_in, c_out);
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_conv_wgrad_simt");
  return MM3D_OK;
}
