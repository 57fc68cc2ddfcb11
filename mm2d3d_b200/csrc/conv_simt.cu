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
// kStrided: a column slice of a wider layer, W rows ld_w and out / add rows ld_out floats apart (otherwise both c_out;
// the layers of up to 256 columns keep the code they have without slicing)
template <int CPL, bool kStrided, class... Epi>
__global__ void __launch_bounds__(kFwdThreads)
k_conv_fwd_simt(const float* __restrict__ in, float* __restrict__ out, const float* __restrict__ W,
                const int32_t* __restrict__ tbl, int64_t tbl_stride, const uint8_t* __restrict__ onehot_off,
                int64_t n_out, int c_in, int c_out, int ld_w, int ld_out, int K, const float* add,
                const __grid_constant__ Epi... epi) {
  extern __shared__ __align__(16) float s_rows[];  // [kWarps][kRows][c_in]
  if constexpr (!kStrided) ld_w = ld_out = c_out;
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
      const float* Wk = W + (int64_t)k * c_in * ld_w;
      if (vec) {
        for (int ci = 0; ci < c_in; ci += 4) {
          float w[4][CPL];
#pragma unroll
          for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int j = 0; j < CPL; ++j) {
              const int co = lane + 32 * j;
              w[q][j] = co < c_out ? __ldg(Wk + (int64_t)(ci + q) * ld_w + co) : 0.f;
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
            w[j] = co < c_out ? __ldg(Wk + (int64_t)ci * ld_w + co) : 0.f;
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
            const int64_t o = (j0 + r) * ld_out + co;
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
constexpr int kMaxTJ = 8;        // c_out <= 128 (wider layers: tiles of at most that, mm3d_conv_wgrad_simt)
constexpr int kSimtWide = 512;   // the widest layer either kernel takes, as slices

// kStrided: a tile of a wider layer, rows ld_in / ld_dout floats apart, dW[k][ci][co] at dW + k dw_k + ci dw_ld + co
// (otherwise c_in, c_out, c_in c_out and c_out: the layers of up to (192, 128) channels keep their code)
template <int TI, int TJ, bool kStrided = false>
__global__ void __launch_bounds__(kWgThreads)
k_conv_wgrad_simt(const float* __restrict__ in, const float* __restrict__ dout, float* __restrict__ dW,
                  const int32_t* __restrict__ tbl, int64_t tbl_stride, const uint8_t* __restrict__ onehot_off,
                  int64_t n_out, int c_in, int c_out, int ld_in, int ld_dout, int64_t dw_k, int dw_ld, int rows_per_chunk) {
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
      if ((((kStrided ? ld_in | ld_dout : 0) | c_in | c_out) & 3) == 0) {
        const int p = threadIdx.x >> 3, l8 = threadIdx.x & 7;
        if (p < nb_pairs) {
          const float4* src_a = reinterpret_cast<const float4*>(in + (int64_t)s_pair_in[b0 + p] * (kStrided ? ld_in : c_in));
          const float4* src_d = reinterpret_cast<const float4*>(dout + (base + s_pair_out[b0 + p]) * (kStrided ? ld_dout : c_out));
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
          const float* src_a = in + (int64_t)s_pair_in[b0 + p] * (kStrided ? ld_in : c_in);
          const float* src_d = dout + (base + s_pair_out[b0 + p]) * (kStrided ? ld_dout : c_out);
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
  float* dWk = kStrided ? dW + k * dw_k : dW + (int64_t)k * c_in * c_out;
#pragma unroll
  for (int i = 0; i < TI; ++i) {
    const int ci = ty + 16 * i;
    if (ci < c_in) {
#pragma unroll
      for (int jj = 0; jj < TJ; ++jj) {
        const int co = tx + 16 * jj;
        if (co < c_out && acc[i][jj] != 0.f) atomicAdd(dWk + (int64_t)ci * (kStrided ? dw_ld : c_out) + co, acc[i][jj]);
      }
    }
  }
}

template <int TI>
int launch_wgrad_tj(int tj, dim3 grid, size_t smem, cudaStream_t stream, const float* in, const float* dout,
                    float* dW, const int32_t* tbl, int64_t tbl_stride, const uint8_t* onehot_off, int64_t n_out,
                    int c_in, int c_out, int ld_in, int ld_dout, int64_t dw_k, int dw_ld, int rows_per_chunk) {
#define WG_CASE(TJ)                                                                                          \
  case TJ:                                                                                                   \
    k_conv_wgrad_simt<TI, TJ><<<grid, kWgThreads, smem, stream>>>(in, dout, dW, tbl, tbl_stride, onehot_off,   \
                                                                 n_out, c_in, c_out, ld_in, ld_dout, dw_k,   \
                                                                 dw_ld, rows_per_chunk);                     \
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
  MM3D_REQUIRE(c_out <= kSimtWide, MM3D_ERR_UNSUPPORTED, "SIMT conv: c_out %d > %d", c_out, kSimtWide);
  MM3D_REQUIRE(c_in <= kSimtWide, MM3D_ERR_UNSUPPORTED, "SIMT conv: c_in %d > %d", c_in, kSimtWide);
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
  // (input rows of more than 384 channels need more than the default 48 KB of dynamic shared memory)
  const size_t smem = sizeof(float) * kWarps * kRows * (size_t)c_in;
  const bool big = smem > 48 * 1024;
  using FwdK = void (*)(const float*, float*, const float*, const int32_t*, int64_t, const uint8_t*, int64_t, int, int, int,
                        int, int, const float*);
  using FwdEpiK = void (*)(const float*, float*, const float*, const int32_t*, int64_t, const uint8_t*, int64_t, int, int,
                           int, int, int, const float*, ConvEpi);
  const int grid = mm3d_grid(mm3d_cdiv(n_out, kRows) * 32, kFwdThreads, 16);
  // output columns beyond 256 (8 per lane): column slices, each reading its columns of W and writing its columns of out
  const int step = mm3d_slice_step(c_out, 32 * 8, 16);
  int launches = W == weight ? 0 : 1;
  for (int co0 = 0; co0 < c_out; co0 += step, ++launches) {
    const int w = c_out - co0 < step ? c_out - co0 : step;
    const float* a = add ? add + co0 : nullptr;
    float* o = out ? out + co0 : nullptr;
    ConvEpi e;
    if (epi) e = epi_columns(*epi, co0);
#define FWD_CASE(CPL, ST)                                                                                   \
  case CPL:                                                                                                 \
    if (epi) {                                                                                              \
      if (big) MM3D_CUDA(cudaFuncSetAttribute((const void*)(FwdEpiK)k_conv_fwd_simt<CPL, ST, ConvEpi>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      k_conv_fwd_simt<CPL, ST, ConvEpi><<<grid, kFwdThreads, smem, stream>>>(in, o, W + co0, tbl, tbl_stride, onehot_off, \
                                                                        n_out, c_in, w, c_out, c_out, K, a, e);   \
    } else {                                                                                                \
      if (big) MM3D_CUDA(cudaFuncSetAttribute((const void*)(FwdK)k_conv_fwd_simt<CPL, ST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      k_conv_fwd_simt<CPL, ST><<<grid, kFwdThreads, smem, stream>>>(in, o, W + co0, tbl, tbl_stride, onehot_off, n_out, \
                                                               c_in, w, c_out, c_out, K, a);                      \
    }                                                                                                       \
    break;
    if (w == c_out) {
      switch ((w + 31) / 32) {
        FWD_CASE(1, false) FWD_CASE(2, false) FWD_CASE(3, false) FWD_CASE(4, false)
        FWD_CASE(5, false) FWD_CASE(6, false) FWD_CASE(7, false) FWD_CASE(8, false)
        default: MM3D_REQUIRE(false, MM3D_ERR_UNSUPPORTED, "SIMT conv: c_out %d", c_out);
      }
    } else {  // (the last slice of 257..272 columns is 113..128 wide, so every width has its instantiation)
      switch ((w + 31) / 32) {
        FWD_CASE(1, true) FWD_CASE(2, true) FWD_CASE(3, true) FWD_CASE(4, true)
        FWD_CASE(5, true) FWD_CASE(6, true) FWD_CASE(7, true) FWD_CASE(8, true)
        default: MM3D_REQUIRE(false, MM3D_ERR_UNSUPPORTED, "SIMT conv: c_out %d", c_out);
      }
    }
#undef FWD_CASE
  }
  mm3d_count_launches(launches);
  MM3D_CHECK_LAUNCH("mm3d_conv_fwd_simt");
  return MM3D_OK;
}

// one launch: input channels [0, c_in) of rows ld_in floats apart, output channels [0, c_out) of rows ld_dout apart,
// dW[k][ci][co] at d_weight + k * dw_k + ci * dw_ld + co
static int wgrad_simt_tile(const float* in, int ld_in, int c_in, const float* d_out, int ld_dout, int c_out, int64_t n_out,
                           float* d_weight, int64_t dw_k, int dw_ld, int K, const int32_t* tbl, int64_t tbl_stride,
                           const uint8_t* onehot_off, cudaStream_t stream) {
  const bool strided = ld_in != c_in || ld_dout != c_out;
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
  if (strided) {
    // the tiles of a wider layer: register tiles of 4, 8 or 12 x 4 or 8 (the kernel masks the channels past c_in /
    // c_out), six instantiations instead of another eighty
#define WG_S(TI, TJ)                                                                                          \
  k_conv_wgrad_simt<TI, TJ, true><<<grid, kWgThreads, smem, stream>>>(                                         \
      in, d_out, d_weight, tbl, tbl_stride, onehot_off, n_out, c_in, c_out, ld_in, ld_dout, dw_k, dw_ld, rows_per_chunk)
    const int si = ti <= 4 ? 4 : ti <= 8 ? 8 : 12;
    if (tj <= 4) {
      if (si == 4) WG_S(4, 4); else if (si == 8) WG_S(8, 4); else WG_S(12, 4);
    } else {
      if (si == 4) WG_S(4, 8); else if (si == 8) WG_S(8, 8); else WG_S(12, 8);
    }
#undef WG_S
    mm3d_count_launches(1);
    return MM3D_OK;
  }
#define WG_TI(TI)                                                                                           \
  case TI:                                                                                                  \
    miss = launch_wgrad_tj<TI>(tj, grid, smem, stream, in, d_out, d_weight, tbl, tbl_stride, onehot_off,     \
                               n_out, c_in, c_out, ld_in, ld_dout, dw_k, dw_ld, rows_per_chunk);            \
    break;
  switch (ti) {
    WG_TI(1) WG_TI(2) WG_TI(3) WG_TI(4) WG_TI(5) WG_TI(6) WG_TI(7) WG_TI(8) WG_TI(10) WG_TI(12)
  }
#undef WG_TI
  MM3D_REQUIRE(miss == 0, MM3D_ERR_UNSUPPORTED, "SIMT wgrad: no kernel for channels (%d,%d)", c_in, c_out);
  mm3d_count_launches(1);
  return MM3D_OK;
}

int mm3d_conv_wgrad_simt(const float* in, int64_t n_in, int c_in, const float* d_out, int64_t n_out, int c_out,
                         float* d_weight, int K, const int32_t* tbl, int64_t tbl_stride,
                         const uint8_t* onehot_off, int accumulate, cudaStream_t stream) {
  (void)n_in;
  MM3D_REQUIRE(c_in <= kSimtWide && c_out <= kSimtWide, MM3D_ERR_UNSUPPORTED,
               "SIMT wgrad: channels (%d,%d) beyond (%d,%d)", c_in, c_out, kSimtWide, kSimtWide);
  if (!accumulate) MM3D_CUDA(cudaMemsetAsync(d_weight, 0, sizeof(float) * (size_t)K * c_in * c_out, stream));
  if (n_out == 0) return MM3D_OK;
  // Channels beyond (192, 128): tiles of at most that, each its own launch adding into its block of d_weight
  const int si = mm3d_slice_step(c_in, 16 * kMaxTI, 16), sj = mm3d_slice_step(c_out, 16 * kMaxTJ, 16);
  for (int ci0 = 0; ci0 < c_in; ci0 += si)
    for (int co0 = 0; co0 < c_out; co0 += sj) {
      const int rc = wgrad_simt_tile(in + ci0, c_in, c_in - ci0 < si ? c_in - ci0 : si, d_out + co0, c_out,
                                     c_out - co0 < sj ? c_out - co0 : sj, n_out, d_weight + (int64_t)ci0 * c_out + co0,
                                     (int64_t)c_in * c_out, c_out, K, tbl, tbl_stride, onehot_off, stream);
      if (rc) return rc;
    }
  MM3D_CHECK_LAUNCH("mm3d_conv_wgrad_simt");
  return MM3D_OK;
}

