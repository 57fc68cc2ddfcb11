// Point-wise prologue and loss around the 3D network (SURVEY 8(f).3):
//
//  * RGB mask (3d_net/model.py:46-48):   s = sigmoid(x . w + b);  x *= s        x [n, c] point features, c small
//  * cross-modal loss (train.py:157-184): mean over points of  sum_c q_c (log q_c - log p_c),
//        p = softmax(pred), q = softmax(target.detach())      pred, target [n, C] logits
//
// Both are a handful of small element-wise / row-reduction launches in the reference; here each direction is one
// launch, one thread per point (rows are 12-80 bytes).  HBM-bound: every tensor is read or written once.
#include "common.cuh"

namespace {

constexpr int kMaxC = 64;

// Deterministic mode (MM3D_DETERMINISTIC): instead of adding its block total to a global FP64 word atomically, every
// CTA stores it to its own slot part[blockIdx.x][...] (the in-block sum in a fixed warp order), and the finalize launch
// that converts the totals to float -- one the default path has too -- sums the slots in CTA order.  At most
// MM3D_DET_CTAS CTAs, independent of the device.
template <int NW>
__device__ __forceinline__ double block_sum_ordered(double v) {  // valid in thread 0
  __shared__ double wsum[NW];
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < NW; ++w) t += wsum[w];
  return t;
}

struct PartOuts {  // where word j of the summed slots goes: the first n[0] words to p[0], the next n[1] to p[1], ...
  float* p[4];
  int n[4];
};

__global__ void k_sum_parts(const double* __restrict__ part, int nparts, int words, double scale, PartOuts o) {
  mm3d_griddep_wait();
  for (int j = threadIdx.x; j < words; j += blockDim.x) {
    double t = 0.0;
    for (int b = 0; b < nparts; ++b) t += part[(int64_t)b * words + j];
    int k = 0, jj = j;
    while (jj >= o.n[k]) jj -= o.n[k++];
    o.p[k][jj] = (float)(t * scale);
  }
}

static inline int det_grid(int64_t g) { return (int)(g < MM3D_DET_CTAS ? g : MM3D_DET_CTAS); }

__global__ void k_rgb_mask_fwd(const float* x, int64_t n, int c, const float* __restrict__ w,
                               const float* __restrict__ b, float* y, float* __restrict__ s_out) {
  mm3d_griddep_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float xr[8];
    float acc = __ldg(b);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      xr[j] = j < c ? x[i * c + j] : 0.f;
      if (j < c) acc = fmaf(xr[j], __ldg(w + j), acc);
    }
    const float s = 1.f / (1.f + expf(-acc));
    s_out[i] = s;
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (j < c) y[i * c + j] = xr[j] * s;
  }
}

// dx = dy s + t w,  t = (dy . x) s (1 - s);   dw = sum_n t x,  db = sum_n t   (FP64 totals, one atomic per CTA)
template <bool DET>
__global__ void k_rgb_mask_bwd(const float* __restrict__ x, const float* __restrict__ s_in, const float* __restrict__ dy,
                               int64_t n, int c, const float* __restrict__ w, float* __restrict__ dx,
                               double* __restrict__ dwb) {
  mm3d_griddep_wait();
  __shared__ double red[kMaxC + 1];
  for (int j = threadIdx.x; j <= c; j += blockDim.x) red[j] = 0.0;
  __syncthreads();
  double loc[9];  // c <= 8 on this path (checked by the host)
#pragma unroll
  for (int j = 0; j < 9; ++j) loc[j] = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float s = __ldg(s_in + i);
    float g = 0.f;
    for (int j = 0; j < c; ++j) g = fmaf(__ldg(dy + i * c + j), __ldg(x + i * c + j), g);
    const float t = g * s * (1.f - s);
    if (dx)
      for (int j = 0; j < c; ++j) dx[i * c + j] = fmaf(t, __ldg(w + j), __ldg(dy + i * c + j) * s);
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (j < c) loc[j] += (double)(t * __ldg(x + i * c + j));
    loc[8] += (double)t;
  }
  if constexpr (DET) {  // dwb = this CTA's slot of c + 1 doubles; 256 threads = 8 warps
    __shared__ double wred[8][9];
#pragma unroll
    for (int j = 0; j < 9; ++j) {
      double v = loc[j];
      for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if ((threadIdx.x & 31) == 0) wred[threadIdx.x >> 5][j] = v;
    }
    __syncthreads();
    if (threadIdx.x <= c) {
      const int j = threadIdx.x == c ? 8 : threadIdx.x;
      double t = 0.0;
      for (int w = 0; w < 8; ++w) t += wred[w][j];
      dwb[(int64_t)blockIdx.x * (c + 1) + threadIdx.x] = t;
    }
  } else {
#pragma unroll
    for (int j = 0; j < 9; ++j) {
      double v = loc[j];
      for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if ((threadIdx.x & 31) == 0 && (j < c || j == 8)) atomicAdd(&red[j == 8 ? c : j], v);
    }
    __syncthreads();
    for (int j = threadIdx.x; j <= c; j += blockDim.x) atomicAdd(dwb + j, red[j]);
  }
}

__global__ void k_f64_to_f32(const double* __restrict__ src, float* __restrict__ dst, int n, double scale) {
  mm3d_griddep_wait();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[i] = (float)(src[i] * scale);
}

// one row: log-softmax of pred and target, KL term, optionally the gradient (p - q) * gscale
__device__ __forceinline__ double kl_row(const float* __restrict__ pr, const float* __restrict__ tg, int C, float* dpred,
                                         float gscale) {
  float mp = -INFINITY, mt = -INFINITY;
  for (int j = 0; j < C; ++j) { mp = fmaxf(mp, __ldg(pr + j)); mt = fmaxf(mt, __ldg(tg + j)); }
  float sp = 0.f, st = 0.f;
  for (int j = 0; j < C; ++j) { sp += expf(__ldg(pr + j) - mp); st += expf(__ldg(tg + j) - mt); }
  const float lsp = logf(sp), lst = logf(st);
  double kl = 0.0;
  for (int j = 0; j < C; ++j) {
    const float logp = __ldg(pr + j) - mp - lsp, logq = __ldg(tg + j) - mt - lst;
    const float q = expf(logq);
    if (q > 0.f) kl += (double)(q * (logq - logp));
    if (dpred) dpred[j] = (expf(logp) - q) * gscale;
  }
  return kl;
}

template <bool DET>
__global__ void k_kl_fwd(const float* __restrict__ pred, const float* __restrict__ target, int64_t n, int C,
                         double* __restrict__ total) {
  mm3d_griddep_wait();
  double loc = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    loc += kl_row(pred + i * C, target + i * C, C, nullptr, 0.f);
  if constexpr (DET) {  // total = this CTA's slot
    const double t = block_sum_ordered<8>(loc);
    if (threadIdx.x == 0) total[blockIdx.x] = t;
  } else {
    for (int o = 16; o; o >>= 1) loc += __shfl_xor_sync(0xffffffffu, loc, o);
    __shared__ double red;
    if (threadIdx.x == 0) red = 0.0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) atomicAdd(&red, loc);
    __syncthreads();
    if (threadIdx.x == 0) atomicAdd(total, red);
  }
}

__global__ void k_kl_bwd(const float* __restrict__ pred, const float* __restrict__ target, int64_t n, int C,
                         const float* __restrict__ dloss, float inv_n, float* __restrict__ dpred) {
  mm3d_griddep_wait();
  const float gs = __ldg(dloss) * inv_n;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    kl_row(pred + i * C, target + i * C, C, dpred + i * C, gs);
}


// ---- the two point-wise heads of the 3D branch and the 3D side of the cross-modal loss in one pass -----------------
//   logit1 = feat W1^T + b1                      Net3DSeg.linear           (3d_net/model.py:38,49)
//   logit2 = feat W2^T + b2                      L2G_classifier_3D.linear_point   (3d_net/model.py:73,85)
//   loss   = mean_n KL(softmax(target_n) || softmax(logit2_n))             (train.py:157-184, loss_3d)
// The reference runs two cuBLAS GEMMs over the [N, 16] features, then log_softmax, softmax, kl_div, sum, mean: seven
// launches that each read or write an [N, C] tensor.  Here the forward reads every feature row once and writes logit1
// (logit2 only if asked for); the backward reads the row, the gradient of logit1 and the target once and produces the
// feature gradient and all four parameter gradients.
constexpr int kHeadMaxF = 32, kHeadMaxC = 20, kHeadTile = 128;

struct HeadsSmem {
  float w1[kHeadMaxC * kHeadMaxF], w2[kHeadMaxC * kHeadMaxF], b1[kHeadMaxC], b2[kHeadMaxC];
};

__device__ __forceinline__ void heads_load_weights(HeadsSmem& s, int f, int C, const float* w1, const float* b1, const float* w2,
                                                   const float* b2) {
  for (int i = threadIdx.x; i < C * f; i += blockDim.x) { s.w1[i] = __ldg(w1 + i); s.w2[i] = __ldg(w2 + i); }
  for (int i = threadIdx.x; i < C; i += blockDim.x) { s.b1[i] = __ldg(b1 + i); s.b2[i] = __ldg(b2 + i); }
}

__device__ __forceinline__ void heads_row(const float* __restrict__ row, int f, float (&fr)[kHeadMaxF]) {
#pragma unroll
  for (int j = 0; j < kHeadMaxF; j += 4) {
    if (j < f) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(row + j));
      fr[j] = v.x; fr[j + 1] = v.y; fr[j + 2] = v.z; fr[j + 3] = v.w;
    } else {
      fr[j] = fr[j + 1] = fr[j + 2] = fr[j + 3] = 0.f;
    }
  }
}

__device__ __forceinline__ float heads_dot(const float (&fr)[kHeadMaxF], const float* __restrict__ w, int f, float b) {
  float acc = b;
#pragma unroll
  for (int j = 0; j < kHeadMaxF; ++j)
    if (j < f) acc = fmaf(fr[j], w[j], acc);
  return acc;
}

template <bool DET>
__global__ void __launch_bounds__(kHeadTile)
k_heads3d_fwd(const float* __restrict__ feat, int64_t n, int f, int C, const float* __restrict__ w1, const float* __restrict__ b1,
              const float* __restrict__ w2, const float* __restrict__ b2, const float* __restrict__ target,
              float* __restrict__ logit1, float* __restrict__ logit2, double* __restrict__ total) {
  __shared__ HeadsSmem s;
  __shared__ double red;
  mm3d_griddep_wait();
  heads_load_weights(s, f, C, w1, b1, w2, b2);
  if (threadIdx.x == 0) red = 0.0;
  __syncthreads();
  double loc = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float fr[kHeadMaxF];
    heads_row(feat + i * f, f, fr);
    float l2[kHeadMaxC];
    float m2 = -INFINITY, mt = -INFINITY;
#pragma unroll
    for (int c = 0; c < kHeadMaxC; ++c) {
      if (c < C) {
        logit1[i * C + c] = heads_dot(fr, s.w1 + c * f, f, s.b1[c]);
        l2[c] = heads_dot(fr, s.w2 + c * f, f, s.b2[c]);
        if (logit2) logit2[i * C + c] = l2[c];
        m2 = fmaxf(m2, l2[c]);
        if (target) mt = fmaxf(mt, __ldg(target + i * C + c));
      }
    }
    if (target) {
      float s2 = 0.f, st = 0.f;
#pragma unroll
      for (int c = 0; c < kHeadMaxC; ++c)
        if (c < C) { s2 += expf(l2[c] - m2); st += expf(__ldg(target + i * C + c) - mt); }
      const float ls2 = logf(s2), lst = logf(st);
#pragma unroll
      for (int c = 0; c < kHeadMaxC; ++c) {
        if (c < C) {
          const float logp = l2[c] - m2 - ls2, logq = __ldg(target + i * C + c) - mt - lst;
          const float q = expf(logq);
          if (q > 0.f) loc += (double)(q * (logq - logp));
        }
      }
    }
  }
  if (total && DET) {  // total = the slots, one per CTA
    const double t = block_sum_ordered<kHeadTile / 32>(loc);
    if (threadIdx.x == 0) total[blockIdx.x] = t;
  } else if (total) {
    for (int o = 16; o; o >>= 1) loc += __shfl_xor_sync(0xffffffffu, loc, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(&red, loc);
    __syncthreads();
    if (threadIdx.x == 0) atomicAdd(total, red);
  }
}

// tot: [C f | C | C f | C] doubles = d_w1, d_b1, d_w2, d_b2 (zero on entry; DET: one such slot per CTA, written)
template <bool DET>
__global__ void __launch_bounds__(kHeadTile)
k_heads3d_bwd(const float* __restrict__ feat, int64_t n, int f, int C, const float* __restrict__ w1, const float* __restrict__ w2,
              const float* __restrict__ b2, const float* __restrict__ target, const float* __restrict__ d_logit1,
              const float* __restrict__ d_logit2, const float* __restrict__ d_loss, float inv_n, float* __restrict__ d_feat,
              double* __restrict__ tot) {
  __shared__ HeadsSmem s;
  __shared__ float sd[kHeadTile][2 * kHeadMaxC + 1];  // per point of the tile: d_logit1 | d_logit2
  __shared__ float sf[kHeadTile][kHeadMaxF + 1];      // ... and its feature row
  mm3d_griddep_wait();
  heads_load_weights(s, f, C, w1, w1 /* b1 is not needed */, w2, b2);
  __syncthreads();
  const float gs = (target && d_loss) ? __ldg(d_loss) * inv_n : 0.f;
  const int n_out = 2 * C * f + 2 * C;  // outputs of the parameter gradients, dealt to the threads round-robin
  float acc[(2 * kHeadMaxC * kHeadMaxF + 2 * kHeadMaxC + kHeadTile - 1) / kHeadTile];
#pragma unroll
  for (int a = 0; a < (int)(sizeof(acc) / sizeof(float)); ++a) acc[a] = 0.f;
  const int64_t tiles = (n + kHeadTile - 1) / kHeadTile;
  for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
    const int64_t i = t * kHeadTile + threadIdx.x;
    float fr[kHeadMaxF], d1[kHeadMaxC], d2[kHeadMaxC];
    if (i < n) {
      heads_row(feat + i * f, f, fr);
      float l2[kHeadMaxC], m2 = -INFINITY, mt = -INFINITY;
#pragma unroll
      for (int c = 0; c < kHeadMaxC; ++c) {
        d1[c] = (c < C && d_logit1) ? __ldg(d_logit1 + i * C + c) : 0.f;
        d2[c] = (c < C && d_logit2) ? __ldg(d_logit2 + i * C + c) : 0.f;
        if (c < C && gs != 0.f) {
          l2[c] = heads_dot(fr, s.w2 + c * f, f, s.b2[c]);
          m2 = fmaxf(m2, l2[c]);
          mt = fmaxf(mt, __ldg(target + i * C + c));
        }
      }
      if (gs != 0.f) {  // d loss / d logit2 = (softmax(logit2) - softmax(target)) * d_loss / n
        float s2 = 0.f, st = 0.f;
#pragma unroll
        for (int c = 0; c < kHeadMaxC; ++c)
          if (c < C) { s2 += expf(l2[c] - m2); st += expf(__ldg(target + i * C + c) - mt); }
#pragma unroll
        for (int c = 0; c < kHeadMaxC; ++c)
          if (c < C) d2[c] += gs * (expf(l2[c] - m2) / s2 - expf(__ldg(target + i * C + c) - mt) / st);
      }
      if (d_feat) {
#pragma unroll
        for (int j = 0; j < kHeadMaxF; ++j) {
          if (j < f) {
            float g = 0.f;
#pragma unroll
            for (int c = 0; c < kHeadMaxC; ++c)
              if (c < C) g = fmaf(d1[c], s.w1[c * f + j], fmaf(d2[c], s.w2[c * f + j], g));
            d_feat[i * f + j] = g;
          }
        }
      }
    }
    __syncthreads();  // (the previous tile's reduction is done with sd / sf)
#pragma unroll
    for (int c = 0; c < kHeadMaxC; ++c) {
      if (c < C) {
        sd[threadIdx.x][c] = i < n ? d1[c] : 0.f;
        sd[threadIdx.x][C + c] = i < n ? d2[c] : 0.f;
      }
    }
#pragma unroll
    for (int j = 0; j < kHeadMaxF; ++j)
      if (j < f) sf[threadIdx.x][j] = i < n ? fr[j] : 0.f;
    __syncthreads();
    // parameter gradients of this tile: output o = (head h, class c, feature j) -> sum_r d_h[r][c] feat[r][j]; the
    // last 2 C outputs are the biases (sum_r d_h[r][c])
    int a = 0;
    for (int o = threadIdx.x; o < n_out; o += kHeadTile, ++a) {
      float v = 0.f;
      if (o < 2 * C * f) {
        const int hc = o / f, j = o - hc * f;
        for (int r = 0; r < kHeadTile; ++r) v = fmaf(sd[r][hc], sf[r][j], v);
      } else {
        const int hc = o - 2 * C * f;
        for (int r = 0; r < kHeadTile; ++r) v += sd[r][hc];
      }
      acc[a] += v;
    }
  }
  int a = 0;
  for (int o = threadIdx.x; o < n_out; o += kHeadTile, ++a) {
    // o indexes [d1 W | d2 W | d1 b | d2 b]; tot is laid out [d_w1 | d_b1 | d_w2 | d_b2]
    int dst;
    if (o < C * f) dst = o;
    else if (o < 2 * C * f) dst = C * f + C + (o - C * f);
    else if (o < 2 * C * f + C) dst = C * f + (o - 2 * C * f);
    else dst = 2 * C * f + C + (o - 2 * C * f - C);
    if (DET) tot[(int64_t)blockIdx.x * n_out + dst] = (double)acc[a];
    else atomicAdd(tot + dst, (double)acc[a]);
  }
}

}  // namespace

// The finalize launch of the deterministic reductions, for other files' kernels that store one row of `words` doubles per
// CTA (the masked InputLayer backward, io_layers.cu): dst[j] = (float) sum of part[b][j] over b < nparts, in CTA order
int mm3d_det_sum_parts(const double* part, int nparts, int words, float* dst, cudaStream_t stream) {
  MM3D_REQUIRE(words > 0 && nparts >= 0 && nparts <= MM3D_DET_CTAS && dst, MM3D_ERR_INVALID, "det_sum_parts: bad arguments");
  const PartOuts o = {{dst, nullptr, nullptr, nullptr}, {words, 0, 0, 0}};
  MM3D_CUDA(mm3d_launch_pdl(k_sum_parts, dim3(1), dim3(32), 0, stream, part, nparts, words, 1.0, o));
  mm3d_count_launches(1);
  return MM3D_OK;
}

extern "C" {

// y = x * sigmoid(x . w + b) row-wise; s_out [n] keeps the gate for the backward pass.  y may be x (in place,
// like the reference's `feats *= mask`): a row is read completely before it is written.
int mm3d_rgb_mask_fwd(const float* x, int64_t n, int c, const float* w, const float* b, float* y, float* s_out,
                      mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(n >= 0 && c > 0 && c <= 8, MM3D_ERR_INVALID, "rgb_mask: 1..8 feature channels supported, got %d", c);
  if (n == 0) return MM3D_OK;
  MM3D_REQUIRE(x && w && b && y && s_out, MM3D_ERR_INVALID, "rgb_mask: null pointer");
  MM3D_CUDA(mm3d_launch_pdl(k_rgb_mask_fwd, dim3(mm3d_grid(n, 256)), dim3(256), 0, stream, x, n, c, w, b, y, s_out));
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_rgb_mask_fwd");
  return MM3D_OK;
}

// x: the UNMASKED features; dx may be NULL (the features are data); dw [c], db [1]; ws: (c + 1) doubles
// flags: MM3D_DETERMINISTIC -> ws: MM3D_DET_CTAS * (c + 1) doubles
int mm3d_rgb_mask_bwd_ex(const float* x, const float* s, const float* dy, int64_t n, int c, const float* w, float* dx,
                         float* dw, float* db, void* ws, size_t ws_bytes, mm3d_stream_t stream_, int flags) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(n >= 0 && c > 0 && c <= 8, MM3D_ERR_INVALID, "rgb_mask: 1..8 feature channels supported, got %d", c);
  MM3D_REQUIRE((flags & ~MM3D_DETERMINISTIC) == 0, MM3D_ERR_INVALID, "rgb_mask: unknown flags %#x", flags);
  const bool det = flags & MM3D_DETERMINISTIC;
  MM3D_REQUIRE(dw && db && ws && ws_bytes >= sizeof(double) * (size_t)(c + 1) * (det ? MM3D_DET_CTAS : 1), MM3D_ERR_WORKSPACE,
               "rgb_mask: workspace too small");
  double* tot = (double*)ws;
  if (det) {
    const int grid = n > 0 ? det_grid(mm3d_grid(n, 256, 2)) : 0;
    if (n > 0) {
      MM3D_REQUIRE(x && s && dy && w, MM3D_ERR_INVALID, "rgb_mask: null pointer");
      MM3D_CUDA(mm3d_launch_pdl(k_rgb_mask_bwd<true>, dim3(grid), dim3(256), 0, stream, x, s, dy, n, c, w, dx, tot));
    }
    const PartOuts o = {{dw, db, nullptr, nullptr}, {c, 1, 0, 0}};
    MM3D_CUDA(mm3d_launch_pdl(k_sum_parts, dim3(1), dim3(32), 0, stream, (const double*)tot, grid, c + 1, 1.0, o));
    mm3d_count_launches(n > 0 ? 2 : 1);
    MM3D_CHECK_LAUNCH("mm3d_rgb_mask_bwd");
    return MM3D_OK;
  }
  MM3D_CUDA(cudaMemsetAsync(tot, 0, sizeof(double) * (size_t)(c + 1), stream));
  if (n > 0) {
    MM3D_REQUIRE(x && s && dy && w, MM3D_ERR_INVALID, "rgb_mask: null pointer");
    MM3D_CUDA(mm3d_launch_pdl(k_rgb_mask_bwd<false>, dim3(mm3d_grid(n, 256, 2)), dim3(256), 0, stream, x, s, dy, n, c, w, dx, tot));
  }
  MM3D_CUDA(mm3d_launch_pdl(k_f64_to_f32, dim3(1), dim3(32), 0, stream, (const double*)tot, dw, c, 1.0));
  MM3D_CUDA(mm3d_launch_pdl(k_f64_to_f32, dim3(1), dim3(32), 0, stream, (const double*)(tot + c), db, 1, 1.0));
  mm3d_count_launches(n > 0 ? 3 : 2);
  MM3D_CHECK_LAUNCH("mm3d_rgb_mask_bwd");
  return MM3D_OK;
}

int mm3d_rgb_mask_bwd(const float* x, const float* s, const float* dy, int64_t n, int c, const float* w, float* dx,
                      float* dw, float* db, void* ws, size_t ws_bytes, mm3d_stream_t stream) {
  return mm3d_rgb_mask_bwd_ex(x, s, dy, n, c, w, dx, dw, db, ws, ws_bytes, stream, 0);
}

// loss[0] = mean_n sum_c q (log q - log p),  p = softmax(pred[n, :]), q = softmax(target[n, :]);  ws: one double
// (flags MM3D_DETERMINISTIC: MM3D_DET_CTAS doubles)
int mm3d_kl_logits_fwd_ex(const float* pred, const float* target, int64_t n, int C, float* loss, void* ws, size_t ws_bytes,
                          mm3d_stream_t stream_, int flags) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(n > 0 && C > 0 && C <= 4096, MM3D_ERR_INVALID, "kl_logits: bad sizes");
  MM3D_REQUIRE((flags & ~MM3D_DETERMINISTIC) == 0, MM3D_ERR_INVALID, "kl_logits: unknown flags %#x", flags);
  const bool det = flags & MM3D_DETERMINISTIC;
  MM3D_REQUIRE(pred && target && loss && ws && ws_bytes >= sizeof(double) * (det ? MM3D_DET_CTAS : 1), MM3D_ERR_WORKSPACE,
               "kl_logits: workspace too small");
  if (det) {
    const int grid = det_grid(mm3d_grid(n, 256, 2));
    MM3D_CUDA(mm3d_launch_pdl(k_kl_fwd<true>, dim3(grid), dim3(256), 0, stream, pred, target, n, C, (double*)ws));
    const PartOuts o = {{loss, nullptr, nullptr, nullptr}, {1, 0, 0, 0}};
    MM3D_CUDA(mm3d_launch_pdl(k_sum_parts, dim3(1), dim3(32), 0, stream, (const double*)ws, grid, 1, 1.0 / (double)n, o));
    mm3d_count_launches(2);
    MM3D_CHECK_LAUNCH("mm3d_kl_logits_fwd");
    return MM3D_OK;
  }
  MM3D_CUDA(cudaMemsetAsync(ws, 0, sizeof(double), stream));
  MM3D_CUDA(mm3d_launch_pdl(k_kl_fwd<false>, dim3(mm3d_grid(n, 256, 2)), dim3(256), 0, stream, pred, target, n, C, (double*)ws));
  MM3D_CUDA(mm3d_launch_pdl(k_f64_to_f32, dim3(1), dim3(32), 0, stream, (const double*)ws, loss, 1, 1.0 / (double)n));
  mm3d_count_launches(2);
  MM3D_CHECK_LAUNCH("mm3d_kl_logits_fwd");
  return MM3D_OK;
}

int mm3d_kl_logits_fwd(const float* pred, const float* target, int64_t n, int C, float* loss, void* ws, size_t ws_bytes,
                       mm3d_stream_t stream) {
  return mm3d_kl_logits_fwd_ex(pred, target, n, C, loss, ws, ws_bytes, stream, 0);
}

// dpred = dloss[0] * (softmax(pred) - softmax(target)) / n   (the target side is detached in the reference)
int mm3d_kl_logits_bwd(const float* pred, const float* target, int64_t n, int C, const float* dloss, float* dpred,
                       mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(n > 0 && C > 0 && C <= 4096, MM3D_ERR_INVALID, "kl_logits: bad sizes");
  MM3D_REQUIRE(pred && target && dloss && dpred, MM3D_ERR_INVALID, "kl_logits: null pointer");
  MM3D_CUDA(mm3d_launch_pdl(k_kl_bwd, dim3(mm3d_grid(n, 256)), dim3(256), 0, stream, pred, target, n, C, dloss,
                            1.f / (float)n, dpred));
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_kl_logits_bwd");
  return MM3D_OK;
}

// The two Linear(f -> C) heads of the 3D branch (weights [C, f] as nn.Linear stores them) and, when `target` is given,
// loss[0] = mean_n KL(softmax(target_n) || softmax(logit2_n)) in one pass over feat [n, f].  logit2 and loss may be NULL.
// f: multiple of 4, <= 32; C <= 20.  ws: one double (flags MM3D_DETERMINISTIC: MM3D_DET_CTAS doubles).
int mm3d_heads3d_fwd_ex(const float* feat, int64_t n, int f, int C, const float* w1, const float* b1, const float* w2,
                        const float* b2, const float* target, float* logit1, float* logit2, float* loss, void* ws,
                        size_t ws_bytes, mm3d_stream_t stream_, int flags) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(n >= 0 && f > 0 && f <= kHeadMaxF && (f & 3) == 0 && C > 0 && C <= kHeadMaxC, MM3D_ERR_INVALID,
               "heads3d: f must be a multiple of 4 up to %d and C at most %d (got %d, %d)", kHeadMaxF, kHeadMaxC, f, C);
  MM3D_REQUIRE((flags & ~MM3D_DETERMINISTIC) == 0, MM3D_ERR_INVALID, "heads3d: unknown flags %#x", flags);
  const bool det = flags & MM3D_DETERMINISTIC;
  MM3D_REQUIRE(!loss || (target && ws && ws_bytes >= sizeof(double) * (det ? MM3D_DET_CTAS : 1)), MM3D_ERR_WORKSPACE,
               "heads3d: the loss needs a target and a workspace");
  if (loss && !det) MM3D_CUDA(cudaMemsetAsync(ws, 0, sizeof(double), stream));
  if (n == 0) {
    if (loss) MM3D_CUDA(cudaMemsetAsync(loss, 0, sizeof(float), stream));
    return MM3D_OK;
  }
  MM3D_REQUIRE(feat && w1 && b1 && w2 && b2 && logit1, MM3D_ERR_INVALID, "heads3d: null pointer");
  MM3D_REQUIRE((((uintptr_t)feat) & 15) == 0, MM3D_ERR_INVALID, "heads3d: feat must be 16-byte aligned");
  const int grid = det ? det_grid(mm3d_grid(n, kHeadTile, 2)) : mm3d_grid(n, kHeadTile, 2);
  MM3D_CUDA(mm3d_launch_pdl(det ? k_heads3d_fwd<true> : k_heads3d_fwd<false>, dim3(grid), dim3(kHeadTile), 0, stream, feat, n, f, C,
                            w1, b1, w2, b2, loss ? target : (const float*)nullptr, logit1, logit2, loss ? (double*)ws : (double*)nullptr));
  mm3d_count_launches(1);
  if (loss && det) {
    const PartOuts o = {{loss, nullptr, nullptr, nullptr}, {1, 0, 0, 0}};
    MM3D_CUDA(mm3d_launch_pdl(k_sum_parts, dim3(1), dim3(32), 0, stream, (const double*)ws, grid, 1, 1.0 / (double)n, o));
    mm3d_count_launches(1);
  } else if (loss) {
    MM3D_CUDA(mm3d_launch_pdl(k_f64_to_f32, dim3(1), dim3(32), 0, stream, (const double*)ws, loss, 1, 1.0 / (double)n));
    mm3d_count_launches(1);
  }
  MM3D_CHECK_LAUNCH("mm3d_heads3d_fwd");
  return MM3D_OK;
}

int mm3d_heads3d_fwd(const float* feat, int64_t n, int f, int C, const float* w1, const float* b1, const float* w2,
                     const float* b2, const float* target, float* logit1, float* logit2, float* loss, void* ws,
                     size_t ws_bytes, mm3d_stream_t stream) {
  return mm3d_heads3d_fwd_ex(feat, n, f, C, w1, b1, w2, b2, target, logit1, logit2, loss, ws, ws_bytes, stream, 0);
}

// Gradients of the above.  d_logit1 / d_logit2: upstream gradients of the two logit tensors ([n, C], either may be NULL);
// d_loss: upstream gradient of the loss ([1], NULL = the loss was not used; needs `target`).  d_feat [n, f] may be NULL.
// d_w1, d_w2 [C, f], d_b1, d_b2 [C] are overwritten.  ws: (2 C f + 2 C) doubles (flags MM3D_DETERMINISTIC:
// MM3D_DET_CTAS times that).
int mm3d_heads3d_bwd_ex(const float* feat, int64_t n, int f, int C, const float* w1, const float* w2, const float* b2,
                        const float* target, const float* d_logit1, const float* d_logit2, const float* d_loss, float* d_feat,
                        float* d_w1, float* d_b1, float* d_w2, float* d_b2, void* ws, size_t ws_bytes, mm3d_stream_t stream_,
                        int flags) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(n >= 0 && f > 0 && f <= kHeadMaxF && (f & 3) == 0 && C > 0 && C <= kHeadMaxC, MM3D_ERR_INVALID,
               "heads3d: f must be a multiple of 4 up to %d and C at most %d (got %d, %d)", kHeadMaxF, kHeadMaxC, f, C);
  MM3D_REQUIRE((flags & ~MM3D_DETERMINISTIC) == 0, MM3D_ERR_INVALID, "heads3d: unknown flags %#x", flags);
  const bool det = flags & MM3D_DETERMINISTIC;
  const size_t words = 2 * (size_t)C * f + 2 * (size_t)C;
  MM3D_REQUIRE(d_w1 && d_b1 && d_w2 && d_b2 && ws && ws_bytes >= sizeof(double) * words * (det ? MM3D_DET_CTAS : 1), MM3D_ERR_WORKSPACE,
               "heads3d: workspace too small");
  MM3D_REQUIRE(!d_loss || target, MM3D_ERR_INVALID, "heads3d: a loss gradient needs the target");
  double* tot = (double*)ws;
  if (det) {
    const int64_t tiles = (n + kHeadTile - 1) / kHeadTile;
    const int grid = n > 0 ? det_grid(tiles) : 0;
    if (n > 0) {
      MM3D_REQUIRE(feat && w1 && w2 && b2, MM3D_ERR_INVALID, "heads3d: null pointer");
      MM3D_REQUIRE((((uintptr_t)feat) & 15) == 0, MM3D_ERR_INVALID, "heads3d: feat must be 16-byte aligned");
      MM3D_CUDA(mm3d_launch_pdl(k_heads3d_bwd<true>, dim3(grid), dim3(kHeadTile), 0, stream, feat, n, f, C, w1, w2, b2, target, d_logit1,
                                d_logit2, d_loss, 1.f / (float)n, d_feat, tot));
    }
    const PartOuts o = {{d_w1, d_b1, d_w2, d_b2}, {C * f, C, C * f, C}};
    MM3D_CUDA(mm3d_launch_pdl(k_sum_parts, dim3(1), dim3(256), 0, stream, (const double*)tot, grid, (int)words, 1.0, o));
    mm3d_count_launches(n > 0 ? 2 : 1);
    MM3D_CHECK_LAUNCH("mm3d_heads3d_bwd");
    return MM3D_OK;
  }
  MM3D_CUDA(cudaMemsetAsync(tot, 0, sizeof(double) * words, stream));
  if (n > 0) {
    MM3D_REQUIRE(feat && w1 && w2 && b2, MM3D_ERR_INVALID, "heads3d: null pointer");
    MM3D_REQUIRE((((uintptr_t)feat) & 15) == 0, MM3D_ERR_INVALID, "heads3d: feat must be 16-byte aligned");
    int64_t tiles = (n + kHeadTile - 1) / kHeadTile;
    const int64_t cap = (int64_t)mm3d_sm_count() * 4;
    MM3D_CUDA(mm3d_launch_pdl(k_heads3d_bwd<false>, dim3((unsigned)(tiles < cap ? tiles : cap)), dim3(kHeadTile), 0, stream, feat, n, f, C, w1, w2, b2,
                              target, d_logit1, d_logit2, d_loss, 1.f / (float)n, d_feat, tot));
    mm3d_count_launches(1);
  }
  MM3D_CUDA(mm3d_launch_pdl(k_f64_to_f32, dim3(1), dim3(256), 0, stream, (const double*)tot, d_w1, C * f, 1.0));
  MM3D_CUDA(mm3d_launch_pdl(k_f64_to_f32, dim3(1), dim3(32), 0, stream, (const double*)(tot + C * f), d_b1, C, 1.0));
  MM3D_CUDA(mm3d_launch_pdl(k_f64_to_f32, dim3(1), dim3(256), 0, stream, (const double*)(tot + C * f + C), d_w2, C * f, 1.0));
  MM3D_CUDA(mm3d_launch_pdl(k_f64_to_f32, dim3(1), dim3(32), 0, stream, (const double*)(tot + 2 * C * f + C), d_b2, C, 1.0));
  mm3d_count_launches(4);
  MM3D_CHECK_LAUNCH("mm3d_heads3d_bwd");
  return MM3D_OK;
}

int mm3d_heads3d_bwd(const float* feat, int64_t n, int f, int C, const float* w1, const float* w2, const float* b2,
                     const float* target, const float* d_logit1, const float* d_logit2, const float* d_loss, float* d_feat,
                     float* d_w1, float* d_b1, float* d_w2, float* d_b2, void* ws, size_t ws_bytes, mm3d_stream_t stream) {
  return mm3d_heads3d_bwd_ex(feat, n, f, C, w1, w2, b2, target, d_logit1, d_logit2, d_loss, d_feat, d_w1, d_b1, d_w2, d_b2, ws,
                             ws_bytes, stream, 0);
}

}  // extern "C"
