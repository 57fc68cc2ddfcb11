// BatchNorm + (leaky) ReLU over the active rows of a sparse tensor (SURVEY A.5; replaces
// SparseConvNet's BatchNormalization_f_train / _f_test / _b, which launch <= 16 thread blocks).
//
// HBM-bound: forward = read x (stats) + read x again (L2) + write y; backward = read x, dy + again (L2) +
// write dx.  Training forward and backward are ONE launch each: per-CTA partial sums -> FP64 atomics ->
// grid-wide barrier (all CTAs co-resident) -> every CTA normalises the rows it summed.
// Layout: a CTA's 256 threads (512 for 257..512 channels that are not multiples of 4) tile (rows_pass x CV) where
// CV = C / VEC channel vectors, so a
// warp reads consecutive float4s of consecutive rows (fully coalesced) and every thread keeps
// one fixed channel vector; per-thread FP32 partials are combined in FP64 (shared, then global
// atomics into 2*C doubles), which makes var = E[x^2] - mean^2 safe.
#include <cuda_bf16.h>
#include <stdlib.h>
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
// Channel counts that are not multiples of 4 take one thread per channel: CTAs of kWideThreads for 257..512 of them
// (the kernels' NT; everything else keeps kThreads)
constexpr int kWideThreads = 512;
// Same-address atomics from ~300 CTAs serialise in L2 (~27 cycles each): the per-channel totals therefore go to one
// of kSlots copies (CTA b adds into copy b % kSlots, every CTA sums the copies after the barrier), the barrier has
// one counter per slot plus a top counter for the slots' last arrivers, and nobody cleans up behind a launch:
// the workspace holds TWO such regions and a launch zeroes the one it does not use -- the next launch on the stream
// uses that one (`parity` alternates per launch).
constexpr int kSlots = 8;

// Row ranges of the groups a training-mode launch normalises separately (grouped BatchNorm statistics): group k is
// rows [lo[k], lo[k + 1]), lo[0] = 0, lo[g] = n.  A plain launch is one group.  Each group gets its own batch mean and
// variance, its own row of save_mean / save_invstd ([g][c]) and its own running-statistics update, in group order; the
// backward's dx terms are per group, d_gamma / d_beta totals over all rows.
struct BnGroups {
  int g;
  int64_t lo[MM3D_BN_MAX_GROUPS + 1];
};

template <int VEC> struct Vec;
template <> struct Vec<4> { using T = float4; };
template <> struct Vec<1> { using T = float; };

template <int VEC> __device__ __forceinline__ void vload(const float* p, float (&v)[VEC]);
template <> __device__ __forceinline__ void vload<4>(const float* p, float (&v)[4]) {
  float4 t = __ldg(reinterpret_cast<const float4*>(p));
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <> __device__ __forceinline__ void vload<1>(const float* p, float (&v)[1]) { v[0] = __ldg(p); }
template <int VEC> __device__ __forceinline__ void vstore(float* p, const float (&v)[VEC]);
template <> __device__ __forceinline__ void vstore<4>(float* p, const float (&v)[4]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
template <> __device__ __forceinline__ void vstore<1>(float* p, const float (&v)[1]) { *p = v[0]; }

// Store for a tensor that a tensor-core convolution gathers: mode 0 = as is, 1 = rounded to TF32 (nearest), 2 = two
// planes `plane` floats apart: hi = tf32(v), lo = tf32(v - hi) (the error-compensated TF32x3 mode), 3 = the
// TF32-rounded FP32 plane (the weight-gradient operand) and, `plane` floats behind the tensor's base, a BF16 plane
// (the gathered operand of the BF16 mode; element i of the tensor at BF16 index i)
template <int VEC>
__device__ __forceinline__ void store_planes(float* base, float* p, float (&v)[VEC], int mode, int64_t plane) {
  if (mode == 0) { vstore<VEC>(p, v); return; }
  if (mode == 3) {
    __nv_bfloat16* b = reinterpret_cast<__nv_bfloat16*>(base + plane) + (p - base);
    if (VEC == 4) {
      const __nv_bfloat162 b01 = __floats2bfloat162_rn(v[0], v[1]), b23 = __floats2bfloat162_rn(v[2 % VEC], v[3 % VEC]);
      uint2 u;
      u.x = *reinterpret_cast<const unsigned int*>(&b01);
      u.y = *reinterpret_cast<const unsigned int*>(&b23);
      *reinterpret_cast<uint2*>(b) = u;
    } else {
#pragma unroll
      for (int j = 0; j < VEC; ++j) b[j] = __float2bfloat16_rn(v[j]);
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j) v[j] = mm3d_rna_tf32(v[j]);
    vstore<VEC>(p, v);
    return;
  }
  float lo[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) {
    const float hi = mm3d_rna_tf32(v[j]);
    lo[j] = mm3d_rna_tf32(v[j] - hi);
    v[j] = hi;
  }
  vstore<VEC>(p, v);
  if (mode == 2) vstore<VEC>(p + plane, lo);
}

// dynamic shared: 2*C doubles (accumulators) -- also reused as 2*C floats of scale/shift
extern __shared__ double s_acc[];

// Block reduction of per-thread FP32 partials (VEC channels each, thread layout rows_pass x cv):
// partials go to shared memory, then one thread per channel sums the rows_pass values in FP64 and
// issues ONE global FP64 atomic per channel and CTA -- or, deterministic (DET), stores it into this CTA's own row
// sums[blockIdx.x * ld ..] (ld: the row length, 2 c per group).
template <int VEC, bool DET = false, int NT = kThreads>
__device__ __forceinline__ void block_flush(const float (&s)[VEC], const float (&q)[VEC], int c, int cv, int rows_pass,
                                            int r, int v, double* __restrict__ sums, int ld) {
  float* part = reinterpret_cast<float*>(s_acc);  // [2][rows_pass][c]
  if (r < rows_pass) {
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      part[r * c + v * VEC + j] = s[j];
      part[(rows_pass + r) * c + v * VEC + j] = q[j];
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * c; i += NT) {
    const int which = i >= c, ch = i - which * c;
    double acc = 0.0;
    for (int rr = 0; rr < rows_pass; ++rr) acc += (double)part[(which * rows_pass + rr) * c + ch];
    if (DET) sums[(int64_t)blockIdx.x * ld + i] = acc;
    else atomicAdd(sums + i, acc);
  }
}

// ---- inference forward: normalise with the running statistics (+ optional copy of them to save_*)
template <int VEC, int NT = kThreads>
__global__ void __launch_bounds__(NT)
k_bn_apply(const float* __restrict__ x, float* __restrict__ y, int64_t n, int c,
           const float* __restrict__ gamma, const float* __restrict__ beta,
           float* running_mean, float* running_var, float* save_mean, float* save_invstd,
           const double* __restrict__ sums, float eps, float momentum, float leak, int training, int round_tf32) {
  float* s_mean = reinterpret_cast<float*>(s_acc);
  float* s_scale = s_mean + c;
  for (int i = threadIdx.x; i < c; i += NT) {
    float mean, invstd;
    if (training) {
      const double m = sums[i] / (double)n;
      double var = sums[c + i] / (double)n - m * m;
      if (var < 0.0) var = 0.0;
      mean = (float)m;
      invstd = (float)(1.0 / sqrt(var + (double)eps));
      if (blockIdx.x == 0) {
        save_mean[i] = mean;
        save_invstd[i] = invstd;
        const double unbiased = var * ((double)n / (double)(n > 1 ? n - 1 : 1));
        running_mean[i] = momentum * running_mean[i] + (1.f - momentum) * mean;
        running_var[i] = momentum * running_var[i] + (1.f - momentum) * (float)unbiased;
      }
    } else {
      mean = running_mean[i];
      invstd = rsqrtf(running_var[i] + eps);
      if (blockIdx.x == 0 && save_mean) { save_mean[i] = mean; save_invstd[i] = invstd; }
    }
    s_mean[i] = mean;
    s_scale[i] = invstd * gamma[i];
  }
  __syncthreads();
  const int cv = c / VEC;
  const int rows_pass = NT / cv;
  const int r = threadIdx.x / cv, v = threadIdx.x - r * cv;
  if (r >= rows_pass) return;
  float mean[VEC], scale[VEC], bet[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) {
    mean[j] = s_mean[v * VEC + j];
    scale[j] = s_scale[v * VEC + j];
    bet[j] = __ldg(beta + v * VEC + j);
  }
  for (int64_t row = (int64_t)blockIdx.x * rows_pass + r; row < n; row += (int64_t)gridDim.x * rows_pass) {
    float t[VEC];
    vload<VEC>(x + row * c + v * VEC, t);
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      const float o = fmaf(t[j] - mean[j], scale[j], bet[j]);
      t[j] = o > 0.f ? o : o * leak;
    }
    store_planes<VEC>(y, y + row * c + v * VEC, t, round_tf32, n * c);
  }
}

// ---- grid-wide barrier for the single-launch kernels below.  All CTAs of these grids are co-resident (bn_grid caps
// the grid by the occupancy API x the device's SM count), so waiting for the others is safe; the wait is bounded anyway
// and raises the device error word instead of hanging.  sync[0..kSlots) count the arrivals of the CTAs of each slot,
// sync[kSlots] the slots that are complete: an arrival contends with ~grid / kSlots others, not with all of them.
__device__ __forceinline__ bool grid_arrive_and_wait(unsigned int* sync, int* err) {
  __shared__ int s_ok;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int slot = blockIdx.x % kSlots;
    const unsigned int expect = (gridDim.x + kSlots - 1 - slot) / kSlots;  // CTAs b < gridDim.x with b % kSlots == slot
    const unsigned int slots_used = gridDim.x < (unsigned)kSlots ? gridDim.x : (unsigned)kSlots;
    if (atomicAdd(sync + slot, 1u) == expect - 1) {
      __threadfence();
      atomicAdd(sync + kSlots, 1u);
    }
    int ok = 0;
    for (unsigned int i = 0; i < (1u << 22); ++i) {
      if (*reinterpret_cast<volatile unsigned int*>(sync + kSlots) >= slots_used) { ok = 1; break; }
      __nanosleep(32);
    }
    if (!ok) mm3d_raise(err);
    s_ok = ok;
    __threadfence();
  }
  __syncthreads();
  return s_ok != 0;
}
// zero the workspace region the NEXT launch will use (this launch does not touch it otherwise)
template <int NT = kThreads>
__device__ __forceinline__ void zero_other(double* other, int words) {
  for (int i = blockIdx.x * NT + threadIdx.x; i < words; i += gridDim.x * NT) other[i] = 0.0;
}
// total of one accumulator over the slot copies
__device__ __forceinline__ double slot_total(const double* sums, int c2, int i) {
  double t = 0.0;
#pragma unroll
  for (int sl = 0; sl < kSlots; ++sl) t += __ldcg(sums + sl * c2 + i);
  return t;
}

// Deterministic totals, between two grid barriers: the CTAs' partial rows [grid][c2] -> tot[c2] in a fixed order.
// Warp w of the grid totals accumulators w, w + 8 grid, ...: lane l sums the rows of CTAs l, l + 32, ... in ascending
// order, then a butterfly over the lanes (the same on every run) combines the 32 sums.  Each row is read once, by one
// CTA, instead of every CTA reading all of them (grid^2 x c2 doubles).
template <int NT = kThreads>
__device__ __forceinline__ void det_totals(const double* rows, double* tot, int c2) {
  const int lane = threadIdx.x & 31, nw = NT / 32;
#pragma unroll 1
  for (int i = blockIdx.x * nw + (threadIdx.x >> 5); i < c2; i += gridDim.x * nw) {
    double t = 0.0;
    const double* src = rows + (size_t)lane * c2 + i;
#pragma unroll 4
    for (int b = lane; b < (int)gridDim.x; b += 32, src += 32 * c2) t += __ldcg(src);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) tot[i] = t;
  }
}

// ---- training forward in ONE launch: statistics, grid barrier, normalise + ReLU.  A CTA re-reads exactly the
// rows it summed, so the second read comes from L2 / L1 instead of HBM.
// DET: the deterministic variant -- `rows` [grid][2 c g] takes the CTAs' partials, `sums` [g][2 c] the totals
// (det_totals between the barrier on `sync` and a second one on sync + kSlots + 1).  Default: `sums` holds kSlots
// copies of [g][2 c].  Each group's rows are strided over the whole grid, one group after the other, so the barriers
// stay two per launch whatever the number of groups.
template <int VEC, bool DET, int NT = kThreads, bool GRP = false>
__global__ void __launch_bounds__(NT)
k_bn_fwd_fused(const float* __restrict__ x, const float* __restrict__ x_hi, int c_lo, float* __restrict__ y, int64_t n, int c,
               const float* __restrict__ gamma, const float* __restrict__ beta,
               float* running_mean, float* running_var, float* save_mean, float* save_invstd,
               double* sums, unsigned int* sync, double* rows, double* other, int other_words, float eps, float momentum,
               float leak, int round_tf32, const BnGroups grp, int* err) {
  mm3d_griddep_launch();
  mm3d_griddep_wait();
  zero_other<NT>(other, other_words);
  const int cv = c / VEC;
  const int rows_pass = NT / cv;
  const int r = threadIdx.x / cv, v = threadIdx.x - r * cv;
  const int64_t stride = (int64_t)gridDim.x * rows_pass;
  const int ng_ = GRP ? grp.g : 1;  // (GRP = false: one group of all rows, the code of an ungrouped launch)
  const int c2 = 2 * c * ng_;       // accumulators of all groups
  // x may be given as two column blocks [x | x_hi] (JoinTable without materialising the concatenation): this
  // thread's channel vector of row i is xb[i * xld]
  const bool hi = c_lo > 0 && v * VEC >= c_lo;
  const float* xb = (x_hi && hi) ? x_hi + (v * VEC - c_lo) : x + v * VEC;
  const int64_t xld = x_hi ? (hi ? c - c_lo : c_lo) : c;
  for (int gi = 0; gi < ng_; ++gi) {
    const int64_t end = GRP ? grp.lo[gi + 1] : n;
    float s[VEC], q[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) s[j] = q[j] = 0.f;
    if (r < rows_pass) {
      int64_t row = (GRP ? grp.lo[gi] : 0) + (int64_t)blockIdx.x * rows_pass + r;
      for (; row + 3 * stride < end; row += 4 * stride) {  // four independent loads in flight
        float t[4][VEC];
#pragma unroll
        for (int u = 0; u < 4; ++u) vload<VEC>(xb + (row + u * stride) * xld, t[u]);
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int j = 0; j < VEC; ++j) { s[j] += t[u][j]; q[j] = fmaf(t[u][j], t[u][j], q[j]); }
      }
      for (; row < end; row += stride) {
        float t[VEC];
        vload<VEC>(xb + row * xld, t);
#pragma unroll
        for (int j = 0; j < VEC; ++j) { s[j] += t[j]; q[j] = fmaf(t[j], t[j], q[j]); }
      }
    }
    if (gi) __syncthreads();  // the previous group's block_flush is done with the shared partials
    if (DET) block_flush<VEC, true, NT>(s, q, c, cv, rows_pass, r, v, rows + gi * 2 * c, c2);
    else block_flush<VEC, false, NT>(s, q, c, cv, rows_pass, r, v, sums + (blockIdx.x % kSlots) * c2 + gi * 2 * c, c2);
  }
  grid_arrive_and_wait(sync, err);
  if (DET) {
    det_totals<NT>(rows, sums, c2);
    grid_arrive_and_wait(sync + kSlots + 1, err);
  }
  float* s_mean = reinterpret_cast<float*>(s_acc);
  float* s_scale = s_mean + c;
  for (int gi = 0; gi < ng_; ++gi) {
    const int64_t begin = GRP ? grp.lo[gi] : 0, end = GRP ? grp.lo[gi + 1] : n, ng = end - begin;
    if (GRP && ng == 0) continue;  // (an empty group changes nothing, as a launch over no rows)
    const double* gs = sums + gi * 2 * c;
    __syncthreads();  // block_flush's (or the previous group's) use of the shared buffer is over
    for (int i = threadIdx.x; i < c; i += NT) {
      const double m = (DET ? __ldcg(gs + i) : slot_total(gs, c2, i)) / (double)ng;
      double var = (DET ? __ldcg(gs + c + i) : slot_total(gs, c2, c + i)) / (double)ng - m * m;
      if (var < 0.0) var = 0.0;
      const float mean = (float)m, invstd = (float)(1.0 / sqrt(var + (double)eps));
      if (blockIdx.x == 0) {  // (one thread per channel: the groups' running updates land in group order)
        save_mean[gi * c + i] = mean;
        save_invstd[gi * c + i] = invstd;
        const double unbiased = var * ((double)ng / (double)(ng > 1 ? ng - 1 : 1));
        running_mean[i] = momentum * running_mean[i] + (1.f - momentum) * mean;
        running_var[i] = momentum * running_var[i] + (1.f - momentum) * (float)unbiased;
      }
      s_mean[i] = mean;
      s_scale[i] = invstd * gamma[i];
    }
    __syncthreads();
    if (r >= rows_pass) continue;
    float mean[VEC], scale[VEC], bet[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      mean[j] = s_mean[v * VEC + j];
      scale[j] = s_scale[v * VEC + j];
      bet[j] = __ldg(beta + v * VEC + j);
    }
    int64_t row = begin + (int64_t)blockIdx.x * rows_pass + r;
    for (; row + 3 * stride < end; row += 4 * stride) {  // four independent loads in flight
      float t[4][VEC];
#pragma unroll
      for (int u = 0; u < 4; ++u) vload<VEC>(xb + (row + u * stride) * xld, t[u]);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          const float o = fmaf(t[u][j] - mean[j], scale[j], bet[j]);
          t[u][j] = o > 0.f ? o : o * leak;
        }
        store_planes<VEC>(y, y + (row + u * stride) * c + v * VEC, t[u], round_tf32, n * c);
      }
    }
    for (; row < end; row += stride) {
      float t[VEC];
      vload<VEC>(xb + row * xld, t);
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const float o = fmaf(t[j] - mean[j], scale[j], bet[j]);
        t[j] = o > 0.f ? o : o * leak;
      }
      store_planes<VEC>(y, y + row * c + v * VEC, t, round_tf32, n * c);
    }
  }
}

// this thread's channels (vector v) of one group's saved statistics; zeros for a thread without a channel vector
template <int VEC>
__device__ __forceinline__ void load_stats(const float* save_mean, const float* save_invstd, const float* gamma,
                                           const float* beta, int v, bool has, float (&mean)[VEC], float (&invstd)[VEC],
                                           float (&scale)[VEC], float (&bet)[VEC]) {
#pragma unroll
  for (int j = 0; j < VEC; ++j) mean[j] = invstd[j] = scale[j] = bet[j] = 0.f;
  if (has) {
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      const int ch = v * VEC + j;
      mean[j] = __ldg(save_mean + ch);
      invstd[j] = __ldg(save_invstd + ch);
      scale[j] = invstd[j] * __ldg(gamma + ch);
      bet[j] = __ldg(beta + ch);
    }
  }
}

// ---- backward in ONE launch: reductions, grid barrier, dx (+ d_gamma / d_beta by CTA 0)
// (DET and the groups: as in k_bn_fwd_fused; save_mean / save_invstd are [g][c], the dx terms per group, d_gamma /
// d_beta the totals over all groups)
template <int VEC, bool DET, int NT = kThreads, bool GRP = false>
__global__ void __launch_bounds__(NT)
k_bn_bwd_fused(const float* __restrict__ x, const float* __restrict__ x_hi, int c_lo, const float* __restrict__ dy,
               float* __restrict__ dx, float* __restrict__ dx_hi, int64_t n, int c,
               const float* __restrict__ gamma, const float* __restrict__ beta,
               const float* __restrict__ save_mean, const float* __restrict__ save_invstd, float leak,
               double* sums, unsigned int* sync, double* rows, double* other, int other_words, float* d_gamma, float* d_beta,
               int training,
               int round_flags, const float* __restrict__ add, int64_t add_ld, const BnGroups grp, int* err) {
  mm3d_griddep_launch();
  mm3d_griddep_wait();
  zero_other<NT>(other, other_words);
  const int cv = c / VEC;
  const int rows_pass = NT / cv;
  const int r = threadIdx.x / cv, v = threadIdx.x - r * cv;
  const int64_t stride = (int64_t)gridDim.x * rows_pass;
  const int ng_ = GRP ? grp.g : 1;  // (GRP = false: one group of all rows, the code of an ungrouped launch)
  const int c2 = 2 * c * ng_;       // accumulators of all groups
  // x may be given as two column blocks [x | x_hi] (JoinTable without materialising the concatenation): this
  // thread's channel vector of row i is xb[i * xld]
  const bool hi = c_lo > 0 && v * VEC >= c_lo;
  const float* xb = (x_hi && hi) ? x_hi + (v * VEC - c_lo) : x + v * VEC;
  const int64_t xld = x_hi ? (hi ? c - c_lo : c_lo) : c;
  float* dxb = (dx_hi && hi) ? dx_hi + (v * VEC - c_lo) : dx + v * VEC;
  const int64_t dxld = dx_hi ? (hi ? c - c_lo : c_lo) : c;
  // round_flags bit 0: dx (or its low column block) feeds a TF32 convolution as d_out -> store RNA-rounded values;
  // bit 1: same for the high column block dx_hi
  // bit 2: those outputs carry a hi and a lo plane (TF32x3 mode), the lo plane n * (row length) floats behind
  // bit 3: ... a TF32-rounded FP32 plane and a BF16 plane behind it (BF16 mode)
  // bit 4: `add` carries a lo plane n * add_ld floats behind its hi plane (a TF32x3 operand): both are added
  const int rnd = (round_flags & ((dx_hi && hi) ? 2 : 1)) ? ((round_flags & 8) ? 3 : (round_flags & 4) ? 2 : 1) : 0;
  float* dx0 = (dx_hi && hi) ? dx_hi : dx;  // base of the tensor this thread writes
  const int64_t dplane = n * dxld;
  float mean[VEC], invstd[VEC], scale[VEC], bet[VEC];
  for (int gi = 0; gi < ng_; ++gi) {
    const int64_t end = GRP ? grp.lo[gi + 1] : n;
    load_stats<VEC>(save_mean + gi * c, save_invstd + gi * c, gamma, beta, v, r < rows_pass, mean, invstd, scale, bet);
    float s[VEC], q[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) s[j] = q[j] = 0.f;
    if (r < rows_pass) {
      int64_t row = (GRP ? grp.lo[gi] : 0) + (int64_t)blockIdx.x * rows_pass + r;
      for (; row < end; row += 2 * stride) {  // two rows (four loads) in flight
        float t[2][VEC], g[2][VEC];
        const bool second = row + stride < end;
        vload<VEC>(xb + row * xld, t[0]);
        vload<VEC>(dy + row * c + v * VEC, g[0]);
        if (second) {
          vload<VEC>(xb + (row + stride) * xld, t[1]);
          vload<VEC>(dy + (row + stride) * c + v * VEC, g[1]);
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          if (u == 1 && !second) break;
#pragma unroll
          for (int j = 0; j < VEC; ++j) {
            const float xc = t[u][j] - mean[j];
            const float o = fmaf(xc, scale[j], bet[j]);
            const float d = o > 0.f ? g[u][j] : g[u][j] * leak;
            s[j] += d;
            q[j] = fmaf(d, xc * invstd[j], q[j]);
          }
        }
      }
    }
    if (gi) __syncthreads();  // the previous group's block_flush is done with the shared partials
    if (DET) block_flush<VEC, true, NT>(s, q, c, cv, rows_pass, r, v, rows + gi * 2 * c, c2);
    else block_flush<VEC, false, NT>(s, q, c, cv, rows_pass, r, v, sums + (blockIdx.x % kSlots) * c2 + gi * 2 * c, c2);
  }
  grid_arrive_and_wait(sync, err);
  if (DET) {
    det_totals<NT>(rows, sums, c2);
    grid_arrive_and_wait(sync + kSlots + 1, err);
  }
  // accumulator i of group gi, totalled over the slot copies
  auto total = [&](int gi, int i) { return DET ? __ldcg(sums + gi * 2 * c + i) : slot_total(sums + gi * 2 * c, c2, i); };
  if (GRP && blockIdx.x == 0)  // (frozen affine parameters: NULL gradient pointers)
    for (int i = threadIdx.x; i < c; i += NT) {
      double tb = 0.0, tg = 0.0;
      for (int gi = 0; gi < ng_; ++gi) {
        tb += total(gi, i);
        tg += total(gi, c + i);
      }
      if (d_beta) d_beta[i] = (float)tb;
      if (d_gamma) d_gamma[i] = (float)tg;
    }
  double* s_tot = s_acc;
  for (int gi = 0; gi < ng_; ++gi) {
    const int64_t begin = GRP ? grp.lo[gi] : 0, end = GRP ? grp.lo[gi + 1] : n, ng = end - begin;
    if (GRP && ng == 0) continue;
    // group gi's totals -> shared memory (block_flush's, or the previous group's, use of the buffer is over)
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * c; i += NT) s_tot[i] = total(gi, i);
    __syncthreads();
    if (!GRP && blockIdx.x == 0)  // (one group: its totals are the gradients)
      for (int i = threadIdx.x; i < c; i += NT) {
        if (d_beta) d_beta[i] = (float)s_tot[i];
        if (d_gamma) d_gamma[i] = (float)s_tot[c + i];
      }
    if (GRP)  // (one group: still in the registers from the reduction)
      load_stats<VEC>(save_mean + gi * c, save_invstd + gi * c, gamma, beta, v, r < rows_pass, mean, invstd, scale, bet);
    float md[VEC], mdx[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) md[j] = mdx[j] = 0.f;
    if (r < rows_pass && training) {
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        md[j] = (float)(s_tot[v * VEC + j] / (double)ng);
        mdx[j] = (float)(s_tot[c + v * VEC + j] / (double)ng);
      }
    }
    if (r >= rows_pass) continue;
    int64_t row = begin + (int64_t)blockIdx.x * rows_pass + r;
    for (; row + stride < end; row += 2 * stride) {  // two rows (four loads) in flight
      float t[2][VEC], g[2][VEC];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        vload<VEC>(xb + (row + u * stride) * xld, t[u]);
        vload<VEC>(dy + (row + u * stride) * c + v * VEC, g[u]);
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          const float xc = t[u][j] - mean[j];
          const float o = fmaf(xc, scale[j], bet[j]);
          const float d = o > 0.f ? g[u][j] : g[u][j] * leak;
          g[u][j] = scale[j] * (d - md[j] - xc * invstd[j] * mdx[j]);
        }
        if (add) {  // dx += another gradient of the same tensor (the U-Net's skip connection), before any rounding
          float a_[VEC];
          vload<VEC>(add + (row + u * stride) * add_ld + v * VEC, a_);
#pragma unroll
          for (int j = 0; j < VEC; ++j) g[u][j] += a_[j];
          if (round_flags & 16) {
            vload<VEC>(add + n * add_ld + (row + u * stride) * add_ld + v * VEC, a_);
#pragma unroll
            for (int j = 0; j < VEC; ++j) g[u][j] += a_[j];
          }
        }
        store_planes<VEC>(dx0, dxb + (row + u * stride) * dxld, g[u], rnd, dplane);
      }
    }
    for (; row < end; row += stride) {
      float t[VEC], g[VEC];
      vload<VEC>(xb + row * xld, t);
      vload<VEC>(dy + row * c + v * VEC, g);
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const float xc = t[j] - mean[j];
        const float o = fmaf(xc, scale[j], bet[j]);
        const float d = o > 0.f ? g[j] : g[j] * leak;
        g[j] = scale[j] * (d - md[j] - xc * invstd[j] * mdx[j]);
      }
      if (add) {
        float a_[VEC];
        vload<VEC>(add + row * add_ld + v * VEC, a_);
#pragma unroll
        for (int j = 0; j < VEC; ++j) g[j] += a_[j];
        if (round_flags & 16) {
          vload<VEC>(add + n * add_ld + row * add_ld + v * VEC, a_);
#pragma unroll
          for (int j = 0; j < VEC; ++j) g[j] += a_[j];
        }
      }
      store_planes<VEC>(dx0, dxb + row * dxld, g, rnd, dplane);
    }
  }
}

// Single-launch kernels wait on each other, so every CTA of the grid must be able to be resident at once: the grid
// is capped at (CTAs per SM the occupancy API reports for this kernel and shared-memory size, at most 2) x (the
// device's real SM count).  Kernels of other streams (the weight-gradient CTAs of the side stream) may delay a
// CTA's start but never depend on this grid, so the barrier always completes; the wait is bounded anyway.
// CTAs per SM the grid may count on.  MM3D_BN_PER_SM overrides it for A/B measurements (bench.py --ab).
static int bn_per_sm_cap() {
  const char* e = getenv("MM3D_BN_PER_SM");
  const int v = e ? atoi(e) : 0;
  return v >= 1 && v <= 8 ? v : 2;
}

template <bool DET, int NT, bool GRP, typename Kernel>
int bn_grid(Kernel kernel, int64_t n, int cv, size_t smem) {
  const int rows_pass = NT / cv;
  int64_t g = mm3d_cdiv(n, (int64_t)rows_pass * 4);  // >= 4 rows per thread when there is enough work
  if (g < 1) g = 1;
  // the query is cached per device and kernel instantiation for the 16 KB upper bound of these kernels' dynamic
  // shared memory (2 * rows_pass * c floats <= 8 KB for every supported c); larger requests are queried directly
  constexpr size_t kSmemBound = 16 * 1024;
  static int cached[64] = {0};  // (DET and GRP are template parameters: the variants of a kernel have the same type)
  int& slot = cached[mm3d_device_slot()];
  int per_sm = smem <= kSmemBound ? slot : 0;
  if (per_sm == 0) {
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, NT, smem <= kSmemBound ? kSmemBound : smem) != cudaSuccess || per_sm < 1) {
      (void)cudaGetLastError();
      per_sm = 1;
    }
    if (smem <= kSmemBound) slot = per_sm;
  }
  if (per_sm > bn_per_sm_cap()) per_sm = bn_per_sm_cap();
  const int64_t cap = (int64_t)mm3d_sm_count() * per_sm;
  return (int)(g < cap ? g : cap);
}

}  // namespace

int* mm3d_device_err_flag();  // conv_tc.cu

// workspace: two regions of [kSlots copies of 2*c doubles of totals | kSlots + 1 barrier counters]
static size_t bn_region_bytes(int c) { return mm3d_align(sizeof(double) * (kSlots * 2 * (size_t)c + 8)); }
extern "C" size_t mm3d_bnrelu_workspace_bytes(int c) { return 2 * bn_region_bytes(c); }
// deterministic variant: two regions of [2*c doubles of totals | two sets of kSlots + 1 barrier counters], then the
// partial rows [grid][2*c] doubles for the largest grid this device can get (every launch overwrites the rows it uses)
static size_t bn_det_region_bytes(int c) {
  return mm3d_align(sizeof(double) * 2 * (size_t)c + sizeof(unsigned int) * 2 * (kSlots + 1));
}
static int64_t bn_max_grid() { return (int64_t)mm3d_sm_count() * bn_per_sm_cap(); }
extern "C" size_t mm3d_bnrelu_workspace_bytes_ex(int c, int flags) {
  if (!(flags & MM3D_DETERMINISTIC)) return mm3d_bnrelu_workspace_bytes(c);
  return 2 * bn_det_region_bytes(c) + sizeof(double) * 2 * (size_t)c * (size_t)bn_max_grid();
}
// the most channels a deterministic workspace of ws_bytes serves: a workspace shared by launches of different widths
// (parity != NULL) lays its two regions out for this many, so that every launch agrees on where the other region is
static int bn_det_capacity(size_t ws_bytes) {
  int64_t c = (int64_t)(ws_bytes / (2 * sizeof(double) * (2 + (size_t)bn_max_grid())));  // (an upper bound)
  while (c > 0 && mm3d_bnrelu_workspace_bytes_ex((int)c, MM3D_DETERMINISTIC) > ws_bytes) --c;
  return (int)c;
}

#define BN_DISPATCH(KERNEL, ...)                                                        \
  do {                                                                                  \
    const int grid = mm3d_grid(n, nt / cv);                                             \
    if (vec4) KERNEL<4><<<grid, kThreads, smem, stream>>>(__VA_ARGS__);                 \
    else if (nt == kThreads) KERNEL<1><<<grid, kThreads, smem, stream>>>(__VA_ARGS__);  \
    else KERNEL<1, kWideThreads><<<grid, kWideThreads, smem, stream>>>(__VA_ARGS__);    \
  } while (0)
#define BN_DISPATCH_PDL_(KERNEL, DET, GRP, ...)                                                                  \
  do {                                                                                                           \
    if (vec4) { const int grid = bn_grid<DET, kThreads, GRP>(KERNEL<4, DET, kThreads, GRP>, n, cv, smem);        \
                MM3D_CUDA(mm3d_launch_pdl(KERNEL<4, DET, kThreads, GRP>, dim3(grid), dim3(kThreads), smem, stream, \
                                          __VA_ARGS__)); }                                                       \
    else if (nt == kThreads) { const int grid = bn_grid<DET, kThreads, GRP>(KERNEL<1, DET, kThreads, GRP>, n, cv, smem); \
                MM3D_CUDA(mm3d_launch_pdl(KERNEL<1, DET, kThreads, GRP>, dim3(grid), dim3(kThreads), smem, stream, \
                                          __VA_ARGS__)); }                                                       \
    else      { const int grid = bn_grid<DET, kWideThreads, GRP>(KERNEL<1, DET, kWideThreads, GRP>, n, cv, smem); \
                MM3D_CUDA(mm3d_launch_pdl(KERNEL<1, DET, kWideThreads, GRP>, dim3(grid), dim3(kWideThreads), smem, \
                                          stream, __VA_ARGS__)); }                                               \
  } while (0)
// several groups take the grouped instantiations (GRP); one group runs the ungrouped code
#define BN_DISPATCH_PDL(KERNEL, DET, ...)                                   \
  do {                                                                      \
    if (grp.g > 1) BN_DISPATCH_PDL_(KERNEL, DET, true, __VA_ARGS__);       \
    else BN_DISPATCH_PDL_(KERNEL, DET, false, __VA_ARGS__);                \
  } while (0)

// The groups a launch runs with: one group of all rows unless a training launch is given several (an eval-mode
// BatchNorm uses the running statistics, so its groups change nothing)
static BnGroups bn_groups(const BnGroups* grp, int64_t n, int training) {
  if (grp && training) return *grp;
  BnGroups one{};
  one.g = 1;
  one.lo[1] = n;
  return one;
}
// host row boundaries of a grouped call -> BnGroups; checks them against n
static int bn_groups_from(int groups, const int64_t* bounds, int64_t n, BnGroups* out) {
  MM3D_REQUIRE(groups >= 1 && groups <= MM3D_BN_MAX_GROUPS, MM3D_ERR_INVALID, "bnrelu: %d groups (1..%d supported)", groups,
               MM3D_BN_MAX_GROUPS);
  MM3D_REQUIRE(bounds && bounds[0] == 0 && bounds[groups] == n, MM3D_ERR_INVALID,
               "bnrelu: group boundaries must run from 0 to n = %lld", (long long)n);
  *out = BnGroups{};
  out->g = groups;
  for (int k = 0; k <= groups; ++k) {
    MM3D_REQUIRE(k == 0 || bounds[k] >= bounds[k - 1], MM3D_ERR_INVALID, "bnrelu: group boundaries must not decrease");
    out->lo[k] = bounds[k];
  }
  return MM3D_OK;
}

// parity == NULL: the workspace is not known to be clean: zero it, use region 0.  Otherwise it is all zero (the kernels
// leave it that way, no memset), and the launches that use it alternate between its two regions by toggling *parity,
// which the caller keeps with the workspace.
// det: the deterministic kernels, workspace mm3d_bnrelu_workspace_bytes_ex(c, MM3D_DETERMINISTIC); with a parity, their
// regions are laid out for the workspace's channel capacity (bn_det_capacity), not for this launch's c
// grp: the row groups of a training launch (NULL: one group); the workspace then serves grp->g * c channels
static int bn_fwd(const float* x, const float* x_hi, int c_lo, float* y, int64_t n, int c, const float* gamma,
                  const float* beta,
                  float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                  float eps, float momentum, float leakiness, int training,
                  void* ws, size_t ws_bytes, int* parity, int round_tf32, cudaStream_t stream, bool det,
                  const BnGroups* grp_in = nullptr) {
  MM3D_REQUIRE(c > 0 && n >= 0, MM3D_ERR_INVALID, "bad sizes");
  const BnGroups grp = bn_groups(grp_in, n, training);
  const int cg = c * grp.g;
  const bool vec4 = (c % 4 == 0) && (c_lo % 4 == 0) && ((((uintptr_t)x | (uintptr_t)x_hi | (uintptr_t)y) & 15) == 0);
  const int cv = vec4 ? c / 4 : c;
  const int nt = (!vec4 && cv > kThreads) ? kWideThreads : kThreads;
  MM3D_REQUIRE(cv <= nt, MM3D_ERR_UNSUPPORTED, "BatchNorm with %d channels not supported", c);
  MM3D_REQUIRE(ws_bytes >= mm3d_bnrelu_workspace_bytes_ex(cg, det ? MM3D_DETERMINISTIC : 0) && ws, MM3D_ERR_WORKSPACE,
               "bnrelu workspace too small");
  MM3D_REQUIRE(!x_hi || (training && c_lo > 0 && c_lo < c), MM3D_ERR_INVALID, "split input needs training mode and 0 < c_lo < c");
  if (n == 0) return MM3D_OK;
  // region `half` is this launch's (all zero: memset below, or zeroed by the previous launch), the other one is
  // zeroed by this launch for the next.  Region size follows the workspace size (the executor shares one workspace
  // among layers of different widths), so consecutive launches agree on where the regions are -- in the deterministic
  // variant through the workspace's channel capacity.
  const size_t region = det ? bn_det_region_bytes(parity ? bn_det_capacity(ws_bytes) : cg) : ws_bytes / 2 / 256 * 256;
  const int half = (parity && training) ? (*parity ^= 1) : 0;  // (only launches that use the workspace alternate)
  double* sums = (double*)((char*)ws + (size_t)half * region);
  double* other = (double*)((char*)ws + (size_t)(half ^ 1) * region);
  unsigned int* sync = (unsigned int*)(sums + (det ? 2 : kSlots * 2) * cg);
  double* rows = det ? (double*)((char*)ws + 2 * region) : nullptr;
  const int other_words = (int)(region / 8);
  const size_t smem = sizeof(double) * 2 * c > sizeof(float) * 2 * (nt / cv) * (size_t)c
                          ? sizeof(double) * 2 * c : sizeof(float) * 2 * (nt / cv) * (size_t)c;
  if (training) {
    MM3D_REQUIRE(save_mean && save_invstd && running_mean && running_var, MM3D_ERR_INVALID, "training needs stat buffers");
    if (!parity) MM3D_CUDA(cudaMemsetAsync(ws, 0, 2 * region, stream));
    if (det)
      BN_DISPATCH_PDL(k_bn_fwd_fused, true, x, x_hi, c_lo, y, n, c, gamma, beta, running_mean, running_var, save_mean,
                      save_invstd, sums, sync, rows, other, other_words, eps, momentum, leakiness, round_tf32, grp,
                      mm3d_device_err_flag());
    else
      BN_DISPATCH_PDL(k_bn_fwd_fused, false, x, x_hi, c_lo, y, n, c, gamma, beta, running_mean, running_var, save_mean,
                      save_invstd, sums, sync, rows, other, other_words, eps, momentum, leakiness, round_tf32, grp,
                      mm3d_device_err_flag());
  } else {
    BN_DISPATCH(k_bn_apply, x, y, n, c, gamma, beta, running_mean, running_var, save_mean, save_invstd, sums, eps,
                momentum, leakiness, training, round_tf32);
  }
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_bnrelu_fwd");
  return MM3D_OK;
}

// groups / bounds: the row groups of a training launch (groups <= 1: one group, bounds unused)
int mm3d_bnrelu_fwd_impl(const float* x, const float* x_hi, int c_lo, float* y, int64_t n, int c, const float* gamma,
                         const float* beta,
                         float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                         float eps, float momentum, float leakiness, int training,
                         void* ws, size_t ws_bytes, int* parity, int round_tf32, cudaStream_t stream, int det,
                         int groups, const int64_t* bounds) {
  BnGroups grp;
  if (groups > 1) {
    const int rc = bn_groups_from(groups, bounds, n, &grp);
    if (rc) return rc;
  }
  return bn_fwd(x, x_hi, c_lo, y, n, c, gamma, beta, running_mean, running_var, save_mean, save_invstd, eps, momentum,
                leakiness, training, ws, ws_bytes, parity, round_tf32, stream, det != 0, groups > 1 ? &grp : nullptr);
}

static int bn_bwd(const float* x, const float* x_hi, int c_lo, const float* dy, float* dx, float* dx_hi,
                  int64_t n, int c, const float* gamma, const float* beta, const float* save_mean, const float* save_invstd,
                  float* d_gamma, float* d_beta, float leakiness, int training,
                  void* ws, size_t ws_bytes, int* parity, int round_flags, const float* add, int64_t add_ld,
                  cudaStream_t stream, bool det, const BnGroups* grp_in = nullptr) {
  MM3D_REQUIRE(c > 0 && n >= 0, MM3D_ERR_INVALID, "bad sizes");
  const BnGroups grp = bn_groups(grp_in, n, training);
  const int cg = c * grp.g;
  const bool vec4 = (c % 4 == 0) && (c_lo % 4 == 0) && (!add || add_ld % 4 == 0) &&
                    ((((uintptr_t)x | (uintptr_t)x_hi | (uintptr_t)dy | (uintptr_t)dx | (uintptr_t)dx_hi | (uintptr_t)add) & 15) == 0);
  const int cv = vec4 ? c / 4 : c;
  const int nt = (!vec4 && cv > kThreads) ? kWideThreads : kThreads;
  MM3D_REQUIRE(cv <= nt, MM3D_ERR_UNSUPPORTED, "BatchNorm with %d channels not supported", c);
  MM3D_REQUIRE(ws_bytes >= mm3d_bnrelu_workspace_bytes_ex(cg, det ? MM3D_DETERMINISTIC : 0) && ws, MM3D_ERR_WORKSPACE,
               "bnrelu workspace too small");
  if (n == 0) {
    if (d_gamma) MM3D_CUDA(cudaMemsetAsync(d_gamma, 0, sizeof(float) * c, stream));
    if (d_beta) MM3D_CUDA(cudaMemsetAsync(d_beta, 0, sizeof(float) * c, stream));
    return MM3D_OK;
  }
  const size_t region = det ? bn_det_region_bytes(parity ? bn_det_capacity(ws_bytes) : cg) : ws_bytes / 2 / 256 * 256;
  const int half = parity ? (*parity ^= 1) : 0;
  double* sums = (double*)((char*)ws + (size_t)half * region);
  double* other = (double*)((char*)ws + (size_t)(half ^ 1) * region);
  unsigned int* sync = (unsigned int*)(sums + (det ? 2 : kSlots * 2) * cg);
  double* rows = det ? (double*)((char*)ws + 2 * region) : nullptr;
  const int other_words = (int)(region / 8);
  if (!parity) MM3D_CUDA(cudaMemsetAsync(ws, 0, 2 * region, stream));
  const size_t smem = sizeof(double) * 2 * c > sizeof(float) * 2 * (nt / cv) * (size_t)c
                          ? sizeof(double) * 2 * c : sizeof(float) * 2 * (nt / cv) * (size_t)c;
  if (det)
    BN_DISPATCH_PDL(k_bn_bwd_fused, true, x, x_hi, c_lo, dy, dx, dx_hi, n, c, gamma, beta, save_mean, save_invstd, leakiness,
                    sums, sync, rows, other, other_words, d_gamma, d_beta, training, round_flags, add, add_ld, grp,
                    mm3d_device_err_flag());
  else
    BN_DISPATCH_PDL(k_bn_bwd_fused, false, x, x_hi, c_lo, dy, dx, dx_hi, n, c, gamma, beta, save_mean, save_invstd, leakiness,
                    sums, sync, rows, other, other_words, d_gamma, d_beta, training, round_flags, add, add_ld, grp,
                    mm3d_device_err_flag());
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_bnrelu_bwd");
  return MM3D_OK;
}

int mm3d_bnrelu_bwd_impl(const float* x, const float* x_hi, int c_lo, const float* dy, float* dx, float* dx_hi,
                         int64_t n, int c, const float* gamma, const float* beta, const float* save_mean, const float* save_invstd,
                         float* d_gamma, float* d_beta, float leakiness, int training,
                         void* ws, size_t ws_bytes, int* parity, int round_flags, const float* add, int64_t add_ld,
                         cudaStream_t stream, int det, int groups, const int64_t* bounds) {
  BnGroups grp;
  if (groups > 1) {
    const int rc = bn_groups_from(groups, bounds, n, &grp);
    if (rc) return rc;
  }
  return bn_bwd(x, x_hi, c_lo, dy, dx, dx_hi, n, c, gamma, beta, save_mean, save_invstd, d_gamma, d_beta, leakiness,
                training, ws, ws_bytes, parity, round_flags, add, add_ld, stream, det != 0, groups > 1 ? &grp : nullptr);
}

extern "C" int mm3d_bnrelu_fwd_ex(const float* x, float* y, int64_t n, int c, const float* gamma, const float* beta,
                                  float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                                  float eps, float momentum, float leakiness, int training,
                                  void* ws, size_t ws_bytes, mm3d_stream_t stream, int flags) {
  MM3D_REQUIRE((flags & ~MM3D_DETERMINISTIC) == 0, MM3D_ERR_INVALID, "bnrelu_fwd: unknown flags %#x", flags);
  return bn_fwd(x, nullptr, 0, y, n, c, gamma, beta, running_mean, running_var, save_mean, save_invstd, eps, momentum,
                leakiness, training, ws, ws_bytes, nullptr, 0, (cudaStream_t)stream, (flags & MM3D_DETERMINISTIC) != 0);
}

extern "C" int mm3d_bnrelu_bwd_ex(const float* x, const float* dy, float* dx, int64_t n, int c, const float* gamma,
                                  const float* beta, const float* save_mean, const float* save_invstd,
                                  float* d_gamma, float* d_beta, float leakiness, int training,
                                  void* ws, size_t ws_bytes, mm3d_stream_t stream, int flags) {
  MM3D_REQUIRE((flags & ~MM3D_DETERMINISTIC) == 0, MM3D_ERR_INVALID, "bnrelu_bwd: unknown flags %#x", flags);
  return bn_bwd(x, nullptr, 0, dy, dx, nullptr, n, c, gamma, beta, save_mean, save_invstd, d_gamma, d_beta, leakiness,
                training, ws, ws_bytes, nullptr, 0, nullptr, 0, (cudaStream_t)stream, (flags & MM3D_DETERMINISTIC) != 0);
}

extern "C" int mm3d_bnrelu_fwd(const float* x, float* y, int64_t n, int c, const float* gamma, const float* beta,
                               float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                               float eps, float momentum, float leakiness, int training,
                               void* ws, size_t ws_bytes, mm3d_stream_t stream) {
  return mm3d_bnrelu_fwd_ex(x, y, n, c, gamma, beta, running_mean, running_var, save_mean, save_invstd, eps, momentum,
                            leakiness, training, ws, ws_bytes, stream, 0);
}

extern "C" int mm3d_bnrelu_bwd(const float* x, const float* dy, float* dx, int64_t n, int c, const float* gamma,
                               const float* beta, const float* save_mean, const float* save_invstd,
                               float* d_gamma, float* d_beta, float leakiness, int training,
                               void* ws, size_t ws_bytes, mm3d_stream_t stream) {
  return mm3d_bnrelu_bwd_ex(x, dy, dx, n, c, gamma, beta, save_mean, save_invstd, d_gamma, d_beta, leakiness, training,
                            ws, ws_bytes, stream, 0);
}

// grouped BatchNorm statistics (include/mm3d.h)
extern "C" size_t mm3d_bnrelu_workspace_bytes_grouped(int c, int groups, int flags) {
  if (c <= 0 || groups < 1 || groups > MM3D_BN_MAX_GROUPS || (flags & ~MM3D_DETERMINISTIC)) return 0;
  return mm3d_bnrelu_workspace_bytes_ex(c * groups, flags);
}

extern "C" int mm3d_bnrelu_fwd_grouped(const float* x, float* y, int64_t n, int c, const float* gamma, const float* beta,
                                       float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                                       float eps, float momentum, float leakiness, int training, void* ws, size_t ws_bytes,
                                       mm3d_stream_t stream, int flags, int groups, const int64_t* bounds) {
  MM3D_REQUIRE((flags & ~MM3D_DETERMINISTIC) == 0, MM3D_ERR_INVALID, "bnrelu_fwd_grouped: unknown flags %#x", flags);
  BnGroups grp;
  const int rc = bn_groups_from(groups, bounds, n, &grp);
  if (rc) return rc;
  return bn_fwd(x, nullptr, 0, y, n, c, gamma, beta, running_mean, running_var, save_mean, save_invstd, eps, momentum,
                leakiness, training, ws, ws_bytes, nullptr, 0, (cudaStream_t)stream, (flags & MM3D_DETERMINISTIC) != 0, &grp);
}

extern "C" int mm3d_bnrelu_bwd_grouped(const float* x, const float* dy, float* dx, int64_t n, int c, const float* gamma,
                                       const float* beta, const float* save_mean, const float* save_invstd,
                                       float* d_gamma, float* d_beta, float leakiness, int training, void* ws,
                                       size_t ws_bytes, mm3d_stream_t stream, int flags, int groups, const int64_t* bounds) {
  MM3D_REQUIRE((flags & ~MM3D_DETERMINISTIC) == 0, MM3D_ERR_INVALID, "bnrelu_bwd_grouped: unknown flags %#x", flags);
  BnGroups grp;
  const int rc = bn_groups_from(groups, bounds, n, &grp);
  if (rc) return rc;
  return bn_bwd(x, nullptr, 0, dy, dx, nullptr, n, c, gamma, beta, save_mean, save_invstd, d_gamma, d_beta, leakiness,
                training, ws, ws_bytes, nullptr, 0, nullptr, 0, (cudaStream_t)stream, (flags & MM3D_DETERMINISTIC) != 0, &grp);
}
