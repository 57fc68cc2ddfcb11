// tcgen05 / TMEM rule-table convolution (forward and dgrad) for sm_100a, driven by a row plan.
//
//   out[j,:] = sum_k in[tbl(j,k),:] . W'[k]          j in a tile of 128 output rows (plan.cuh)
//
// Output-stationary implicit GEMM with block-sparse K.  A CTA owns tiles of 128 output rows in
// plan order; the reduction runs over the tile's NON-EMPTY offsets only (tile_mask), each offset
// cut into K-blocks of 32 input channels (= one 128-byte shared-memory row; the last block of an
// offset may be 16 channels wide).  For every K-block the 128 gathered rows (zero where the
// neighbour is absent) form a K-major SWIZZLE_128B tile that tcgen05.mma (M=128, N=C_out,
// kind::tf32) multiplies with the matching block of the pre-swizzled weight image, accumulating all
// offsets of the tile in one TMEM accumulator.  No atomics, no read-modify-write of `out`, each
// output row stored once; the result does not depend on which rows share a tile.
//
// Warp roles ((S+5) warps):   warps 0..S-1    gather producers, warp w OWNS ring stage w: 16-byte
//                                             cp.async per (row, chunk), zero fill for absent rows,
//                                             plus the bulk copy of the K-block's weight block
//                             warps S..S+3    epilogue (TMEM lanes -> registers -> out[perm[row]])
//                             warp  S+4       MMA issuer (one lane) + TMEM allocator
// Pipelines (mbarriers):      ring     a_full[S] (32 cp.async arrivals + expect_tx of the weight block)
//                                      / a_empty[S] (tcgen05.commit)
//                             accum    acc_full[2] (tcgen05.commit)       / acc_empty[2] (128 arrivals)
// The accumulator is double buffered in TMEM, so the epilogue of tile i overlaps the MMAs of i+1.
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdlib.h>
#include <string.h>

#include <type_traits>

#include "epilogue.cuh"
#include "plan.cuh"
#include "tc_common.cuh"

namespace {

using namespace tc;

constexpr int kTileM = 128;
constexpr int kKBlock = 32;                 // tf32 elements per 128-byte row of a K-block
constexpr int kStageBytes = kTileM * 128;   // one A stage = one K-block of 128 rows = 16 KB
constexpr int kEntBytes = kTileM * 4;       // the K-block's 128 table entries
constexpr int kEpilogue = 128;
constexpr int kMaxStages = 8;

struct TcParams {
  CUtensorMap tmap;   // `in` as a [n_in, c_in] float32 tensor, box {32 channels, 1 row}, SWIZZLE_128B (TMA gather path)
  int use_tma;        // 1: producers gather rows with cp.async.bulk.tensor tile::gather4, 0: 16-byte cp.async
  int oob_row;        // a row index outside the tensor (= n_in): TMA zero-fills it
  const float* in;
  float* out;
  const float* wimg;  // [K][nb][n_pad][32] tf32, rows 128-byte swizzled
  const int32_t* perm;
  const uint32_t* tile_mask;
  const int32_t* order;
  const int32_t* tbl;
  int64_t tstride;
  int c_in, c_out, K;
  int ld_in;    // row stride of `in` / `in_lo` in 4-byte units (c_in, or c_in / 2 for BF16, unless a channel slice)
  int ld_out;   // row stride of `out` / `add` in floats (c_out unless a column slice)
  int img_nb, img_rows;  // block stride of the weight image: its K-blocks per offset and rows per block (nb, n_pad unless sliced)
  int nb;       // K-blocks per offset = ceil(c_in / 32)
  int last_w;   // 16-byte chunks of an offset's last block (8, or 4 when c_in % 32 == 16)
  int S;        // ring stages = producer warps
  int n_pad, num_tiles, tmem_cols;
  int n_local;  // tiles per CTA (upper bound) = ceil(num_tiles / grid)
  const float* add;  // epilogue: out[row] = acc + add[row] (NULL: out = acc; add == out accumulates)
  int x3;         // TF32x3 mode: every stage also holds the lo planes of the gathered rows and of the weight block, and
                  // an item is three products into the same accumulator: hi.Whi + lo.Whi + hi.Wlo
 const float* in_lo;
  const float* wimg_lo;
  int bf16;       // BF16 mode: `in` and the weight image hold BF16 elements (64 channels per 128-byte K-block), kind::f16
  int split;      // MMA issuer warps with their own accumulators (2, or 1 when 4 accumulators do not fit TMEM)
  int max_items;  // capacity of the shared-memory item list = n_local * K * nb
  int* err;
#ifdef MM3D_TRACE
  long long* trace;  // development builds: clock64 stamps of one CTA's roles, [role][64 records][4], then
                     // [4096 + 2 cta]: globaltimer at every CTA's start (after the dependency wait) and end
  int trace_cta;     // ... which CTA's roles (MM3D_TC_TRACE_CTA)
#endif
};

// the inference form (mm3d_unet_topo_infer): the epilogue writes its value to the destinations of `epi` (epilogue.cuh)
// instead of `out`.  The default kernel is the instantiation with TcParams, whose code the inference form leaves as it is.
struct TcEpiParams : TcParams {
  ConvEpi epi;
};

#ifdef MM3D_TRACE
#define TRACE(role, rec, slot)                                                                                   \
  do {                                                                                                           \
    if (p.trace && (int)blockIdx.x == p.trace_cta && lane == 0 && (rec) < 64) p.trace[(((role) * 64) + (rec)) * 4 + (slot)] = clock64(); \
  } while (0)
#else
#define TRACE(role, rec, slot) do {} while (0)
#endif

// Weight image: one [n_pad][32] block per (offset, channel block); element (n, e) of block (k, j) is
// Wsel(k)[32 j + e][n] (0 beyond c_in / c_out), tf32-rounded, the 16-byte chunks of every 128-byte
// row XOR-swizzled with (n & 7): exactly the bytes a SWIZZLE_128B K-major B tile has in shared
// memory, so the kernel bulk-copies it verbatim.
// lo != 0: the image of the weights' TF32 remainder, tf32(w - tf32(w)) (second term of the error-compensated mode)
__device__ __forceinline__ float wimg_value(float v, int lo) {
  const float hi = to_tf32(v);
  return lo ? to_tf32(v - hi) : hi;
}

// bf16 != 0: BF16 elements, 64 channels per 128-byte row (8 per 16-byte chunk), round to nearest even
__device__ __forceinline__ void wimg_element(const float* __restrict__ w, float* __restrict__ img, int64_t i, int K, int c_in,
                                             int c_out, int nb, int n_pad, int transposed, int mirror, int lo, int bf16) {
  const int per_row = bf16 ? 2 * kKBlock : kKBlock, per_chunk = bf16 ? 8 : 4;
  const int e_sw = (int)(i % per_row);
  const int n = (int)((i / per_row) % n_pad);
  const int blk = (int)(i / ((int64_t)per_row * n_pad));
  const int k = blk / nb, j = blk - k * nb;
  const int chunk = (e_sw / per_chunk) ^ (n & 7);  // un-swizzle: which logical chunk lives here
  const int ci = j * per_row + chunk * per_chunk + (e_sw % per_chunk);
  float v = 0.f;
  if (ci < c_in && n < c_out) {
    const int ks = mirror ? K - 1 - k : k;
    v = transposed ? __ldg(w + ((int64_t)ks * c_out + n) * c_in + ci)   // forward weight is [K][c_out][c_in]
                   : __ldg(w + ((int64_t)ks * c_in + ci) * c_out + n);  // [K][c_in][c_out]
  }
  if (bf16) reinterpret_cast<__nv_bfloat16*>(img)[i] = __float2bfloat16_rn(v);
  else img[i] = wimg_value(v, lo);
}

__global__ void k_weight_image(const float* __restrict__ w, float* __restrict__ img, int K, int c_in, int c_out, int nb,
                               int n_pad, int transposed, int mirror, int lo, int bf16) {
  const int64_t total = (int64_t)K * nb * n_pad * (bf16 ? 2 * kKBlock : kKBlock);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x)
    wimg_element(w, img, i, K, c_in, c_out, nb, n_pad, transposed, mirror, lo, bf16);
}

// Several weight images in one launch (the whole network's, built once per direction by the executor).
struct WImgItem {
  const float* w;
  float* img;
  int K, c_in, c_out, nb, n_pad, transposed, mirror, lo, bf16, block0;
};
constexpr int kMaxImgBatch = 32;
struct WImgBatch {
  int n;
  WImgItem item[kMaxImgBatch];
};
__global__ void k_weight_images(const __grid_constant__ WImgBatch b) {
  mm3d_griddep_wait();
  int i = 0;
  while (i + 1 < b.n && (int)blockIdx.x >= b.item[i + 1].block0) ++i;
  const WImgItem& it = b.item[i];
  const int64_t total = (int64_t)it.K * it.nb * it.n_pad * (it.bf16 ? 2 * kKBlock : kKBlock);
  const int nblk = (i + 1 < b.n ? b.item[i + 1].block0 : (int)gridDim.x) - it.block0;
  for (int64_t e = (int64_t)((int)blockIdx.x - it.block0) * blockDim.x + threadIdx.x; e < total; e += (int64_t)nblk * blockDim.x)
    wimg_element(it.w, it.img, e, it.K, it.c_in, it.c_out, it.nb, it.n_pad, it.transposed, it.mirror, it.lo, it.bf16);
}

// ---- the kernel --------------------------------------------------------------------------------
// Every CTA first writes the list of its ITEMS into shared memory: its tiles (dealt from the plan's cost-ordered
// list) x the set bits of each tile's mask (ascending offset) x the nb channel blocks of an offset, 16 bits per
// item (local tile << 8 | offset << 3 | channel block).  The roles then index that list instead of each walking
// the masks again: measured with clock64 stamps, the per-item walk cost every producer ~1000 cycles and the MMA
// warp ~170 of its ~600 cycles per item, and that single MMA warp was what bounded every layer.
//
// Warp roles (14 warps):   warps 0..7     gather producers: warp w < S owns ring stage w and fills items w, w + S, ...
//                                         (item i lives in stage i % S): the K-block's 128 gathered rows -- TMA tile::gather4 (one
//                                         instruction per lane = 4 rows) for whole 32-channel blocks, 16-byte
//                                         cp.async for 16-channel tails -- plus the bulk copy of its weight block
//                          warps 8..11    epilogue (TMEM lanes -> registers -> out[perm[row]])
//                          warps 12, 13   MMA issuers: warp m issues the items with i % 2 == m into ITS OWN
//                                         accumulator (split K inside the CTA; S is even, so ring stage s is only
//                                         ever consumed by warp s % 2, in order); the epilogue adds the two
// Pipelines (mbarriers):   ring     a_full[S] (33 arrivals + expect_tx bytes)  / a_empty[S] (tcgen05.commit)
//                          accum    acc_full[2] (one tcgen05.commit per issuer) / acc_empty[2] (128 arrivals)
// The accumulator pair is double buffered in TMEM, so the epilogue of tile i overlaps the MMAs of i+1.
constexpr int kProducers = 8;
constexpr int kThreads = (kProducers + 6) * 32;

__device__ __forceinline__ int item_tile(uint32_t it) { return (int)(it >> 8); }
__device__ __forceinline__ int item_k(uint32_t it) { return (int)((it >> 3) & 31u); }
__device__ __forceinline__ int item_j(uint32_t it) { return (int)(it & 7u); }

template <class P>
__global__ void __launch_bounds__(kThreads, 2)
k_conv_tc(const __grid_constant__ P p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const int S = p.S;
  // carve: [A stages][B stages][entry rows (one per producer warp)][tile masks | tile indices | item0][items][barriers]
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t b_bytes = (uint32_t)p.n_pad * 128u;
  const uint32_t b_stride = (b_bytes + 1023u) & ~1023u;
  const uint32_t a_base = smem_base;
  const uint32_t a_stage = (uint32_t)(1 + p.x3) * kStageBytes, b_stage = (uint32_t)(1 + p.x3) * b_stride;  // [hi | lo]
  const uint32_t b_base = a_base + (uint32_t)S * a_stage;
  const uint32_t e_base = b_base + (uint32_t)S * b_stage;
  const uint32_t m_base = e_base + (uint32_t)kProducers * kEntBytes;
  const uint32_t i_base = m_base + (((uint32_t)(3 * p.n_local + 1) * 4u + 15u) & ~15u);
  const uint32_t bar_base = i_base + (((uint32_t)p.max_items * 2u + 15u) & ~15u);
  uint32_t* lmask = reinterpret_cast<uint32_t*>(smem + (m_base - smem_base));  // [n_local] masks, [n_local] tiles, [n_local + 1] item0
  uint16_t* items = reinterpret_cast<uint16_t*>(smem + (i_base - smem_base));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (bar_base - smem_base));
  auto a_full = [&](int s) { return bar_base + 8u * (uint32_t)s; };
  auto a_empty = [&](int s) { return bar_base + 8u * (uint32_t)(kMaxStages + s); };
  auto acc_full = [&](int s) { return bar_base + 8u * (uint32_t)(2 * kMaxStages + s); };
  auto acc_empty = [&](int s) { return bar_base + 8u * (uint32_t)(2 * kMaxStages + 2 + s); };
  constexpr int kNumBars = 2 * kMaxStages + 4;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(bars + kNumBars);
  volatile int* abort_flag = reinterpret_cast<volatile int*>(bars + kNumBars + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int split = p.split;  // 2: two issuers with their own accumulators; 1: warp 12 alone

  // ---- one-time setup.  Nothing before mm3d_griddep_wait() touches global memory (the previous kernel of the
  // stream may still be running: programmatic dependent launch).
  mm3d_griddep_launch();
  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(a_full(s), 33);  // 32 lane arrivals (cp.async completion or plain) + 1 expect_tx arrival
      mbar_init(a_empty(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(acc_full(s), (uint32_t)split);
      mbar_init(acc_empty(s), kEpilogue);
    }
    *abort_flag = 0;
    fence_barrier_init();
  }
  if (warp == kProducers + 4) tmem_alloc(smem_u32((const void*)tmem_slot), (uint32_t)p.tmem_cols);
  mm3d_griddep_wait();
#ifdef MM3D_TRACE
  if (p.trace && threadIdx.x == 0) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    p.trace[4096 + 2 * blockIdx.x] = (long long)gt;
  }
#endif
  // this CTA's tiles (mm3d_plan_local_tile), their masks and the item list
  int n_local = p.n_local;
  if (mm3d_plan_local_tile(p.order, p.num_tiles, (int)gridDim.x, (int)blockIdx.x, n_local - 1) < 0) --n_local;
  uint32_t* ltile = lmask + p.n_local;
  uint32_t* item0 = lmask + 2 * p.n_local;
  for (int i = threadIdx.x; i < n_local; i += blockDim.x) {
    const int t = mm3d_plan_local_tile(p.order, p.num_tiles, (int)gridDim.x, (int)blockIdx.x, i);
    lmask[i] = __ldg(p.tile_mask + t);
    ltile[i] = (uint32_t)t;
  }
  __syncthreads();
  if (warp == 0) {  // exclusive scan of the tiles' item counts
    uint32_t run = 0;
    for (int b0 = 0; b0 < n_local; b0 += 32) {
      const int i = b0 + lane;
      const uint32_t c = i < n_local ? (uint32_t)(__popc(lmask[i]) * p.nb) : 0u;
      uint32_t inc = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t x = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += x;
      }
      if (i < n_local) item0[i] = run + inc - c;
      run += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) item0[n_local] = run;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n_local; i += blockDim.x) {
    uint32_t at = item0[i];
    for (uint32_t rem = lmask[i]; rem; rem &= rem - 1) {
      const uint32_t k = (uint32_t)(__ffs(rem) - 1);
      for (int j = 0; j < p.nb; ++j) items[at++] = (uint16_t)(((uint32_t)i << 8) | (k << 3) | (uint32_t)j);
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_items = (int)item0[n_local];

  if (warp < kProducers) {
    // =================================================================== gather producers
    // Warp w < S OWNS ring stage w and fills items w, w + S, w + 2 S, ... (warps >= S idle): consecutive waits of a
    // warp on its stage's barriers are then consecutive phases, which is what a parity wait can tell apart.
    if (warp >= S) goto done;
    const uint32_t ent = e_base + (uint32_t)warp * kEntBytes;
    int i = warp;
    int4 e = make_int4(-1, -1, -1, -1);  // entries of rows 4*lane .. 4*lane+3 of the current item
    uint32_t cur = 0;
    if (i < n_items) {
      cur = items[i];
      e = __ldg(reinterpret_cast<const int4*>(p.tbl + (int64_t)item_k(cur) * p.tstride + (int64_t)ltile[item_tile(cur)] * kTileM) + lane);
    }
    while (i < n_items) {
      const int k = item_k(cur), j = item_j(cur);
      const int inext = i + S;
      int4 en = make_int4(-1, -1, -1, -1);  // the next item's entries are in flight while this one is copied
      uint32_t nxt = 0;
      if (inext < n_items) {
        nxt = items[inext];
        en = __ldg(reinterpret_cast<const int4*>(p.tbl + (int64_t)item_k(nxt) * p.tstride + (int64_t)ltile[item_tile(nxt)] * kTileM) + lane);
      }
      const int s = warp;
      const uint32_t stage = a_base + (uint32_t)s * a_stage;
      TRACE(warp, i / S, 0);
      if (!mbar_wait(a_empty(s), (((uint32_t)i / (uint32_t)S) & 1u) ^ 1u, abort_flag)) goto done;
      TRACE(warp, i / S, 1);
      const int w = (j == p.nb - 1) ? p.last_w : 8;  // 16-byte chunks of this block's rows
      const bool tma = p.use_tma && w == 8;
      if (lane == 0) {  // this K-block's weight block rides on the same barrier as the gathered rows
        mbar_arrive_expect_tx(a_full(s), (uint32_t)(1 + p.x3) * b_bytes + (tma ? (uint32_t)kStageBytes : 0u));
        bulk_g2s(b_base + (uint32_t)s * b_stage, p.wimg + ((size_t)k * p.img_nb + j) * p.img_rows * kKBlock, b_bytes, a_full(s));
        if (p.x3)
          bulk_g2s(b_base + (uint32_t)s * b_stage + b_stride, p.wimg_lo + ((size_t)k * p.img_nb + j) * p.img_rows * kKBlock, b_bytes, a_full(s));
      }
      if (tma) {
        // One tile::gather4 per lane: rows 4 lane .. 4 lane + 3 of the K-block (128 bytes each, swizzled by the TMA
        // unit, zeros for absent rows = an out-of-bounds row coordinate) -- the whole 16 KB stage is ONE warp
        // instruction, no per-row address arithmetic in the SM.
        tma_gather4(stage + (uint32_t)lane * 512u, &p.tmap, j * kKBlock, e.x < 0 ? p.oob_row : e.x, e.y < 0 ? p.oob_row : e.y,
                    e.z < 0 ? p.oob_row : e.z, e.w < 0 ? p.oob_row : e.w, a_full(s));
        mbar_arrive(a_full(s));
      } else {
        asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(ent + (uint32_t)lane * 16u), "r"(e.x), "r"(e.y), "r"(e.z), "r"(e.w) : "memory");
        __syncwarp();
        // (addresses in 4-byte units: a K-block is 128 bytes of a row in both element types)
        const uint32_t row_units = (uint32_t)p.ld_in;
        const float* src0 = p.in + j * kKBlock;
        if (w == 8)      gather_block<8, false>(stage, ent, p.in, src0, row_units, lane);
        else if (w == 4) gather_block<4, false>(stage, ent, p.in, src0, row_units, lane);
        else if (w == 2) gather_block<2, false>(stage, ent, p.in, src0, row_units, lane);
        else             gather_block<8, false>(stage, ent, p.in, src0, row_units, lane, w);  // (6: BF16 rows of 48 mod 64 channels)
        if (p.x3) {  // the same rows of the lo plane, behind the hi block
          const float* src1 = p.in_lo + j * kKBlock;
          if (w == 8) gather_block<8, false>(stage + kStageBytes, ent, p.in_lo, src1, row_units, lane);
          else        gather_block<4, false>(stage + kStageBytes, ent, p.in_lo, src1, row_units, lane);
        }
        cp_async_arrive(a_full(s));
        __syncwarp();  // the entry row is rewritten by the next item
      }
      TRACE(warp, i / S, 2);
      e = en;
      cur = nxt;
      i = inext;
    }
  } else if (warp < kProducers + 4) {
    // =================================================================== epilogue
    const int ew = warp & 3;  // a warp may only touch TMEM lanes 32*(warp%4) .. +31
    for (uint32_t tile_iter = 0; tile_iter < (uint32_t)n_local; ++tile_iter) {
      const int ab = (int)(tile_iter & 1u);
      const int tile = (int)ltile[tile_iter];
      const int row = __ldg(p.perm + (int64_t)tile * kTileM + ew * 32 + lane);
      // which issuers had items of this tile (an accumulator nobody wrote holds the previous tile's values)
      const uint32_t i0 = item0[tile_iter], i1 = item0[tile_iter + 1];
      const bool two = split == 2 && i1 - i0 >= 2;
      const int only = (int)(i0 & 1u) & (split - 1);  // the issuer of a one-item tile
      if (ew == 0) TRACE(kProducers + 1, tile_iter, 0);
      if (!mbar_wait_sleep(acc_full(ab), (tile_iter >> 1) & 1u, abort_flag, 100)) goto done;
      if (ew == 0) TRACE(kProducers + 1, tile_iter, 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(ab * split * p.n_pad);
      for (int c0 = 0; c0 < p.n_pad; c0 += 16) {
        float acc[16];
        tmem_ld16(taddr + (uint32_t)((two ? 0 : only) * p.n_pad + c0), acc);
        if (two) {
          float acc1[16];
          tmem_ld16(taddr + (uint32_t)(p.n_pad + c0), acc1);
#pragma unroll
          for (int q = 0; q < 16; ++q) acc[q] += acc1[q];
        }
        if constexpr (std::is_same<P, TcEpiParams>::value) {
          if (row >= 0) {
            const float* add = p.add ? p.add + (int64_t)row * p.ld_out + c0 : nullptr;
            if (((p.c_out | p.ld_out) & 3) == 0) {
#pragma unroll
              for (int jj = 0; jj < 16; jj += 4)
                if (c0 + jj < p.c_out) {
                  float v[4] = {acc[jj], acc[jj + 1], acc[jj + 2], acc[jj + 3]};
                  if (add) {
                    const float4 t = *reinterpret_cast<const float4*>(add + jj);
                    v[0] += t.x; v[1] += t.y; v[2] += t.z; v[3] += t.w;
                  }
                  epi_store<4>(p.epi, row, c0 + jj, v);
                }
            } else {
#pragma unroll
              for (int jj = 0; jj < 16; ++jj)
                if (c0 + jj < p.c_out) {
                  const float v[1] = {add ? add[jj] + acc[jj] : acc[jj]};
                  epi_store<1>(p.epi, row, c0 + jj, v);
                }
            }
          }
        } else if (row >= 0) {
          float* dst = p.out + (int64_t)row * p.ld_out + c0;
          if (((p.c_out | p.ld_out) & 3) == 0) {
#pragma unroll
            for (int jj = 0; jj < 16; jj += 4)
              if (c0 + jj < p.c_out) {
                float4 o = make_float4(acc[jj], acc[jj + 1], acc[jj + 2], acc[jj + 3]);
                if (p.add) {  // (each row is owned by one thread: a plain read-modify-write when add == out)
                  const float4 t = *reinterpret_cast<const float4*>(p.add + (int64_t)row * p.ld_out + c0 + jj);
                  o.x += t.x; o.y += t.y; o.z += t.z; o.w += t.w;
                }
                *reinterpret_cast<float4*>(dst + jj) = o;
              }
          } else {
#pragma unroll
            for (int jj = 0; jj < 16; ++jj)
              if (c0 + jj < p.c_out) dst[jj] = p.add ? p.add[(int64_t)row * p.ld_out + c0 + jj] + acc[jj] : acc[jj];
          }
        }
      }
      tc_fence_before();
      mbar_arrive(acc_empty(ab));
      if (ew == 0) TRACE(kProducers + 1, tile_iter, 2);
    }
  } else {
    // =================================================================== MMA issuers: the whole warp runs the loop
    // (warp-uniform control flow), one elected lane issues.  Issuer m takes the items with i % split == m.
    const int m = warp - (kProducers + 4);
    if (m < split) {
      const uint32_t idesc = p.bf16 ? make_idesc_bf16(kTileM, p.n_pad) : make_idesc_tf32(kTileM, p.n_pad);
      const uint64_t desc0 = make_desc_sw128(0);
      uint32_t n_mine = 0;
      (void)n_mine;
      for (uint32_t tile_iter = 0; tile_iter < (uint32_t)n_local; ++tile_iter) {
        const int ab = (int)(tile_iter & 1u);
        const int i0 = (int)item0[tile_iter], i1 = (int)item0[tile_iter + 1];
        TRACE(kProducers + 2 + m, n_mine, 3);
        if (!mbar_wait(acc_empty(ab), ((tile_iter >> 1) & 1u) ^ 1u, abort_flag)) goto done;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)((ab * split + m) * p.n_pad);
        uint32_t acc = 0u;
        int i = i0 + (((i0 & (split - 1)) == m) ? 0 : 1);
        if (split == 1) i = i0;
        for (; i < i1; i += split) {
          const int s = i % S;
          const int ksteps = (item_j(items[i]) == p.nb - 1 ? p.last_w : 8) >> 1;
          TRACE(kProducers + 2 + m, n_mine, 0);
          if (!mbar_wait(a_full(s), ((uint32_t)i / (uint32_t)S) & 1u, abort_flag)) goto done;
          TRACE(kProducers + 2 + m, n_mine, 1);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t a_desc = desc0 + desc_addr(a_base + (uint32_t)s * a_stage);
            const uint64_t b_desc = desc0 + desc_addr(b_base + (uint32_t)s * b_stage);
            if (p.bf16) {  // K-steps of 16 BF16 elements = 32 bytes (1..4 per block)
              umma_f16(d_tmem, a_desc, b_desc, idesc, acc);
#pragma unroll
              for (int q = 1; q < 4; ++q)
                if (q < ksteps) umma_f16(d_tmem, a_desc + 2 * q, b_desc + 2 * q, idesc, 1u);
            } else {
              umma_tf32(d_tmem, a_desc, b_desc, idesc, acc);
              umma_tf32(d_tmem, a_desc + 2, b_desc + 2, idesc, 1u);  // +32 bytes per K-step of 8
              if (ksteps == 4) {
                umma_tf32(d_tmem, a_desc + 4, b_desc + 4, idesc, 1u);
                umma_tf32(d_tmem, a_desc + 6, b_desc + 6, idesc, 1u);
              }
            }
            if (p.x3) {  // + lo.Whi + hi.Wlo (the lo blocks sit one block behind the hi ones)
              const uint64_t a_lo = a_desc + (kStageBytes >> 4), b_lo = b_desc + (b_stride >> 4);
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                if (q < ksteps) {
                  umma_tf32(d_tmem, a_lo + 2 * q, b_desc + 2 * q, idesc, 1u);
                  umma_tf32(d_tmem, a_desc + 2 * q, b_lo + 2 * q, idesc, 1u);
                }
              }
            }
            umma_commit(a_empty(s));  // frees the stage and its weight block
          }
          __syncwarp();
          TRACE(kProducers + 2 + m, n_mine, 2);
          ++n_mine;
          acc = 1u;
        }
        if (elect_one()) umma_commit(acc_full(ab));  // (arrives at once when this issuer had no item of the tile)
        __syncwarp();
      }
    }
  }
done:
  asm volatile("cp.async.wait_all;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0 && *abort_flag) mm3d_raise(p.err);
#ifdef MM3D_TRACE
  if (p.trace && threadIdx.x == 0) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    p.trace[4096 + 2 * blockIdx.x + 1] = (long long)gt;
  }
#endif
  if (warp == kProducers + 4) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

int pow2_cols(int n) {
  int c = 32;
  while (c < n) c <<= 1;
  return c;
}

}  // namespace

// ---- host entry points used by capi.cu -------------------------------------------------------
#ifdef MM3D_TRACE
static long long* g_trace = nullptr;
extern "C" __attribute__((visibility("default"))) void mm3d_debug_set_trace(long long* p) { g_trace = p; }
long long* mm3d_debug_trace_ptr() { return g_trace; }
#endif

// Tensor map of a row-major [rows, c] float32 feature tensor for row gathers: box = {32 channels, 1 row} (a
// tile::gather4 moves 4 such rows), 128-byte swizzle -- plain for K-major MMA operands, 32-byte-atom for the MN-major
// ones of the weight-gradient kernel.  Columns past c and rows past `rows` read as zeros.  false = TMA not available
// (the kernels then gather with cp.async).
bool mm3d_encode_rows_tmap(CUtensorMap* tm, const float* base, int64_t rows, int c, bool atom32) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeFn)f;
    else
      (void)cudaGetLastError();
  }
  if (!fn || (((uintptr_t)base) & 15) != 0 || (c % 4) != 0) return false;
  const cuuint64_t dims[2] = {(cuuint64_t)c, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)c * 4};
  const cuuint32_t box[2] = {32, 1};
  const cuuint32_t estr[2] = {1, 1};
  return fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            atom32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// One launch takes up to kSliceIn input channels (8 K-blocks: the item's 3-bit block index) and kSliceOut output
// columns (the double-buffered accumulator in 512 TMEM columns).  Wider layers, up to kWide channels on either side,
// run as slices (mm3d_conv_fwd_tc_img): output-column slices of near-equal multiples of 16, each a contiguous row
// range of every block of the full-width weight image; input-channel slices of kSliceIn that accumulate through the
// epilogue's addend.  The reference widths are one slice, the same launch as without slicing.
constexpr int kSliceIn = 256, kSliceOut = 256, kWide = 512;

// geometry of the full-width weight image
static int tc_geometry(int c_in, int c_out, int K, int* nb, int* n_pad, int bf16 = 0) {
  *nb = bf16 ? (c_in + 63) / 64 : (c_in + 31) / 32;
  *n_pad = (c_out + 15) / 16 * 16;
  // input rows are cut into 128-byte blocks with an optional 64-byte tail
  return (*n_pad <= kWide && (c_in % 16) == 0 && c_in <= kWide && K <= 32) ? 0 : 1;
}

// 1 when the tcgen05 kernel handles this shape
int mm3d_conv_tc_supported(int c_in, int c_out, int K) {
  int nb, n_pad;
  return tc_geometry(c_in, c_out, K, &nb, &n_pad) == 0;
}

size_t mm3d_conv_tc_workspace_bytes(int c_in, int c_out, int K) {
  int nb, n_pad;
  if (tc_geometry(c_in, c_out, K, &nb, &n_pad)) return 0;
  return mm3d_align((size_t)K * nb * n_pad * 128);  // weight image
}

// Sticky per-device error words (mm3d_raise, common.cuh) in MAPPED PINNED host memory: a kernel whose bounded wait
// timed out (never in a correct build; it turns a would-be GPU hang into a reportable error) or that met an
// out-of-image lift index stores 1 there, and the host reads the words without any CUDA call or synchronisation --
// the executor polls them at every forward / backward call.
static int* g_err_host[64] = {nullptr};
static int* g_err_dev[64] = {nullptr};
int* mm3d_device_err_flag() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  if (!g_err_dev[dev]) {
    int* h = nullptr;
    if (cudaHostAlloc(&h, 64, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }
    for (int i = 0; i < 16; ++i) h[i] = 0;
    int* d = nullptr;
    if (cudaHostGetDevicePointer(&d, h, 0) != cudaSuccess) { (void)cudaGetLastError(); cudaFreeHost(h); return nullptr; }
    g_err_host[dev] = h;
    g_err_dev[dev] = d;
  }
  return g_err_dev[dev];
}

static int g_sm_count[64] = {0};
int mm3d_sm_count() {
  const int dev = mm3d_device_slot();
  if (!g_sm_count[dev]) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) { (void)cudaGetLastError(); n = MM3D_NUM_SMS; }
    g_sm_count[dev] = n;
  }
  return g_sm_count[dev];
}

// Bits: 1 = a kernel pipeline / grid barrier timed out, 2 = a lift index outside the image.  Reads and clears the
// current device's words; no synchronisation (callers that want everything enqueued so far synchronise first).
extern "C" int mm3d_take_device_error(void) {
  if (!mm3d_device_err_flag()) return -1;
  volatile int* h = g_err_host[mm3d_device_slot()];
  int v = 0;
  if (h[0]) { v |= 1; h[0] = 0; }
  if (h[1]) { v |= 2; h[1] = 0; }
  return v;
}

// images of several layers in one launch; descs[i] = {weight, image buffer (mm3d_conv_tc_workspace_bytes), K, c_in,
// c_out, flags}
int mm3d_conv_tc_build_images(const float* const* weights, float* const* images, const int* K, const int* c_in,
                              const int* c_out, const int* flags, int n, cudaStream_t stream) {
  for (int first = 0; first < n; first += kMaxImgBatch) {
    WImgBatch b;
    b.n = 0;
    int blocks = 0;
    for (int i = first; i < n && i < first + kMaxImgBatch; ++i) {
      WImgItem& it = b.item[b.n++];
      it.bf16 = (flags[i] & MM3D_CONV_BF16) ? 1 : 0;
      MM3D_REQUIRE(tc_geometry(c_in[i], c_out[i], K[i], &it.nb, &it.n_pad, it.bf16) == 0, MM3D_ERR_UNSUPPORTED,
                   "tcgen05 conv: unsupported shape c_in %d c_out %d K %d", c_in[i], c_out[i], K[i]);
      it.w = weights[i]; it.img = images[i]; it.K = K[i]; it.c_in = c_in[i]; it.c_out = c_out[i];
      it.transposed = (flags[i] & MM3D_CONV_TRANSPOSE_W) ? 1 : 0;
      it.mirror = (flags[i] & MM3D_CONV_MIRROR_K) ? 1 : 0;
      it.lo = (flags[i] & MM3D_CONV_WEIGHT_LO) ? 1 : 0;
      it.block0 = blocks;
      int nb_blocks = (int)mm3d_cdiv((int64_t)it.K * it.nb * it.n_pad * (it.bf16 ? 2 * kKBlock : kKBlock), 256 * 8);
      blocks += nb_blocks < 1 ? 1 : nb_blocks;
    }
    if (blocks == 0) continue;
    MM3D_CUDA(mm3d_launch_pdl(k_weight_images, dim3(blocks), dim3(256), 0, stream, b));
    mm3d_count_launches(1);
    MM3D_CHECK_LAUNCH("mm3d_conv_tc_build_images");
  }
  return MM3D_OK;
}

int mm3d_conv_fwd_tc_img(const float* in, int64_t n_in, int c_in, float* out, int64_t n_out, int c_out,
                         const float* wimg, int K, const void* plan, int64_t plan_cap, const float* add, cudaStream_t stream,
                         const float* wimg_lo = nullptr, int bf16 = 0, const ConvEpi* epi = nullptr);

int mm3d_conv_fwd_tc(const float* in, int64_t n_in, int c_in, float* out, int64_t n_out, int c_out,
                     const float* weight, int K, const void* plan, int64_t plan_cap, int flags, void* ws,
                     size_t ws_bytes, cudaStream_t stream) {
  int nb, n_pad;
  const int bf16 = (flags & MM3D_CONV_BF16) ? 1 : 0;
  MM3D_REQUIRE(tc_geometry(c_in, c_out, K, &nb, &n_pad, bf16) == 0, MM3D_ERR_UNSUPPORTED,
               "tcgen05 conv: unsupported shape c_in %d c_out %d K %d", c_in, c_out, K);
  MM3D_REQUIRE(!(bf16 && (flags & MM3D_CONV_X3)), MM3D_ERR_INVALID, "tcgen05 conv: BF16 and TF32x3 exclude each other");
  MM3D_REQUIRE(ws && ws_bytes >= mm3d_conv_tc_workspace_bytes(c_in, c_out, K) * ((flags & MM3D_CONV_X3) ? 2 : 1), MM3D_ERR_WORKSPACE,
               "tcgen05 conv: workspace too small");
  const bool tr = (flags & MM3D_CONV_TRANSPOSE_W) != 0, mir = (flags & MM3D_CONV_MIRROR_K) != 0;
  MM3D_REQUIRE(tr || !mir, MM3D_ERR_UNSUPPORTED, "MIRROR_K without TRANSPOSE_W not implemented");
  if (n_out == 0) return MM3D_OK;
  float* wimg = (float*)ws;
  k_weight_image<<<mm3d_grid((int64_t)K * nb * n_pad * (bf16 ? 2 * kKBlock : kKBlock), 256), 256, 0, stream>>>(
      weight, wimg, K, c_in, c_out, nb, n_pad, tr ? 1 : 0, mir ? 1 : 0, 0, bf16);
  mm3d_count_launches(1);
  // BF16 mode: `in` holds an FP32 plane and, n_in * c_in floats behind it, the BF16 plane that is gathered
  if (bf16) return mm3d_conv_fwd_tc_img(in + n_in * (int64_t)c_in, n_in, c_in, out, n_out, c_out, wimg, K, plan, plan_cap, nullptr, stream, nullptr, 1);
  if (!(flags & MM3D_CONV_X3)) return mm3d_conv_fwd_tc_img(in, n_in, c_in, out, n_out, c_out, wimg, K, plan, plan_cap, nullptr, stream);
  // Error-compensated mode: `in` holds two planes, hi = tf32(x) and lo = tf32(x - hi) ([n_in, c_in] each), the
  // workspace two weight images; out = hi.Whi + lo.Whi + hi.Wlo, accumulated in FP32 (the dropped lo.Wlo term and the
  // roundings of the lo parts are ~2^-22 relative)
  float* wimg_lo = wimg + mm3d_conv_tc_workspace_bytes(c_in, c_out, K) / sizeof(float);
  k_weight_image<<<mm3d_grid((int64_t)K * nb * n_pad * kKBlock, 256), 256, 0, stream>>>(weight, wimg_lo, K, c_in, c_out, nb,
                                                                                    n_pad, tr ? 1 : 0, mir ? 1 : 0, 1, 0);
  mm3d_count_launches(1);
  return mm3d_conv_fwd_tc_img(in, n_in, c_in, out, n_out, c_out, wimg, K, plan, plan_cap, nullptr, stream, wimg_lo);
}

template <class P>
static int set_conv_tc_attributes() {
  static bool once_dev[64] = {false};
  bool& once = once_dev[mm3d_device_slot()];
  if (!once) {
    MM3D_CUDA(cudaFuncSetAttribute(k_conv_tc<P>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
    MM3D_CUDA(cudaFuncSetAttribute(k_conv_tc<P>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    once = true;
  }
  return MM3D_OK;
}

// One launch over a slice: input channels [ci0, ci0 + c_in) of rows ld_in units apart (in / in_lo at ci0), output
// columns [co0, co0 + c_out) of rows ld_out floats apart (out / add / wimg / wimg_lo / epi already at the slice)
static int conv_tc_launch(const float* in, const float* in_lo, int ld_in, int64_t n_in, int c_in, float* out, int ld_out,
                          int64_t n_out, int c_out, const float* wimg, const float* wimg_lo, int img_nb, int img_rows, int K,
                          const Mm3dPlanView& pv, const float* add, cudaStream_t stream, int bf16, const ConvEpi* epi,
                          bool whole) {
  const int nb = bf16 ? (c_in + 63) / 64 : (c_in + 31) / 32, n_pad = (c_out + 15) / 16 * 16;
  TcParams p;
  p.in = in; p.out = out; p.wimg = wimg;
  p.perm = pv.perm; p.tile_mask = pv.tile_mask; p.order = pv.order; p.tbl = pv.tbl; p.tstride = pv.stride;
  p.c_in = c_in; p.c_out = c_out; p.K = K; p.nb = nb;
  p.ld_in = ld_in; p.ld_out = ld_out; p.img_nb = img_nb; p.img_rows = img_rows;
  // chunks of an offset's last block: TF32 rows are whole 64-byte pieces, BF16 rows whole 32-byte pieces
  p.last_w = bf16 ? ((c_in % 64) ? (c_in % 64) / 8 : 8) : ((c_in % 32) == 16 ? 4 : 8);
  p.bf16 = bf16;
  p.n_pad = n_pad;
  p.num_tiles = (int)mm3d_cdiv(n_out, kTileM);
  p.err = mm3d_device_err_flag();
  p.add = add;
  p.x3 = wimg_lo ? 1 : 0;
  p.in_lo = in_lo;
  p.wimg_lo = wimg_lo;
#ifdef MM3D_TRACE
  p.trace = g_trace;
  p.trace_cta = getenv("MM3D_TC_TRACE_CTA") ? atoi(getenv("MM3D_TC_TRACE_CTA")) : 0;
#endif
  p.use_tma = 0;
  p.oob_row = (int)n_in;
  // Row gathers: 16-byte cp.async by default.  MM3D_TC_GATHER=tma selects TMA tile::gather4 for whole 32-channel
  // blocks instead (one instruction per 4 rows, no address arithmetic in the SM): measured on B200 it is on par
  // for 64+ input channels and slower for 32 (the TMA unit takes ~4 cycles per 128-byte row and is shared by the SM's
  // CTAs), 1 % slower over the whole step -- kept selectable for that comparison (DESIGN.md section 7).
  static const bool want_tma = [] { const char* e = getenv("MM3D_TC_GATHER"); return e && strcmp(e, "tma") == 0; }();
  if (want_tma && whole && !wimg_lo && !bf16 && n_in > 0 && n_in < (1ll << 31) - 1) {
    p.use_tma = mm3d_encode_rows_tmap(&p.tmap, in, n_in, c_in, /*atom32=*/false) ? 1 : 0;
  }
  const uint32_t b_stride = ((uint32_t)n_pad * 128u + 1023u) & ~1023u;
  const size_t per_stage = ((size_t)kStageBytes + b_stride) * (wimg_lo ? 2 : 1);
  if (int rc = epi ? set_conv_tc_attributes<TcEpiParams>() : set_conv_tc_attributes<TcParams>()) return rc;
  // Two issuer warps with their own accumulators (double buffered: 4 x n_pad TMEM columns) whenever they fit.
  // Two CTAs per SM when the layer has more tiles than SMs, each CTA's accumulators fit half the TMEM and half the
  // shared memory still holds a ring of >= 4 stages; one CTA per SM with a deeper ring otherwise.  S is even (ring
  // stage s is consumed by issuer s % 2).
  const int sms = mm3d_sm_count();
  p.split = 4 * n_pad <= 512 ? 2 : 1;
  p.tmem_cols = pow2_cols(2 * p.split * n_pad);
  const size_t fixed = 1024 + (size_t)kProducers * kEntBytes + 8 * (2 * kMaxStages + 4) + 64 + 64;
  const int two = (int)((108 * 1024 - fixed) / per_stage), one = (int)((218 * 1024 - fixed) / per_stage);
  // (measured: two CTAs per SM win for one-block layers (c_in <= 32), one CTA with the deeper ring from 64 channels on)
  int per_sm = (p.num_tiles > sms && nb == 1 && two >= 4 && 2 * p.tmem_cols <= 512) ? 2 : 1;
  if (const char* e = getenv("MM3D_TC_PER_SM")) {  // A/B measurements: 2 = two CTAs per SM wherever they fit
    if (atoi(e) == 2 && p.num_tiles > sms && two >= 2 && 2 * p.tmem_cols <= 512) per_sm = 2;
    if (atoi(e) == 1) per_sm = 1;
  }
  int S = per_sm == 2 ? two : one;
  if (S > kMaxStages) S = kMaxStages;
  S &= ~1;
  MM3D_REQUIRE(S >= 2, MM3D_ERR_UNSUPPORTED, "tcgen05 conv: a K-block of %d output channels does not fit the ring", n_pad);
  p.S = S;
  const size_t smem_fixed = fixed + (size_t)S * per_stage;
  // Per-CTA lists (tile masks / indices / first items: 12 bytes per tile; items: 2 bytes each) live in shared memory
  // next to the ring.  Row counts whose lists do not fit are processed in several launches over consecutive pieces of
  // the plan's tile order (tiles are independent).
  const size_t list_budget = (per_sm == 2 ? 110 * 1024 : 224 * 1024) - smem_fixed;
  const size_t per_tile = 12 + 2 * (size_t)K * nb;
  int64_t max_local = (int64_t)((list_budget - 64) / per_tile);
  if (max_local > 255) max_local = 255;  // (8 bits of local tile index per item)
  MM3D_REQUIRE(max_local >= 1, MM3D_ERR_UNSUPPORTED, "tcgen05 conv: no shared memory left for the item list");
  const int all_tiles = p.num_tiles;
  const int64_t max_tiles = max_local * sms * per_sm;
  for (int64_t start = 0; start < all_tiles; start += max_tiles) {
    const int cnt = (int)(all_tiles - start < max_tiles ? all_tiles - start : max_tiles);
    p.order = pv.order + start;
    p.num_tiles = cnt;
    int grid = sms * per_sm;
    if (grid > cnt) grid = cnt;
    p.n_local = (cnt + grid - 1) / grid;
    p.max_items = p.n_local * K * nb;
    const size_t smem = smem_fixed + (((size_t)(3 * p.n_local + 1) * 4 + 15) & ~(size_t)15) + (((size_t)p.max_items * 2 + 15) & ~(size_t)15);
    MM3D_REQUIRE(smem <= 226 * 1024, MM3D_ERR_UNSUPPORTED, "tcgen05 conv: shared memory budget exceeded");
    if (epi) {
      TcEpiParams pe;
      static_cast<TcParams&>(pe) = p;
      pe.epi = *epi;
      MM3D_CUDA(mm3d_launch_pdl(k_conv_tc<TcEpiParams>, dim3(grid), dim3(kThreads), smem, stream, pe));
    } else {
      MM3D_CUDA(mm3d_launch_pdl(k_conv_tc<TcParams>, dim3(grid), dim3(kThreads), smem, stream, p));
    }
    mm3d_count_launches(1);
  }
  return MM3D_OK;
}

// the convolution proper, from a prebuilt weight image
// wimg_lo != NULL: the TF32x3 form -- `in` carries a lo plane n_in * c_in floats behind the hi one, wimg_lo is the image of
// the weights' TF32 remainder, and every item is three products (one launch, one gather of both planes)
// epi != NULL: the inference form -- the epilogue writes to epi's destinations; `out` is not written,
// except for the partial sums of the input-channel slices before the last when c_in > kSliceIn
int mm3d_conv_fwd_tc_img(const float* in, int64_t n_in, int c_in, float* out, int64_t n_out, int c_out,
                         const float* wimg, int K, const void* plan, int64_t plan_cap, const float* add, cudaStream_t stream,
                         const float* wimg_lo, int bf16, const ConvEpi* epi) {
  int nb, n_pad;
  MM3D_REQUIRE(!(bf16 && wimg_lo), MM3D_ERR_INVALID, "tcgen05 conv: BF16 and TF32x3 exclude each other");
  MM3D_REQUIRE(tc_geometry(c_in, c_out, K, &nb, &n_pad, bf16) == 0, MM3D_ERR_UNSUPPORTED,
               "tcgen05 conv: unsupported shape c_in %d c_out %d K %d", c_in, c_out, K);
  MM3D_REQUIRE(n_out < (1ll << 31) && n_in * (int64_t)c_in < (1ll << 32), MM3D_ERR_UNSUPPORTED,
               "tcgen05 conv: tensor too large for 32-bit element offsets");
  MM3D_REQUIRE(plan && plan_cap >= n_out, MM3D_ERR_INVALID, "tcgen05 conv: needs a row plan covering n_out rows");
  MM3D_REQUIRE((((uintptr_t)in | (uintptr_t)out | (uintptr_t)wimg | (uintptr_t)add) & 15) == 0, MM3D_ERR_INVALID,
               "tcgen05 conv: pointers must be 16-byte aligned");
  if (epi && (c_out & 3) == 0) {  // the epilogue stores whole float4s (BF16 planes: 8-byte groups of four)
    MM3D_REQUIRE(epi->n >= 1 && epi->n <= kEpiDsts, MM3D_ERR_INVALID, "tcgen05 conv: %d epilogue destinations", epi->n);
    for (int i = 0; i < epi->n; ++i) {
      const EpiDst& d = epi->d[i];
      const uintptr_t a = (d.store == 4 ? 0 : (uintptr_t)d.p) | (d.store == 2 ? (uintptr_t)d.p2 : 0);
      MM3D_REQUIRE((d.ld & 3) == 0 && (a & 15) == 0 && (d.store < 3 || ((uintptr_t)d.p2 & 7) == 0), MM3D_ERR_INVALID,
                   "tcgen05 conv: epilogue destination %d not aligned for vector stores (ld %d)", i, d.ld);
    }
  }
  if (n_out == 0) return MM3D_OK;
  const Mm3dPlanView pv = mm3d_plan_view(plan, plan_cap);
  const int col_step = mm3d_slice_step(c_out, kSliceOut, 16);
  const int units = bf16 ? 2 : 1;  // channels per 4-byte unit of `in`
  const int per_blk = bf16 ? 2 * kKBlock : kKBlock;
  MM3D_REQUIRE(!epi || c_in <= kSliceIn || out, MM3D_ERR_INVALID,
               "tcgen05 conv: the inference form of c_in %d > %d needs `out` for the partial sums", c_in, kSliceIn);
  for (int co0 = 0; co0 < c_out; co0 += col_step) {
    const int w = c_out - co0 < col_step ? c_out - co0 : col_step;
    ConvEpi e;
    if (epi) e = epi_columns(*epi, co0);
    for (int ci0 = 0; ci0 < c_in; ci0 += kSliceIn) {
      const int cw = c_in - ci0 < kSliceIn ? c_in - ci0 : kSliceIn;
      const bool last = ci0 + cw == c_in;
      // input slices after the first add to the partial sum in `out`; only the last one runs the inference epilogue
      const float* a = ci0 ? out + co0 : add ? add + co0 : nullptr;
      const size_t img_off = ((size_t)(ci0 / per_blk) * n_pad + co0) * kKBlock;
      int rc = conv_tc_launch(in + ci0 / units, in + n_in * (int64_t)c_in + ci0, c_in / units, n_in, cw,
                              out ? out + co0 : nullptr, c_out, n_out, w, wimg + img_off, wimg_lo ? wimg_lo + img_off : nullptr,
                              nb, n_pad, K, pv, a, stream, bf16, epi && last ? &e : nullptr, w == c_out && cw == c_in);
      if (rc) return rc;
    }
  }
  MM3D_CHECK_LAUNCH("mm3d_conv_fwd_tc");
  return MM3D_OK;
}
