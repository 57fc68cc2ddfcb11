// tcgen05 / TMEM weight gradient of the rule-table convolution for sm_100a, driven by a row plan.
//
//   dW[k][ci][co] = sum_j in[tbl(j,k)][ci] * dout[j][co]
//
// Per tile of 128 output rows (plan order) and NON-EMPTY offset k this is one small GEMM whose reduction
// runs over the tile's rows:
//   dW[k] [ci x co] += A_{tile,k}^T [ci x 128] . G_tile [128 x co]
// A = the gathered, zero-filled input rows (the stage the forward kernel builds, here with the
// 32-byte-granule swizzle that MN-major tf32 operands require, SWIZZLE_128B_BASE32B), G = the tile's 128
// dout rows.  Both operands are MN-major; the MMA's K dimension is the tile's rows (16 tcgen05.mma of K = 8
// per item), M = the gathered input channels (64 or 128 accumulator lanes; c_in > 128 is cut into two
// M-blocks), N = c_out.  An accumulator therefore costs c_out TMEM columns per offset (not c_in, as with the
// roles the other way round): the decoder layers (c_in = 2 c_out) keep twice as many offsets resident.  A CTA
// covers a GROUP of offsets whose accumulators fit the 512 columns -- all 27 for the 16-channel layers -- and
// the dout tile is loaded once per (tile, group).  ONE pipeline item = (tile, offset, M-block) with all its
// channel blocks: 16 MMAs of M x c_out x 8 per hand-shake.  Accumulators stay in TMEM for the whole kernel
// and are added to dW once at the end, each lane (= input channel) flushing its contiguous c_out floats with
// red.global.add.v4.f32.  Offsets are dealt to groups by class (centre, faces, edges, corners); how many
// CTAs a group gets is decided in the kernel from the plan's per-offset tile counts.
//
// Warp roles (13 warps): 0..7 producers (each owns 16 rows of every stage: gathers A, and the dout tile when
// a new tile starts), 8..11 epilogue (TMEM -> red.add), 12 MMA issuer + TMEM allocator.
#include <cstdlib>
#include "plan.cuh"
#include "tc_common.cuh"

namespace {

using namespace tc;

constexpr int kTileM = 128;
constexpr int kBlockBytes = kTileM * 128;  // one 32-channel block of 128 rows
constexpr int kMaxStages = 6;
constexpr int kMaxGBufs = 4;
constexpr int kProducers = 8;              // producer warps; each owns 128 / 8 = 16 rows of every item
constexpr int kRowsPerWarp = kTileM / kProducers;
constexpr int kThreads = (kProducers + 5) * 32;

struct WgParams {
  const float* in;
  const float* dout;
  float* dw;
  const int32_t* perm;
  const uint32_t* tile_mask;
  const int32_t* order;
  const uint32_t* off_tiles;
  const int32_t* tbl;
  int64_t tstride;
  int c_in, c_out, K;
  int ld_in, ld_dout;  // row strides of `in` / `dout` in 4-byte units (c_in, c_out; halved for BF16 planes; wider for a slice)
  int dw_ld;           // dW[k] row stride (c_out unless a slice)
  int64_t dw_k;        // dW offset stride (c_in * c_out unless a slice)
  int nmb;          // M-blocks per offset: 1, or 2 when c_in > 128
  int cm;           // input channels per M-block = c_in / nmb
  int nbi;          // 32-channel shared-memory blocks of one item = ceil(cm / 32)
  int last_w;       // 16-byte chunks of an item's last block (8, or 4 when cm % 32 == 16)
  int mm;           // UMMA M: 64 (cm <= 64) or 128
  int gblocks;      // 32-channel blocks of the dout tile = ceil(c_out / 32)
  int g_last_w;     // 16-byte chunks of its last block
  int S, gbufs;
  int num_tiles, tmem_cols;
  int n_local;      // tiles per CTA (upper bound: every group gets at least ceil(num_tiles / n_local) CTAs)
  int max_items;    // two-ring variant: capacity of one ring's item list
  int bf16;         // two-ring variant: `in` / `dout` are BF16 planes (64 channels per 128-byte block), kind::f16 MMAs of K = 16 rows
  int groups;       // offset groups; group g owns the offsets of gmask[g]; its CTAs are decided in the kernel
  uint32_t gmask[32];
  int* err;
  // deterministic variant: CTA b stores its accumulators to slab + b * slab_cta ([gk][c_in][c_out] floats), CTA 0 the
  // group -> first-CTA table to slab_cta0 [groups + 1]; k_wgrad_reduce sums them
  float* slab;
  int* slab_cta0;
  int64_t slab_cta;
#ifdef MM3D_TRACE
  long long* trace;  // development builds: clock64 stamps of CTA 0's roles, [role][64 records][4]
#endif
};

#ifdef MM3D_TRACE
#define TRACE(role, rec, slot)                                                                                   \
  do {                                                                                                           \
    if (p.trace && blockIdx.x == 0 && lane == 0 && (rec) < 64) p.trace[(((role) * 64) + (rec)) * 4 + (slot)] = clock64(); \
  } while (0)
#else
#define TRACE(role, rec, slot) do {} while (0)
#endif

// tiles of this CTA that contain at least one offset of its group, in order
struct TileWalk {
  const uint32_t* lmask;  // shared memory: [n_local] (mask & group) of this CTA's tiles, then [n_local] tile indices
  int n_local, lt, tile;
  uint32_t m;
  __device__ __forceinline__ void seek() {
    while (lt < n_local) {
      m = lmask[lt];
      if (m) { tile = (int)lmask[n_local + lt]; return; }
      ++lt;
    }
    m = 0;
  }
  __device__ __forceinline__ void init(const uint32_t* local_masks, int n_loc) {
    lmask = local_masks; n_local = n_loc; lt = 0; tile = 0;
    seek();
  }
  __device__ __forceinline__ bool valid() const { return lt < n_local; }
  __device__ __forceinline__ void next_tile() { ++lt; seek(); }
};

// items = (tile, offset, M-block) over TileWalk
struct ItemWalk {
  TileWalk t;
  int nmb, k, h;
  uint32_t rem;
  bool first;  // first item of its tile (the dout tile is loaded with it)
  __device__ __forceinline__ void init(const WgParams& p, const uint32_t* local_masks, int n_loc) {
    t.init(local_masks, n_loc); nmb = p.nmb; h = 0; rem = t.m; k = rem ? __ffs(rem) - 1 : 0; first = true;
  }
  __device__ __forceinline__ bool valid() const { return t.valid(); }
  __device__ __forceinline__ void next() {
    first = false;
    if (++h < nmb) return;
    h = 0;
    rem &= rem - 1;
    if (!rem) { t.next_tile(); rem = t.m; first = true; }
    k = rem ? __ffs(rem) - 1 : 0;
  }
};

// This warp's 16 rows of one operand tile (gathered input rows or dout rows): `nblk` 32-channel blocks, kBlockBytes
// apart, the last one 16 channels wide when `last_half`.  Lanes 0..15 hold the 16 source rows in `rowv` (negative =
// absent: zeros).  Row indices and source pointers are resolved ONCE per pass (4 shuffles + 4 address computations for
// the full-width blocks) and every block then costs one cp.async per pass: the copies go out back to back instead of
// each behind its own shuffle -> compare -> multiply chain (measured: the producers, not the MMA issuer, bound the
// kernel, at ~100 cycles per copy).  Full blocks: 8 lanes per row, 4 rows per pass; the 16-channel tail: 4 lanes per
// row, 8 rows per pass, a quarter-warp holding rows x and x + 2 (their 32-byte granules do not share banks).
__device__ __forceinline__ void gather_rows16(uint32_t tile_base, int row0, int rowv, const float* __restrict__ src0,
                                              uint32_t row_floats, int nblk, bool last_half, int lane) {
  const int nfull = last_half ? nblk - 1 : nblk;
  {
    const int c = lane & 7, rsub = lane >> 3;
    const float* ptr[4];
    uint32_t dst[4];
    bool absent[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int rl = u * 4 + rsub;
      const int row = __shfl_sync(0xffffffffu, rowv, rl);
      const int r = row0 + rl;
      absent[u] = row < 0;
      ptr[u] = src0 + (size_t)(uint32_t)max(row, 0) * row_floats + c * 4;
      dst[u] = tile_base + (uint32_t)r * 128u + swz_base32(c, r);
    }
#pragma unroll 1
    for (int j = 0; j < nfull; ++j) {
#pragma unroll
      for (int u = 0; u < 4; ++u) cp_async16_zfill(dst[u] + (uint32_t)j * kBlockBytes, ptr[u] + j * 32, absent[u]);
    }
  }
  if (last_half) {
    const int c = lane & 3, q = lane >> 2;
    const int rsub = (q & 4) | ((q & 1) << 1) | ((q >> 1) & 1);
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int rl = u * 8 + rsub;
      const int row = __shfl_sync(0xffffffffu, rowv, rl);
      const int r = row0 + rl;
      cp_async16_zfill(tile_base + (uint32_t)nfull * kBlockBytes + (uint32_t)r * 128u + swz_base32(c, r),
                       src0 + (size_t)(uint32_t)max(row, 0) * row_floats + nfull * 32 + c * 4, row < 0);
    }
  }
}

__device__ __forceinline__ void red_add_v4(float* dst, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// Deterministic epilogue (epilogue warp ew): this CTA's accumulators of EVERY offset of its group -> its own slab with
// plain stores, zeros for the offsets it never touched (their TMEM columns were never written), so that the reduction
// can sum a fixed set of CTAs without knowing which of them saw which offset.  Slab row = kidx (the offset's rank in
// the group), then the dW[k] layout [c_in][c_out].
__device__ __forceinline__ void flush_to_slab(const WgParams& p, uint32_t tmem_base, int ew, int lane, uint32_t gmask,
                                              uint32_t seen) {
  const int ci = p.mm == 128 ? ew * 32 + lane : ew * 16 + lane;
  const bool lane_ok = (p.mm == 128 || lane < 16) && ci < p.cm;
  float* slab = p.slab + (int64_t)blockIdx.x * p.slab_cta;
  int kidx = 0;
  for (uint32_t rem = gmask; rem; rem &= rem - 1, ++kidx) {
    const bool touched = (seen >> (__ffs(rem) - 1)) & 1u;
    for (int h = 0; h < p.nmb; ++h) {
      const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)((kidx * p.nmb + h) * p.c_out);
      float* dst = slab + ((int64_t)kidx * p.c_in + h * p.cm + ci) * p.c_out;
      for (int c0 = 0; c0 < p.c_out; c0 += 16) {
        float acc[16];
        if (touched) tmem_ld16(taddr + (uint32_t)c0, acc);  // (warp-uniform: every lane takes part)
        else {
#pragma unroll
          for (int q = 0; q < 16; ++q) acc[q] = 0.f;
        }
        if (lane_ok) {
#pragma unroll
          for (int q = 0; q < 16; q += 4)
            *reinterpret_cast<float4*>(dst + c0 + q) = make_float4(acc[q], acc[q + 1], acc[q + 2], acc[q + 3]);
        }
      }
    }
  }
}

// Deterministic variant, second launch: dW[k] = (accumulate ? dW[k] : 0) + sum of the slabs of the CTAs of the group
// that owns k, in ascending CTA index, in FP32.  Which CTAs those are comes from the plan, the shapes and the SM count
// only (the table the first launch's CTA 0 wrote), never from timing.
struct WgReduceParams {
  const float* slab;
  const int* cta0;
  float* dw;
  int64_t slab_cta;
  int c_in, c_out, K, accumulate, groups;
  int dw_ld;
  int64_t dw_k;
  uint32_t gmask[32];  // as WgParams::gmask
};

__global__ void __launch_bounds__(256)
k_wgrad_reduce(const WgReduceParams r) {
  const int64_t per_k = (int64_t)r.c_in * r.c_out;  // (a multiple of 256: float4 pieces never straddle an offset)
  const int64_t n4 = (int64_t)r.K * per_k / 4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(4 * i / per_k);
    const int64_t e = 4 * i - k * per_k;
    int g = 0;  // the group that owns k, and k's rank in it (constant indices: the table stays in parameter space)
    uint32_t gm = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (j < r.groups && ((r.gmask[j] >> k) & 1u)) { g = j; gm = r.gmask[j]; }
    const int b0 = __ldg(r.cta0 + g), b1 = __ldg(r.cta0 + g + 1);
    const float* src = r.slab + (int64_t)__popc(gm & ((1u << k) - 1u)) * per_k + e;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int b = b0; b < b1; ++b) {
      const float4 v = __ldcs(reinterpret_cast<const float4*>(src + (int64_t)b * r.slab_cta));
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    const int ci = (int)e / r.c_out, co = (int)e - ci * r.c_out;  // (a slice's per_k is at most 256 x 256)
    float4* d = reinterpret_cast<float4*>(r.dw + k * r.dw_k + (int64_t)ci * r.dw_ld + co);
    if (r.accumulate) {
      const float4 o = *d;
      s = make_float4(o.x + s.x, o.y + s.y, o.z + s.z, o.w + s.w);
    }
    *d = s;
  }
}

template <bool kDet>
__global__ void __launch_bounds__(kThreads, 1)
k_wgrad_tc(const WgParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const int S = p.S;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t a_bytes = (uint32_t)p.nbi * kBlockBytes;      // one stage: the item's channel blocks, LBO apart
  const uint32_t g_bytes = (uint32_t)p.gblocks * kBlockBytes;  // dout tile: blocks of [128 rows][32 channels]
  const uint32_t a_base = smem_base;
  // (an M = 64 operand reads 2 blocks even when the item has one: the block past the stage is the next stage or the
  // first dout buffer, and only feeds accumulator lanes >= cm, which nobody reads; M = 128 items have 3 or 4 blocks
  // and the same holds for the 4th)
  const uint32_t g_base = a_base + (uint32_t)S * a_bytes;
  const uint32_t m_base = g_base + (uint32_t)p.gbufs * g_bytes;  // (mask & group) and index of this CTA's tiles
  const uint32_t bar_base = m_base + (((uint32_t)p.n_local * 8u + 15u) & ~15u);
  uint32_t* lmask = reinterpret_cast<uint32_t*>(smem + (m_base - smem_base));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (bar_base - smem_base));
  auto a_full = [&](int s) { return bar_base + 8u * (uint32_t)s; };
  auto a_empty = [&](int s) { return bar_base + 8u * (uint32_t)(kMaxStages + s); };
  auto g_full = [&](int s) { return bar_base + 8u * (uint32_t)(2 * kMaxStages + s); };
  auto g_empty = [&](int s) { return bar_base + 8u * (uint32_t)(2 * kMaxStages + kMaxGBufs + s); };
  const uint32_t acc_full = bar_base + 8u * (uint32_t)(2 * kMaxStages + 2 * kMaxGBufs);
  constexpr int kNumBars = 2 * kMaxStages + 2 * kMaxGBufs + 1;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(bars + kNumBars);
  volatile int* abort_flag = reinterpret_cast<volatile int*>(bars + kNumBars + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  mm3d_griddep_launch();
  mm3d_griddep_wait();  // (everything below reads the plan; the wgrad stream's kernels follow each other closely)
  // ---- CTAs -> offset groups in proportion to the groups' work, from the plan's per-offset tile counts
  // (every CTA computes the same table; lane g of warp 0 owns group g): cost = nbi nmb * sum_k tiles(k) for the
  // gathers and MMAs + gblocks * max_k tiles(k) for the dout tiles.
  __shared__ int s_cta0[33];
  if (warp == 0) {
    const int nctas = (int)gridDim.x;
    float cost = 0.f;
    if (lane < p.groups) {
      uint32_t sum = 0, mx = 0;
      for (uint32_t r = p.gmask[lane]; r; r &= r - 1) {
        const uint32_t c = __ldg(p.off_tiles + (__ffs(r) - 1));
        sum += c;
        mx = max(mx, c);
      }
      cost = (float)((uint32_t)(p.nbi * p.nmb) * sum + (uint32_t)p.gblocks * mx) + 1.f;
    }
    float total = cost;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
    const int min_ct = (p.num_tiles + p.n_local - 1) / p.n_local;
    int ct = 0;
    if (lane < p.groups) ct = max(min_ct, min(p.num_tiles, (int)((float)nctas * cost / total)));
    int used = ct;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) used += __shfl_xor_sync(0xffffffffu, used, o);
    for (int guard = 0; used != nctas && guard < 4 * 148; ++guard) {
      // hand out spare CTAs to the group with the most work per CTA / take surplus from the one with the least
      const bool add = used < nctas;
      float load = -1.f;
      if (lane < p.groups && (add ? ct < p.num_tiles : ct > min_ct)) load = add ? cost / (float)ct : (float)ct / cost;
      float best = load;
      int who = lane;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int ow = __shfl_xor_sync(0xffffffffu, who, o);
        if (ob > best || (ob == best && ow < who)) { best = ob; who = ow; }
      }
      if (best < 0.f) break;
      if (lane == who) ct += add ? 1 : -1;
      used += add ? 1 : -1;
    }
    int incl = ct;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int x = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += x;
    }
    s_cta0[lane + 1] = incl;
    if (lane == 0) s_cta0[0] = 0;
  }
  __syncthreads();
  if (kDet && blockIdx.x == 0 && threadIdx.x <= p.groups) p.slab_cta0[threadIdx.x] = s_cta0[threadIdx.x];
  int grp = 0;  // this CTA's offset group, its index among the group's CTAs and their number
  while (grp + 1 < p.groups && (int)blockIdx.x >= s_cta0[grp + 1]) ++grp;
  const uint32_t gmask = p.gmask[grp];
  const int split = (int)blockIdx.x - s_cta0[grp], splits = s_cta0[grp + 1] - s_cta0[grp];
  if (split >= splits) return;  // (only if the shares could not be made to add up: more CTAs than tiles)

  int n_local = p.n_local;
  while (n_local > 0 && mm3d_plan_local_tile(p.order, p.num_tiles, splits, split, n_local - 1) < 0) --n_local;
  for (int i = threadIdx.x; i < n_local; i += blockDim.x) {
    const int t = mm3d_plan_local_tile(p.order, p.num_tiles, splits, split, i);
    lmask[i] = __ldg(p.tile_mask + t) & gmask;
    lmask[n_local + i] = (uint32_t)t;
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(a_full(s), kProducers * 32);
      mbar_init(a_empty(s), 1);
    }
    for (int s = 0; s < kMaxGBufs; ++s) {
      mbar_init(g_full(s), kProducers * 32);
      mbar_init(g_empty(s), 1);
    }
    mbar_init(acc_full, 1);
    *abort_flag = 0;
    fence_barrier_init();
  }
  if (warp == kProducers + 4) tmem_alloc(smem_u32((const void*)tmem_slot), (uint32_t)p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < kProducers) {
    // =================================================================== producers: warp w owns rows 16 w .. 16 w + 15
    const int row0 = warp * kRowsPerWarp;
    ItemWalk it;
    it.init(p, lmask, n_local);
    uint32_t n_item = 0, gi = 0;
    // lanes 0..15: this warp's 16 table entries of the current item / its 16 dout rows of the current tile
    int e = -1, pr = -1;
    if (it.valid() && lane < kRowsPerWarp) {
      e = __ldg(p.tbl + (int64_t)it.k * p.tstride + (int64_t)it.t.tile * kTileM + row0 + lane);
      pr = __ldg(p.perm + (int64_t)it.t.tile * kTileM + row0 + lane);
    }
    while (it.valid()) {
      const int h = it.h;
      const bool first = it.first;
      it.next();
      // the next item's entries (and, at a tile change, its dout rows) are in flight while this one is copied
      int en = -1, prn = pr;
      if (it.valid() && lane < kRowsPerWarp) {
        en = it.h ? e : __ldg(p.tbl + (int64_t)it.k * p.tstride + (int64_t)it.t.tile * kTileM + row0 + lane);
        if (it.first) prn = __ldg(p.perm + (int64_t)it.t.tile * kTileM + row0 + lane);
      }
      TRACE(warp, n_item, 0);
      if (first) {  // the tile's dout rows, shared by all offsets of the group
        const int buf = (int)(gi % (uint32_t)p.gbufs);
        if (!mbar_wait(g_empty(buf), ((gi / (uint32_t)p.gbufs) & 1u) ^ 1u, abort_flag)) goto done;
        const uint32_t gb = g_base + (uint32_t)buf * g_bytes;
        gather_rows16(gb, row0, pr, p.dout, (uint32_t)p.ld_dout, p.gblocks, p.g_last_w == 4, lane);
        cp_async_arrive(g_full(buf));
        ++gi;
      }
      const int s = (int)(n_item % (uint32_t)S);
      TRACE(warp, n_item, 1);
      if (!mbar_wait(a_empty(s), ((n_item / (uint32_t)S) & 1u) ^ 1u, abort_flag)) goto done;
      TRACE(warp, n_item, 2);
      const uint32_t stage = a_base + (uint32_t)s * a_bytes;
      gather_rows16(stage, row0, e, p.in + h * p.cm, (uint32_t)p.ld_in, p.nbi, p.last_w == 4, lane);
      cp_async_arrive(a_full(s));
      TRACE(warp, n_item, 3);
      e = en;
      pr = prn;
      ++n_item;
    }
  } else if (warp < kProducers + 4) {
    // =================================================================== epilogue: TMEM -> dW (+=)
    const int ew = warp & 3;  // a warp may only touch TMEM lanes 32*(warp%4) .. +31
    // offsets this CTA touched = OR of its tiles' masks (the MMA issuer derives the same set)
    uint32_t seen = 0;
    for (int i = lane; i < n_local; i += 32) seen |= lmask[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) seen |= __shfl_xor_sync(0xffffffffu, seen, o);
    if (seen == 0) {
      if constexpr (kDet) flush_to_slab(p, tmem_base, ew, lane, gmask, 0u);
      goto done;
    }
    if (!mbar_wait_sleep(acc_full, 0u, abort_flag, 1000)) goto done;
    if (ew == 0) TRACE(kProducers + 2, 0, 0);
    tc_fence_after();
    if constexpr (kDet) {
      flush_to_slab(p, tmem_base, ew, lane, gmask, seen);
      tc_fence_before();
      goto done;
    }
    // accumulator row (= input channel of the M-block) of this thread: M=128 -> lane i holds row i; M=64 -> row m
    // sits in lane 32*(m/16) + m%16 (16 lanes per sub-partition)
    const int ci = p.mm == 128 ? ew * 32 + lane : ew * 16 + lane;
    const bool lane_ok = (p.mm == 128 || lane < 16) && ci < p.cm;
    // every CTA of a group flushes the same addresses: start each at a different offset so that the L2
    // atomic units do not serialise on one line at a time
    const int rot = (int)((unsigned)split * 5u % 32u);
    const uint32_t hi = seen & ~((1u << rot) - 1u), lo = seen & ((1u << rot) - 1u);
    for (int part = 0; part < 2; ++part)
    for (uint32_t rem = part ? lo : hi; rem; rem &= rem - 1) {
      const int k = __ffs(rem) - 1;
      const int kidx = __popc(gmask & ((1u << k) - 1u));
      for (int h = 0; h < p.nmb; ++h) {
        const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)((kidx * p.nmb + h) * p.c_out);
        float* dst = p.dw + k * p.dw_k + (int64_t)(h * p.cm + ci) * p.dw_ld;
        for (int c0 = 0; c0 < p.c_out; c0 += 16) {
          float acc[16];
          tmem_ld16(taddr + (uint32_t)c0, acc);
          if (lane_ok) {
#pragma unroll
            for (int q = 0; q < 16; q += 4)
              if (acc[q] != 0.f || acc[q + 1] != 0.f || acc[q + 2] != 0.f || acc[q + 3] != 0.f)
                red_add_v4(dst + c0 + q, acc[q], acc[q + 1], acc[q + 2], acc[q + 3]);
          }
        }
      }
    }
    if (ew == 0) TRACE(kProducers + 2, 0, 1);
    tc_fence_before();
  } else {
    // =================================================================== MMA issuer: the whole warp walks the
    // items (warp-uniform control flow), one elected lane issues
    const uint32_t idesc = make_idesc_tf32(p.mm, p.c_out, 1, 1);
    const uint64_t desc0 = make_desc_sw128_base32(0, kBlockBytes, 512);
    ItemWalk it;
    it.init(p, lmask, n_local);
    uint32_t gi = 0, seen = 0, n_item = 0;
    bool ok = true, any = false;
    int buf = 0;
    while (it.valid()) {
      if (it.first) {
        buf = (int)(gi % (uint32_t)p.gbufs);
        if (!mbar_wait(g_full(buf), (gi / (uint32_t)p.gbufs) & 1u, abort_flag)) { ok = false; break; }
      }
      const int s = (int)(n_item % (uint32_t)S);
      TRACE(kProducers + 1, n_item, 0);
      if (!mbar_wait(a_full(s), (n_item / (uint32_t)S) & 1u, abort_flag)) { ok = false; break; }
      TRACE(kProducers + 1, n_item, 1);
      tc_fence_after();
      const int k = it.k, h = it.h;
      it.next();
      const bool tile_done = !it.valid() || it.first;
      if (elect_one()) {
        const uint64_t a_desc = desc0 + desc_addr(a_base + (uint32_t)s * a_bytes);
        const uint64_t g_desc = desc0 + desc_addr(g_base + (uint32_t)buf * g_bytes);
        const uint32_t d_tmem = tmem_base + (uint32_t)((__popc(gmask & ((1u << k) - 1u)) * p.nmb + h) * p.c_out);
        // per K-step of 8 rows: two 4-row swizzle atoms (SBO = 512 B, 1024 B per step); 32-wide M / N blocks are
        // LBO = 16 KB apart
        umma_tf32(d_tmem, a_desc, g_desc, idesc, (seen >> k) & 1u);
#pragma unroll
        for (int r8 = 1; r8 < 16; ++r8) umma_tf32(d_tmem, a_desc + r8 * 64, g_desc + r8 * 64, idesc, 1u);
        umma_commit(a_empty(s));
        if (tile_done) umma_commit(g_empty(buf));
      }
      __syncwarp();
      TRACE(kProducers + 1, n_item, 2);
      if (h == p.nmb - 1) seen |= 1u << k;
      if (tile_done) ++gi;
      any = true;
      ++n_item;
    }
    if (ok && any && elect_one()) umma_commit(acc_full);
    __syncwarp();
  }
done:
  asm volatile("cp.async.wait_all;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0 && *abort_flag) mm3d_raise(p.err);
  if (warp == kProducers + 4) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}


// ---- narrow layers: two rings -----------------------------------------------------------------------------------
// For items of one 32-channel block (c_in <= 32) the kernel above is bound by per-item latencies, not by data: its
// single issuer needs ~650 cycles for the 16 small MMAs of an item and its 8 cooperating producer warps ~1100 cycles
// per item (exposed table-entry latency, a 256-arrival barrier) -- measured with clock64 stamps.  This variant runs
// TWO independent rings inside the CTA, each with its own MMA issuer warp: the offsets of the CTA's group are dealt to
// the rings by their tile counts (so every accumulator keeps a single writer), ring m owns the stages s with
// s % 2 == m, and every producer warp OWNS one stage and fills whole items alone (32 arrivals, the next item's
// entries in flight while the current one is copied).  One more warp loads the dout tiles, which both rings share.
//
// Warp roles (14 warps): 0..5 item producers (warp w = stage w, ring w & 1), 6 dout-tile loader, 7 idle,
// 8..11 epilogue (TMEM -> red.add at the end), 12 / 13 MMA issuers of ring 0 / 1 (12 also allocates TMEM).
constexpr int kRingStages = 6;
constexpr int kRingThreads = 14 * 32;
constexpr int kRingEntBytes = kTileM * 4;

template <bool kDet>
__global__ void __launch_bounds__(kRingThreads, 1)
k_wgrad_tc_rings(const WgParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const int S = p.S, R = p.S / 2;  // 6 stages (4 when an item has two channel blocks)
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t a_bytes = (uint32_t)p.nbi * kBlockBytes;
  const uint32_t g_bytes = (uint32_t)p.gblocks * kBlockBytes;
  const uint32_t a_base = smem_base;
  const uint32_t g_base = a_base + (uint32_t)S * a_bytes;  // (the block past the last stage is the first dout buffer: see above)
  const uint32_t e_base = g_base + (uint32_t)p.gbufs * g_bytes;       // entry rows of warps 0..6
  const uint32_t m_base = e_base + 7u * kRingEntBytes;                 // [n_local] masks, [n_local] tiles
  const uint32_t f_base = m_base + (uint32_t)p.n_local * 8u;           // [2][n_local + 1] first item of a tile, per ring
  const uint32_t i_base = f_base + (uint32_t)(p.n_local + 1) * 8u;     // [2][max_items] items (tile << 5 | offset), 16 bits
  const uint32_t bar_base = (i_base + (uint32_t)p.max_items * 4u + 15u) & ~15u;
  uint32_t* cmask = reinterpret_cast<uint32_t*>(smem + (m_base - smem_base));
  uint32_t* ctile = cmask + p.n_local;
  uint32_t* first = reinterpret_cast<uint32_t*>(smem + (f_base - smem_base));
  uint16_t* items = reinterpret_cast<uint16_t*>(smem + (i_base - smem_base));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (bar_base - smem_base));
  auto a_full = [&](int s) { return bar_base + 8u * (uint32_t)s; };
  auto a_empty = [&](int s) { return bar_base + 8u * (uint32_t)(kMaxStages + s); };
  auto g_full = [&](int s) { return bar_base + 8u * (uint32_t)(2 * kMaxStages + s); };
  auto g_empty = [&](int s) { return bar_base + 8u * (uint32_t)(2 * kMaxStages + kMaxGBufs + s); };
  const uint32_t acc_full = bar_base + 8u * (uint32_t)(2 * kMaxStages + 2 * kMaxGBufs);
  constexpr int kNumBars = 2 * kMaxStages + 2 * kMaxGBufs + 1;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(bars + kNumBars);
  volatile int* abort_flag = reinterpret_cast<volatile int*>(bars + kNumBars + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  mm3d_griddep_launch();
  mm3d_griddep_wait();
#ifdef MM3D_TRACE
  if (p.trace && threadIdx.x == 0) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    p.trace[4096 + 2 * blockIdx.x] = (long long)gt;
  }
#endif
  // ---- CTAs -> offset groups (as in k_wgrad_tc) and the group's offsets -> rings, both from the plan's per-offset
  // tile counts; every CTA computes the same tables
  __shared__ int s_cta0[33];
  __shared__ uint32_t s_ring1[32];  // per group: the offsets of ring 1
  __shared__ int s_byrank[32];
  __shared__ uint32_t s_cnt[32];
  __shared__ int s_ne;
  if (warp == 0) {
    const int nctas = (int)gridDim.x;
    // lane k: tile count of offset k (one load), and its rank by descending count (ties: lower offset first)
    const uint32_t cnt = lane < p.K ? __ldg(p.off_tiles + lane) : 0u;
    int rank = 0;
#pragma unroll
    for (int o = 0; o < 32; ++o) {
      const uint32_t oc = __shfl_sync(0xffffffffu, cnt, o);
      if (o < p.K && (oc > cnt || (oc == cnt && o < lane))) ++rank;
    }
    if (lane < p.K) {
      s_byrank[rank] = lane;
      s_cnt[lane] = cnt;
    }
    __syncwarp();
    float cost = 0.f;
    if (lane < p.groups) {
      // this group's offsets by descending tile count, each to the lighter ring
      uint32_t sum = 0, mx = 0, r1 = 0, w0 = 0, w1 = 0;
      const uint32_t gm = p.gmask[lane];
      for (int r = 0; r < p.K; ++r) {
        const int k = s_byrank[r];
        if (!((gm >> k) & 1u)) continue;
        const uint32_t c = s_cnt[k];
        sum += c;
        mx = max(mx, c);
        if (w1 <= w0) { r1 |= 1u << k; w1 += c + 1; } else w0 += c + 1;
      }
      cost = (float)((uint32_t)p.nbi * sum + (uint32_t)p.gblocks * mx) + 1.f;
      s_ring1[lane] = r1;
    }
    float total = cost;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
    const int min_ct = (p.num_tiles + p.n_local - 1) / p.n_local;
    int ct = 0;
    if (lane < p.groups) ct = max(min_ct, min(p.num_tiles, (int)((float)nctas * cost / total)));
    int used = ct;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) used += __shfl_xor_sync(0xffffffffu, used, o);
    for (int guard = 0; used != nctas && guard < 4 * 148; ++guard) {
      const bool add = used < nctas;
      float load = -1.f;
      if (lane < p.groups && (add ? ct < p.num_tiles : ct > min_ct)) load = add ? cost / (float)ct : (float)ct / cost;
      float best = load;
      int who = lane;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int ow = __shfl_xor_sync(0xffffffffu, who, o);
        if (ob > best || (ob == best && ow < who)) { best = ob; who = ow; }
      }
      if (best < 0.f) break;
      if (lane == who) ct += add ? 1 : -1;
      used += add ? 1 : -1;
    }
    int incl = ct;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int x = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += x;
    }
    s_cta0[lane + 1] = incl;
    if (lane == 0) s_cta0[0] = 0;
  }
  __syncthreads();
  if (kDet && blockIdx.x == 0 && threadIdx.x <= p.groups) p.slab_cta0[threadIdx.x] = s_cta0[threadIdx.x];
  int grp = 0;
  while (grp + 1 < p.groups && (int)blockIdx.x >= s_cta0[grp + 1]) ++grp;
  const uint32_t gmask = p.gmask[grp], ring1 = s_ring1[grp];
  const int split = (int)blockIdx.x - s_cta0[grp], splits = s_cta0[grp + 1] - s_cta0[grp];
  if (split >= splits) return;

  int n_local = p.n_local;
  while (n_local > 0 && mm3d_plan_local_tile(p.order, p.num_tiles, splits, split, n_local - 1) < 0) --n_local;
  for (int i = threadIdx.x; i < n_local; i += blockDim.x) {
    const int t = mm3d_plan_local_tile(p.order, p.num_tiles, splits, split, i);
    cmask[i] = __ldg(p.tile_mask + t) & gmask;
    ctile[i] = (uint32_t)t;
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(a_full(s), 32);
      mbar_init(a_empty(s), 1);
    }
    for (int s = 0; s < kMaxGBufs; ++s) {
      mbar_init(g_full(s), 32);
      mbar_init(g_empty(s), 2);  // both issuers are done with the tile
    }
    mbar_init(acc_full, 2);
    *abort_flag = 0;
    fence_barrier_init();
  }
  if (warp == 12) tmem_alloc(smem_u32((const void*)tmem_slot), (uint32_t)p.tmem_cols);
  __syncthreads();
  if (warp == 0) {
    // tiles without an offset of this group drop out (in place: a chunk is read before anything of it is rewritten) ...
    int base = 0;
    for (int b0 = 0; b0 < n_local; b0 += 32) {
      const int i = b0 + lane;
      const uint32_t m = i < n_local ? cmask[i] : 0u, t = i < n_local ? ctile[i] : 0u;
      const uint32_t bal = __ballot_sync(0xffffffffu, m != 0u);
      __syncwarp();
      if (m) {
        const int pos = base + __popc(bal & ((1u << lane) - 1u));
        cmask[pos] = m;
        ctile[pos] = t;
      }
      base += __popc(bal);
      __syncwarp();
    }
    const int ne = base;
    if (lane == 0) s_ne = ne;
    // ... and each ring's first item of every remaining tile (exclusive scans of the per-tile item counts)
    uint32_t run0 = 0, run1 = 0;
    for (int b0 = 0; b0 < ne; b0 += 32) {
      const int i = b0 + lane;
      const uint32_t m = i < ne ? cmask[i] : 0u;
      const uint32_t c0 = (uint32_t)__popc(m & ~ring1), c1 = (uint32_t)__popc(m & ring1);
      uint32_t i0 = c0, i1 = c1;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t x0 = __shfl_up_sync(0xffffffffu, i0, o), x1 = __shfl_up_sync(0xffffffffu, i1, o);
        if (lane >= o) { i0 += x0; i1 += x1; }
      }
      if (i < ne) {
        first[i] = run0 + i0 - c0;
        first[p.n_local + 1 + i] = run1 + i1 - c1;
      }
      run0 += __shfl_sync(0xffffffffu, i0, 31);
      run1 += __shfl_sync(0xffffffffu, i1, 31);
    }
    if (lane == 0) {
      first[ne] = run0;
      first[p.n_local + 1 + ne] = run1;
    }
  }
  __syncthreads();
  const int ne = s_ne;
  for (int t = threadIdx.x; t < ne; t += blockDim.x) {
    const uint32_t m = cmask[t];
    uint32_t at0 = first[t], at1 = (uint32_t)p.max_items + first[p.n_local + 1 + t];
    for (uint32_t rem = m & ~ring1; rem; rem &= rem - 1) items[at0++] = (uint16_t)(((uint32_t)t << 5) | (uint32_t)(__ffs(rem) - 1));
    for (uint32_t rem = m & ring1; rem; rem &= rem - 1) items[at1++] = (uint16_t)(((uint32_t)t << 5) | (uint32_t)(__ffs(rem) - 1));
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < S) {
    // =================================================================== item producers: warp w owns stage w
    const int m = warp & 1, q = warp >> 1;
    const uint16_t* list = items + (size_t)m * p.max_items;
    const int n_items = (int)first[m * (p.n_local + 1) + ne];
    const uint32_t ent = e_base + (uint32_t)warp * kRingEntBytes;
    const uint32_t stage = a_base + (uint32_t)warp * a_bytes;
    int e[4] = {-1, -1, -1, -1};  // table entries of rows lane, 32 + lane, 64 + lane, 96 + lane of the current item
    int i = q;
    if (i < n_items) {
      const uint32_t it = list[i];
      const int32_t* src = p.tbl + (int64_t)(it & 31u) * p.tstride + (int64_t)ctile[it >> 5] * kTileM + lane;
#pragma unroll
      for (int r = 0; r < 4; ++r) e[r] = __ldg(src + 32 * r);
    }
    for (uint32_t use = 0; i < n_items; i += R, ++use) {
      int en[4] = {-1, -1, -1, -1};  // the next item's entries are in flight while this one is copied
      if (i + R < n_items) {
        const uint32_t it = list[i + R];
        const int32_t* src = p.tbl + (int64_t)(it & 31u) * p.tstride + (int64_t)ctile[it >> 5] * kTileM + lane;
#pragma unroll
        for (int r = 0; r < 4; ++r) en[r] = __ldg(src + 32 * r);
      }
      TRACE(warp, use, 0);
      if (!mbar_wait(a_empty(warp), (use & 1u) ^ 1u, abort_flag)) goto done;
      TRACE(warp, use, 1);
#pragma unroll
      for (int r = 0; r < 4; ++r)
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(ent + (uint32_t)(32 * r + lane) * 4u), "r"(e[r]) : "memory");
      __syncwarp();
      for (int jb = 0; jb < p.nbi; ++jb) {
        // (BF16: plain 128-byte swizzle, rows of c_in / 2 four-byte units, the last block's missing chunks zero-filled)
        if (p.bf16) gather_block<8, false>(stage + (uint32_t)jb * kBlockBytes, ent, p.in, p.in + jb * 32, (uint32_t)p.ld_in, lane, jb == p.nbi - 1 ? p.last_w : 8);
        else if (jb == p.nbi - 1 && p.last_w == 4) gather_block<4, true>(stage + (uint32_t)jb * kBlockBytes, ent, p.in, p.in + jb * 32, (uint32_t)p.ld_in, lane);
        else gather_block<8, true>(stage + (uint32_t)jb * kBlockBytes, ent, p.in, p.in + jb * 32, (uint32_t)p.ld_in, lane);
      }
      cp_async_arrive(a_full(warp));
      __syncwarp();  // the entry row is rewritten by the next item
      TRACE(warp, use, 2);
#pragma unroll
      for (int r = 0; r < 4; ++r) e[r] = en[r];
    }
  } else if (warp == 6) {
    // =================================================================== dout tiles, shared by both rings
    const uint32_t ent = e_base + 6u * kRingEntBytes;
    int e[4] = {-1, -1, -1, -1};
    if (ne > 0) {
#pragma unroll
      for (int r = 0; r < 4; ++r) e[r] = __ldg(p.perm + (int64_t)ctile[0] * kTileM + 32 * r + lane);
    }
    for (int t = 0; t < ne; ++t) {
      int en[4] = {-1, -1, -1, -1};
      if (t + 1 < ne) {
#pragma unroll
        for (int r = 0; r < 4; ++r) en[r] = __ldg(p.perm + (int64_t)ctile[t + 1] * kTileM + 32 * r + lane);
      }
      const int buf = t % p.gbufs;
      if (!mbar_wait(g_empty(buf), (((uint32_t)t / (uint32_t)p.gbufs) & 1u) ^ 1u, abort_flag)) goto done;
#pragma unroll
      for (int r = 0; r < 4; ++r)
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(ent + (uint32_t)(32 * r + lane) * 4u), "r"(e[r]) : "memory");
      __syncwarp();
      const uint32_t gb = g_base + (uint32_t)buf * g_bytes;
      for (int jb = 0; jb < p.gblocks; ++jb) {
        if (p.bf16) gather_block<8, false>(gb + (uint32_t)jb * kBlockBytes, ent, p.dout, p.dout + jb * 32, (uint32_t)p.ld_dout, lane, jb == p.gblocks - 1 ? p.g_last_w : 8);
        else if (jb == p.gblocks - 1 && p.g_last_w == 4) gather_block<4, true>(gb + (uint32_t)jb * kBlockBytes, ent, p.dout, p.dout + jb * 32, (uint32_t)p.ld_dout, lane);
        else gather_block<8, true>(gb + (uint32_t)jb * kBlockBytes, ent, p.dout, p.dout + jb * 32, (uint32_t)p.ld_dout, lane);
      }
      cp_async_arrive(g_full(buf));
      __syncwarp();
#pragma unroll
      for (int r = 0; r < 4; ++r) e[r] = en[r];
    }
  } else if (warp >= 8 && warp < 12) {
    // =================================================================== epilogue: TMEM -> dW (+=)
    const int ew = warp & 3;
    uint32_t seen = 0;
    for (int i = lane; i < ne; i += 32) seen |= cmask[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) seen |= __shfl_xor_sync(0xffffffffu, seen, o);
    if (seen == 0) {
      if constexpr (kDet) flush_to_slab(p, tmem_base, ew, lane, gmask, 0u);
      goto done;
    }
    if (!mbar_wait_sleep(acc_full, 0u, abort_flag, 1000)) goto done;
    if (ew == 0) TRACE(kProducers + 2, 0, 0);
    tc_fence_after();
    if constexpr (kDet) {
      flush_to_slab(p, tmem_base, ew, lane, gmask, seen);
      tc_fence_before();
      goto done;
    }
    const int ci = p.mm == 128 ? ew * 32 + lane : ew * 16 + lane;
    const bool lane_ok = (p.mm == 128 || lane < 16) && ci < p.cm;
    const int rot = (int)((unsigned)split * 5u % 32u);
    const uint32_t hi = seen & ~((1u << rot) - 1u), lo = seen & ((1u << rot) - 1u);
    for (int part = 0; part < 2; ++part)
    for (uint32_t rem = part ? lo : hi; rem; rem &= rem - 1) {
      const int k = __ffs(rem) - 1;
      const int kidx = __popc(gmask & ((1u << k) - 1u));
      const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(kidx * p.c_out);
      float* dst = p.dw + k * p.dw_k + (int64_t)ci * p.dw_ld;
      for (int c0 = 0; c0 < p.c_out; c0 += 16) {
        float acc[16];
        tmem_ld16(taddr + (uint32_t)c0, acc);
        if (lane_ok) {
#pragma unroll
          for (int qq = 0; qq < 16; qq += 4)
            if (acc[qq] != 0.f || acc[qq + 1] != 0.f || acc[qq + 2] != 0.f || acc[qq + 3] != 0.f)
              red_add_v4(dst + c0 + qq, acc[qq], acc[qq + 1], acc[qq + 2], acc[qq + 3]);
        }
      }
    }
    if (ew == 0) TRACE(kProducers + 2, 0, 1);
    tc_fence_before();
  } else if (warp >= 12) {
    // =================================================================== MMA issuers: ring m = warp - 12
    const int m = warp - 12;
    const uint16_t* list = items + (size_t)m * p.max_items;
    const uint32_t* fst = first + m * (p.n_local + 1);
    // TF32: MN-major operands need the 32-byte-granule swizzle (4-row atoms, 8 rows = 1024 bytes per K-step);
    // BF16: the plain 128-byte swizzle (8-row atoms, K = 16 rows = 2048 bytes per instruction)
    const uint32_t idesc = p.bf16 ? make_idesc_bf16(p.mm, p.c_out, 1, 1) : make_idesc_tf32(p.mm, p.c_out, 1, 1);
    const uint64_t desc0 = p.bf16 ? make_desc_sw128(0, kBlockBytes, 1024) : make_desc_sw128_base32(0, kBlockBytes, 512);
    uint32_t seen = 0;
    bool ok = true;
    for (int t = 0; t < ne && ok; ++t) {
      const int buf = t % p.gbufs;
      if (!mbar_wait(g_full(buf), ((uint32_t)t / (uint32_t)p.gbufs) & 1u, abort_flag)) { ok = false; break; }
      const uint64_t g_desc = desc0 + desc_addr(g_base + (uint32_t)buf * g_bytes);
      for (uint32_t i = fst[t]; i < fst[t + 1]; ++i) {
        const int s = 2 * (int)(i % (uint32_t)R) + m;
        TRACE(kProducers + 3 + m, i, 0);
        if (!mbar_wait(a_full(s), (i / (uint32_t)R) & 1u, abort_flag)) { ok = false; break; }
        TRACE(kProducers + 3 + m, i, 1);
        tc_fence_after();
        const int k = (int)(list[i] & 31u);
        if (elect_one()) {
          const uint64_t a_desc = desc0 + desc_addr(a_base + (uint32_t)s * a_bytes);
          const uint32_t d_tmem = tmem_base + (uint32_t)(__popc(gmask & ((1u << k) - 1u)) * p.c_out);
          if (p.bf16) {
            umma_f16(d_tmem, a_desc, g_desc, idesc, (seen >> k) & 1u);
#pragma unroll
            for (int r16 = 1; r16 < 8; ++r16) umma_f16(d_tmem, a_desc + r16 * 128, g_desc + r16 * 128, idesc, 1u);
          } else {
            umma_tf32(d_tmem, a_desc, g_desc, idesc, (seen >> k) & 1u);
#pragma unroll
            for (int r8 = 1; r8 < 16; ++r8) umma_tf32(d_tmem, a_desc + r8 * 64, g_desc + r8 * 64, idesc, 1u);
          }
          umma_commit(a_empty(s));
        }
        __syncwarp();
        TRACE(kProducers + 3 + m, i, 2);
        seen |= 1u << k;
      }
      if (!ok) break;
      if (elect_one()) umma_commit(g_empty(buf));  // (arrives at once when this ring had no item of the tile)
      __syncwarp();
    }
    if (ok && elect_one()) umma_commit(acc_full);
    __syncwarp();
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
  if (warp == 12) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

}  // namespace

int* mm3d_device_err_flag();  // conv_tc.cu
#ifdef MM3D_TRACE
long long* mm3d_debug_trace_ptr();  // conv_tc.cu
#endif

// one launch's shape (wgrad_tc_slice)
static int wgrad_slice_supported(int c_in, int c_out, int K) {
  if ((c_in % 16) != 0 || c_in < 16 || c_in > 256 || (c_out % 16) != 0 || c_out < 16 || c_out > 256 || K > 32) return 0;
  const int nmb = c_in > 128 ? 2 : 1;
  if (nmb == 2 && (c_in % 32) != 0) return 0;  // halves must stay whole 64-byte pieces
  return nmb * c_out <= 512;
}

// Layers wider than 256 channels on either side (up to 512) run as (input slice) x (output slice) launches, each a
// shape wgrad_slice_supported takes, each writing its own block of dW: output slices of near-equal multiples of 16,
// input slices of 256 channels and a remainder (cut at 128 when it is not a whole number of 64-byte M-block halves).
// The shapes of 256 channels or fewer are one launch, as without slicing.
constexpr int kWgSlice = 256, kWgWide = 512;
static int wgrad_in_slice(int rem) {
  if (rem > kWgSlice) return kWgSlice;
  return (rem <= 128 || rem % 32 == 0) ? rem : 128;
}
static bool wgrad_sliced(int c_in, int c_out) { return c_in > kWgSlice || c_out > kWgSlice; }

int mm3d_conv_wgrad_tc_supported(int c_in, int c_out, int K) {
  if (!wgrad_sliced(c_in, c_out)) return wgrad_slice_supported(c_in, c_out, K);
  if (c_in > kWgWide || c_out > kWgWide || (c_out % 16) != 0) return 0;
  const int co_step = mm3d_slice_step(c_out, kWgSlice, 16);
  for (int ci0 = 0, w; ci0 < c_in; ci0 += w) {
    w = wgrad_in_slice(c_in - ci0);
    for (int co0 = 0; co0 < c_out; co0 += co_step)
      if (!wgrad_slice_supported(w, c_out - co0 < co_step ? c_out - co0 : co_step, K)) return 0;
  }
  return 1;
}

// offsets per group: as many (offset, M-block) accumulators of c_out TMEM columns as fit the 512 columns
static int wgrad_group_size(int c_in, int c_out, int K) {
  const int gk = 512 / (c_out * (c_in > 128 ? 2 : 1));
  return gk < K ? gk : K;
}

// Launch grid of both kernels: one CTA per SM, at least one per offset group
static int wgrad_ctas(int c_in, int c_out, int K) {
  const int gk = wgrad_group_size(c_in, c_out, K), groups = (K + gk - 1) / gk;
  const int sms = mm3d_sm_count();
  return sms < groups ? groups : sms;
}

// Deterministic variant's workspace: the group -> first-CTA table (256 bytes), then one slab of gk * c_in * c_out floats
// per CTA (at most 512 TMEM columns x 128 lanes = 256 KB).  Independent of the row count; 0 for shapes the kernels do
// not take.
static size_t wgrad_slice_slab_bytes(int c_in, int c_out, int K) {
  return 256 + (size_t)wgrad_ctas(c_in, c_out, K) * wgrad_group_size(c_in, c_out, K) * c_in * c_out * sizeof(float);
}
// (sliced layers: the largest slice's, the slices run one after the other through the same workspace)
size_t mm3d_conv_wgrad_tc_slab_bytes(int c_in, int c_out, int K) {
  if (!mm3d_conv_wgrad_tc_supported(c_in, c_out, K)) return 0;
  if (!wgrad_sliced(c_in, c_out)) return wgrad_slice_slab_bytes(c_in, c_out, K);
  size_t most = 0;
  const int co_step = mm3d_slice_step(c_out, kWgSlice, 16);
  for (int ci0 = 0, w; ci0 < c_in; ci0 += w) {
    w = wgrad_in_slice(c_in - ci0);
    for (int co0 = 0; co0 < c_out; co0 += co_step) {
      const size_t b = wgrad_slice_slab_bytes(w, c_out - co0 < co_step ? c_out - co0 : co_step, K);
      if (b > most) most = b;
    }
  }
  return most;
}

// One launch (and the deterministic variant's reductions) over a slice: input channels of rows ld_in units apart,
// output channels of rows ld_dout units apart, dW block (k, ci, co) at d_weight + k * dw_k + ci * dw_ld + co
static int wgrad_tc_slice(const float* in, int ld_in, int c_in, const float* d_out, int ld_dout, int64_t n_out, int c_out,
                          float* d_weight, int64_t dw_k, int dw_ld, int K, const Mm3dPlanView& pv, int accumulate,
                          cudaStream_t stream, int bf16, void* slab) {
  const bool det = slab != nullptr;
  WgParams p;
  p.in = in; p.dout = d_out; p.dw = d_weight;
  p.perm = pv.perm; p.tile_mask = pv.tile_mask; p.order = pv.order; p.off_tiles = pv.off_tiles; p.tbl = pv.tbl;
  p.tstride = pv.stride;
  p.c_in = c_in; p.c_out = c_out; p.K = K;
  p.ld_in = ld_in; p.ld_dout = ld_dout; p.dw_k = dw_k; p.dw_ld = dw_ld;
  p.nmb = c_in > 128 ? 2 : 1;
  p.cm = c_in / p.nmb;
  p.bf16 = bf16;
  if (bf16) {
    if (p.nmb != 1 || getenv("MM3D_WGRAD_NO_BF16")) return MM3D_ERR_UNSUPPORTED;  // (quietly: the caller falls back)
    p.nbi = (p.cm + 63) / 64;
    p.last_w = (p.cm % 64) ? (p.cm % 64) / 8 : 8;
    p.gblocks = (c_out + 63) / 64;
    p.g_last_w = (c_out % 64) ? (c_out % 64) / 8 : 8;
  } else {
    p.nbi = (p.cm + 31) / 32;
    p.last_w = (p.cm % 32) == 16 ? 4 : 8;
    p.gblocks = (c_out + 31) / 32;
    p.g_last_w = (c_out % 32) == 16 ? 4 : 8;
  }
  p.mm = p.cm <= 64 ? 64 : 128;
  p.num_tiles = (int)mm3d_cdiv(n_out, kTileM);
  const int gk = wgrad_group_size(c_in, c_out, K);  // TMEM: c_out accumulator columns per (offset, M-block)
  const int groups = (K + gk - 1) / gk;
  int cols = 32;
  while (cols < gk * p.nmb * c_out) cols <<= 1;
  p.tmem_cols = cols;
  // one CTA per SM: ring stages and dout-tile buffers from what fits into shared memory
  const size_t a_bytes = (size_t)p.nbi * kBlockBytes, g_bytes = (size_t)p.gblocks * kBlockBytes;
  const size_t fixed = 1024 + 8 * (2 * kMaxStages + 2 * kMaxGBufs + 1) + 64;
  const size_t budget = 218 * 1024 - fixed;  // (the rest, >= 8 KB, holds the CTA's tile list)
  p.gbufs = 2;
  p.max_items = 0;
  p.S = budget > 2 * g_bytes ? (int)((budget - 2 * g_bytes) / a_bytes) : 0;
  if (p.S < 2) {
    p.gbufs = 1;
    p.S = budget > g_bytes ? (int)((budget - g_bytes) / a_bytes) : 0;
  }
  MM3D_REQUIRE(p.S >= 1, MM3D_ERR_UNSUPPORTED, "tcgen05 wgrad: shared memory budget exceeded");
  if (p.S > kMaxStages) p.S = kMaxStages;
  while (p.gbufs < kMaxGBufs && (size_t)p.S * a_bytes + (size_t)(p.gbufs + 1) * g_bytes <= budget) ++p.gbufs;
  const size_t smem_fixed = fixed + (size_t)p.S * a_bytes + (size_t)p.gbufs * g_bytes;
  p.err = mm3d_device_err_flag();
  p.slab_cta0 = det ? (int*)slab : nullptr;
  p.slab = det ? (float*)((char*)slab + 256) : nullptr;
  p.slab_cta = (int64_t)gk * c_in * c_out;
#ifdef MM3D_TRACE
  p.trace = mm3d_debug_trace_ptr();
#endif
  // Offsets -> groups and CTAs -> groups by expected work.  How often an offset occurs is data dependent; as a
  // prior, the centre of a 3^3 table is present for every row, faces often, edges sometimes, corners rarely.
  // Heaviest offsets are dealt first, each to the lightest group with a free accumulator slot; then every group
  // gets CTAs in proportion to its weight (its tiles are split among them).
  {
    float w[32];
    int idx[32];
    for (int k = 0; k < K; ++k) {
      idx[k] = k;
      w[k] = 1.f;
      if (K == 27) {
        const int cls = abs(k / 9 - 1) + abs((k / 3) % 3 - 1) + abs(k % 3 - 1);
        w[k] = cls == 0 ? 1.f : cls == 1 ? 0.4f : cls == 2 ? 0.15f : 0.03f;
      }
    }
    for (int a = 0; a < K; ++a)
      for (int b = a + 1; b < K; ++b)
        if (w[idx[b]] > w[idx[a]]) { const int t = idx[a]; idx[a] = idx[b]; idx[b] = t; }
    float gw[32];
    int gn[32];
    for (int g = 0; g < groups; ++g) { gw[g] = 0.f; gn[g] = 0; p.gmask[g] = 0; }
    for (int a = 0; a < K; ++a) {
      int best = -1;
      for (int g = 0; g < groups; ++g)
        if (gn[g] < gk && (best < 0 || gw[g] < gw[best])) best = g;
      p.gmask[best] |= 1u << idx[a];
      gw[best] += w[idx[a]] + 0.05f;  // + per-tile cost of loading the dout tile
      ++gn[best];
    }
    p.groups = groups;
  }
  // CTA shares of the groups are computed in the kernel from measured offset frequencies; here only the bound
  // on tiles per CTA (size of the shared-memory tile list): every group gets >= ceil(num_tiles / n_local) CTAs
  const int total_ctas = wgrad_ctas(c_in, c_out, K);
  int per_group_min = total_ctas / groups / 3;
  if (per_group_min < 1) per_group_min = 1;
  MM3D_REQUIRE(smem_fixed + 1024 <= 226 * 1024, MM3D_ERR_UNSUPPORTED, "tcgen05 wgrad: shared memory budget exceeded");
  // deterministic variant: after each launch, its slabs -> d_weight (the first piece honours `accumulate`, later
  // pieces add to it)
  WgReduceParams rp;
  if (det) {
    rp.slab = p.slab; rp.cta0 = p.slab_cta0; rp.dw = d_weight; rp.slab_cta = p.slab_cta;
    rp.c_in = c_in; rp.c_out = c_out; rp.K = K; rp.groups = groups;
    rp.dw_k = dw_k; rp.dw_ld = dw_ld;
    for (int g = 0; g < 32; ++g) rp.gmask[g] = g < groups ? p.gmask[g] : 0u;
  }
  const int reduce_grid = (int)mm3d_cdiv((int64_t)K * c_in * c_out / 4, 256);
  auto reduce = [&](bool first) {
    rp.accumulate = first ? accumulate : 1;
    k_wgrad_reduce<<<reduce_grid < 4 * MM3D_NUM_SMS ? reduce_grid : 4 * MM3D_NUM_SMS, 256, 0, stream>>>(rp);
    mm3d_count_launches(1);
  };
  static bool once_dev[2][64] = {{false}};
  bool& once = once_dev[det][mm3d_device_slot()];
  auto* const k_tc = det ? k_wgrad_tc<true> : k_wgrad_tc<false>;
  if (!once) {
    MM3D_CUDA(cudaFuncSetAttribute(k_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
    MM3D_CUDA(cudaFuncSetAttribute(k_tc, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    once = true;
  }
  // Narrow layers (one 32-channel block per item): the two-ring kernel.  MM3D_WGRAD_RINGS_NBI overrides the widest
  // item it takes (in 32-channel blocks; 0 = never), for A/B measurements.
  int ring_nbi = 1;
  if (const char* e = getenv("MM3D_WGRAD_RINGS_NBI")) ring_nbi = atoi(e);
  const int all_tiles = p.num_tiles;
  if (bf16) ring_nbi = 2;
  if (p.nmb == 1 && p.nbi <= ring_nbi) {
    static bool once_r[2][64] = {{false}};
    bool& once2 = once_r[det][mm3d_device_slot()];
    auto* const k_rings = det ? k_wgrad_tc_rings<true> : k_wgrad_tc_rings<false>;
    if (!once2) {
      MM3D_CUDA(cudaFuncSetAttribute(k_rings, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
      MM3D_CUDA(cudaFuncSetAttribute(k_rings, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
      once2 = true;
    }
    int gbufs = 4;
    const int ring_s = p.nbi == 1 ? kRingStages : 4;
    const size_t ring_fixed = 1024 + (size_t)ring_s * a_bytes + 7 * kRingEntBytes + 8 * (2 * kMaxStages + 2 * kMaxGBufs + 1) + 64 + 64;
    while (gbufs > 1 && ring_fixed + (size_t)gbufs * g_bytes + 16 * 1024 > 226 * 1024) --gbufs;
    if (ring_fixed + (size_t)gbufs * g_bytes + 16 * 1024 <= 226 * 1024) {
      p.gbufs = gbufs;
      p.S = ring_s;
      const size_t fixed_r = ring_fixed + (size_t)gbufs * g_bytes;
      const size_t per_tile = 8 + 8 + 4 * (size_t)gk;  // mask + index, two first-item entries, two lists of 16-bit items
      int64_t max_local_r = (int64_t)((226 * 1024 - fixed_r - 64) / per_tile);
      if (max_local_r > 2047) max_local_r = 2047;  // (11 bits of local tile index per item)
      if (const char* e = getenv("MM3D_WGRAD_MAX_LOCAL")) {
        const int64_t v = atoll(e);
        if (v >= 2 && v < max_local_r) max_local_r = v;
      }
      const int64_t max_tiles_r = max_local_r * per_group_min;
      for (int64_t start = 0; start < all_tiles; start += max_tiles_r) {
        const int cnt = (int)(all_tiles - start < max_tiles_r ? all_tiles - start : max_tiles_r);
        p.order = pv.order + start;
        p.num_tiles = cnt;
        p.n_local = (cnt + per_group_min - 1) / per_group_min;
        p.max_items = p.n_local * gk;
        const size_t smem = fixed_r + (size_t)p.n_local * 8 + (size_t)(p.n_local + 1) * 8 + (size_t)p.max_items * 4 + 32;
        MM3D_REQUIRE(smem <= 226 * 1024, MM3D_ERR_UNSUPPORTED, "tcgen05 wgrad: shared memory budget exceeded");
        MM3D_CUDA(mm3d_launch_pdl(k_rings, dim3((unsigned)total_ctas), dim3(kRingThreads), smem, stream, p));
        mm3d_count_launches(1);
        if (det) reduce(start == 0);
      }
      MM3D_CHECK_LAUNCH("mm3d_conv_wgrad_tc");
      return MM3D_OK;
    }
  }
  if (bf16) return MM3D_ERR_UNSUPPORTED;
  // The kernel keeps the list of a CTA's tiles (index + mask, 8 bytes each) in shared memory.  Row counts whose list
  // does not fit next to the stages are processed in several launches over consecutive pieces of the plan's tile
  // order (the kernel only ever adds into d_weight, so the pieces simply accumulate).
  int64_t max_local = (int64_t)((226 * 1024 - smem_fixed) / 8) & ~(int64_t)1;
  if (const char* e = getenv("MM3D_WGRAD_MAX_LOCAL")) {  // tests: force the multi-launch path at small sizes
    const int64_t v = atoll(e);
    if (v >= 2 && v < max_local) max_local = v & ~(int64_t)1;
  }
  const int64_t max_tiles = max_local * per_group_min;
  for (int64_t start = 0; start < all_tiles; start += max_tiles) {
    const int cnt = (int)(all_tiles - start < max_tiles ? all_tiles - start : max_tiles);
    p.order = pv.order + start;
    p.num_tiles = cnt;
    p.n_local = (cnt + per_group_min - 1) / per_group_min;
    const size_t smem = smem_fixed + ((size_t)p.n_local * 8 + 15) / 16 * 16;
    MM3D_CUDA(mm3d_launch_pdl(k_tc, dim3((unsigned)total_ctas), dim3(kThreads), smem, stream, p));
    mm3d_count_launches(1);
    if (det) reduce(start == 0);
  }
  MM3D_CHECK_LAUNCH("mm3d_conv_wgrad_tc");
  return MM3D_OK;
}

// bf16 != 0: `in` / `d_out` point at BF16 planes ([rows, c] bfloat16); only shapes the two-ring kernel takes
// (c_in <= 128), MM3D_ERR_UNSUPPORTED otherwise (the caller then runs the TF32 kernel on the FP32 planes)
// slab != NULL: the deterministic variant (slab_bytes >= mm3d_conv_wgrad_tc_slab_bytes): every launch is followed by
// k_wgrad_reduce, which adds that launch's slabs into d_weight, so the pieces of a long tile list reduce in piece order
// (and the slices of a wide layer in slice order)
int mm3d_conv_wgrad_tc(const float* in, int64_t n_in, int c_in, const float* d_out, int64_t n_out, int c_out,
                       float* d_weight, int K, const void* plan, int64_t plan_cap, int accumulate,
                       cudaStream_t stream, int bf16, void* slab, size_t slab_bytes) {
  MM3D_REQUIRE(mm3d_conv_wgrad_tc_supported(c_in, c_out, K), MM3D_ERR_UNSUPPORTED,
               "tcgen05 wgrad: unsupported shape c_in %d c_out %d K %d", c_in, c_out, K);
  MM3D_REQUIRE(n_out < (1ll << 31) && n_in * (int64_t)c_in < (1ll << 32) && n_out * (int64_t)c_out < (1ll << 32),
               MM3D_ERR_UNSUPPORTED, "tcgen05 wgrad: tensor too large for 32-bit element offsets");
  MM3D_REQUIRE(plan && plan_cap >= n_out, MM3D_ERR_INVALID, "tcgen05 wgrad: needs a row plan covering n_out rows");
  MM3D_REQUIRE((((uintptr_t)in | (uintptr_t)d_out | (uintptr_t)d_weight) & 15) == 0, MM3D_ERR_INVALID,
               "tcgen05 wgrad: pointers must be 16-byte aligned");
  const bool det = slab != nullptr;
  MM3D_REQUIRE(!det || slab_bytes >= mm3d_conv_wgrad_tc_slab_bytes(c_in, c_out, K), MM3D_ERR_WORKSPACE,
               "deterministic wgrad: workspace %zu bytes < %zu (mm3d_conv_wgrad_workspace_bytes)", slab_bytes,
               mm3d_conv_wgrad_tc_slab_bytes(c_in, c_out, K));
  MM3D_REQUIRE(((uintptr_t)slab & 15) == 0, MM3D_ERR_INVALID, "deterministic wgrad: workspace must be 16-byte aligned");
  // the BF16 form only where every slice has one M-block (decided before anything runs: the caller falls back to the
  // TF32 kernel for the whole layer)
  if (bf16 && (c_in > 128 || getenv("MM3D_WGRAD_NO_BF16"))) return MM3D_ERR_UNSUPPORTED;
  // (the deterministic variant's reduction overwrites d_weight itself when !accumulate)
  if (!accumulate && (!det || n_out == 0))
    MM3D_CUDA(cudaMemsetAsync(d_weight, 0, sizeof(float) * (size_t)K * c_in * c_out, stream));
  if (n_out == 0) return MM3D_OK;
  const Mm3dPlanView pv = mm3d_plan_view(plan, plan_cap);
  const int units = bf16 ? 2 : 1;  // channels per 4-byte unit of the operands
  const int co_step = wgrad_sliced(c_in, c_out) ? mm3d_slice_step(c_out, kWgSlice, 16) : c_out;
  for (int ci0 = 0, w; ci0 < c_in; ci0 += w) {
    w = wgrad_sliced(c_in, c_out) ? wgrad_in_slice(c_in - ci0) : c_in;
    for (int co0 = 0; co0 < c_out; co0 += co_step) {
      const int wo = c_out - co0 < co_step ? c_out - co0 : co_step;
      // (slices write disjoint blocks of d_weight: each honours `accumulate` as the whole layer would)
      const int rc = wgrad_tc_slice(in + ci0 / units, c_in / units, w, d_out + co0 / units, c_out / units, n_out, wo,
                                    d_weight + (int64_t)ci0 * c_out + co0, (int64_t)c_in * c_out, c_out, K, pv,
                                    accumulate || !det, stream, bf16, slab);
      if (rc) return rc;
    }
  }
  return MM3D_OK;
}
