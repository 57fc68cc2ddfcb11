// Structure builders: voxel hash, first-occurrence numbering, level pyramid, rule tables.
//
// Replaces SparseConvNet's CPU-only Metadata<3> (SURVEY.md 2.2 / 8(a) a5,a7,a12).  Everything
// is HBM/L2-bound integer work on the GPU: an open-addressing hash per level (linear probing,
// load <= 0.5), ids = rank of first occurrence obtained with atomicMin(item index) per slot +
// a prefix scan over the "I am the first occurrence" flags -- NOT atomic tickets -- so voxel
// rows are bit-identical to SparseConvNet's `nActive++` order on every run.
// Row counts stay on the device; the host only passes capacities.
#include "augment.cuh"
#include "common.cuh"

namespace {

constexpr int kScanThreads = 256;
constexpr int kItemsPerThread = 4;
constexpr int kItemsPerBlock = kScanThreads * kItemsPerThread;  // 1024

__device__ __forceinline__ uint32_t pow2ceil_u32(uint32_t v) {
  return v <= 1 ? 1u : 1u << (32 - __clz(v - 1));
}

// ---- per-level setup: probe mask from the (device-side) item count, zero the output count
__global__ void k_setup(const int32_t* __restrict__ n_dev, int64_t n_host, int64_t hash_cap,
                        int32_t* hash_mask_dev, int32_t* n_out_dev, int32_t* n_items_dev) {
  mm3d_griddep_wait();  // programmatic dependent launch: the previous kernel's writes are visible from here
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    int64_t n = n_dev ? (int64_t)*n_dev : n_host;
    uint32_t want = pow2ceil_u32((uint32_t)(2 * n < 32 ? 32 : 2 * n));
    if ((int64_t)want > hash_cap) want = (uint32_t)hash_cap;  // host sized cap for the capacity bound
    *hash_mask_dev = (int32_t)(want - 1);
    *n_out_dev = 0;
    *n_items_dev = (int32_t)n;
  }
}

__global__ void k_clear(uint64_t* __restrict__ hash_keys, int32_t* __restrict__ slot_min,
                        const int32_t* __restrict__ hash_mask_dev, const int32_t* __restrict__ n_items_dev,
                        int32_t* __restrict__ fill_buf, int fill_planes, int64_t fill_stride, int32_t fill_val) {
  mm3d_griddep_wait();  // programmatic dependent launch: the previous kernel's writes are visible from here
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nth = (int64_t)gridDim.x * blockDim.x;
  const int64_t slots = (int64_t)(uint32_t)*hash_mask_dev + 1;
  for (int64_t s = tid; s < slots; s += nth) {
    hash_keys[s] = MM3D_KEY_EMPTY;
    slot_min[s] = 0x7fffffff;
  }
  const int64_t n = *n_items_dev;
  for (int p = 0; p < fill_planes; ++p)
    for (int64_t i = tid; i < n; i += nth) fill_buf[p * fill_stride + i] = fill_val;
}

struct SrcCoords {
  const int64_t* coords;
  int spatial;
  int32_t* status;
  __device__ __forceinline__ uint64_t operator()(int64_t i) const {
    const longlong2* p = reinterpret_cast<const longlong2*>(coords) + 2 * i;
    longlong2 xy = __ldg(p), zb = __ldg(p + 1);
    if ((uint64_t)xy.x >= (uint64_t)spatial || (uint64_t)xy.y >= (uint64_t)spatial ||
        (uint64_t)zb.x >= (uint64_t)spatial || (uint64_t)zb.y >= 32768ull) {
      atomicOr(status, MM3D_STATUS_BAD_COORD);
      // clamp so the structure stays well formed; the host raises on the status bit
      xy.x &= 0xFFFF; xy.y &= 0xFFFF; zb.x &= 0xFFFF; zb.y &= 0x7FFF;
    }
    return mm3d_pack_key((uint64_t)xy.x, (uint64_t)xy.y, (uint64_t)zb.x, (uint64_t)zb.y);
  }
};

// Raw float points (metres) as the item source: rotation, scaling, min-shift, random translation, cast and
// receptive-field test of the reference's augment_and_scale_3d + loader filter (augment.cuh) are evaluated on the fly,
// so the int64 [N, 4] coordinate tensor between the two never exists (SURVEY 8(f).1).  A point outside the receptive
// field is what the reference drops before the collate: it raises MM3D_STATUS_DROPPED (the caller rebuilds from the
// filtered points -- row numbering must not see it) and is held at a clamped coordinate so the build stays well formed.
struct SrcPoints {
  const float* pts;
  const int64_t* offs;
  int B;
  const float* rot;
  float scale;
  int full_scale;
  const double* u;
  const uint32_t* mm;
  uint8_t* keep;
  float* min_value;
  double* offset;
  int32_t* status;
  __device__ __forceinline__ uint64_t operator()(int64_t i) const {
    const int b = mm3d_sample_of(offs, B, i);
    long long q[3];
    const bool ok = mm3d_point_voxel(pts, offs, b, i, rot, scale, full_scale, u, mm, min_value, offset, q);
    keep[i] = ok ? 1 : 0;
    if (!ok) {
      atomicOr(status, MM3D_STATUS_DROPPED);
#pragma unroll
      for (int j = 0; j < 3; ++j) q[j] = q[j] < 0 ? 0 : (q[j] >= full_scale ? full_scale - 1 : q[j]);
    }
    return mm3d_pack_key((uint64_t)q[0], (uint64_t)q[1], (uint64_t)q[2], (uint64_t)b);
  }
};

struct SrcCoarsen {
  const uint64_t* fine_keys;
  __device__ __forceinline__ uint64_t operator()(int64_t i) const {
    uint64_t k = __ldg(fine_keys + i);
    return mm3d_pack_key((uint64_t)(mm3d_key_x(k) >> 1), (uint64_t)(mm3d_key_y(k) >> 1),
                         (uint64_t)(mm3d_key_z(k) >> 1), mm3d_key_b(k));
  }
};

// ---- insert every item; remember its slot; slot_min = smallest item index that hit the slot
template <class Src>
__global__ void k_insert(Src src, const int32_t* __restrict__ n_items_dev, uint64_t* hash_keys,
                         int32_t* slot_min, const int32_t* __restrict__ hash_mask_dev,
                         int32_t* __restrict__ item_slot) {
  mm3d_griddep_wait();  // programmatic dependent launch: the previous kernel's writes are visible from here
  const int64_t n = *n_items_dev;
  const uint32_t mask = (uint32_t)*hash_mask_dev;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t key = src(i);
    uint32_t s = mm3d_hash(key) & mask;
    while (true) {
      unsigned long long prev = atomicCAS(reinterpret_cast<unsigned long long*>(hash_keys + s),
                                          (unsigned long long)MM3D_KEY_EMPTY, (unsigned long long)key);
      if (prev == MM3D_KEY_EMPTY || prev == key) break;
      s = (s + 1) & mask;
    }
    item_slot[i] = (int32_t)s;
    atomicMin(slot_min + s, (int32_t)i);
  }
}

__device__ __forceinline__ int block_exclusive_scan(int v, int* total) {
  // 256 threads; returns the exclusive prefix of v over the block, *total = block sum
  __shared__ int warp_sums[kScanThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += t;
  }
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  int woff = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < kScanThreads / 32; ++w) {
    int s = warp_sums[w];
    if (w < warp) woff += s;
    tot += s;
  }
  __syncthreads();
  *total = tot;
  return woff + incl - v;
}

// flags of the 4 consecutive items a thread owns (bit j set = item is a first occurrence)
__device__ __forceinline__ int thread_flags(const int32_t* __restrict__ item_slot,
                                            const int32_t* __restrict__ slot_min, int64_t base, int64_t n) {
  int f = 0;
  if (base + kItemsPerThread <= n) {
    int4 s = *reinterpret_cast<const int4*>(item_slot + base);
    f |= (slot_min[s.x] == (int32_t)(base + 0)) << 0;
    f |= (slot_min[s.y] == (int32_t)(base + 1)) << 1;
    f |= (slot_min[s.z] == (int32_t)(base + 2)) << 2;
    f |= (slot_min[s.w] == (int32_t)(base + 3)) << 3;
  } else {
    for (int j = 0; j < kItemsPerThread; ++j)
      if (base + j < n) f |= (slot_min[item_slot[base + j]] == (int32_t)(base + j)) << j;
  }
  return f;
}

__global__ void __launch_bounds__(kScanThreads)
k_count(const int32_t* __restrict__ item_slot, const int32_t* __restrict__ slot_min,
        const int32_t* __restrict__ n_items_dev, int32_t* __restrict__ block_sums) {
  mm3d_griddep_wait();  // programmatic dependent launch: the previous kernel's writes are visible from here
  const int64_t n = *n_items_dev;
  const int64_t base = (int64_t)blockIdx.x * kItemsPerBlock + threadIdx.x * kItemsPerThread;
  int c = base < n ? __popc(thread_flags(item_slot, slot_min, base, n)) : 0;
  int total;
  block_exclusive_scan(c, &total);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// exclusive scan of the per-block counts by ONE block (counts are few: n_cap / 1024)
__global__ void __launch_bounds__(kScanThreads)
k_scan_blocks(int32_t* __restrict__ block_sums, int nblocks, int32_t* __restrict__ n_out_dev) {
  mm3d_griddep_wait();  // programmatic dependent launch: the previous kernel's writes are visible from here
  int carry = 0;
  for (int base = 0; base < nblocks; base += kScanThreads) {
    int i = base + threadIdx.x;
    int v = i < nblocks ? block_sums[i] : 0;
    int total;
    int ex = block_exclusive_scan(v, &total);
    if (i < nblocks) block_sums[i] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0) *n_out_dev = carry;
}

__global__ void __launch_bounds__(kScanThreads)
k_assign(const int32_t* __restrict__ item_slot, const int32_t* __restrict__ slot_min,
         const int32_t* __restrict__ n_items_dev, const int32_t* __restrict__ block_offs,
         const uint64_t* __restrict__ hash_keys, int32_t* __restrict__ hash_vals,
         uint64_t* __restrict__ uniq_keys) {
  mm3d_griddep_wait();  // programmatic dependent launch: the previous kernel's writes are visible from here
  const int64_t n = *n_items_dev;
  const int64_t base = (int64_t)blockIdx.x * kItemsPerBlock + threadIdx.x * kItemsPerThread;
  const int f = base < n ? thread_flags(item_slot, slot_min, base, n) : 0;
  int total;
  int rank = block_offs[blockIdx.x] + block_exclusive_scan(__popc(f), &total);
#pragma unroll
  for (int j = 0; j < kItemsPerThread; ++j) {
    if (f & (1 << j)) {
      const int32_t s = item_slot[base + j];
      hash_vals[s] = rank;
      uniq_keys[rank] = hash_keys[s];
      ++rank;
    }
  }
}

// ---- ids of all items + the level-specific by-products
__global__ void k_ids_level0(const int32_t* __restrict__ item_slot, const int32_t* __restrict__ hash_vals,
                             const int32_t* __restrict__ n_items_dev, int32_t* __restrict__ p2v,
                             int32_t* __restrict__ npts) {
  mm3d_griddep_wait();  // programmatic dependent launch: the previous kernel's writes are visible from here
  const int64_t n = *n_items_dev;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t v = hash_vals[item_slot[i]];
    p2v[i] = v;
    atomicAdd(npts + v, 1);
  }
}

__global__ void k_ids_coarsen(const int32_t* __restrict__ item_slot, const int32_t* __restrict__ hash_vals,
                              const int32_t* __restrict__ n_items_dev, const uint64_t* __restrict__ fine_keys,
                              int32_t* __restrict__ parent, uint8_t* __restrict__ off,
                              int32_t* __restrict__ child_tbl, int64_t tbl_stride) {
  mm3d_griddep_wait();  // programmatic dependent launch: the previous kernel's writes are visible from here
  const int64_t n = *n_items_dev;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t q = hash_vals[item_slot[i]];
    const uint64_t k = __ldg(fine_keys + i);
    const int o = ((mm3d_key_x(k) & 1) * 2 + (mm3d_key_y(k) & 1)) * 2 + (mm3d_key_z(k) & 1);
    parent[i] = q;
    off[i] = (uint8_t)o;
    child_tbl[(int64_t)o * tbl_stride + q] = (int32_t)i;  // (q, o) is unique: no race
  }
}

// ---- 3^3 neighbour table, offset-major: one thread per (k, row), rows fastest => coalesced.  The table is symmetric
// (row j is the neighbour of row i at offset k exactly when i is the neighbour of j at offset 26 - k), so only the
// offsets 0..12 are probed: a hit also writes the mirrored entry, and the mirrored half is pre-filled with -1 by the
// launch's memset -- 13 hash probes per voxel instead of 26.  blockIdx.y = k: no 64-bit division per entry.
__global__ void k_nbr27(const uint64_t* __restrict__ keys, const int32_t* __restrict__ n_dev, int spatial,
                        const uint64_t* __restrict__ hash_keys, const int32_t* __restrict__ hash_vals,
                        const int32_t* __restrict__ hash_mask_dev, int32_t* __restrict__ tbl, int64_t tbl_stride) {
  mm3d_griddep_wait();  // programmatic dependent launch: the previous kernel's writes are visible from here
  const int64_t n = *n_dev;
  const uint32_t mask = (uint32_t)*hash_mask_dev;
  const int k = (int)blockIdx.y;  // 0..13
  const int dx = k / 9 - 1, dy = (k / 3) % 3 - 1, dz = k % 3 - 1;
  for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < n; row += (int64_t)gridDim.x * blockDim.x) {
    if (k == 13) {
      tbl[(int64_t)13 * tbl_stride + row] = (int32_t)row;
      continue;
    }
    const uint64_t key = __ldg(keys + row);
    const int x = mm3d_key_x(key) + dx, y = mm3d_key_y(key) + dy, z = mm3d_key_z(key) + dz;
    int32_t r = -1;
    if ((unsigned)x < (unsigned)spatial && (unsigned)y < (unsigned)spatial && (unsigned)z < (unsigned)spatial)
      r = mm3d_hash_find(hash_keys, hash_vals, mask, mm3d_pack_key((uint64_t)x, (uint64_t)y, (uint64_t)z, mm3d_key_b(key)));
    tbl[(int64_t)k * tbl_stride + row] = r;
    if (r >= 0) tbl[(int64_t)(26 - k) * tbl_stride + r] = (int32_t)row;  // (r, 26 - k) is unique: no race
  }
}

struct UniqueWs {
  int32_t* item_slot;   // [n_cap]
  int32_t* slot_min;    // [hash_cap]
  int32_t* block_sums;  // [nblocks]
  int32_t* n_items;     // [1]
  int nblocks;
};

size_t unique_ws_bytes(int64_t n_cap) {
  int64_t hash_cap = mm3d_hash_capacity(n_cap);
  int64_t nblocks = mm3d_cdiv(n_cap > 0 ? n_cap : 1, kItemsPerBlock);
  return mm3d_align(4 * (size_t)(n_cap + 4)) + mm3d_align(4 * (size_t)hash_cap) +
         mm3d_align(4 * (size_t)nblocks) + 256;
}

int carve_ws(void* ws, size_t ws_bytes, int64_t n_cap, int64_t hash_cap, UniqueWs* out) {
  MM3D_REQUIRE(ws != nullptr && ws_bytes >= unique_ws_bytes(n_cap), MM3D_ERR_WORKSPACE,
               "unique workspace too small: have %zu need %zu", ws_bytes, unique_ws_bytes(n_cap));
  MM3D_REQUIRE(hash_cap >= mm3d_hash_capacity(n_cap), MM3D_ERR_INVALID,
               "hash_cap %lld < required %lld", (long long)hash_cap, (long long)mm3d_hash_capacity(n_cap));
  MM3D_REQUIRE(((uintptr_t)ws & 15) == 0, MM3D_ERR_INVALID, "workspace must be 16-byte aligned");
  char* p = (char*)ws;
  out->nblocks = (int)mm3d_cdiv(n_cap > 0 ? n_cap : 1, kItemsPerBlock);
  out->item_slot = (int32_t*)p;  p += mm3d_align(4 * (size_t)(n_cap + 4));
  out->slot_min = (int32_t*)p;   p += mm3d_align(4 * (size_t)mm3d_hash_capacity(n_cap));
  out->block_sums = (int32_t*)p; p += mm3d_align(4 * (size_t)out->nblocks);
  out->n_items = (int32_t*)p;
  return MM3D_OK;
}

// Group row boundaries (grouped BatchNorm statistics): several batches built as one structure, group k's scans with
// batch indices [batch_start[k], batch_start[k + 1]).  Its points precede group k + 1's and every level numbers its rows
// by first occurrence, so each group is one contiguous row range at every level and "batch >= batch_start[k]" is false
// then true along the rows: boundary k is the first row where it holds (a binary search).  blockIdx.x = level.
struct GroupLevels {
  const uint64_t* keys[MM3D_MAX_GROUP_LEVELS];
};
__global__ void k_group_bounds(const __grid_constant__ GroupLevels lv, const int32_t* __restrict__ counts,
                               const int64_t* __restrict__ batch_start, int groups, int32_t* __restrict__ bounds) {
  mm3d_griddep_wait();
  const int l = blockIdx.x;
  const int64_t n = counts[l];
  for (int k = threadIdx.x; k <= groups; k += blockDim.x) {
    int64_t lo = 0, hi = n;  // boundary k in [lo, hi]
    if (k == 0) hi = 0;
    else if (k < groups) {
      const int64_t b = batch_start[k];
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if ((int64_t)(lv.keys[l][mid] >> 48) >= b) hi = mid;
        else lo = mid + 1;
      }
    }
    bounds[l * (groups + 1) + k] = (int32_t)hi;
  }
}

}  // namespace

// bounds[l (groups + 1) + k]: the first row of group k at level l (bounds[.. + groups] = the level's row count)
extern "C" int mm3d_group_bounds(const uint64_t* const* keys, const int32_t* counts, int levels, const int64_t* batch_start,
                                 int groups, int32_t* bounds, mm3d_stream_t stream) {
  MM3D_REQUIRE(levels >= 1 && levels <= MM3D_MAX_GROUP_LEVELS && groups >= 1 && keys && counts && bounds &&
                   (groups == 1 || batch_start),
               MM3D_ERR_INVALID, "group_bounds: bad arguments");
  GroupLevels lv{};
  for (int l = 0; l < levels; ++l) lv.keys[l] = keys[l];
  MM3D_CUDA(mm3d_launch_pdl(k_group_bounds, dim3(levels), dim3(32), 0, (cudaStream_t)stream, lv, counts, batch_start, groups,
                            bounds));
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_group_bounds");
  return MM3D_OK;
}

extern "C" int64_t mm3d_hash_capacity(int64_t n) {
  int64_t want = 2 * (n > 16 ? n : 16);
  int64_t cap = 32;
  while (cap < want) cap <<= 1;
  return cap + 1;  // +1: the last int32 of hash_vals holds the probe mask of the built table
}

extern "C" size_t mm3d_unique_workspace_bytes(int64_t n) { return unique_ws_bytes(n); }

// hash_vals[hash_cap - 1] stores the probe mask chosen on the device (see k_setup).
static inline int32_t* mask_slot(int32_t* hash_vals, int64_t hash_cap) { return hash_vals + (hash_cap - 1); }

extern "C" int mm3d_voxelize(const int64_t* coords, int64_t n_points, int spatial_size,
                             uint64_t* hash_keys, int32_t* hash_vals, int64_t hash_cap,
                             int32_t* p2v, uint64_t* vox_keys, int32_t* npts, int32_t* n_vox_dev,
                             int32_t* status_dev, void* ws, size_t ws_bytes, mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(n_points >= 0 && n_points < (1ll << 30), MM3D_ERR_INVALID, "n_points out of range");
  MM3D_REQUIRE(spatial_size > 0 && spatial_size <= 65536, MM3D_ERR_INVALID, "spatial_size must be in (0, 65536]");
  MM3D_REQUIRE(((uintptr_t)coords & 15) == 0, MM3D_ERR_INVALID, "coords must be 16-byte aligned");
  UniqueWs w;
  int rc = carve_ws(ws, ws_bytes, n_points, hash_cap, &w);
  if (rc) return rc;
  int32_t* mask_dev = mask_slot(hash_vals, hash_cap);
  MM3D_CUDA(mm3d_launch_pdl(k_setup, dim3(1), dim3(32), 0, stream, nullptr, n_points, hash_cap - 1, mask_dev, n_vox_dev, w.n_items));
  MM3D_CUDA(mm3d_launch_pdl(k_clear, dim3(mm3d_grid(hash_cap, 256)), dim3(256), 0, stream, hash_keys, w.slot_min, mask_dev, w.n_items, npts, 1, 0, 0));
  if (n_points > 0) {
    SrcCoords src{coords, spatial_size, status_dev};
    MM3D_CUDA(mm3d_launch_pdl(k_insert<SrcCoords>, dim3(mm3d_grid(n_points, 256)), dim3(256), 0, stream, src, w.n_items, hash_keys, w.slot_min, mask_dev, w.item_slot));
    MM3D_CUDA(mm3d_launch_pdl(k_count, dim3(w.nblocks), dim3(kScanThreads), 0, stream, w.item_slot, w.slot_min, w.n_items, w.block_sums));
    MM3D_CUDA(mm3d_launch_pdl(k_scan_blocks, dim3(1), dim3(kScanThreads), 0, stream, w.block_sums, w.nblocks, n_vox_dev));
    MM3D_CUDA(mm3d_launch_pdl(k_assign, dim3(w.nblocks), dim3(kScanThreads), 0, stream, w.item_slot, w.slot_min, w.n_items, w.block_sums,
                                                     hash_keys, hash_vals, vox_keys));
    MM3D_CUDA(mm3d_launch_pdl(k_ids_level0, dim3(mm3d_grid(n_points, 256)), dim3(256), 0, stream, w.item_slot, hash_vals, w.n_items, p2v, npts));
  }
  mm3d_count_launches(n_points > 0 ? 7 : 2);
  MM3D_CHECK_LAUNCH("mm3d_voxelize");
  return MM3D_OK;
}

extern "C" size_t mm3d_voxelize_points_workspace_bytes(int64_t n, int B) {
  return unique_ws_bytes(n) + mm3d_align(sizeof(uint32_t) * 6 * (size_t)(B > 0 ? B : 1));
}

extern "C" int mm3d_voxelize_points(const float* points, const int64_t* sample_offsets, int B, int64_t n_points,
                                    const float* rot, float scale, int full_scale, const double* transl_u,
                                    uint8_t* keep, float* min_value, double* offset,
                                    uint64_t* hash_keys, int32_t* hash_vals, int64_t hash_cap,
                                    int32_t* p2v, uint64_t* vox_keys, int32_t* npts, int32_t* n_vox_dev,
                                    int32_t* status_dev, void* ws, size_t ws_bytes, mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(n_points >= 0 && n_points < (1ll << 30), MM3D_ERR_INVALID, "n_points out of range");
  MM3D_REQUIRE(B > 0 && B <= 32768, MM3D_ERR_INVALID, "voxelize_points: B must be in (0, 32768]");
  MM3D_REQUIRE(full_scale > 0 && full_scale <= 65536, MM3D_ERR_INVALID, "full_scale must be in (0, 65536]");
  MM3D_REQUIRE(ws_bytes >= mm3d_voxelize_points_workspace_bytes(n_points, B), MM3D_ERR_WORKSPACE,
               "voxelize_points: workspace too small");
  MM3D_REQUIRE(n_points == 0 || (points && sample_offsets && rot && keep && min_value && offset), MM3D_ERR_INVALID,
               "voxelize_points: null pointer");
  UniqueWs w;
  int rc = carve_ws(ws, ws_bytes, n_points, hash_cap, &w);
  if (rc) return rc;
  uint32_t* mm = (uint32_t*)((char*)ws + unique_ws_bytes(n_points));
  int32_t* mask_dev = mask_slot(hash_vals, hash_cap);
  MM3D_CUDA(mm3d_launch_pdl(k_setup, dim3(1), dim3(32), 0, stream, nullptr, n_points, hash_cap - 1, mask_dev, n_vox_dev, w.n_items));
  MM3D_CUDA(mm3d_launch_pdl(k_clear, dim3(mm3d_grid(hash_cap, 256)), dim3(256), 0, stream, hash_keys, w.slot_min, mask_dev, w.n_items, npts, 1, 0, 0));
  if (n_points > 0) {
    rc = mm3d_launch_minmax(points, sample_offsets, B, n_points, rot, scale, mm, stream);
    if (rc) return rc;
    SrcPoints src{points, sample_offsets, B, rot, scale, full_scale, transl_u, mm, keep, min_value, offset, status_dev};
    MM3D_CUDA(mm3d_launch_pdl(k_insert<SrcPoints>, dim3(mm3d_grid(n_points, 256)), dim3(256), 0, stream, src, w.n_items, hash_keys, w.slot_min, mask_dev, w.item_slot));
    MM3D_CUDA(mm3d_launch_pdl(k_count, dim3(w.nblocks), dim3(kScanThreads), 0, stream, w.item_slot, w.slot_min, w.n_items, w.block_sums));
    MM3D_CUDA(mm3d_launch_pdl(k_scan_blocks, dim3(1), dim3(kScanThreads), 0, stream, w.block_sums, w.nblocks, n_vox_dev));
    MM3D_CUDA(mm3d_launch_pdl(k_assign, dim3(w.nblocks), dim3(kScanThreads), 0, stream, w.item_slot, w.slot_min, w.n_items, w.block_sums,
                                                     hash_keys, hash_vals, vox_keys));
    MM3D_CUDA(mm3d_launch_pdl(k_ids_level0, dim3(mm3d_grid(n_points, 256)), dim3(256), 0, stream, w.item_slot, hash_vals, w.n_items, p2v, npts));
  }
  mm3d_count_launches(n_points > 0 ? 7 : 2);
  MM3D_CHECK_LAUNCH("mm3d_voxelize_points");
  return MM3D_OK;
}

extern "C" int mm3d_coarsen(const uint64_t* fine_keys, const int32_t* n_fine_dev, int64_t n_fine_cap,
                            uint64_t* hash_keys, int32_t* hash_vals, int64_t hash_cap,
                            int32_t* parent, uint8_t* off, uint64_t* coarse_keys,
                            int32_t* child_tbl, int64_t tbl_stride, int32_t* n_coarse_dev,
                            void* ws, size_t ws_bytes, mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(n_fine_cap >= 0 && n_fine_cap < (1ll << 30), MM3D_ERR_INVALID, "n_fine_cap out of range");
  MM3D_REQUIRE(tbl_stride >= n_fine_cap, MM3D_ERR_INVALID, "tbl_stride must be >= n_fine_cap");
  UniqueWs w;
  int rc = carve_ws(ws, ws_bytes, n_fine_cap, hash_cap, &w);
  if (rc) return rc;
  int32_t* mask_dev = mask_slot(hash_vals, hash_cap);
  MM3D_CUDA(mm3d_launch_pdl(k_setup, dim3(1), dim3(32), 0, stream, n_fine_dev, 0, hash_cap - 1, mask_dev, n_coarse_dev, w.n_items));
  // child table: -1 over (at most) n_fine rows of each of the 8 planes; coarse rows <= fine rows
  MM3D_CUDA(mm3d_launch_pdl(k_clear, dim3(mm3d_grid(hash_cap, 256)), dim3(256), 0, stream, hash_keys, w.slot_min, mask_dev, w.n_items,
                                                        child_tbl, 8, tbl_stride, -1));
  if (n_fine_cap > 0) {
    SrcCoarsen src{fine_keys};
    MM3D_CUDA(mm3d_launch_pdl(k_insert<SrcCoarsen>, dim3(mm3d_grid(n_fine_cap, 256)), dim3(256), 0, stream, src, w.n_items, hash_keys, w.slot_min, mask_dev, w.item_slot));
    MM3D_CUDA(mm3d_launch_pdl(k_count, dim3(w.nblocks), dim3(kScanThreads), 0, stream, w.item_slot, w.slot_min, w.n_items, w.block_sums));
    MM3D_CUDA(mm3d_launch_pdl(k_scan_blocks, dim3(1), dim3(kScanThreads), 0, stream, w.block_sums, w.nblocks, n_coarse_dev));
    MM3D_CUDA(mm3d_launch_pdl(k_assign, dim3(w.nblocks), dim3(kScanThreads), 0, stream, w.item_slot, w.slot_min, w.n_items, w.block_sums,
                                                     hash_keys, hash_vals, coarse_keys));
    MM3D_CUDA(mm3d_launch_pdl(k_ids_coarsen, dim3(mm3d_grid(n_fine_cap, 256)), dim3(256), 0, stream, w.item_slot, hash_vals, w.n_items, fine_keys,
                                                                 parent, off, child_tbl, tbl_stride));
  }
  mm3d_count_launches(n_fine_cap > 0 ? 7 : 2);
  MM3D_CHECK_LAUNCH("mm3d_coarsen");
  return MM3D_OK;
}

extern "C" int mm3d_build_nbr27(const uint64_t* keys, const int32_t* n_dev, int64_t n_cap, int spatial_size,
                                const uint64_t* hash_keys, const int32_t* hash_vals, int64_t hash_cap,
                                int32_t* nbr_tbl, int64_t tbl_stride, mm3d_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MM3D_REQUIRE(tbl_stride >= n_cap, MM3D_ERR_INVALID, "tbl_stride must be >= n_cap");
  MM3D_REQUIRE(spatial_size > 0 && spatial_size <= 65536, MM3D_ERR_INVALID, "spatial_size must be in (0, 65536]");
  if (n_cap > 0) {
    // the mirrored half (offsets 14..26) starts as "no neighbour"; hits of the probed half fill it in
    MM3D_CUDA(cudaMemsetAsync(nbr_tbl + 14 * tbl_stride, 0xFF, sizeof(int32_t) * (size_t)13 * tbl_stride, stream));
    MM3D_CUDA(mm3d_launch_pdl(k_nbr27, dim3(mm3d_grid(n_cap, 256, 8), 14), dim3(256), 0, stream, keys, n_dev, spatial_size, hash_keys,
                              hash_vals, hash_vals + (hash_cap - 1), nbr_tbl, tbl_stride));
  }
  mm3d_count_launches(n_cap > 0 ? 1 : 0);
  MM3D_CHECK_LAUNCH("mm3d_build_nbr27");
  return MM3D_OK;
}
