// Group-by-key lists of the deterministic mode: for n entries with keys in [0, n_keys) (key < 0 = no key), the
// CSR pair start[n_keys + 1], list[<= n] with each key's entries in ASCENDING entry index.  The segmented sums that
// replace the scatter-adds (InputLayer forward, OutputLayer backward, lift backward) read a key's entries in that
// order, so their results do not depend on the order in which any atomic landed.
//
//   count (integer atomics, or the caller's counts) -> exclusive scan -> scatter with atomic cursors
//   -> sort every segment by entry index
// The scatter order is arbitrary; the sort makes the result unique.  One thread sorts a segment in place: insertion sort
// up to kGbShortSeg entries (the common case: points of one voxel or pixel), heapsort above, so a segment of k entries
// costs O(k log k) steps on its thread and no scratch memory.
#include "common.cuh"

namespace {

constexpr int kGbThreads = 256, kGbItems = 4, kGbTile = kGbThreads * kGbItems, kGbShortSeg = 32;

__device__ __forceinline__ int gb_block_exclusive_scan(int v, int* total) {
  __shared__ int warp_sums[kGbThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += t;
  }
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  int woff = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < kGbThreads / 32; ++w) {
    const int s = warp_sums[w];
    if (w < warp) woff += s;
    tot += s;
  }
  __syncthreads();
  *total = tot;
  return woff + incl - v;
}

__global__ void k_gb_count(const int32_t* __restrict__ key, int64_t n, int32_t* __restrict__ cnt) {
  mm3d_griddep_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t k = __ldg(key + i);
    if (k >= 0) atomicAdd(cnt + k, 1);
  }
}

// per tile of kGbTile counts: its sum
__global__ void __launch_bounds__(kGbThreads)
k_gb_tile_sums(const int32_t* __restrict__ cnt, int64_t n_keys, int32_t* __restrict__ tile_sums) {
  mm3d_griddep_wait();
  const int64_t base = (int64_t)blockIdx.x * kGbTile + (int64_t)threadIdx.x * kGbItems;
  int s = 0;
#pragma unroll
  for (int j = 0; j < kGbItems; ++j)
    if (base + j < n_keys) s += __ldg(cnt + base + j);
  int total;
  gb_block_exclusive_scan(s, &total);
  if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

// exclusive scan of the tile sums by one block; start[n_keys] = the grand total
__global__ void __launch_bounds__(kGbThreads)
k_gb_scan_tiles(int32_t* __restrict__ tile_sums, int n_tiles, int32_t* __restrict__ start, int64_t n_keys) {
  mm3d_griddep_wait();
  int carry = 0;
  for (int b = 0; b < n_tiles; b += kGbThreads) {
    const int i = b + threadIdx.x;
    const int v = i < n_tiles ? tile_sums[i] : 0;
    int total;
    const int ex = gb_block_exclusive_scan(v, &total);
    if (i < n_tiles) tile_sums[i] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0) start[n_keys] = carry;
}

// start[k] = exclusive prefix of the counts; cursor[k] = start[k] (the scatter's atomic cursors)
__global__ void __launch_bounds__(kGbThreads)
k_gb_scan_write(const int32_t* __restrict__ cnt, int64_t n_keys, const int32_t* __restrict__ tile_offs,
                int32_t* __restrict__ start, int32_t* __restrict__ cursor) {
  mm3d_griddep_wait();
  const int64_t base = (int64_t)blockIdx.x * kGbTile + (int64_t)threadIdx.x * kGbItems;
  int c[kGbItems], s = 0;
#pragma unroll
  for (int j = 0; j < kGbItems; ++j) {
    c[j] = base + j < n_keys ? __ldg(cnt + base + j) : 0;
    s += c[j];
  }
  int total;
  int run = tile_offs[blockIdx.x] + gb_block_exclusive_scan(s, &total);
#pragma unroll
  for (int j = 0; j < kGbItems; ++j) {
    if (base + j < n_keys) {
      start[base + j] = run;
      cursor[base + j] = run;
    }
    run += c[j];
  }
}

__global__ void k_gb_scatter(const int32_t* __restrict__ key, int64_t n, int32_t* __restrict__ cursor,
                             int32_t* __restrict__ list) {
  mm3d_griddep_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t k = __ldg(key + i);
    if (k >= 0) list[atomicAdd(cursor + k, 1)] = (int32_t)i;
  }
}

// max-heap sift-down of a[i] within a[0 .. n)
__device__ __forceinline__ void gb_sift_down(int32_t* a, int32_t i, int32_t n) {
  const int32_t v = a[i];
  for (int32_t c = 2 * i + 1; c < n; c = 2 * i + 1) {
    if (c + 1 < n && a[c + 1] > a[c]) ++c;
    if (a[c] <= v) break;
    a[i] = a[c];
    i = c;
  }
  a[i] = v;
}

// every segment sorted ascending (one thread per key)
__global__ void k_gb_sort(const int32_t* __restrict__ start, int64_t n_keys, int32_t* __restrict__ list) {
  mm3d_griddep_wait();
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n_keys; k += (int64_t)gridDim.x * blockDim.x) {
    const int32_t b = __ldg(start + k), e = __ldg(start + k + 1);
    if (e - b > kGbShortSeg) {  // heapsort
      int32_t* a = list + b;
      const int32_t n = e - b;
      for (int32_t i = n / 2 - 1; i >= 0; --i) gb_sift_down(a, i, n);
      for (int32_t m = n - 1; m > 0; --m) {
        const int32_t t = a[0];
        a[0] = a[m];
        a[m] = t;
        gb_sift_down(a, 0, m);
      }
      continue;
    }
    for (int32_t i = b + 1; i < e; ++i) {
      const int32_t v = list[i];
      int32_t j = i - 1;
      while (j >= b && list[j] > v) {
        list[j + 1] = list[j];
        --j;
      }
      list[j + 1] = v;
    }
  }
}

}  // namespace

size_t mm3d_group_by_workspace_bytes(int64_t n_keys) {
  const int64_t n_tiles = mm3d_cdiv(n_keys > 0 ? n_keys : 1, kGbTile);
  return 2 * mm3d_align(sizeof(int32_t) * (size_t)(n_keys > 0 ? n_keys : 1)) + mm3d_align(sizeof(int32_t) * (size_t)n_tiles);
}

int mm3d_group_by(const int32_t* key, const int32_t* counts, int64_t n, int64_t n_keys, int32_t* start, int32_t* list,
                  void* ws, size_t ws_bytes, cudaStream_t stream) {
  MM3D_REQUIRE(n >= 0 && n < (1ll << 31) && n_keys >= 0 && n_keys < (1ll << 31), MM3D_ERR_INVALID,
               "group-by: %lld entries / %lld keys out of range", (long long)n, (long long)n_keys);
  MM3D_REQUIRE(start && ws && ws_bytes >= mm3d_group_by_workspace_bytes(n_keys), MM3D_ERR_WORKSPACE,
               "group-by: workspace too small");
  if (n_keys == 0) {
    MM3D_CUDA(cudaMemsetAsync(start, 0, sizeof(int32_t), stream));
    return MM3D_OK;
  }
  char* w = (char*)ws;
  int32_t* cursor = (int32_t*)w;
  int32_t* cnt = (int32_t*)(w + mm3d_align(sizeof(int32_t) * (size_t)n_keys));
  int32_t* tile_sums = (int32_t*)(w + 2 * mm3d_align(sizeof(int32_t) * (size_t)n_keys));
  const int n_tiles = (int)mm3d_cdiv(n_keys, kGbTile);
  int launches = 0;
  if (!counts) {
    MM3D_REQUIRE(n == 0 || key, MM3D_ERR_INVALID, "group-by: null key array");
    MM3D_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (size_t)n_keys, stream));
    if (n > 0) {
      MM3D_CUDA(mm3d_launch_pdl(k_gb_count, dim3(mm3d_grid(n, 256)), dim3(256), 0, stream, key, n, cnt));
      ++launches;
    }
    counts = cnt;
  }
  MM3D_CUDA(mm3d_launch_pdl(k_gb_tile_sums, dim3(n_tiles), dim3(kGbThreads), 0, stream, counts, n_keys, tile_sums));
  MM3D_CUDA(mm3d_launch_pdl(k_gb_scan_tiles, dim3(1), dim3(kGbThreads), 0, stream, tile_sums, n_tiles, start, n_keys));
  MM3D_CUDA(mm3d_launch_pdl(k_gb_scan_write, dim3(n_tiles), dim3(kGbThreads), 0, stream, counts, n_keys,
                            (const int32_t*)tile_sums, start, cursor));
  launches += 3;
  if (n > 0) {
    MM3D_REQUIRE(key && list, MM3D_ERR_INVALID, "group-by: null key or list array");
    MM3D_CUDA(mm3d_launch_pdl(k_gb_scatter, dim3(mm3d_grid(n, 256)), dim3(256), 0, stream, key, n, cursor, list));
    MM3D_CUDA(mm3d_launch_pdl(k_gb_sort, dim3(mm3d_grid(n_keys, 256)), dim3(256), 0, stream, (const int32_t*)start, n_keys, list));
    launches += 2;
  }
  mm3d_count_launches(launches);
  MM3D_CHECK_LAUNCH("mm3d_group_by");
  return MM3D_OK;
}

// ---------------------------------------------------------------------------------- C ABI: voxel point lists
extern "C" size_t mm3d_point_csr_workspace_bytes(int64_t n_vox) { return mm3d_group_by_workspace_bytes(n_vox); }

extern "C" int mm3d_point_csr(const int32_t* p2v, const int32_t* npts, int64_t n_points, int64_t n_vox, int32_t* vox_start,
                              int32_t* vox_pts, void* ws, size_t ws_bytes, mm3d_stream_t stream) {
  MM3D_REQUIRE(n_vox == 0 || npts, MM3D_ERR_INVALID, "point_csr: null npts");
  return mm3d_group_by(p2v, npts, n_points, n_vox, vox_start, vox_pts, ws, ws_bytes, (cudaStream_t)stream);
}
