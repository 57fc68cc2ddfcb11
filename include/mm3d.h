/*
 * mm3d.h -- C ABI of libmm3d.so, the B200 (sm_100a) implementation of MM2D3D's 3D-branch
 * hot path.  This is the drop-in boundary: it sits where SparseConvNet's pybind module
 * `sparseconvnet.SCN` sits under the reference's `import sparseconvnet as scn`
 * (/root/reference/experiments_USA_SING/rgbd_rgbxyz_sigmoid_for_rgb/3d_net/scn_unet.py:1,
 * constructors at :38-52,:56-81,:113-117) and where the advanced-indexing lift sits in
 * 2d_net/model.py:131-137,:166-173.  SparseConvNet (facebookresearch/SparseConvNet@dcf6a7ff,
 * environment.yml:37) is not vendored, so the "replaces" notes below name its pybind entry
 * points as listed in SURVEY.md section 8(b).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless named *_host;
 *   - the caller owns every buffer (PyTorch tensors in the shipped host code); scratch comes
 *     from the caller through (ws, ws_bytes) with a *_workspace_bytes() query per op;
 *   - every call is stream-ordered on `stream` (a cudaStream_t) and never synchronises the host;
 *   - returns MM3D_OK or an error code; mm3d_last_error() gives the thread-local message;
 *   - features are row-major float32 [rows, channels]; weights are SparseConvNet's
 *     [K, C_in, C_out] (its parameter tensor [K, 1, C_in, C_out] with groups == 1);
 *   - rule tables are offset-major int32 `tbl[k * tbl_stride + out_row]` = input row or -1.
 */
#ifndef MM3D_H_
#define MM3D_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MM3D_ABI_VERSION 8

#define MM3D_OK 0
#define MM3D_ERR_INVALID 1     /* bad argument */
#define MM3D_ERR_CUDA 2        /* a CUDA runtime call or launch failed */
#define MM3D_ERR_WORKSPACE 3   /* workspace too small */
#define MM3D_ERR_UNSUPPORTED 4 /* shape / mode not implemented by this build */

/* arithmetic modes of the convolution kernels */
#define MM3D_MODE_FP32 0 /* SIMT FP32 FMA -- the parity mode (1e-4) */
#define MM3D_MODE_TF32 1 /* tcgen05 kind::tf32, FP32 accumulate in TMEM (1e-2) */
#define MM3D_MODE_BF16 2 /* tcgen05 kind::f16 with BF16 gathered operands and weights, FP32 accumulate (1e-2 per
                          * op): forward, dgrad and weight gradient move half the bytes of the TF32 mode.  The gathered
                          * operands (`in` of mm3d_conv_fwd; `in` and `d_out` of mm3d_conv_wgrad) carry an FP32 plane of
                          * [rows, c] floats (TF32-rounded values) and, rows * c floats behind it, a BF16 plane of
                          * [rows, c] bfloat16 (mm3d_split_bf16).  mm3d_conv_wgrad reads the BF16 planes for c_in <= 128
                          * and falls back to the TF32 kernel on the FP32 planes above that */
#define MM3D_MODE_TF32X3 3 /* tcgen05, three error-compensated TF32 products (hi.hi + lo.hi + hi.lo), FP32 accumulate:
                            * FP32-grade results (1e-4 bar) on the tensor cores.  The gathered operands (`in` of
                            * mm3d_conv_fwd; `in` and `d_out` of mm3d_conv_wgrad) carry TWO planes of [rows, c] floats,
                            * hi = tf32(x) then lo = tf32(x - hi) (mm3d_split_tf32) */

/* Deterministic mode: the `flags` bit of the *_ex entry points below.  With it, an op whose default form adds into
 * its output with floating-point atomics (so that the result depends on the order in which they land) sums in a
 * fixed order instead and returns the same bits on every run.  The scatter-adds of the point -> voxel and point ->
 * pixel sums become segmented sums over group-by-key lists (mm3d_point_csr, mm3d_lift_csr and the *_csr ops); the
 * small FP64 totals (RGB-mask weight gradient, KL loss, heads3d loss and weight gradients) keep one partial vector per
 * CTA, at most MM3D_DET_CTAS CTAs, summed in CTA order by the launch that converts them to float. */
#define MM3D_DETERMINISTIC 0x100
#define MM3D_DET_CTAS 592

/* flags of mm3d_conv_fwd */
#define MM3D_CONV_TRANSPOSE_W 1 /* use W[k]^T: weight is [K, c_out, c_in] as stored by the forward layer (dgrad) */
#define MM3D_CONV_MIRROR_K 2    /* use W[K-1-k] for table column k (submanifold dgrad) */

typedef void* mm3d_stream_t; /* cudaStream_t */

#if defined(__GNUC__)
#define MM3D_API __attribute__((visibility("default")))
#else
#define MM3D_API
#endif

MM3D_API int mm3d_abi_version(void);
MM3D_API const char* mm3d_last_error(void);
/* 1 if the running device is compute capability 10.x (tcgen05 paths usable), 0 otherwise, <0 on error */
MM3D_API int mm3d_device_supports_tc(void);
/* number of CUDA kernels this library has launched in this process (for the benchmark's gpu_launches) */
MM3D_API long long mm3d_kernel_launches(void);
/* Returns (and clears) the current device's sticky error bits: 1 = a kernel's bounded internal wait (mbarrier
 * pipeline, BatchNorm grid barrier) timed out -- its results are garbage; 2 = mm3d_lift2d_* met an index outside
 * the image (that point was skipped).  0 = none, <0 = could not be read.  The bits live in mapped pinned host
 * memory, so this call neither synchronises nor touches the device: it reports what the kernels that have
 * finished so far raised (synchronise first to cover everything enqueued).  The Python host polls it at every
 * network forward / backward and raises. */
MM3D_API int mm3d_take_device_error(void);

/* ------------------------------------------------------------------------------------------
 * Structure: replaces SparseConvNet's CPU-only Metadata<3> (InputLayer rules,
 * SubmanifoldConvolution_SgsToRules, Convolution_InputSgsToRulesAndOutputSgs).
 *
 * Keys are b<<48 | x<<32 | y<<16 | z.  Rows are numbered by first occurrence (SURVEY A.2/A.4),
 * computed with an open-addressing hash + atomicMin + prefix scan, so ids are deterministic.
 * Row counts are data dependent: they are written to DEVICE ints; sizes passed from the host
 * are capacities (upper bounds).  status_dev is OR-ed with MM3D_STATUS_* bits.
 * ---------------------------------------------------------------------------------------- */
#define MM3D_STATUS_BAD_COORD 1 /* a coordinate outside [0, spatial_size) or batch outside [0, 32768) */
#define MM3D_STATUS_DROPPED 2   /* mm3d_voxelize_points: a point fell outside the receptive field (see there) */

/* number of hash slots needed for up to n keys (power of two, load <= 0.5) */
MM3D_API int64_t mm3d_hash_capacity(int64_t n);
/* scratch bytes of mm3d_voxelize / mm3d_coarsen for up to n items */
MM3D_API size_t mm3d_unique_workspace_bytes(int64_t n);

/* InputLayer structure (replaces the rule-building half of SCN InputLayer_updateOutput):
 * coords int64 [n_points,4] = (x,y,z,batch).  Outputs: p2v[n_points] voxel row of each point,
 * vox_keys[<=n_points] key of each voxel row, npts[<=n_points] points per voxel,
 * *n_vox_dev the voxel count; (hash_keys, hash_vals)[hash_cap] the level-0 grid. */
MM3D_API int mm3d_voxelize(const int64_t* coords, int64_t n_points, int spatial_size,
                  uint64_t* hash_keys, int32_t* hash_vals, int64_t hash_cap,
                  int32_t* p2v, uint64_t* vox_keys, int32_t* npts, int32_t* n_vox_dev,
                  int32_t* status_dev, void* ws, size_t ws_bytes, mm3d_stream_t stream);

/* Stride-2/size-2 structure (replaces Convolution_InputSgsToRulesAndOutputSgs): from the fine
 * rows (fine_keys[*n_fine_dev], capacity n_fine_cap) build the coarse grid, parent[fine row],
 * off[fine row] in 0..7 and the offset-major child table child_tbl[8][tbl_stride]. */
MM3D_API int mm3d_coarsen(const uint64_t* fine_keys, const int32_t* n_fine_dev, int64_t n_fine_cap,
                 uint64_t* hash_keys, int32_t* hash_vals, int64_t hash_cap,
                 int32_t* parent, uint8_t* off, uint64_t* coarse_keys,
                 int32_t* child_tbl, int64_t tbl_stride, int32_t* n_coarse_dev,
                 void* ws, size_t ws_bytes, mm3d_stream_t stream);

/* 3^3 submanifold rules (replaces SubmanifoldConvolution_SgsToRules): offset-major table
 * nbr_tbl[27][tbl_stride]; column k = ((dx+1)*3+(dy+1))*3+(dz+1). */
MM3D_API int mm3d_build_nbr27(const uint64_t* keys, const int32_t* n_dev, int64_t n_cap, int spatial_size,
                     const uint64_t* hash_keys, const int32_t* hash_vals, int64_t hash_cap,
                     int32_t* nbr_tbl, int64_t tbl_stride, mm3d_stream_t stream);
/* Row boundaries of batch groups (grouped BatchNorm statistics, mm3d_unet_topo_forward_grouped): the structure holds
 * `groups` batches one after the other, group k's scans with batch indices in [batch_start[k], batch_start[k + 1])
 * (device int64 [groups + 1]), and its points before group k + 1's.  keys: HOST array of the levels' device key arrays,
 * counts: device int32, level l's row count at counts[l].  Writes the device int32 bounds[levels][groups + 1], level l's
 * group k = rows [bounds[l (groups + 1) + k], ... + 1).  One launch, no host synchronisation. */
#define MM3D_MAX_GROUP_LEVELS 16
MM3D_API int mm3d_group_bounds(const uint64_t* const* keys, const int32_t* counts, int levels, const int64_t* batch_start,
                      int groups, int32_t* bounds, mm3d_stream_t stream);


/* Row plan of a rule table, used by the tensor-core convolution modes: the table's output rows
 * ordered by neighbour mask (stable radix sort per 8192-row chunk), the table permuted into that
 * order and one offset mask per tile of 128 rows, so the kernels skip (tile, offset) blocks without
 * any input.  Built once per table (no SparseConvNet counterpart: its rule books are per-offset pair
 * lists); every layer, direction and gradient that uses the table shares it.  `tbl`, `tbl_stride`,
 * `onehot_off` as in mm3d_conv_fwd; the row count is read from *n_dev (<= n_cap).  Results of the
 * convolutions do not depend on the plan's row order. */
MM3D_API size_t mm3d_plan_bytes(int64_t n_cap, int K);
MM3D_API int mm3d_build_plan(const int32_t* tbl, int64_t tbl_stride, const uint8_t* onehot_off,
                    const int32_t* n_dev, int64_t n_cap, int K, void* plan, size_t plan_bytes,
                    mm3d_stream_t stream);
/* Several plans in ONE launch (the tables of all levels of a forward: their builds are independent and each
 * keeps only a few SMs busy).  n_rows_hint: the row count if the host knows it (sizes the launch; 0 = use
 * n_cap); the authoritative count is still *n_dev and must not exceed the hint. */
typedef struct mm3d_plan_desc {
  const int32_t* tbl;
  int64_t tbl_stride;
  const uint8_t* onehot_off;
  const int32_t* n_dev;
  int64_t n_cap;
  int64_t n_rows_hint;
  int K;
  void* plan;
  size_t plan_bytes;
} mm3d_plan_desc;
MM3D_API int mm3d_build_plans(const mm3d_plan_desc* descs_host, int n_plans, mm3d_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Points (metres) -> voxel coordinates: the reference's augment_and_scale_3d
 * (lib/utils/augmentation_3d.py:83-158) + integer cast + receptive-field filter
 * (lib/dataset/nuscenes_dataloader.py:312-327) for a collated batch.  points float32 [n,3]; sample_offsets
 * int64 [B+1]; rot float32 [B,3,3] (applied as points.dot(rot)); transl_u float64 [B,3] uniform draws of the
 * random translation or NULL (transl=False).  Outputs: coords int64 [n,4] (x,y,z,sample), keep uint8 [n]
 * (inside [0, full_scale)^3), min_value float32 [B,3], offset float64 [B,3] -- what the reference returns.
 * ---------------------------------------------------------------------------------------- */
MM3D_API size_t mm3d_scale_points_workspace_bytes(int B);
MM3D_API int mm3d_scale_points(const float* points, const int64_t* sample_offsets, int B, int64_t n, const float* rot,
                      float scale, int full_scale, const double* transl_u, int64_t* coords, uint8_t* keep,
                      float* min_value, double* offset, void* ws, size_t ws_bytes, mm3d_stream_t stream);

/* The two steps above in one: raw float points straight into the voxel hash (SURVEY 8(f).1) -- the reference's
 * augment_and_scale_3d + cast + filter (same files/lines as mm3d_scale_points, same device arithmetic) feeding
 * scn.InputLayer(3, full_scale, mode) (3d_net/scn_unet.py:108), without the int64 [n,4] coordinate tensor in between.
 * Arguments as in mm3d_scale_points (no coords output) followed by those of mm3d_voxelize (spatial size = full_scale).
 * The reference drops points outside [0, full_scale)^3 BEFORE the collate; when any point of the batch is outside,
 * MM3D_STATUS_DROPPED is OR-ed into *status_dev, keep[] marks the survivors and the structure built here must be
 * discarded: rebuild with mm3d_scale_points + mm3d_voxelize on the kept points (mm2d3d_b200.augment does). */
MM3D_API size_t mm3d_voxelize_points_workspace_bytes(int64_t n, int B);
MM3D_API int mm3d_voxelize_points(const float* points, const int64_t* sample_offsets, int B, int64_t n_points,
                         const float* rot, float scale, int full_scale, const double* transl_u,
                         uint8_t* keep, float* min_value, double* offset,
                         uint64_t* hash_keys, int32_t* hash_vals, int64_t hash_cap,
                         int32_t* p2v, uint64_t* vox_keys, int32_t* npts, int32_t* n_vox_dev,
                         int32_t* status_dev, void* ws, size_t ws_bytes, mm3d_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * I/O layers (replace SCN InputLayer_updateOutput/updateGradInput, OutputLayer_*).
 * mode 4 = mean of a voxel's points, 3 = sum.
 * ---------------------------------------------------------------------------------------- */
MM3D_API int mm3d_input_fwd(const float* feats, const int32_t* p2v, const int32_t* npts, int64_t n_points,
                   int64_t n_vox, int c, int mode, float* out_vox, mm3d_stream_t stream);
MM3D_API int mm3d_input_bwd(const float* d_vox, const int32_t* p2v, const int32_t* npts, int64_t n_points,
                   int c, int mode, float* d_feats, mm3d_stream_t stream);
/* InputLayer with the RGB-mask prologue of Net3DSeg.forward (3d_net/model.py:46-48) folded in: the voxel rows of
 * feats * sigmoid(feats . w + b) without the masked [N, c] tensor; c == 3; wb = [w_0, w_1, w_2, b] (device);
 * s_out [n_points] keeps the gates.  Backward: d_feats may be NULL; d_wb [c + 1] = (d_w, d_b), overwritten; feats are the
 * UNMASKED features; ws: (c + 1) doubles. */
MM3D_API int mm3d_input_masked_fwd(const float* feats, const int32_t* p2v, const int32_t* npts, int64_t n_points,
                          int64_t n_vox, int c, int mode, const float* wb, float* out_vox, float* s_out,
                          mm3d_stream_t stream);
MM3D_API int mm3d_input_masked_bwd(const float* d_vox, const float* feats, const float* s, const int32_t* p2v,
                          const int32_t* npts, int64_t n_points, int c, int mode, const float* wb, float* d_feats,
                          float* d_wb, void* ws, size_t ws_bytes, mm3d_stream_t stream);
MM3D_API int mm3d_output_fwd(const float* vox, const int32_t* p2v, int64_t n_points, int c, float* out,
                    mm3d_stream_t stream);
MM3D_API int mm3d_output_bwd(const float* d_out, const int32_t* p2v, int64_t n_points, int64_t n_vox, int c,
                    float* d_vox, mm3d_stream_t stream);
/* Deterministic forms (MM3D_DETERMINISTIC).  mm3d_point_csr: the points of every voxel in ascending point index,
 * vox_pts[vox_start[v] .. vox_start[v + 1]) (vox_start [n_vox + 1], vox_pts [n_points]), from p2v and npts of
 * mm3d_voxelize; ws: mm3d_point_csr_workspace_bytes(n_vox).  The lists depend only on p2v, so a structure builds
 * them once for all its forward and backward passes.  Cost: linear in points and voxels, except that one thread sorts
 * each voxel's list (O(k log k) for k points), so a voxel holding a large share of all points serialises that part. */
MM3D_API size_t mm3d_point_csr_workspace_bytes(int64_t n_vox);
MM3D_API int mm3d_point_csr(const int32_t* p2v, const int32_t* npts, int64_t n_points, int64_t n_vox, int32_t* vox_start,
                   int32_t* vox_pts, void* ws, size_t ws_bytes, mm3d_stream_t stream);
/* mm3d_input_fwd / mm3d_output_bwd over those lists: every voxel row is written once (no memset, no atomics).  Mode 4
 * sums f / count in point order, so a voxel of one point gets the bits of mm3d_input_fwd. */
MM3D_API int mm3d_input_fwd_csr(const float* feats, const int32_t* vox_start, const int32_t* vox_pts, int64_t n_vox, int c,
                       int mode, float* out_vox, mm3d_stream_t stream);
MM3D_API int mm3d_output_bwd_csr(const float* d_out, const int32_t* vox_start, const int32_t* vox_pts, int64_t n_vox, int c,
                        float* d_vox, mm3d_stream_t stream);
/* The masked InputLayer over those lists: every voxel row and every point's gate s_out[p] written once (no memset, no
 * atomics); a voxel of one point gets the bits of mm3d_input_masked_fwd. */
MM3D_API int mm3d_input_masked_fwd_csr(const float* feats, const int32_t* vox_start, const int32_t* vox_pts, int64_t n_vox,
                              int c, int mode, const float* wb, float* out_vox, float* s_out, mm3d_stream_t stream);
/* flags 0 = mm3d_input_masked_bwd.  MM3D_DETERMINISTIC: d_feats as there (per point); d_wb from one FP64 row per CTA
 * summed in CTA order instead of FP64 atomics -- ws: MM3D_DET_CTAS * (c + 1) doubles. */
MM3D_API int mm3d_input_masked_bwd_ex(const float* d_vox, const float* feats, const float* s, const int32_t* p2v,
                             const int32_t* npts, int64_t n_points, int c, int mode, const float* wb, float* d_feats,
                             float* d_wb, void* ws, size_t ws_bytes, mm3d_stream_t stream, int flags);

/* ------------------------------------------------------------------------------------------
 * Rule-table convolution (replaces SubmanifoldConvolution_/Convolution_/Deconvolution_
 * updateOutput and _backward):
 *     out[j,:] = sum_k  in[tbl(j,k), :] . Wsel(k)            j < n_out
 * tbl(j,k) = tbl[k*tbl_stride + j] for a dense table, or, when onehot_off != NULL,
 * (onehot_off[j] == k ? tbl[j] : -1) with tbl = parent[] (the deconvolution's table).
 * Wsel(k) = W[k] ([c_in, c_out]), or with flags: W[k]^T and/or W[K-1-k].
 * The three layer types and their gradients are all instances (DESIGN.md section 3).
 * `plan` (with the capacity it was built for) is the table's row plan; the tensor-core modes
 * require it, MM3D_MODE_FP32 ignores it (may be NULL).
 * ---------------------------------------------------------------------------------------- */
MM3D_API size_t mm3d_conv_workspace_bytes(int64_t n_in, int64_t n_out, int c_in, int c_out, int K, int mode);
MM3D_API int mm3d_conv_fwd(const float* in, int64_t n_in, int c_in, float* out, int64_t n_out, int c_out,
                  const float* weight, int K, const int32_t* tbl, int64_t tbl_stride,
                  const uint8_t* onehot_off, const void* plan, int64_t plan_cap, int flags, int mode,
                  void* ws, size_t ws_bytes, mm3d_stream_t stream);
/* Tensor-core modes: the gathered operand (`in` of mm3d_conv_fwd, `in` and `d_out` of mm3d_conv_wgrad) is read by
 * a kind::tf32 MMA, which ignores the low 13 mantissa bits.  Callers get round-to-nearest instead of truncation by
 * passing tensors whose values are already TF32 (mm3d_round_tf32; the whole-network executor's producers -- BatchNorm,
 * skip-gradient sum, stem padding -- store rounded values themselves).  Weights are rounded inside. */
MM3D_API int mm3d_round_tf32(const float* in, float* out, int64_t n, mm3d_stream_t stream);
/* out[0..n) = tf32(in), out[n..2n) = tf32(in - tf32(in)): the two operand planes of MM3D_MODE_TF32X3 */
MM3D_API int mm3d_split_tf32(const float* in, float* out, int64_t n, mm3d_stream_t stream);
/* out[0..n) = tf32(in) (float32) and, starting at float index n, n bfloat16 values bf16(in) (round to nearest even):
 * the two operand planes of MM3D_MODE_BF16; `out` holds 2 n floats, the BF16 plane fills the first half of the second n */
MM3D_API int mm3d_split_bf16(const float* in, float* out, int64_t n, mm3d_stream_t stream);
/* d_weight[k] (+)= sum_j in[tbl(j,k)]^T . d_out[j]   ([K, c_in, c_out]); accumulate=0 overwrites */
MM3D_API int mm3d_conv_wgrad(const float* in, int64_t n_in, int c_in, const float* d_out, int64_t n_out,
                    int c_out, float* d_weight, int K, const int32_t* tbl, int64_t tbl_stride,
                    const uint8_t* onehot_off, const void* plan, int64_t plan_cap, int accumulate, int mode,
                    void* ws, size_t ws_bytes, mm3d_stream_t stream);
/* flags 0 = mm3d_conv_wgrad (ws unused).  MM3D_DETERMINISTIC (tensor-core modes, shapes the tcgen05 kernels take; else
 * MM3D_ERR_UNSUPPORTED -- the FP32 mode and an unpadded stem run the SIMT kernel, which has no such form): every CTA
 * stores its accumulators into its own slab of ws with plain stores, and a second launch adds the slabs of the CTAs
 * of each offset to d_weight in ascending CTA order.  Which CTAs those are depends on the row plan, the shapes and the
 * device's SM count, so the bits are the same on every run on one device model.  ws: mm3d_conv_wgrad_workspace_bytes
 * -- 0 with flags 0, and also 0 (no deterministic form) for the FP32 mode and shapes the tcgen05 kernels do not take;
 * otherwise at most (SM count) x 256 KB, whatever n_out. */
MM3D_API size_t mm3d_conv_wgrad_workspace_bytes(int64_t n_out, int c_in, int c_out, int K, int mode, int flags);
MM3D_API int mm3d_conv_wgrad_ex(const float* in, int64_t n_in, int c_in, const float* d_out, int64_t n_out,
                       int c_out, float* d_weight, int K, const int32_t* tbl, int64_t tbl_stride,
                       const uint8_t* onehot_off, const void* plan, int64_t plan_cap, int accumulate, int mode,
                       void* ws, size_t ws_bytes, mm3d_stream_t stream, int flags);

/* ------------------------------------------------------------------------------------------
 * BatchNorm + (leaky) ReLU over active rows (replaces BatchNormalization_updateOutput/_backward).
 * momentum is SparseConvNet's (weight of the old running value, 0.9).  ws: 2*c doubles.
 * ---------------------------------------------------------------------------------------- */
MM3D_API size_t mm3d_bnrelu_workspace_bytes(int c);
MM3D_API int mm3d_bnrelu_fwd(const float* x, float* y, int64_t n, int c, const float* gamma, const float* beta,
                    float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                    float eps, float momentum, float leakiness, int training,
                    void* ws, size_t ws_bytes, mm3d_stream_t stream);
MM3D_API int mm3d_bnrelu_bwd(const float* x, const float* dy, float* dx, int64_t n, int c, const float* gamma,
                    const float* beta, const float* save_mean, const float* save_invstd,
                    float* d_gamma, float* d_beta, float leakiness, int training,
                    void* ws, size_t ws_bytes, mm3d_stream_t stream);
/* flags 0 = the functions above.  MM3D_DETERMINISTIC: the reductions over rows (batch statistics of the training
 * forward; d_beta / d_gamma and the terms of dx of every backward) store one FP64 partial row per CTA, and the totals
 * are summed in a fixed order, so save_mean / save_invstd, the running statistics, y, dx, d_gamma and d_beta are the
 * same bits on every run.  The grid comes from the occupancy API, the SM count and MM3D_BN_PER_SM: the bits are per
 * device model and per setting.  ws: mm3d_bnrelu_workspace_bytes_ex(c, flags), sized for the largest grid the current
 * device can get (flags 0: mm3d_bnrelu_workspace_bytes). */
MM3D_API size_t mm3d_bnrelu_workspace_bytes_ex(int c, int flags);
MM3D_API int mm3d_bnrelu_fwd_ex(const float* x, float* y, int64_t n, int c, const float* gamma, const float* beta,
                       float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                       float eps, float momentum, float leakiness, int training,
                       void* ws, size_t ws_bytes, mm3d_stream_t stream, int flags);
MM3D_API int mm3d_bnrelu_bwd_ex(const float* x, const float* dy, float* dx, int64_t n, int c, const float* gamma,
                       const float* beta, const float* save_mean, const float* save_invstd,
                       float* d_gamma, float* d_beta, float leakiness, int training,
                       void* ws, size_t ws_bytes, mm3d_stream_t stream, int flags);
/* Grouped BatchNorm statistics: the rows are `groups` consecutive ranges [bounds[k], bounds[k + 1]) (bounds: HOST
 * array of groups + 1 row indices, 0 = bounds[0] <= ... <= bounds[groups] = n), and a training forward normalises each
 * range as if it were its own mm3d_bnrelu_fwd_ex call, in range order: its own batch mean and biased variance, its own
 * row of save_mean / save_invstd (both [groups][c]) and its own running-statistics update (unbiased with the range's
 * row count; an empty range changes nothing).  The backward's dx is per range; d_gamma / d_beta total all rows.  Eval
 * mode (training = 0) normalises with the running statistics, so the groups change nothing there (save_* are then [c]).
 * 1 <= groups <= MM3D_BN_MAX_GROUPS; with groups = 1 the launches, workspace and results are those of the _ex
 * functions.  ws: mm3d_bnrelu_workspace_bytes_grouped(c, groups, flags) (0 = bad arguments). */
#define MM3D_BN_MAX_GROUPS 8
MM3D_API size_t mm3d_bnrelu_workspace_bytes_grouped(int c, int groups, int flags);
MM3D_API int mm3d_bnrelu_fwd_grouped(const float* x, float* y, int64_t n, int c, const float* gamma, const float* beta,
                            float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                            float eps, float momentum, float leakiness, int training,
                            void* ws, size_t ws_bytes, mm3d_stream_t stream, int flags, int groups,
                            const int64_t* bounds);
MM3D_API int mm3d_bnrelu_bwd_grouped(const float* x, const float* dy, float* dx, int64_t n, int c, const float* gamma,
                            const float* beta, const float* save_mean, const float* save_invstd,
                            float* d_gamma, float* d_beta, float leakiness, int training,
                            void* ws, size_t ws_bytes, mm3d_stream_t stream, int flags, int groups,
                            const int64_t* bounds);

/* ------------------------------------------------------------------------------------------
 * 2D->3D lift (replaces the per-sample advanced indexing of 2d_net/model.py:131-137):
 * out[n,:] = fmap[b(n), :, idx[n,0], idx[n,1]]; the [B, C, H, W] map is addressed through its element strides
 * (sb, sc, sh, sw), so a channels-last map -- what cuDNN produces for the 2D network, and the layout in which a
 * pixel's C values are one contiguous piece -- is read in place; sample_offsets int64 [B+1] gives the
 * row range of each sample in the concatenated idx; dtype 0=f32 1=f16 2=bf16 (map and out).
 * Backward scatter-adds into d_fmap (caller zero-fills), duplicates accumulate.
 * ---------------------------------------------------------------------------------------- */
MM3D_API int mm3d_lift2d_fwd(const void* fmap, int dtype, int B, int C, int H, int W, int64_t sb, int64_t sc, int64_t sh,
                    int64_t sw, const int64_t* idx, const int64_t* sample_offsets, int64_t n, void* out, mm3d_stream_t stream);
MM3D_API int mm3d_lift2d_bwd(const void* d_out, int dtype, int B, int C, int H, int W, int64_t sb, int64_t sc, int64_t sh,
                    int64_t sw, const int64_t* idx, const int64_t* sample_offsets, int64_t n, void* d_fmap, mm3d_stream_t stream);
/* Bilinear variant -- an extension, the reference only gathers at integer pixels (2d_net/model.py:131-137): uv float32
 * [n,2] = (row, col) in pixel units, pixel centres at the integers; out[n,:] = the blend of the four neighbouring pixels,
 * a neighbour outside the map contributing zero (torch.nn.functional.grid_sample, mode "bilinear", padding_mode "zeros",
 * align_corners=True, on the normalised coordinates).  Backward: gradient of the map only (the coordinates are data). */
MM3D_API int mm3d_lift2d_bilinear_fwd(const void* fmap, int dtype, int B, int C, int H, int W, int64_t sb, int64_t sc,
                             int64_t sh, int64_t sw, const float* uv, const int64_t* sample_offsets, int64_t n, void* out,
                             mm3d_stream_t stream);
MM3D_API int mm3d_lift2d_bilinear_bwd(const void* d_out, int dtype, int B, int C, int H, int W, int64_t sb, int64_t sc,
                             int64_t sh, int64_t sw, const float* uv, const int64_t* sample_offsets, int64_t n, void* d_fmap,
                             mm3d_stream_t stream);
/* Deterministic forms of the two backward passes (MM3D_DETERMINISTIC).  mm3d_lift_csr groups the lift's entries by
 * pixel key (b H + r) W + c: with idx (uv NULL) the entries are the points, indices normalised as mm3d_lift2d_bwd
 * takes them (an index outside the map gets no entry and raises device-error bit 2); with uv (idx NULL) they are the
 * (point, tap) pairs 4 p + q of the bilinear lift, q = 2 (row step) + (column step), a tap outside the map or of weight
 * zero dropped.  pix_start [B H W + 1], pix_ent [n] (idx) or [4 n] (uv), each pixel's entries in ascending order;
 * ws: mm3d_lift_csr_workspace_bytes(B, H, W, n, uv != NULL); cost as for mm3d_point_csr, per pixel.  The *_bwd_csr ops sum every pixel's entries in that
 * order in FP32, round once to the map's dtype and store into the caller's zero-filled d_fmap (strides as in
 * mm3d_lift2d_fwd); uv of the bilinear form is the one the lists were built from. */
MM3D_API size_t mm3d_lift_csr_workspace_bytes(int B, int H, int W, int64_t n, int bilinear);
MM3D_API int mm3d_lift_csr(const int64_t* idx, const float* uv, const int64_t* sample_offsets, int B, int H, int W, int64_t n,
                  int32_t* pix_start, int32_t* pix_ent, void* ws, size_t ws_bytes, mm3d_stream_t stream);
MM3D_API int mm3d_lift2d_bwd_csr(const void* d_out, int dtype, int B, int C, int H, int W, int64_t sb, int64_t sc, int64_t sh,
                        int64_t sw, const int32_t* pix_start, const int32_t* pix_ent, void* d_fmap, mm3d_stream_t stream);
MM3D_API int mm3d_lift2d_bilinear_bwd_csr(const void* d_out, int dtype, int B, int C, int H, int W, int64_t sb, int64_t sc,
                                 int64_t sh, int64_t sw, const float* uv, const int32_t* pix_start, const int32_t* pix_ent,
                                 void* d_fmap, mm3d_stream_t stream);

/* Point values -> image (the loaders' sparse depth and 2D label maps, lib/dataset/nuscenes_dataloader.py:275-278):
 * out[b, idx[i,0], idx[i,1]] = vals[i] over a map pre-filled with `fill`; where several points share a pixel the
 * last one wins, like numpy's indexed assignment.  idx int64 [n,2] (row, col), sample_offsets int64 [B+1],
 * out float32 [B,H,W]; ws: mm3d_raster2d_workspace_bytes. */
MM3D_API size_t mm3d_raster2d_workspace_bytes(int B, int H, int W);
MM3D_API int mm3d_raster2d(const int64_t* idx, const int64_t* sample_offsets, int B, int H, int W, int64_t n,
                  const float* vals, float fill, float* out, void* ws, size_t ws_bytes, mm3d_stream_t stream);

/* Point-wise prologue and loss around the 3D network (SURVEY 8(f).3).
 * RGB mask, 3d_net/model.py:46-48:  s = sigmoid(x . w + b); y = x * s   (x, y float32 [n, c], c <= 8; w [c], b [1];
 * s_out [n] keeps the gate for the backward pass; y may be x).  Backward: dx (may be NULL) [n, c], dw [c], db [1];
 * x is the UNMASKED input; ws: (c + 1) doubles. */
MM3D_API int mm3d_rgb_mask_fwd(const float* x, int64_t n, int c, const float* w, const float* b, float* y, float* s_out,
                      mm3d_stream_t stream);
MM3D_API int mm3d_rgb_mask_bwd(const float* x, const float* s, const float* dy, int64_t n, int c, const float* w, float* dx,
                      float* dw, float* db, void* ws, size_t ws_bytes, mm3d_stream_t stream);
/* flags 0 = mm3d_rgb_mask_bwd; MM3D_DETERMINISTIC: ws MM3D_DET_CTAS * (c + 1) doubles */
MM3D_API int mm3d_rgb_mask_bwd_ex(const float* x, const float* s, const float* dy, int64_t n, int c, const float* w, float* dx,
                         float* dw, float* db, void* ws, size_t ws_bytes, mm3d_stream_t stream, int flags);
/* Cross-modal loss, train.py:157-184:  loss[0] = mean over the n rows of sum_c q_c (log q_c - log p_c) with
 * p = softmax(pred[n, :]), q = softmax(target[n, :]) (target detached); pred, target float32 [n, C] logits; ws: one
 * double.  Backward: dpred = dloss[0] * (p - q) / n. */
MM3D_API int mm3d_kl_logits_fwd(const float* pred, const float* target, int64_t n, int C, float* loss, void* ws, size_t ws_bytes,
                       mm3d_stream_t stream);
/* flags 0 = mm3d_kl_logits_fwd; MM3D_DETERMINISTIC: ws MM3D_DET_CTAS doubles */
MM3D_API int mm3d_kl_logits_fwd_ex(const float* pred, const float* target, int64_t n, int C, float* loss, void* ws,
                          size_t ws_bytes, mm3d_stream_t stream, int flags);
MM3D_API int mm3d_kl_logits_bwd(const float* pred, const float* target, int64_t n, int C, const float* dloss, float* dpred,
                       mm3d_stream_t stream);
/* The two point-wise heads of the 3D branch and the 3D side of the cross-modal loss in ONE pass over the features
 * (3d_net/model.py:38,49 `linear`; :73,85 `L2G_classifier_3D.linear_point`; train.py:157-184 `loss_3d`):
 *   logit1 = feat w1^T + b1,   logit2 = feat w2^T + b2,   loss[0] = mean_n KL(softmax(target_n) || softmax(logit2_n))
 * feat float32 [n, f] (f a multiple of 4, <= 32, 16-byte aligned), w1 / w2 [C, f] and b1 / b2 [C] as nn.Linear stores
 * them (C <= 20), target [n, C] logits (detached).  logit2 and loss may be NULL (then target may be NULL); ws: 1 double.
 * Backward: d_logit1 / d_logit2 [n, C] upstream gradients (either may be NULL), d_loss [1] (NULL = loss unused);
 * d_feat [n, f] (may be NULL), d_w1 / d_w2 [C, f], d_b1 / d_b2 [C] overwritten; ws: (2 C f + 2 C) doubles. */
MM3D_API int mm3d_heads3d_fwd(const float* feat, int64_t n, int f, int C, const float* w1, const float* b1, const float* w2,
                     const float* b2, const float* target, float* logit1, float* logit2, float* loss, void* ws,
                     size_t ws_bytes, mm3d_stream_t stream);
MM3D_API int mm3d_heads3d_bwd(const float* feat, int64_t n, int f, int C, const float* w1, const float* w2, const float* b2,
                     const float* target, const float* d_logit1, const float* d_logit2, const float* d_loss, float* d_feat,
                     float* d_w1, float* d_b1, float* d_w2, float* d_b2, void* ws, size_t ws_bytes, mm3d_stream_t stream);
/* flags 0 = the functions above; MM3D_DETERMINISTIC: ws MM3D_DET_CTAS doubles (forward with a loss) and
 * MM3D_DET_CTAS * (2 C f + 2 C) doubles (backward) */
MM3D_API int mm3d_heads3d_fwd_ex(const float* feat, int64_t n, int f, int C, const float* w1, const float* b1, const float* w2,
                        const float* b2, const float* target, float* logit1, float* logit2, float* loss, void* ws,
                        size_t ws_bytes, mm3d_stream_t stream, int flags);
MM3D_API int mm3d_heads3d_bwd_ex(const float* feat, int64_t n, int f, int C, const float* w1, const float* w2, const float* b2,
                        const float* target, const float* d_logit1, const float* d_logit2, const float* d_loss,
                        float* d_feat, float* d_w1, float* d_b1, float* d_w2, float* d_b2, void* ws, size_t ws_bytes,
                        mm3d_stream_t stream, int flags);

/* ------------------------------------------------------------------------------------------
 * Whole-network executor: UNetSCN (3d_net/scn_unet.py:36-126) forward and backward as one call each -- the
 * same kernels as above, driven natively instead of from ~110 Python autograd nodes (about twice that with
 * block_reps == 2).  Every configuration of the constructor's block topology is covered: block_reps >= 1 blocks per
 * pre / post group, VGG blocks (residual == 0) or pre-activation residual blocks (residual == 1), whose
 * NetworkInNetwork shortcut runs as a K = 1 rule-table convolution.  The mm3d_unet_* functions are the
 * reference configuration (block_reps == 1, VGG) of the mm3d_unet_topo_* ones.  level_desc:
 * MM3D_LEVEL_DESC_WORDS int64 per level {rows, nbr table ptr, table stride, parent ptr, off ptr, child ptr, plan of
 * the 3^3 table, plan of the child table, plan of the (parent, off) table, plan capacity} (plans may be 0 in
 * MM3D_MODE_FP32).  params / grads: HOST arrays of device pointers in module-tree order:
 *   stem.w | per level: pre blocks [dn_bn{gamma,beta,running_mean,running_var} dn.w <deeper level>
 *   up_bn{4} up.w post blocks] | head_bn{4}
 * with a VGG block = bn{4} smc.w and a residual block = [nin.w] bn{4} smc.w bn{4} smc.w (the NetworkInNetwork
 * weight [a, b] only where the block changes the channel count: the first post block of a level).
 * (mm3d_unet_topo_num_params slots; grads ignore the running-stat slots.)  act: activations kept from forward to
 * backward; tmp: backward temporaries, mm3d_unet_topo_bwd_bytes, which is the exact need.  Forward and backward check
 * every buffer against its query before they issue any CUDA call and return MM3D_ERR_WORKSPACE when one is short.
 * ---------------------------------------------------------------------------------------- */
#define MM3D_LEVEL_DESC_WORDS 10
MM3D_API int64_t mm3d_unet_topo_num_params(int num_planes, int block_reps, int residual);
MM3D_API size_t mm3d_unet_topo_act_bytes(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                const int64_t* level_desc, int64_t n_points);
MM3D_API size_t mm3d_unet_topo_bwd_bytes(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                const int64_t* level_desc, int64_t n_points);
MM3D_API size_t mm3d_unet_topo_scratch_bytes(int in_channels, int m, int num_planes, int block_reps, int residual, int mode);
/* the reference configuration: block_reps = 1, residual = 0 */
MM3D_API int64_t mm3d_unet_num_params(int num_planes);
MM3D_API size_t mm3d_unet_act_bytes(int in_channels, int m, int num_planes, int mode, const int64_t* level_desc,
                           int64_t n_points);
MM3D_API size_t mm3d_unet_bwd_bytes(int in_channels, int m, int num_planes, int mode, const int64_t* level_desc,
                           int64_t n_points);
MM3D_API size_t mm3d_unet_scratch_bytes(int in_channels, int m, int num_planes, int mode);
/* Optional RGB-mask prologue (3d_net/model.py:46-48, feats *= sigmoid(linear_rgb_mask(feats))) folded into the
 * network's InputLayer (mm3d_input_masked_fwd / _bwd); NULL = the features are used as they are.  Forward reads wb and
 * writes s; backward reads wb, s, feats (the UNMASKED features of the forward) and writes d_wb, using ws. */
typedef struct {
  const float* wb;    /* [in_channels + 1] device: the Linear(in_channels, 1) weight, then its bias */
  float* s;           /* [n_points] gates */
  const float* feats; /* backward only */
  float* d_wb;        /* backward only: [in_channels + 1] gradient of wb, overwritten */
  void* ws;           /* backward only: (in_channels + 1) doubles; MM3D_DETERMINISTIC: MM3D_DET_CTAS * (in_channels + 1) */
  size_t ws_bytes;
} mm3d_unet_mask;
MM3D_API int mm3d_unet_topo_forward(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                           int training, float eps, float momentum, const int64_t* level_desc, int64_t n_points,
                           const int32_t* p2v, const int32_t* npts, const float* feats, float* out, void* const* params,
                           void* act, size_t act_bytes, void* scratch, size_t scratch_bytes, const mm3d_unet_mask* mask,
                           mm3d_stream_t stream);
MM3D_API int mm3d_unet_topo_backward(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                            int training, const int64_t* level_desc, int64_t n_points, const int32_t* p2v,
                            const int32_t* npts, const float* d_out, float* d_feats, void* const* params,
                            void* const* grads, void* act, size_t act_bytes, void* tmp, size_t tmp_bytes, void* scratch,
                            size_t scratch_bytes, const mm3d_unet_mask* mask, mm3d_stream_t stream);
MM3D_API int mm3d_unet_forward(int in_channels, int m, int num_planes, int mode, int training, float eps, float momentum,
                      const int64_t* level_desc, int64_t n_points, const int32_t* p2v, const int32_t* npts,
                      const float* feats, float* out, void* const* params, void* act, size_t act_bytes,
                      void* scratch, size_t scratch_bytes, const mm3d_unet_mask* mask, mm3d_stream_t stream);
MM3D_API int mm3d_unet_backward(int in_channels, int m, int num_planes, int mode, int training,
                       const int64_t* level_desc, int64_t n_points, const int32_t* p2v, const int32_t* npts,
                       const float* d_out, float* d_feats, void* const* params, void* const* grads,
                       void* act, size_t act_bytes, void* tmp, size_t tmp_bytes, void* scratch,
                       size_t scratch_bytes, const mm3d_unet_mask* mask, mm3d_stream_t stream);
/* flags 0 = the mm3d_unet_topo_* functions above (vox_start / vox_pts unused).  MM3D_DETERMINISTIC: a training step
 * whose outputs, gradients and running statistics are the same bits on every run on one device model --
 *   InputLayer forward and OutputLayer backward over the voxels' point lists vox_start / vox_pts (mm3d_point_csr,
 *   required), the masked InputLayer backward's mask gradient in CTA order (mask->ws as documented there), every
 *   BatchNorm in its deterministic form, and every weight gradient through mm3d_conv_wgrad_ex's fixed-order form with
 *   slabs in the scratch buffer (mm3d_unet_topo_scratch_bytes_ex with the same flags).
 * A weight gradient without such a form (mm3d_conv_wgrad_workspace_bytes(..., MM3D_DETERMINISTIC) == 0: every one of
 * the fp32 mode, and channel counts the tcgen05 kernels do not take) runs its default kernel; the caller decides
 * beforehand whether that is acceptable. */
MM3D_API size_t mm3d_unet_topo_scratch_bytes_ex(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                       int flags);
MM3D_API int mm3d_unet_topo_forward_ex(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                              int training, float eps, float momentum, const int64_t* level_desc, int64_t n_points,
                              const int32_t* p2v, const int32_t* npts, const int32_t* vox_start, const int32_t* vox_pts,
                              const float* feats, float* out, void* const* params, void* act, size_t act_bytes,
                              void* scratch, size_t scratch_bytes, const mm3d_unet_mask* mask, mm3d_stream_t stream,
                              int flags);
MM3D_API int mm3d_unet_topo_backward_ex(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                               int training, const int64_t* level_desc, int64_t n_points, const int32_t* p2v,
                               const int32_t* npts, const int32_t* vox_start, const int32_t* vox_pts, const float* d_out,
                               float* d_feats, void* const* params, void* const* grads, void* act, size_t act_bytes,
                               void* tmp, size_t tmp_bytes, void* scratch, size_t scratch_bytes,
                               const mm3d_unet_mask* mask, mm3d_stream_t stream, int flags);
/* Grouped BatchNorm statistics (mm3d_bnrelu_fwd_grouped): several batches through one structure, one forward and one
 * backward, each normalised as if it had been its own call.  The rows of every level are `groups` consecutive ranges,
 * bounds: HOST int64 [num_planes][groups + 1], level l's group k = rows [bounds[l (groups + 1) + k], ... + 1), each
 * level's running from 0 to its row count.  A training forward is then the same as one mm3d_unet_topo_forward_ex call
 * per group, in group order: every BatchNorm normalises a group's rows with that group's statistics and updates the
 * running statistics once per group.  The backward gives each group's feature gradient as its own call would and the
 * parameter (and mask) gradients summed over the groups.  Eval mode: the groups change nothing.  1 <= groups <=
 * MM3D_BN_MAX_GROUPS; groups == 1 (bounds may then be NULL) is the _ex call.  The saved statistics grow to [groups][C]:
 * act and scratch come from the _grouped queries (mm3d_unet_topo_bwd_bytes does not depend on the groups). */
typedef struct {
  int groups;
  const int64_t* bounds;
} mm3d_unet_groups;
MM3D_API size_t mm3d_unet_topo_act_bytes_grouped(int in_channels, int m, int num_planes, int block_reps, int residual,
                                        int mode, const int64_t* level_desc, int64_t n_points, int groups);
MM3D_API size_t mm3d_unet_topo_scratch_bytes_grouped(int in_channels, int m, int num_planes, int block_reps, int residual,
                                            int mode, int flags, int groups);
MM3D_API int mm3d_unet_topo_forward_grouped(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                   int training, float eps, float momentum, const int64_t* level_desc, int64_t n_points,
                                   const int32_t* p2v, const int32_t* npts, const int32_t* vox_start,
                                   const int32_t* vox_pts, const float* feats, float* out, void* const* params, void* act,
                                   size_t act_bytes, void* scratch, size_t scratch_bytes, const mm3d_unet_mask* mask,
                                   mm3d_stream_t stream, int flags, const mm3d_unet_groups* groups);
MM3D_API int mm3d_unet_topo_backward_grouped(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                    int training, const int64_t* level_desc, int64_t n_points, const int32_t* p2v,
                                    const int32_t* npts, const int32_t* vox_start, const int32_t* vox_pts,
                                    const float* d_out, float* d_feats, void* const* params, void* const* grads, void* act,
                                    size_t act_bytes, void* tmp, size_t tmp_bytes, void* scratch, size_t scratch_bytes,
                                    const mm3d_unet_mask* mask, mm3d_stream_t stream, int flags,
                                    const mm3d_unet_groups* groups);
/* Inference forward: the eval-mode forward (BatchNorm with the running statistics, training = 0) without anything a
 * backward would read.  Every BatchNorm+ReLU is applied in the epilogue of the convolution that produces its input and
 * the JoinTable concatenations are never materialised; the output is the same bits as mm3d_unet_topo_forward_ex with
 * training = 0 and the same flags.  ws: one device workspace of mm3d_unet_topo_infer_bytes (the exact need: the
 * tensors this call writes, the forward weight images and the BatchNorm scales); a short one gives MM3D_ERR_WORKSPACE
 * before any CUDA call.  flags: 0 or MM3D_DETERMINISTIC (InputLayer over the voxels' point lists vox_start / vox_pts).
 * params as above (running statistics read, nothing written); mask: wb and s as in the forward. */
MM3D_API size_t mm3d_unet_topo_infer_bytes(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                  const int64_t* level_desc, int64_t n_points, int flags);
MM3D_API int mm3d_unet_topo_infer(int in_channels, int m, int num_planes, int block_reps, int residual, int mode, float eps,
                         const int64_t* level_desc, int64_t n_points, const int32_t* p2v, const int32_t* npts,
                         const int32_t* vox_start, const int32_t* vox_pts, const float* feats, float* out,
                         void* const* params, void* ws, size_t ws_bytes, const mm3d_unet_mask* mask, mm3d_stream_t stream,
                         int flags);

#ifdef __cplusplus
}
#endif
#endif /* MM3D_H_ */
