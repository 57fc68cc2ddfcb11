// Whole-network executor: UNetSCN forward and backward as ONE C-ABI call each.
//
// The per-layer entry points are enough for a drop-in, but driving ~110 autograd nodes from
// Python costs ~8 ms of host time per step -- as much as the GPU work itself.  The executor walks
// the U-Net topology of 3d_net/scn_unet.py:36-84 natively, for any number of blocks per level
// (block_reps) and for VGG or pre-activation residual blocks, and issues the same kernels the modules use.  One
// walk over the module tree (`Carve`) assigns the parameter slots and lays out every activation, every backward
// temporary and the scratch buffer in the caller's workspaces; forward, backward and the size queries all run it.
//
//   level l (p = m(l+1), q = m(l+2)):
//     X_l --[block p->p] x reps--> Y_l                                           ("pre" blocks)
//     if l < L-1:  Y_l --BN--> B_l --Conv 2/2--> X_{l+1} ... R_{l+1} --BN--> E_l --Deconv 2/2--> F_l
//                  J_l = [Y_l | F_l] --block 2p->p--> --[block p->p] x (reps-1)--> R_l   ("post" blocks)
//     else         R_l = Y_l
//   VGG block:      x --BN--> A --SMC--> out
//   residual block: x --BN--> A --SMC--> H --BN--> A2 --SMC(+ shortcut)--> out, shortcut = x (a == b) or
//                   NetworkInNetwork(x) (a != b: only the first post block, on J), run as a K = 1 rule-table
//                   convolution over an identity row plan; the add happens in the second SMC's epilogue
//   stem: V (InputLayer mean) --SMC(in->m)--> X_0 ;  head: R_0 --BN--> Z --OutputLayer--> out
//
// Parameter pointers come in the module tree's order (Appendix B of SURVEY.md):
//   stem.w | per level: pre blocks [dn_bn{gamma,beta,rmean,rvar} dn.w <deeper level> up_bn{4} up.w post blocks]
//   | head_bn{4};  VGG block: bn{4} smc.w;  residual block: [nin.w] bn{4} smc.w bn{4} smc.w
#include <cuda_bf16.h>
#include <stdlib.h>

#include <cstring>
#include <vector>

#include "common.cuh"
#include "epilogue.cuh"
#include "plan.cuh"

// bnrelu.cu
int mm3d_bnrelu_fwd_impl(const float* x, const float* x_hi, int c_lo, float* y, int64_t n, int c, const float* gamma,
                         const float* beta, float* running_mean, float* running_var, float* save_mean,
                         float* save_invstd, float eps, float momentum, float leakiness, int training, void* ws,
                         size_t ws_bytes, int* parity, int round_tf32, cudaStream_t stream, int det, int groups,
                         const int64_t* bounds);
int mm3d_bnrelu_bwd_impl(const float* x, const float* x_hi, int c_lo, const float* dy, float* dx, float* dx_hi,
                         int64_t n, int c, const float* gamma, const float* beta, const float* save_mean,
                         const float* save_invstd, float* d_gamma, float* d_beta, float leakiness, int training,
                         void* ws, size_t ws_bytes, int* parity, int round_flags, const float* add, int64_t add_ld,
                         cudaStream_t stream, int det, int groups, const int64_t* bounds);

// conv_tc.cu
size_t mm3d_conv_tc_workspace_bytes(int c_in, int c_out, int K);
int mm3d_conv_tc_supported(int c_in, int c_out, int K);
int mm3d_conv_tc_build_images(const float* const* weights, float* const* images, const int* K, const int* c_in,
                              const int* c_out, const int* flags, int n, cudaStream_t stream);
int mm3d_conv_fwd_tc_img(const float* in, int64_t n_in, int c_in, float* out, int64_t n_out, int c_out,
                         const float* wimg, int K, const void* plan, int64_t plan_cap, const float* add, cudaStream_t stream,
                         const float* wimg_lo = nullptr, int bf16 = 0, const ConvEpi* epi = nullptr);
// conv_simt.cu
int mm3d_conv_fwd_simt(const float* in, int64_t n_in, int c_in, float* out, int64_t n_out, int c_out,
                       const float* weight, int K, const int32_t* tbl, int64_t tbl_stride,
                       const uint8_t* onehot_off, int flags, void* ws, size_t ws_bytes, cudaStream_t stream,
                       const float* add, const ConvEpi* epi = nullptr);

namespace {

struct LevelMeta {
  int64_t n;
  const int32_t* nbr;
  int64_t tstride;
  const int32_t* parent;
  const uint8_t* off;
  const int32_t* child;
  const void *plan_smc, *plan_down, *plan_up;  // row plans of the three tables (tensor-core modes)
  int64_t plan_cap;
};

// hands out consecutive 256-byte aligned pieces of a buffer; a NULL base only counts the bytes
struct Bump {
  char* base;
  size_t off;
  void* bytes(size_t n) {
    size_t o = off;
    off += mm3d_align(n);
    return base ? base + o : nullptr;
  }
  float* f(int64_t n, int64_t c) { return (float*)bytes(sizeof(float) * (size_t)n * (size_t)c); }
};

// one convolution of the network: its weight's parameter slot, kernel volume and channels (the stem's c_in is cin_k,
// as the kernels see it)
struct ConvInfo {
  int pidx, K, c_in, c_out, smc;
};

// one VGG or residual block, a -> b channels
struct BlockBufs {
  int a, b;
  int pidx;            // first parameter slot
  float *A, *s1;       // first BatchNorm's output (operand form) and its save_mean | save_invstd ([2][G][a])
  float *H, *A2, *s2;  // residual: first SMC's output, second BatchNorm's output (operand form), its save
  float* out;          // [n, b]
  // backward: gradients w.r.t. A, A2, H (operand form), the NetworkInNetwork's input, and the block's input (operand
  // form; the level's d_X for its first pre block, none for its first post block, which writes d_J and d_F)
  float *d_A, *d_A2, *d_H, *d_S, *d_x;
};

struct LevelBufs {
  float *X, *Y, *B, *E, *F, *J, *R;
  float* Jop;           // NiN shortcut: J in operand form (== J in FP32 mode)
  float *s_dn, *s_up;   // BN save_mean | save_invstd ([2][G][C])
  void* id_plan;        // NiN shortcut: identity row plan of the level's rows (capacity n)
  int dn, up;           // first parameter slot of the down and the up branch (BatchNorm, then the convolution at + 4)
  std::vector<BlockBufs> pre, post;
  // backward: gradients w.r.t. J ([n, 2p]; a split join writes only its skip half, [n, p]), F, Y (skip + branch),
  // E, R_{l+1} and X_{l+1} (all three of the next level's rows), and B.  All but d_J, d_E and d_B in operand form.
  float *d_J, *d_F, *d_Yskip, *d_E, *d_Rn, *d_Xn, *d_B;
};

struct Net {
  int L, m, cin, cin_k;  // cin_k = stem input channels as seen by the kernels (padded to 16 in TC modes)
  int reps, res;         // blocks per pre / post group; residual blocks
  int mode;
  int flags;  // MM3D_DETERMINISTIC or 0
  // grouped BatchNorm statistics: G row groups, level l's group k = rows [gb[l (G + 1) + k], gb[l (G + 1) + k + 1]);
  // every saved statistic is [G][C] (mean) then [G][C] (invstd)
  int G = 1;
  std::vector<int64_t> gb;
  std::vector<LevelMeta> lv;
  std::vector<LevelBufs> b;
  float *V, *Vp, *Z, *s_head;
  float* wide_sum = nullptr;  // inference forward: partial sums of the tcgen05 input-channel slices (c_in > 256)
  float *d_Z, *d_R0, *d_X0, *d_Vp;        // backward: gradients w.r.t. Z, R_0, X_0 (operand form) and Vp
  float *d_wp = nullptr, *d_V = nullptr;  // backward, padded stem input only: gradients w.r.t. wp and V
  int head, n_params;                     // the head BatchNorm's first parameter slot; the number of slots
  std::vector<ConvInfo> convs;            // every convolution, in slot order
  std::vector<std::pair<int, int>> bns;   // every BatchNorm's first parameter slot and channels, in slot order
  size_t bn_channels = 0;                 // of all BatchNorms (each has a gamma and a beta gradient)
  // The scratch buffer: [convolution workspace | weight images | BatchNorm workspace | padded stem weight], and in the
  // deterministic mode behind that [deterministic BatchNorm workspace | weight-gradient slabs].  Weight images
  // (tensor-core modes): every layer's, for this call's direction, built by one launch up front.  BatchNorm workspace:
  // totals and barrier counters, zeroed at the start of each call; the kernels keep it clean.  Weight-gradient slabs:
  // one region for the largest convolution -- every weight gradient runs on one stream, one after the other.
  void *conv_ws, *img_ws, *bn_ws, *wg_ws = nullptr;
  size_t conv_ws_bytes, img_ws_bytes, bn_ws_bytes, wg_ws_bytes = 0;
  float* wp;  // the stem weight with zeros for the padded input channels (cin_k != cin only)
  int64_t n_points;
  bool det() const { return (flags & MM3D_DETERMINISTIC) != 0; }
  int planes(int l) const { return m * (l + 1); }
  const int64_t* bounds(int l) const { return G > 1 ? gb.data() + (size_t)l * (G + 1) : nullptr; }
  // TF32x3 mode: every tensor a convolution gathers carries a hi and a lo plane ([rows, c] floats each)
  // BF16 mode: an FP32 plane (TF32-rounded: the weight-gradient operand) and a BF16 plane behind it (what forward and
  // dgrad gather; it only fills the first half of its plane)
  int pl() const { return (mode == MM3D_MODE_TF32X3 || mode == MM3D_MODE_BF16) ? 2 : 1; }
  // how a producer stores a tensor that a convolution gathers (bnrelu.cu store_planes / k_pad_cols)
  int rmode() const { return mode == MM3D_MODE_TF32X3 ? 2 : mode == MM3D_MODE_BF16 ? 3 : mode == MM3D_MODE_TF32 ? 1 : 0; }
  bool x3() const { return mode == MM3D_MODE_TF32X3; }
  bool bf16() const { return mode == MM3D_MODE_BF16; }
  bool nin(int a, int b) const { return res && a != b; }
};

// One walk over the module tree, in its order: it assigns the parameter slots with a running counter, lists the
// convolutions, counts the BatchNorm channels, and carves the activations out of `act` and the backward temporaries
// out of `tmp`.  A NULL base only sizes (the queries, and `tmp` in the forward).
struct Carve {
  Net& net;
  Bump &act, &tmp;
  int pi = 0;  // next parameter slot

  int bn(int ch) {
    net.bn_channels += ch;
    net.bns.push_back({pi, ch});
    pi += 4;  // gamma, beta, running mean, running var
    return pi - 4;
  }
  void conv(int K, int c_in, int c_out, int smc) { net.convs.push_back({pi++, K, c_in, c_out, smc}); }

  BlockBufs block(int64_t n, int a, int b) {
    const int pl = net.pl();
    BlockBufs k{};
    k.a = a; k.b = b; k.pidx = pi;
    if (net.nin(a, b)) {
      conv(1, a, b, 0);
      k.d_S = tmp.f(n, a);
    }
    bn(a);
    conv(27, a, b, 1);
    k.A = act.f(n, (int64_t)a * pl);
    k.s1 = act.f(2 * net.G, a);
    k.d_A = tmp.f(n, a);
    if (net.res) {
      bn(b);
      conv(27, b, b, 1);
      k.H = act.f(n, b);
      k.A2 = act.f(n, (int64_t)b * pl);
      k.s2 = act.f(2 * net.G, b);
      k.d_A2 = tmp.f(n, b);
      k.d_H = tmp.f(n, (int64_t)b * pl);
    }
    k.out = act.f(n, b);
    return k;
  }

  // level l; d_X: the gradient w.r.t. its input X_l, carved by the caller
  void level(int l, float* d_X) {
    const int64_t n = net.lv[l].n;
    const int p = net.planes(l), pl = net.pl();
    LevelBufs& B = net.b[l];
    B.X = act.f(n, p);
    for (int r = 0; r < net.reps; ++r) {
      B.pre.push_back(block(n, p, p));
      B.pre.back().d_x = r ? tmp.f(n, (int64_t)p * pl) : d_X;
    }
    B.Y = B.pre.back().out;
    if (l + 1 == net.L) {
      B.R = B.Y;
      return;
    }
    const int q = net.planes(l + 1);
    const int64_t nc = net.lv[l + 1].n;
    B.dn = bn(p);
    conv(8, p, q, 0);
    B.B = act.f(n, (int64_t)p * pl);
    B.s_dn = act.f(2 * net.G, p);
    B.d_B = tmp.f(n, p);
    B.d_Xn = tmp.f(nc, (int64_t)q * pl);
    level(l + 1, B.d_Xn);
    B.up = bn(q);
    conv(8, q, p, 0);
    B.E = act.f(nc, (int64_t)q * pl);
    B.s_up = act.f(2 * net.G, q);
    B.d_Rn = tmp.f(nc, (int64_t)q * pl);
    B.d_E = tmp.f(nc, q);
    B.F = act.f(n, p);
    B.J = act.f(n, 2 * p);
    B.Jop = B.J;
    if (net.nin(2 * p, p)) {
      if (net.mode != MM3D_MODE_FP32) B.Jop = act.f(n, (int64_t)2 * p * pl);
      B.id_plan = act.bytes(mm3d_plan_size(n, 1));
    }
    B.d_J = tmp.f(n, 2 * p);
    B.d_F = tmp.f(n, (int64_t)p * pl);
    B.d_Yskip = tmp.f(n, (int64_t)p * pl);
    for (int r = 0; r < net.reps; ++r) {
      B.post.push_back(block(n, r ? p : 2 * p, p));
      if (r) B.post.back().d_x = tmp.f(n, (int64_t)p * pl);
    }
    B.R = B.post.back().out;
  }

  void run() {
    const int64_t n0 = net.lv[0].n;
    const int pl = net.pl();
    net.V = act.f(n0, net.cin);
    net.Vp = (net.cin_k != net.cin || pl == 2) ? act.f(n0, (int64_t)net.cin_k * pl) : net.V;
    net.d_Vp = tmp.f(n0, net.cin_k);
    if (net.cin_k != net.cin) {
      net.d_V = tmp.f(n0, net.cin);
      net.d_wp = tmp.f(27, (int64_t)net.cin_k * net.m);
    }
    conv(27, net.cin_k, net.m, 1);  // the stem
    net.d_X0 = tmp.f(n0, (int64_t)net.m * pl);
    net.b.assign(net.L, LevelBufs());
    level(0, net.d_X0);
    net.head = bn(net.m);
    net.n_params = pi;
    net.Z = act.f(n0, net.m);
    net.s_head = act.f(2 * net.G, net.m);
    net.d_Z = tmp.f(n0, net.m);
    net.d_R0 = tmp.f(n0, (int64_t)net.m * pl);
  }
};

// the region of the weight images: the larger direction's images (the forward's alone without `backward`), twice in
// TF32x3 mode (hi and lo)
size_t img_region_bytes(const Net& net, bool backward = true) {
  if (net.mode == MM3D_MODE_FP32) return 0;
  size_t fwd = 0, bwd = 0;
  for (const ConvInfo& ci : net.convs) {  // (0 bytes for a shape the tensor cores do not take)
    fwd += mm3d_align(mm3d_conv_tc_workspace_bytes(ci.c_in, ci.c_out, ci.K));
    if (backward) bwd += mm3d_align(mm3d_conv_tc_workspace_bytes(ci.c_out, ci.c_in, ci.K));
  }
  return (fwd > bwd ? fwd : bwd) * (net.x3() ? 2 : 1);
}

// the layout of the scratch buffer (after the walk: it needs the convolution list), the same in forward, backward and
// the size query
void carve_scratch(Net& net, Bump& bp) {
  size_t conv = 0;
  for (const ConvInfo& ci : net.convs) {
    const size_t s = mm3d_conv_workspace_bytes(0, 0, ci.c_in, ci.c_out, ci.K, net.mode);  // (covers dgrad and wgrad)
    if (s > conv) conv = s;
  }
  net.conv_ws_bytes = conv;
  net.conv_ws = bp.bytes(conv);
  net.img_ws_bytes = img_region_bytes(net);
  net.img_ws = bp.bytes(net.img_ws_bytes);
  // (the groups' accumulators side by side: G times the widest layer's)
  net.bn_ws_bytes = mm3d_bnrelu_workspace_bytes(2 * net.m * net.L * net.G);
  net.bn_ws = bp.bytes(net.bn_ws_bytes);
  net.wp = net.cin_k != net.cin ? bp.f(27, (int64_t)net.cin_k * net.m) : nullptr;
  if (!net.det()) return;
  // (behind the default layout, which stays as it is; the default BatchNorm workspace is then unused)
  net.bn_ws_bytes = mm3d_bnrelu_workspace_bytes_ex(2 * net.m * net.L * net.G, MM3D_DETERMINISTIC);
  net.bn_ws = bp.bytes(net.bn_ws_bytes);
  size_t wg = 0;
  for (const ConvInfo& ci : net.convs) {  // (0 for a convolution without a deterministic form: it keeps the default)
    const size_t s = mm3d_conv_wgrad_workspace_bytes(0, ci.c_in, ci.c_out, ci.K, net.mode, MM3D_DETERMINISTIC);
    if (s > wg) wg = s;
  }
  net.wg_ws_bytes = wg;
  net.wg_ws = bp.bytes(wg);
}

// Identity row plans (NetworkInNetwork as a K = 1 rule-table convolution): perm = iota (-1 past the rows), one
// offset per tile, tiles in natural order, table = perm.  All levels' plans in one launch (blockIdx.y = level).
constexpr int kMaxIdPlans = 16;
struct IdPlans {
  void* plan[kMaxIdPlans];
  int64_t rows[kMaxIdPlans];
};
__global__ void k_identity_plans(const __grid_constant__ IdPlans ps) {
  mm3d_griddep_launch();
  mm3d_griddep_wait();
  char* base = (char*)ps.plan[blockIdx.y];
  if (!base) return;
  const int64_t n = ps.rows[blockIdx.y];
  const int64_t T = mm3d_plan_tiles(n);
  int32_t* perm = (int32_t*)base;
  uint32_t* mask = (uint32_t*)(base + mm3d_plan_off_mask(n));
  int32_t* order = (int32_t*)(base + mm3d_plan_off_order(n));
  uint32_t* off_tiles = (uint32_t*)(base + mm3d_plan_off_cnt(n));
  int32_t* tbl = (int32_t*)(base + mm3d_plan_off_tbl(n));
  const int64_t step = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < T * 128; i += step) {
    const int32_t v = i < n ? (int32_t)i : -1;
    perm[i] = v;
    tbl[i] = v;
    if (i < T) {
      mask[i] = 1u;
      order[i] = (int32_t)i;
    }
    if (i < 32) off_tiles[i] = i == 0 ? (uint32_t)T : 0u;
  }
}

__global__ void k_copy_cols(const float* __restrict__ src, int64_t n, int c_src, float* __restrict__ dst, int c_dst,
                            int dst_col0, int ncols, int src_col0) {
  mm3d_griddep_launch();
  mm3d_griddep_wait();
  // dst[r, dst_col0 + j] = src[r, src_col0 + j], j < ncols  (other dst columns untouched)
  if (((ncols | c_src | c_dst | dst_col0 | src_col0) & 3) == 0) {  // whole float4s (every layer of the network)
    const int nv = ncols >> 2;
    const int64_t total = n * nv;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
      const int64_t r = i / nv;
      const int j = (int)(i - r * nv) << 2;
      *reinterpret_cast<float4*>(dst + r * c_dst + dst_col0 + j) =
          __ldg(reinterpret_cast<const float4*>(src + r * c_src + src_col0 + j));
    }
    return;
  }
  const int64_t total = n * ncols;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / ncols;
    const int j = (int)(i - r * ncols);
    dst[r * c_dst + dst_col0 + j] = __ldg(src + r * c_src + src_col0 + j);
  }
}

// JoinTable: J = [A | B] (both [n, p], p a multiple of 4) in one pass
__global__ void k_concat2(const float* __restrict__ a, const float* __restrict__ b, int64_t n, int p, float* __restrict__ j_out) {
  mm3d_griddep_launch();
  mm3d_griddep_wait();
  const int pv = p >> 2;
  const int64_t total = n * 2 * pv;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / (2 * pv);
    const int v = (int)(i - r * 2 * pv);  // float4 column of J
    const float* src = v < pv ? a + r * p + (v << 2) : b + r * p + ((v - pv) << 2);
    *reinterpret_cast<float4*>(j_out + r * 2 * p + (v << 2)) = __ldg(reinterpret_cast<const float4*>(src));
  }
}

__global__ void k_pad_cols(const float* __restrict__ src, int64_t n, int c_src, float* __restrict__ dst, int c_dst,
                           int round_tf32) {
  mm3d_griddep_launch();
  mm3d_griddep_wait();
  // dst[r, j] = j < c_src ? src[r, j] : 0   (c_dst >= c_src: pad;  c_dst < c_src: slice); optionally RNA-rounded to
  // TF32 (the padded stem input is the A operand of a kind::tf32 MMA)
  const int64_t total = n * c_dst;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / c_dst;
    const int j = (int)(i - r * c_dst);
    float v = j < c_src ? __ldg(src + r * c_src + j) : 0.f;
    if (round_tf32) {
      const float hi = mm3d_rna_tf32(v);
      if (round_tf32 == 2) dst[total + i] = mm3d_rna_tf32(v - hi);  // lo plane (TF32x3 mode)
      if (round_tf32 == 3) reinterpret_cast<__nv_bfloat16*>(dst + total)[i] = __float2bfloat16_rn(v);  // BF16 plane
      v = hi;
    }
    dst[i] = v;
  }
}

// out = RNA-rounded-to-TF32(in), whole float4s + tail (module-by-module path: operands of a TF32 convolution that
// were not produced by one of this library's rounding producers)
__global__ void k_round_tf32(const float* __restrict__ in, float* __restrict__ out, int64_t n) {
  mm3d_griddep_launch();
  mm3d_griddep_wait();
  const int64_t nv = n >> 2;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (int64_t)gridDim.x * blockDim.x) {
    float4 v = __ldg(reinterpret_cast<const float4*>(in) + i);
    v.x = mm3d_rna_tf32(v.x); v.y = mm3d_rna_tf32(v.y); v.z = mm3d_rna_tf32(v.z); v.w = mm3d_rna_tf32(v.w);
    reinterpret_cast<float4*>(out)[i] = v;
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) out[(nv << 2) + threadIdx.x] = mm3d_rna_tf32(__ldg(in + (nv << 2) + threadIdx.x));
}

// Backward runs the weight gradients on a second stream: a layer's wgrad only feeds the optimiser, while its
// dgrad is on the critical chain, and neither kernel fills the GPU alone at the deeper levels.
struct SideStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[64];
  int n_ev = 0, next = 0;
  bool ok = false;
};
SideStream* side_stream() {
  static SideStream pool[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  SideStream& s = pool[dev];
  if (!s.ok) {
    if (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    for (s.n_ev = 0; s.n_ev < 64; ++s.n_ev)
      if (cudaEventCreateWithFlags(&s.ev[s.n_ev], cudaEventDisableTiming) != cudaSuccess) return nullptr;
    s.ok = true;
  }
  return &s;
}

struct Ctx {
  Net* net;
  void* const* params;
  void* const* grads;  // backward only
  cudaStream_t stream;
  float eps, momentum;
  int training;
  int rc;
  SideStream* side = nullptr;  // backward only; NULL = everything on `stream`
  int bn_parity = 0;  // which half of bn_ws the BatchNorms of this call alternate to (bnrelu.cu); bn_ws is zeroed first
  const char *grad_lo = nullptr, *grad_hi = nullptr;  // span of the caller's gradient buffers when contiguous
  int wgrad_acc = 0;  // 1: the weight-gradient buffers were zeroed by one memset up front, wgrad kernels accumulate
  std::vector<const float*> img_key;  // weight pointer ...
  std::vector<const float*> img_val;  // ... -> its image
  std::vector<const float*> img_lo;   // ... -> the image of its TF32 remainder (TF32x3 mode)
};

// stream for a layer's weight gradient: the side stream once everything enqueued on the main stream so far
// (the layer's d_out) is done
cudaStream_t wgrad_stream(Ctx& c) {
  if (!c.side || c.rc) return c.stream;
  cudaEvent_t e = c.side->ev[c.side->next++ % c.side->n_ev];
  if (cudaEventRecord(e, c.stream) != cudaSuccess || cudaStreamWaitEvent(c.side->stream, e, 0) != cudaSuccess) {
    mm3d_set_error("unet backward: could not fork the weight-gradient stream");
    c.rc = MM3D_ERR_CUDA;
    return c.stream;
  }
  return c.side->stream;
}

// Timing experiments only: a library built with -DMM3D_ABLATION reads MM3D_ABL_SKIP, a list of kernel families the
// executor then does not launch (any of "bn", "wgrad", "conv" = forward + dgrad); results are garbage.  The
// product build has no such switch.
#ifdef MM3D_ABLATION
bool abl_skip(const char* what) {
  static const char* e = getenv("MM3D_ABL_SKIP");
  return e && strstr(e, what) != nullptr;
}
#else
constexpr bool abl_skip(const char*) { return false; }
#endif

#define EX(call)                   \
  do {                             \
    if (c.rc == 0) c.rc = (call);  \
  } while (0)

#ifdef MM3D_TRACE
// development builds: an event after every operation of the main stream; mm3d_debug_dump_marks() prints the time
// between consecutive events of the last forward + backward
struct Mark { const char* name; int level; cudaEvent_t ev; };
static std::vector<Mark> g_marks;
static bool g_marks_on = false;
static void trace_mark(cudaStream_t s, const char* name, int level) {
  if (!g_marks_on) return;
  Mark m{name, level, nullptr};
  cudaEventCreate(&m.ev);
  cudaEventRecord(m.ev, s);
  g_marks.push_back(m);
}
#define MARK(name, level) trace_mark(c.stream, name, level)
#else
#define MARK(name, level) do {} while (0)
#endif

const float* P(Ctx& c, int i) { return (const float*)c.params[i]; }
float* Gp(Ctx& c, int i) { return (float*)c.grads[i]; }

// x_hi != NULL: the input is the column blocks [x | x_hi] ([n, c_lo] and [n, ch - c_lo]) -- JoinTable without
// materialising the concatenation (training mode only)
// Tensor-core modes: every tensor that a kind::tf32 MMA reads as its gathered operand (activations in forward and
// wgrad, d_out in dgrad and wgrad) is stored RNA-rounded to TF32 by the kernel that PRODUCES it, so that the
// tensor core's truncation of the low mantissa bits is exact.  `to_conv`: the output feeds a convolution.
bool tc_mode(const Ctx& c) { return c.net->mode != MM3D_MODE_FP32; }

// l: the level whose rows x holds (its group boundaries)
void bn_fwd(Ctx& c, int pidx, int l, const float* x, float* y, int64_t n, int ch, float* save, const float* x_hi = nullptr,
            int c_lo = 0, bool to_conv = true) {
  if (abl_skip("bn")) return;
  const Net& net = *c.net;
  EX(mm3d_bnrelu_fwd_impl(x, x_hi, c_lo, y, n, ch, P(c, pidx), P(c, pidx + 1), (float*)c.params[pidx + 2], (float*)c.params[pidx + 3],
                          save, save + (int64_t)net.G * ch, c.eps, c.momentum, 0.f, c.training, net.bn_ws, net.bn_ws_bytes,
                          &c.bn_parity, tc_mode(c) && to_conv ? net.rmode() : 0, c.stream, net.det(), net.G, net.bounds(l)));
}
// round: bit 0 = dx (its low column block when split) feeds a convolution as d_out, bit 1 = dx_hi does
// add (rows add_ld floats apart): another gradient of the same tensor, summed into dx before it is stored;
// add_lo: `add` is a TF32x3 operand whose lo plane (n * add_ld floats behind) is summed too
void bn_bwd(Ctx& c, int pidx, int l, const float* x, const float* dy, float* dx, int64_t n, int ch, const float* save,
            int round, const float* x_hi = nullptr, int c_lo = 0, float* dx_hi = nullptr, const float* add = nullptr,
            int64_t add_ld = 0, bool add_lo = false) {
  if (abl_skip("bn")) return;
  const Net& net = *c.net;
  const int flags = tc_mode(c) ? (round | (net.x3() ? 4 : net.bf16() ? 8 : 0) | (add_lo ? 16 : 0)) : 0;
  EX(mm3d_bnrelu_bwd_impl(x, x_hi, c_lo, dy, dx, dx_hi, n, ch, P(c, pidx), P(c, pidx + 1), save, save + (int64_t)net.G * ch,
                          Gp(c, pidx), Gp(c, pidx + 1), 0.f, c.training, net.bn_ws, net.bn_ws_bytes, &c.bn_parity, flags, add,
                          add_ld, c.stream, net.det(), net.G, net.bounds(l)));
}
// NIN: NetworkInNetwork, a K = 1 convolution over the level's identity row plan
enum Kind { SMC, DOWN, UP, NIN };

const float* find_img(const Ctx& c, const float* w) {
  for (size_t i = 0; i < c.img_key.size(); ++i)
    if (c.img_key[i] == w) return c.img_val[i];
  return nullptr;
}
const float* find_img_lo(const Ctx& c, const float* w) {
  for (size_t i = 0; i < c.img_key.size() && i < c.img_lo.size(); ++i)
    if (c.img_key[i] == w) return c.img_lo[i];
  return nullptr;
}
// One rule-table convolution from prebuilt weight images.  TF32x3 mode: hi.Whi + lo.Whi + hi.Wlo inside one launch (`in`
// carries the lo plane n_in * c_in floats behind the hi one, both planes are gathered into every ring stage).
// add != NULL: out = conv + add (add == out accumulates); epi != NULL: the value goes to epi's destinations instead of out
int conv_img(const Ctx& c, const float* in, int64_t n_in, int c_in, float* out, int64_t n_out, int c_out, const float* im,
             const float* im_lo, int K, const void* plan, int64_t plan_cap, const float* add = nullptr,
             const ConvEpi* epi = nullptr) {
  if (c.net->x3() && !im_lo) { mm3d_set_error("tf32x3: missing lo weight image"); return MM3D_ERR_INVALID; }
  if (c.net->bf16())  // the BF16 plane sits n_in * c_in floats behind the FP32 one
    return mm3d_conv_fwd_tc_img(in + n_in * (int64_t)c_in, n_in, c_in, out, n_out, c_out, im, K, plan, plan_cap, add, c.stream, nullptr, 1,
                                epi);
  return mm3d_conv_fwd_tc_img(in, n_in, c_in, out, n_out, c_out, im, K, plan, plan_cap, add, c.stream, c.net->x3() ? im_lo : nullptr,
                              0, epi);
}

// the rule table of a layer type at FINE level l, as the convolutions take it
struct Table {
  int K;
  const int32_t* tbl;
  int64_t stride;
  const uint8_t* onehot;
  const void* plan;
  int64_t cap;
  int64_t n_in, n_out;
};
Table table(const Ctx& c, Kind kind, int l) {
  const LevelMeta& f = c.net->lv[l];
  const int64_t nc = l + 1 < c.net->L ? c.net->lv[l + 1].n : 0;
  switch (kind) {
    case SMC: return {27, f.nbr, f.tstride, nullptr, f.plan_smc, f.plan_cap, f.n, f.n};
    case DOWN: return {8, f.child, f.tstride, nullptr, f.plan_down, f.plan_cap, f.n, nc};
    case UP: return {8, f.parent, 0, f.off, f.plan_up, f.plan_cap, nc, f.n};
    default: {
      const void* plan = c.net->b[l].id_plan;
      return {1, mm3d_plan_view(plan, f.n).tbl, mm3d_plan_tiles(f.n) * 128, nullptr, plan, f.n, f.n, f.n};
    }
  }
}
// the table of the transposed layer (dgrad): SMC and NIN are their own transpose, DOWN <-> UP
Table table_t(const Ctx& c, Kind kind, int l) {
  Table t = table(c, kind == DOWN ? UP : kind == UP ? DOWN : kind, l);
  return t;
}

// forward of layer type `kind` whose FINE level is l; add != NULL: out = conv + add (add may be out)
void conv_fwd(Ctx& c, Kind kind, int l, const float* in, int c_in, float* out, int c_out, const float* w,
              const float* add = nullptr) {
  if (abl_skip("conv")) return;
  const Table t = table(c, kind, l);
  if (const float* im = find_img(c, w)) {  // prebuilt weight image: the tcgen05 kernel directly
    EX(conv_img(c, in, t.n_in, c_in, out, t.n_out, c_out, im, find_img_lo(c, w), t.K, t.plan, t.cap, add));
    return;
  }
  if (add) {  // (no weight image: FP32 mode, or a TF32 shape the tensor cores do not take) the SIMT kernel with the addend
    if (c.net->x3() || c.net->bf16()) {
      mm3d_set_error("unet: conv c_in %d c_out %d has no tensor-core weight image in this mode", c_in, c_out);
      if (c.rc == 0) c.rc = MM3D_ERR_UNSUPPORTED;
      return;
    }
    EX(mm3d_conv_fwd_simt(in, t.n_in, c_in, out, t.n_out, c_out, w, t.K, t.tbl, t.stride, t.onehot, 0, c.net->conv_ws,
                          c.net->conv_ws_bytes, c.stream, add));
  } else
    EX(mm3d_conv_fwd(in, t.n_in, c_in, out, t.n_out, c_out, w, t.K, t.tbl, t.stride, t.onehot, t.plan, t.cap, 0,
                     c.net->mode, c.net->conv_ws, c.net->conv_ws_bytes, c.stream));
}
// dgrad (d_in from d_out) and wgrad of the same layer; c_in / c_out are the FORWARD layer's
void conv_bwd(Ctx& c, Kind kind, int l, const float* in, int c_in, const float* d_out, int c_out, const float* w,
              float* d_in, float* d_w) {
  const int md = c.net->mode;
  const Table t = table(c, kind, l), tt = table_t(c, kind, l);
  cudaStream_t ws = wgrad_stream(c);  // d_out is complete on the main stream at this point
  const float* im = find_img(c, w);   // prebuilt dgrad image (tensor-core modes)
  const float* il = find_img_lo(c, w);
  // parameter gradients inside the caller's (pre-zeroed) flat buffer accumulate; temporaries are overwritten
  const int acc = c.wgrad_acc && c.grad_lo <= (const char*)d_w && (const char*)d_w < c.grad_hi;
  const bool do_wg = !abl_skip("wgrad") && d_w != nullptr, do_dg = !abl_skip("conv") && d_in != nullptr;  // (frozen weight: no d_w)
  // The weight gradient (side stream) is enqueued before the data gradient.  (Measured with the in-process A/B of
  // bench.py on the final kernels: the order makes no difference, 2.959 vs 2.958 ms per step -- the step is bound by
  // the total work of both streams, not by which kernel gets the SMs first.)
  // Deterministic mode: the fixed-order form through the slab region wherever the shape has one (the caller learns
  // beforehand which do not: the fp32 mode, channels that are not multiples of 16); the others keep the default.
  const bool det_wg = c.net->det() && mm3d_conv_wgrad_workspace_bytes(t.n_out, c_in, c_out, t.K, md, MM3D_DETERMINISTIC) > 0;
  if (do_wg && det_wg)
    EX(mm3d_conv_wgrad_ex(in, t.n_in, c_in, d_out, t.n_out, c_out, d_w, t.K, t.tbl, t.stride, t.onehot, t.plan, t.cap, acc,
                          md, c.net->wg_ws, c.net->wg_ws_bytes, ws, MM3D_DETERMINISTIC));
  else if (do_wg)
    EX(mm3d_conv_wgrad(in, t.n_in, c_in, d_out, t.n_out, c_out, d_w, t.K, t.tbl, t.stride, t.onehot, t.plan, t.cap, acc,
                       md, nullptr, 0, ws));
  if (im && do_dg)
    EX(conv_img(c, d_out, t.n_out, c_out, d_in, t.n_in, c_in, im, il, t.K, tt.plan, tt.cap));
  else if (do_dg)
    EX(mm3d_conv_fwd(d_out, t.n_out, c_out, d_in, t.n_in, c_in, w, t.K, tt.tbl, tt.stride, tt.onehot, tt.plan, tt.cap,
                     MM3D_CONV_TRANSPOSE_W | (kind == SMC ? MM3D_CONV_MIRROR_K : 0), md, c.net->conv_ws, c.net->conv_ws_bytes,
                     c.stream));
}

// main stream waits for everything enqueued on the side stream so far
void join_side(Ctx& c) {
  if (!c.side || c.rc) return;
  cudaEvent_t e = c.side->ev[c.side->next++ % c.side->n_ev];
  if (cudaEventRecord(e, c.side->stream) != cudaSuccess || cudaStreamWaitEvent(c.stream, e, 0) != cudaSuccess) {
    mm3d_set_error("unet backward: could not join the weight-gradient stream");
    c.rc = MM3D_ERR_CUDA;
  }
}

void launch_copy_cols(Ctx& c, const float* src, int64_t n, int c_src, float* dst, int c_dst, int col0, int ncols) {
  if (n == 0 || c.rc) return;
  if (mm3d_launch_pdl(k_copy_cols, dim3(mm3d_grid(n * ncols / 4 + 1, 256)), dim3(256), 0, c.stream, src, n, c_src, dst, c_dst, col0, ncols, 0) != cudaSuccess) c.rc = MM3D_ERR_CUDA;
  mm3d_count_launches(1);
}
void launch_pad_cols(Ctx& c, const float* src, int64_t n, int c_src, float* dst, int c_dst, int round_tf32 = 0) {
  if (n == 0 || c.rc) return;
  if (mm3d_launch_pdl(k_pad_cols, dim3(mm3d_grid(n * c_dst, 256)), dim3(256), 0, c.stream, src, n, c_src, dst, c_dst, round_tf32) != cudaSuccess) c.rc = MM3D_ERR_CUDA;
  mm3d_count_launches(1);
}
// JoinTable: j = [y | f] ([n, p] each)
void launch_join(Ctx& c, const float* y, const float* f, int64_t n, int p, float* j) {
  if ((p & 3) == 0) {
    if (n && !c.rc) {
      if (mm3d_launch_pdl(k_concat2, dim3(mm3d_grid(n * p / 2 + 1, 256)), dim3(256), 0, c.stream, y, f, n, p, j) != cudaSuccess)
        c.rc = MM3D_ERR_CUDA;
      mm3d_count_launches(1);
    }
  } else {
    launch_copy_cols(c, y, n, p, j, 2 * p, 0, p);
    launch_copy_cols(c, f, n, p, j, 2 * p, p, p);
  }
}

// One launch builds the weight images of every layer for this direction (dgrad: W^T, mirrored for 3^3 layers).
int build_images(Ctx& c, bool backward, const float* w_stem) {
  const Net& net = *c.net;
  if (net.mode == MM3D_MODE_FP32) return MM3D_OK;
  std::vector<const float*> w;
  std::vector<float*> img;
  std::vector<int> K, ci, co, fl;
  char* at = (char*)net.img_ws;
  for (const ConvInfo& x : net.convs) {
    const int a = backward ? x.c_out : x.c_in, b = backward ? x.c_in : x.c_out;
    if (!mm3d_conv_tc_supported(a, b, x.K)) continue;
    const size_t bytes = mm3d_align(mm3d_conv_tc_workspace_bytes(a, b, x.K));
    MM3D_REQUIRE((size_t)(at - (char*)net.img_ws) + bytes <= net.img_ws_bytes, MM3D_ERR_WORKSPACE, "weight image region too small");
    w.push_back(x.pidx == 0 ? w_stem : (const float*)c.params[x.pidx]);
    img.push_back((float*)at);
    K.push_back(x.K); ci.push_back(a); co.push_back(b);
    fl.push_back((backward ? (MM3D_CONV_TRANSPOSE_W | (x.smc ? MM3D_CONV_MIRROR_K : 0)) : 0) | (net.bf16() ? MM3D_CONV_BF16 : 0));
    at += bytes;
  }
  int rc = mm3d_conv_tc_build_images(w.data(), img.data(), K.data(), ci.data(), co.data(), fl.data(), (int)w.size(), c.stream);
  if (rc) return rc;
  c.img_key.assign(w.begin(), w.end());
  c.img_val.assign(img.begin(), img.end());
  c.img_lo.clear();
  if (net.x3()) {  // the images of the weights' TF32 remainders, behind the hi images
    std::vector<float*> lo;
    for (size_t i = 0; i < w.size(); ++i) {
      const size_t bytes = mm3d_align(mm3d_conv_tc_workspace_bytes(ci[i], co[i], K[i]));
      MM3D_REQUIRE((size_t)(at - (char*)net.img_ws) + bytes <= net.img_ws_bytes, MM3D_ERR_WORKSPACE, "weight image region too small");
      lo.push_back((float*)at);
      at += bytes;
      fl[i] |= MM3D_CONV_WEIGHT_LO;
    }
    rc = mm3d_conv_tc_build_images(w.data(), lo.data(), K.data(), ci.data(), co.data(), fl.data(), (int)w.size(), c.stream);
    if (rc) return rc;
    c.img_lo.assign(lo.begin(), lo.end());
  }
  return MM3D_OK;
}

// the identity row plans of every level with a NetworkInNetwork shortcut, one launch
void build_identity_plans(Ctx& c) {
  const Net& net = *c.net;
  IdPlans ps{};
  int64_t most = 0;
  bool any = false;
  for (int l = 0; l < net.L && l < kMaxIdPlans; ++l) {
    ps.plan[l] = net.b[l].id_plan;
    ps.rows[l] = net.lv[l].n;
    if (ps.plan[l]) {
      any = true;
      if (net.lv[l].n > most) most = net.lv[l].n;
    }
  }
  if (!any || c.rc) return;
  if (net.L > kMaxIdPlans) { mm3d_set_error("unet: more than %d levels", kMaxIdPlans); c.rc = MM3D_ERR_UNSUPPORTED; return; }
  const int blocks = mm3d_grid(mm3d_plan_tiles(most) * 128 + 1, 256);
  if (mm3d_launch_pdl(k_identity_plans, dim3(blocks, net.L), dim3(256), 0, c.stream, ps) != cudaSuccess) c.rc = MM3D_ERR_CUDA;
  mm3d_count_launches(1);
}

// A block's forward.  x: its input [n, a]; the first post block of a level (join) reads [Y | F] instead.
void block_fwd(Ctx& c, int l, const BlockBufs& k, const float* x, bool join) {
  Net& net = *c.net;
  LevelBufs& B = net.b[l];
  const int64_t n = net.lv[l].n;
  const int o = net.nin(k.a, k.b) ? 1 : 0;
  const int bn1 = k.pidx + o;
  if (join) {
    const int p = k.b;
    const bool split = (p & 3) == 0 && c.training;  // JoinTable never materialised: BatchNorm reads [Y | F] directly
    // the shortcut gathers J: it is written (the BatchNorm of an unsplit join reads the unrounded J)
    if (!split || o) launch_join(c, B.Y, B.F, n, p, split ? B.Jop : B.J);
    if (split) bn_fwd(c, bn1, l, B.Y, k.A, n, 2 * p, k.s1, B.F, p);
    else bn_fwd(c, bn1, l, B.J, k.A, n, 2 * p, k.s1);
    if (o && tc_mode(c))  // J in operand form (rounded; + second plane)
      launch_pad_cols(c, split ? B.Jop : B.J, n, 2 * p, B.Jop, 2 * p, net.rmode());
    MARK("bn_fwd post", l);
  } else {
    bn_fwd(c, bn1, l, x, k.A, n, k.a, k.s1);
    MARK("bn_fwd block", l);
  }
  if (!net.res) {
    conv_fwd(c, SMC, l, k.A, k.a, k.out, k.b, P(c, k.pidx + 4));
    MARK("smc_fwd block", l);
    return;
  }
  conv_fwd(c, SMC, l, k.A, k.a, k.H, k.b, P(c, bn1 + 4));
  bn_fwd(c, bn1 + 5, l, k.H, k.A2, n, k.b, k.s2);
  if (o) {  // NetworkInNetwork shortcut writes `out`, the second convolution adds onto it
    conv_fwd(c, NIN, l, B.Jop, k.a, k.out, k.b, P(c, k.pidx));
    conv_fwd(c, SMC, l, k.A2, k.b, k.out, k.b, P(c, bn1 + 9), k.out);
  } else {  // identity shortcut: the block input is the second convolution's addend
    conv_fwd(c, SMC, l, k.A2, k.b, k.out, k.b, P(c, bn1 + 9), x);
  }
  MARK("residual block fwd", l);
}

void level_fwd(Ctx& c, int l) {
  Net& net = *c.net;
  LevelBufs& B = net.b[l];
  const int64_t n = net.lv[l].n;
  const int p = net.planes(l);
  const float* x = B.X;
  for (const BlockBufs& k : B.pre) {
    block_fwd(c, l, k, x, false);
    x = k.out;
  }
  if (l + 1 < net.L) {
    const int q = net.planes(l + 1);
    bn_fwd(c, B.dn, l, B.Y, B.B, n, p, B.s_dn);
    MARK("bn_fwd dn", l);
    conv_fwd(c, DOWN, l, B.B, p, net.b[l + 1].X, q, P(c, B.dn + 4));
    MARK("down_fwd", l);
    level_fwd(c, l + 1);
    bn_fwd(c, B.up, l + 1, net.b[l + 1].R, B.E, net.lv[l + 1].n, q, B.s_up);
    MARK("bn_fwd up", l);
    conv_fwd(c, UP, l, B.E, q, B.F, p, P(c, B.up + 4));
    MARK("up_fwd", l);
    for (size_t r = 0; r < B.post.size(); ++r) block_fwd(c, l, B.post[r], r ? B.post[r - 1].out : nullptr, r == 0);
  }
}

// A block's backward.  d_o: gradient w.r.t. its output (operand form); writes k.d_x, the gradient w.r.t. its input,
// in operand form.  The first post block (join) instead writes the skip half d_J[:, :p] (unrounded; all of d_J
// when the join is not split) and d_F, the deconvolution's d_out (operand form).
void block_bwd(Ctx& c, int l, const BlockBufs& k, const float* x, const float* d_o, bool join) {
  Net& net = *c.net;
  LevelBufs& B = net.b[l];
  const int64_t n = net.lv[l].n;
  const int o = net.nin(k.a, k.b) ? 1 : 0;
  const int bn1 = k.pidx + o;
  const float* add = nullptr;  // the shortcut's gradient, summed into the first BatchNorm's backward
  int64_t add_ld = 0;
  bool add_lo = false;
  if (!net.res) {
    conv_bwd(c, SMC, l, k.A, k.a, d_o, k.b, P(c, k.pidx + 4), k.d_A, Gp(c, k.pidx + 4));
  } else {
    conv_bwd(c, SMC, l, k.A2, k.b, d_o, k.b, P(c, bn1 + 9), k.d_A2, Gp(c, bn1 + 9));
    bn_bwd(c, bn1 + 5, l, k.H, k.d_A2, k.d_H, n, k.b, k.s2, 1);
    conv_bwd(c, SMC, l, k.A, k.a, k.d_H, k.b, P(c, bn1 + 4), k.d_A, Gp(c, bn1 + 4));
    if (o) {
      conv_bwd(c, NIN, l, B.Jop, k.a, d_o, k.b, P(c, k.pidx), k.d_S, Gp(c, k.pidx));
      add = k.d_S;
      add_ld = k.a;
    } else {  // identity: d_o itself, FP32-exact in TF32x3 mode through its lo plane
      add = d_o;
      add_ld = k.b;
      add_lo = net.x3();
    }
  }
  MARK("block conv bwd", l);
  if (!join) {
    bn_bwd(c, bn1, l, x, k.d_A, k.d_x, n, k.a, k.s1, 1, nullptr, 0, nullptr, add, add_ld, add_lo);
    MARK("bn_bwd block", l);
    return;
  }
  const int p = k.b;
  if ((p & 3) == 0 && c.training) {  // as in the forward: [Y | F] was never concatenated
    bn_bwd(c, bn1, l, B.Y, k.d_A, B.d_J, n, 2 * p, k.s1, 2, B.F, p, B.d_F, add, add_ld);  // d_F is the deconvolution's d_out
  } else {
    bn_bwd(c, bn1, l, B.J, k.d_A, B.d_J, n, 2 * p, k.s1, 0, nullptr, 0, nullptr, add, add_ld);  // (eval-mode backward: d_F stays unrounded)
    // d_F = d_J[:, p:]; the skip half is combined with the branch gradient further down
    if (n && !c.rc) {
      if (mm3d_launch_pdl(k_copy_cols, dim3(mm3d_grid(n * p / 4 + 1, 256)), dim3(256), 0, c.stream, (const float*)B.d_J, n, 2 * p, B.d_F, p, 0, p, p) != cudaSuccess) c.rc = MM3D_ERR_CUDA;
      mm3d_count_launches(1);
      if (tc_mode(c)) launch_pad_cols(c, B.d_F, n, p, B.d_F, p, net.rmode());  // round in place (+ second plane): d_F is the deconvolution's d_out
    }
  }
  MARK("bn_bwd post", l);
}

// d_R: gradient w.r.t. the level's output R_l (operand form); writes the gradient w.r.t. X_l, B.pre[0].d_x.
void level_bwd(Ctx& c, int l, const float* d_R) {
  Net& net = *c.net;
  LevelBufs& B = net.b[l];
  const int64_t n = net.lv[l].n;
  const int p = net.planes(l);
  const float* d_Y = d_R;
  if (l + 1 < net.L) {
    const int q = net.planes(l + 1);
    const int64_t nc = net.lv[l + 1].n;
    const float* d_o = d_R;
    for (size_t r = B.post.size() - 1; r >= 1; --r) {
      block_bwd(c, l, B.post[r], B.post[r - 1].out, d_o, false);
      d_o = B.post[r].d_x;
    }
    block_bwd(c, l, B.post[0], nullptr, d_o, true);
    conv_bwd(c, UP, l, B.E, q, B.d_F, p, P(c, B.up + 4), B.d_E, Gp(c, B.up + 4));
    MARK("up_dgrad", l);
    bn_bwd(c, B.up, l + 1, net.b[l + 1].R, B.d_E, B.d_Rn, nc, q, B.s_up, 1);
    MARK("bn_bwd up", l);
    level_bwd(c, l + 1, B.d_Rn);
    conv_bwd(c, DOWN, l, B.B, p, B.d_Xn, q, P(c, B.dn + 4), B.d_B, Gp(c, B.dn + 4));
    MARK("down_dgrad", l);
    // d_Y = d_J[:, :p] (the skip half of the join's gradient) + the branch gradient: summed inside the BatchNorm
    // backward of the down-branch, stored rounded (it is the pre-block convolution's d_out)
    const bool split = (p & 3) == 0 && c.training;
    bn_bwd(c, B.dn, l, B.Y, B.d_B, B.d_Yskip, n, p, B.s_dn, 1, nullptr, 0, nullptr, B.d_J, split ? p : 2 * p);
    MARK("bn_bwd dn", l);
    d_Y = B.d_Yskip;
  }
  for (size_t r = B.pre.size(); r-- > 0;) {
    block_bwd(c, l, B.pre[r], r ? B.pre[r - 1].out : B.X, d_Y, false);
    d_Y = B.pre[r].d_x;
  }
}

int fill_net(Net& net, int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
             const int64_t* level_desc, int64_t n_points, int flags = 0, const mm3d_unet_groups* groups = nullptr) {
  MM3D_REQUIRE((flags & ~MM3D_DETERMINISTIC) == 0, MM3D_ERR_INVALID, "unet: unknown flags %#x", flags);
  MM3D_REQUIRE(num_planes >= 1 && num_planes <= 16 && m > 0 && in_channels > 0, MM3D_ERR_INVALID, "bad network shape");
  MM3D_REQUIRE(block_reps >= 1 && block_reps <= 16 && (residual == 0 || residual == 1), MM3D_ERR_INVALID,
               "bad block topology: block_reps %d residual %d", block_reps, residual);
  MM3D_REQUIRE(mode == MM3D_MODE_FP32 || mode == MM3D_MODE_TF32 || mode == MM3D_MODE_TF32X3 || mode == MM3D_MODE_BF16, MM3D_ERR_UNSUPPORTED,
               "conv mode %d not implemented in this build", mode);
  net.L = num_planes; net.m = m; net.cin = in_channels; net.mode = mode; net.n_points = n_points;
  net.reps = block_reps; net.res = residual; net.flags = flags;
  // tensor-core kernels gather rows in 64-byte pieces: pad the stem input to a multiple of 16 channels
  net.cin_k = in_channels;
  if (mode != MM3D_MODE_FP32) net.cin_k = (in_channels + 15) / 16 * 16;
  net.lv.assign(num_planes, LevelMeta{});
  for (int l = 0; l < num_planes && level_desc; ++l) {
    const int64_t* d = level_desc + MM3D_LEVEL_DESC_WORDS * l;
    net.lv[l] = LevelMeta{d[0], (const int32_t*)d[1], d[2], (const int32_t*)d[3], (const uint8_t*)d[4], (const int32_t*)d[5],
                          (const void*)d[6], (const void*)d[7], (const void*)d[8], d[9]};
  }
  if (groups) {  // (a NULL bounds array only sizes: the queries)
    MM3D_REQUIRE(groups->groups >= 1 && groups->groups <= MM3D_BN_MAX_GROUPS, MM3D_ERR_INVALID,
                 "unet: %d groups (1..%d supported)", groups->groups, MM3D_BN_MAX_GROUPS);
    net.G = groups->groups;
    if (groups->bounds && net.G > 1) {
      net.gb.assign(groups->bounds, groups->bounds + (size_t)num_planes * (net.G + 1));
      for (int l = 0; l < num_planes && level_desc; ++l) {
        const int64_t* b = net.gb.data() + (size_t)l * (net.G + 1);
        MM3D_REQUIRE(b[0] == 0 && b[net.G] == net.lv[l].n, MM3D_ERR_INVALID,
                     "unet: level %d's group boundaries must run from 0 to its %lld rows", l, (long long)net.lv[l].n);
        for (int k = 1; k <= net.G; ++k)
          MM3D_REQUIRE(b[k] >= b[k - 1], MM3D_ERR_INVALID, "unet: level %d's group boundaries decrease", l);
      }
    }
  }
  return MM3D_OK;
}

// What the walk and the scratch layout need of each of the caller's three buffers.  A NULL base only sizes.
struct Sizes {
  size_t act, tmp, scratch;
};
Sizes lay_out(Net& net, void* act, void* tmp, void* scratch) {
  Bump a{(char*)act, 0}, t{(char*)tmp, 0}, s{(char*)scratch, 0};
  Carve{net, a, t}.run();
  carve_scratch(net, s);
  return {a.off, t.off, s.off};
}

// The InputLayer (+ the folded RGB mask) into net.V, the stem input in operand form (net.Vp) and the stem weight as the
// kernels see it, which is returned
const float* input_stage(Ctx& c, int64_t n_points, const int32_t* p2v, const int32_t* npts, const int32_t* vox_start,
                         const int32_t* vox_pts, const float* feats, const mm3d_unet_mask* mask) {
  Net& net = *c.net;
  const int64_t n0 = net.lv[0].n;
  if (mask) {  // the RGB-mask prologue of Net3DSeg.forward folded into the point -> voxel scatter
    if (net.det())
      EX(mm3d_input_masked_fwd_csr(feats, vox_start, vox_pts, n0, net.cin, 4, mask->wb, net.V, mask->s, c.stream));
    else
      EX(mm3d_input_masked_fwd(feats, p2v, npts, n_points, n0, net.cin, 4, mask->wb, net.V, mask->s, c.stream));
  } else if (net.det()) {
    EX(mm3d_input_fwd_csr(feats, vox_start, vox_pts, n0, net.cin, 4, net.V, c.stream));
  } else {
    EX(mm3d_input_fwd(feats, p2v, npts, n_points, n0, net.cin, 4, net.V, c.stream));
  }
  MARK("input_fwd", -1);
  const float* w_stem = P(c, 0);
  if (net.Vp != net.V)  // pad the stem input to whole 64-byte pieces; rounded to TF32 (+ lo plane in TF32x3 mode)
    launch_pad_cols(c, net.V, n0, net.cin, net.Vp, net.cin_k, net.rmode());
  else if (tc_mode(c) && n0 > 0 && !c.rc) {
    // (stem input already a whole number of 64-byte pieces: round the InputLayer output in place)
    if (mm3d_launch_pdl(k_round_tf32, dim3(mm3d_grid(n0 * net.cin / 4 + 1, 256)), dim3(256), 0, c.stream, (const float*)net.V, net.V, n0 * (int64_t)net.cin) != cudaSuccess) c.rc = MM3D_ERR_CUDA;
    mm3d_count_launches(1);
  }
  if (net.cin_k != net.cin) {  // zero input channels for the stem weight too
    launch_pad_cols(c, w_stem, 27, net.cin * net.m, net.wp, net.cin_k * net.m);
    w_stem = net.wp;
  }
  return w_stem;
}

// ---- inference forward (eval-mode BatchNorm, nothing kept for a backward) ---------------------------------------------
// Every BatchNorm+ReLU runs in the epilogue of the convolution that produces its input (epilogue.cuh): a tensor is
// written straight into the normalised operand forms its consumers gather, and the JoinTable [Y | F] is never
// materialised -- Y and F each write their column block of the first post block's normalised input (rows 2p floats
// apart) and, with residual blocks, of J in operand form, which the NetworkInNetwork shortcut gathers.  Destinations
// per tensor (at most kEpiDsts = 3):
//   a block's input (stem / down output / previous block's output): the block's first BatchNorm -> A; residual:
//     + raw (the identity shortcut's addend)
//   Y (the last pre block's output, not the deepest level): down BatchNorm -> B, the first post block's BatchNorm ->
//     AJ[:, :p]; residual: + J[:, :p] in operand form
//   F (the deconvolution's output): AJ[:, p:]; residual: + J[:, p:] in operand form
//   R (a level's output): the parent's up BatchNorm -> E, or at level 0 the head BatchNorm -> Z (FP32, for the
//     OutputLayer)
//   residual blocks: first SMC -> the second BatchNorm -> A2; NetworkInNetwork -> S (raw, the second SMC's addend)
// No standalone BatchNorm or join launch remains, in any block topology.
struct IBlock {
  float *A, *xr, *A2, *S;  // normalised input (operand form), raw input, second normalised input, shortcut output
};
struct ILevel {
  std::vector<IBlock> pre, post;
  float *B, *E, *AJ, *Jop;  // down input, up input (the next level's rows), first post block's input [n, 2p], J (operand form)
};
struct InferLayout {
  std::vector<ILevel> lv;
  std::vector<float*> scale;  // per BatchNorm (at its first slot): rsqrtf(running_var + eps) * gamma
};

// The workspace walk: sizes (NULL ws) and lays out everything the inference forward writes -- the InputLayer output and
// stem input, each convolution's destinations, the identity row plans, the forward weight images, the padded stem
// weight and the BatchNorm scales.  Returns the bytes it needs.
size_t infer_layout(Net& net, InferLayout& IL, void* ws) {
  Bump none{nullptr, 0}, none2{nullptr, 0};
  Carve{net, none, none2}.run();  // (parameter slots, the convolution and BatchNorm lists; no buffers)
  Bump a{(char*)ws, 0};
  const int pl = net.pl();
  const int64_t n0 = net.lv[0].n;
  net.V = a.f(n0, net.cin);
  net.Vp = (net.cin_k != net.cin || pl == 2) ? a.f(n0, (int64_t)net.cin_k * pl) : net.V;
  IL.lv.assign(net.L, ILevel());
  auto block = [&](int64_t n, int a_ch, int b_ch) {
    IBlock k{};
    k.A = a.f(n, (int64_t)a_ch * pl);
    if (net.res) {
      if (a_ch == b_ch) k.xr = a.f(n, a_ch);
      else k.S = a.f(n, b_ch);
      k.A2 = a.f(n, (int64_t)b_ch * pl);
    }
    return k;
  };
  for (int l = 0; l < net.L; ++l) {
    const int64_t n = net.lv[l].n;
    const int p = net.planes(l);
    ILevel& I = IL.lv[l];
    for (int r = 0; r < net.reps; ++r) I.pre.push_back(block(n, p, p));
    if (l + 1 == net.L) continue;
    I.B = a.f(n, (int64_t)p * pl);
    I.E = a.f(net.lv[l + 1].n, (int64_t)net.planes(l + 1) * pl);
    for (int r = 0; r < net.reps; ++r) {
      if (r == 0) {
        IBlock k{};
        k.A = I.AJ = a.f(n, (int64_t)2 * p * pl);
        if (net.res) {
          I.Jop = a.f(n, (int64_t)2 * p * pl);
          net.b[l].id_plan = a.bytes(mm3d_plan_size(n, 1));
          k.S = a.f(n, p);
          k.A2 = a.f(n, (int64_t)p * pl);
        }
        I.post.push_back(k);
      } else {
        I.post.push_back(block(n, p, p));
      }
    }
  }
  net.Z = a.f(n0, net.m);
  // A tensor-core convolution of more than 256 input channels runs as input slices whose partial sum goes through
  // memory before the last slice's epilogue: one buffer of the largest such output.  Every convolution producing level
  // l's rows has at most planes(l) output and 2 planes(l) input channels.
  int64_t wide = 0;
  for (int l = 0; l < net.L && net.mode != MM3D_MODE_FP32; ++l)
    if (2 * net.planes(l) > 256 && net.lv[l].n * net.planes(l) > wide) wide = net.lv[l].n * net.planes(l);
  net.wide_sum = wide ? a.f(wide, 1) : nullptr;
  net.img_ws_bytes = img_region_bytes(net, false);
  net.img_ws = a.bytes(net.img_ws_bytes);
  net.wp = net.cin_k != net.cin ? a.f(27, (int64_t)net.cin_k * net.m) : nullptr;
  IL.scale.assign(net.n_params, nullptr);
  for (const auto& bn : net.bns) IL.scale[bn.first] = a.f(1, bn.second);
  return a.off;
}

// the scales of every BatchNorm, one CTA each, in as few launches as the list takes (one for the usual networks)
constexpr int kMaxBnScales = 128;
struct BnScales {
  const float* gamma[kMaxBnScales];
  const float* var[kMaxBnScales];
  float* scale[kMaxBnScales];
  int c[kMaxBnScales];
  float eps;
};
__global__ void k_bn_scales(const __grid_constant__ BnScales b) {
  mm3d_griddep_launch();
  mm3d_griddep_wait();
  const int i = blockIdx.x;
  for (int ch = threadIdx.x; ch < b.c[i]; ch += blockDim.x) b.scale[i][ch] = rsqrtf(b.var[i][ch] + b.eps) * b.gamma[i][ch];
}
void bn_scales(Ctx& c, const InferLayout& IL) {
  const auto& bns = c.net->bns;
  for (size_t first = 0; first < bns.size() && !c.rc; first += kMaxBnScales) {
    BnScales b;
    b.eps = c.eps;
    int k = 0;
    for (size_t i = first; i < bns.size() && k < kMaxBnScales; ++i, ++k) {
      const int s = bns[i].first;
      b.gamma[k] = P(c, s);
      b.var[k] = P(c, s + 3);
      b.scale[k] = IL.scale[s];
      b.c[k] = bns[i].second;
    }
    if (mm3d_launch_pdl(k_bn_scales, dim3(k), dim3(128), 0, c.stream, b) != cudaSuccess) c.rc = MM3D_ERR_CUDA;
    mm3d_count_launches(1);
  }
}

struct Infer {
  Ctx& c;
  const InferLayout& IL;
  Net& net;

  // how a tensor that a convolution gathers is stored: the store_planes forms, except that the BF16 mode's FP32 plane
  // (the weight gradients' operand) is not written
  int op() const { return net.bf16() ? 4 : net.rmode(); }
  // column block col0.. of the [rows, ld] tensor t (planes rows * ld floats apart), in store form `store`; bn >= 0:
  // normalised with the BatchNorm of that first slot (its channels col0..)
  EpiDst dst(float* t, int64_t rows, int ld, int col0, int store, int bn = -1) const {
    EpiDst d{};
    d.p = t + col0;
    d.ld = ld;
    d.store = store;
    if (store == 2) d.p2 = t + rows * ld + col0;
    if (store >= 3) d.p2 = reinterpret_cast<__nv_bfloat16*>(t + rows * ld) + col0;
    if (bn >= 0) {
      d.mean = P(c, bn + 2) + col0;
      d.scale = IL.scale[bn] + col0;
      d.beta = P(c, bn + 1) + col0;
    }
    return d;
  }
  int bn1(const BlockBufs& k) const { return k.pidx + (net.nin(k.a, k.b) ? 1 : 0); }
  // the destinations of a block's input
  ConvEpi input_of(int l, const BlockBufs& k, const IBlock& ib) const {
    const int64_t n = net.lv[l].n;
    ConvEpi e{};
    e.d[e.n++] = dst(ib.A, n, k.a, 0, op(), bn1(k));
    if (net.res) e.d[e.n++] = dst(ib.xr, n, k.a, 0, 0);
    return e;
  }
  // R_l, the output of level l
  ConvEpi level_output(int l) const {
    ConvEpi e{};
    if (l == 0) e.d[e.n++] = dst(net.Z, net.lv[0].n, net.m, 0, 0, net.head);
    else e.d[e.n++] = dst(IL.lv[l - 1].E, net.lv[l].n, net.planes(l), 0, op(), net.b[l - 1].up);
    return e;
  }
  // Y (pre = true) or F: their column block of the join
  ConvEpi join_half(int l, bool pre) const {
    const int64_t n = net.lv[l].n;
    const int p = net.planes(l), col0 = pre ? 0 : p;
    const ILevel& I = IL.lv[l];
    ConvEpi e{};
    if (pre) e.d[e.n++] = dst(I.B, n, p, 0, op(), net.b[l].dn);
    e.d[e.n++] = dst(I.AJ, n, 2 * p, col0, op(), bn1(net.b[l].post[0]));
    if (net.res) e.d[e.n++] = dst(I.Jop, n, 2 * p, col0, op());
    return e;
  }

  void conv(Kind kind, int l, const float* in, int c_in, int c_out, const float* w, const float* add, const ConvEpi& e) {
    if (abl_skip("conv")) return;
    const Table t = table(c, kind, l);
    if (const float* im = find_img(c, w)) {
      EX(conv_img(c, in, t.n_in, c_in, c_in > 256 ? net.wide_sum : nullptr, t.n_out, c_out, im, find_img_lo(c, w), t.K, t.plan,
                  t.cap, add, &e));
    } else if (net.x3() || net.bf16()) {
      mm3d_set_error("unet: conv c_in %d c_out %d has no tensor-core weight image in this mode", c_in, c_out);
      if (c.rc == 0) c.rc = MM3D_ERR_UNSUPPORTED;
    } else {  // FP32 mode, or a TF32 shape the tensor cores do not take
      EX(mm3d_conv_fwd_simt(in, t.n_in, c_in, nullptr, t.n_out, c_out, w, t.K, t.tbl, t.stride, t.onehot, 0, nullptr, 0,
                            c.stream, add, &e));
    }
  }

  void block(int l, const BlockBufs& k, const IBlock& ib, const ConvEpi& out) {
    const int64_t n = net.lv[l].n;
    if (!net.res) {
      conv(SMC, l, ib.A, k.a, k.b, P(c, k.pidx + 4), nullptr, out);
      return;
    }
    const int b1 = bn1(k);
    ConvEpi e{};
    e.d[e.n++] = dst(ib.A2, n, k.b, 0, op(), b1 + 5);
    conv(SMC, l, ib.A, k.a, k.b, P(c, b1 + 4), nullptr, e);
    if (net.nin(k.a, k.b)) {
      ConvEpi s{};
      s.d[s.n++] = dst(ib.S, n, k.b, 0, 0);
      conv(NIN, l, IL.lv[l].Jop, k.a, k.b, P(c, k.pidx), nullptr, s);
    }
    conv(SMC, l, ib.A2, k.b, k.b, P(c, b1 + 9), net.nin(k.a, k.b) ? ib.S : ib.xr, out);
  }

  void level(int l) {
    const LevelBufs& B = net.b[l];
    const ILevel& I = IL.lv[l];
    const bool deepest = l + 1 == net.L;
    for (int r = 0; r < net.reps; ++r)
      block(l, B.pre[r], I.pre[r],
            r + 1 < net.reps ? input_of(l, B.pre[r + 1], I.pre[r + 1]) : deepest ? level_output(l) : join_half(l, true));
    MARK("pre blocks (infer)", l);
    if (deepest) return;
    const int p = net.planes(l), q = net.planes(l + 1);
    conv(DOWN, l, I.B, p, q, P(c, B.dn + 4), nullptr, input_of(l + 1, net.b[l + 1].pre[0], IL.lv[l + 1].pre[0]));
    level(l + 1);
    conv(UP, l, I.E, q, p, P(c, B.up + 4), nullptr, join_half(l, false));
    for (int r = 0; r < net.reps; ++r)
      block(l, B.post[r], I.post[r], r + 1 < net.reps ? input_of(l, B.post[r + 1], I.post[r + 1]) : level_output(l));
    MARK("post blocks (infer)", l);
  }
};

}  // namespace

extern "C" {

// level_desc: MM3D_LEVEL_DESC_WORDS int64 per level = {n rows, nbr table ptr, table stride, parent ptr, off ptr,
// child ptr, plan of the 3^3 table, plan of the child table, plan of the (parent, off) table, plan capacity}
MM3D_API int64_t mm3d_unet_topo_num_params(int num_planes, int block_reps, int residual) {
  Net net;
  if (fill_net(net, 1, 1, num_planes, block_reps, residual, MM3D_MODE_FP32, nullptr, 0)) return -1;
  lay_out(net, nullptr, nullptr, nullptr);
  return net.n_params;
}
MM3D_API int64_t mm3d_unet_num_params(int num_planes) { return mm3d_unet_topo_num_params(num_planes, 1, 0); }

MM3D_API size_t mm3d_unet_topo_act_bytes_grouped(int in_channels, int m, int num_planes, int block_reps, int residual,
                                                 int mode, const int64_t* level_desc, int64_t n_points, int groups) {
  Net net;
  const mm3d_unet_groups g{groups, nullptr};
  if (!level_desc || fill_net(net, in_channels, m, num_planes, block_reps, residual, mode, level_desc, n_points, 0, &g)) return 0;
  return lay_out(net, nullptr, nullptr, nullptr).act + 256;
}
MM3D_API size_t mm3d_unet_topo_act_bytes(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                         const int64_t* level_desc, int64_t n_points) {
  return mm3d_unet_topo_act_bytes_grouped(in_channels, m, num_planes, block_reps, residual, mode, level_desc, n_points, 1);
}
MM3D_API size_t mm3d_unet_act_bytes(int in_channels, int m, int num_planes, int mode, const int64_t* level_desc,
                                    int64_t n_points) {
  return mm3d_unet_topo_act_bytes(in_channels, m, num_planes, 1, 0, mode, level_desc, n_points);
}

MM3D_API size_t mm3d_unet_topo_bwd_bytes(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                         const int64_t* level_desc, int64_t n_points) {
  Net net;
  if (!level_desc || fill_net(net, in_channels, m, num_planes, block_reps, residual, mode, level_desc, n_points)) return 0;
  return lay_out(net, nullptr, nullptr, nullptr).tmp;
}
MM3D_API size_t mm3d_unet_bwd_bytes(int in_channels, int m, int num_planes, int mode, const int64_t* level_desc,
                                    int64_t n_points) {
  return mm3d_unet_topo_bwd_bytes(in_channels, m, num_planes, 1, 0, mode, level_desc, n_points);
}

MM3D_API size_t mm3d_unet_topo_scratch_bytes_grouped(int in_channels, int m, int num_planes, int block_reps, int residual,
                                                     int mode, int flags, int groups) {
  Net net;
  const mm3d_unet_groups g{groups, nullptr};
  if (fill_net(net, in_channels, m, num_planes, block_reps, residual, mode, nullptr, 0, flags, &g)) return 0;
  return lay_out(net, nullptr, nullptr, nullptr).scratch;  // (independent of the row counts)
}
MM3D_API size_t mm3d_unet_topo_scratch_bytes_ex(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                               int flags) {
  return mm3d_unet_topo_scratch_bytes_grouped(in_channels, m, num_planes, block_reps, residual, mode, flags, 1);
}
MM3D_API size_t mm3d_unet_topo_scratch_bytes(int in_channels, int m, int num_planes, int block_reps, int residual, int mode) {
  return mm3d_unet_topo_scratch_bytes_ex(in_channels, m, num_planes, block_reps, residual, mode, 0);
}
MM3D_API size_t mm3d_unet_scratch_bytes(int in_channels, int m, int num_planes, int mode) {
  return mm3d_unet_topo_scratch_bytes(in_channels, m, num_planes, 1, 0, mode);
}

MM3D_API int mm3d_unet_topo_forward_grouped(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                            int training, float eps, float momentum, const int64_t* level_desc,
                                            int64_t n_points, const int32_t* p2v, const int32_t* npts,
                                            const int32_t* vox_start, const int32_t* vox_pts, const float* feats, float* out,
                                            void* const* params, void* act, size_t act_bytes, void* scratch,
                                            size_t scratch_bytes, const mm3d_unet_mask* mask, mm3d_stream_t stream_, int flags,
                                            const mm3d_unet_groups* groups) {
  MM3D_REQUIRE(!groups || groups->groups == 1 || groups->bounds, MM3D_ERR_INVALID, "unet forward: groups without boundaries");
  MM3D_REQUIRE(level_desc, MM3D_ERR_INVALID, "unet forward: no level descriptors");
  MM3D_REQUIRE(!mask || (mask->wb && (n_points == 0 || mask->s)), MM3D_ERR_INVALID, "unet forward: incomplete mask descriptor");
  MM3D_REQUIRE(!(flags & MM3D_DETERMINISTIC) || (vox_start && vox_pts), MM3D_ERR_INVALID,
               "unet forward: the deterministic mode needs the voxels' point lists (mm3d_point_csr)");
  Net net;
  int rc = fill_net(net, in_channels, m, num_planes, block_reps, residual, mode, level_desc, n_points, flags, groups);
  if (rc) return rc;
  const Sizes need = lay_out(net, act, nullptr, scratch);  // (no backward temporaries)
  MM3D_REQUIRE(act_bytes >= need.act, MM3D_ERR_WORKSPACE, "activation workspace too small: need %zu have %zu", need.act, act_bytes);
  MM3D_REQUIRE(scratch_bytes >= need.scratch, MM3D_ERR_WORKSPACE, "unet scratch too small: need %zu have %zu", need.scratch,
               scratch_bytes);
  Ctx c{&net, params, nullptr, (cudaStream_t)stream_, eps, momentum, training, 0};
  MM3D_CUDA(cudaMemsetAsync(net.bn_ws, 0, net.bn_ws_bytes, c.stream));
  const int64_t n0 = net.lv[0].n;
  MARK("fwd start", -1);
  const float* w_stem = input_stage(c, n_points, p2v, npts, vox_start, vox_pts, feats, mask);
  EX(build_images(c, false, w_stem));
  build_identity_plans(c);  // (kept in `act`: the backward reuses them)
  MARK("pad + weight images", -1);
  conv_fwd(c, SMC, 0, net.Vp, net.cin_k, net.b[0].X, m, w_stem);
  MARK("stem fwd", -1);
  level_fwd(c, 0);
  bn_fwd(c, net.head, 0, net.b[0].R, net.Z, n0, m, net.s_head, nullptr, 0, /*to_conv=*/false);
  MARK("bn_fwd head", -1);
  EX(mm3d_output_fwd(net.Z, p2v, n_points, m, out, c.stream));
  MARK("output_fwd", -1);
  return c.rc;
}

MM3D_API int mm3d_unet_topo_forward_ex(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                       int training, float eps, float momentum, const int64_t* level_desc, int64_t n_points,
                                       const int32_t* p2v, const int32_t* npts, const int32_t* vox_start,
                                       const int32_t* vox_pts, const float* feats, float* out, void* const* params, void* act,
                                       size_t act_bytes, void* scratch, size_t scratch_bytes, const mm3d_unet_mask* mask,
                                       mm3d_stream_t stream_, int flags) {
  return mm3d_unet_topo_forward_grouped(in_channels, m, num_planes, block_reps, residual, mode, training, eps, momentum,
                                        level_desc, n_points, p2v, npts, vox_start, vox_pts, feats, out, params, act,
                                        act_bytes, scratch, scratch_bytes, mask, stream_, flags, nullptr);
}

MM3D_API int mm3d_unet_topo_forward(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                    int training, float eps, float momentum, const int64_t* level_desc, int64_t n_points,
                                    const int32_t* p2v, const int32_t* npts, const float* feats, float* out,
                                    void* const* params, void* act, size_t act_bytes, void* scratch, size_t scratch_bytes,
                                    const mm3d_unet_mask* mask, mm3d_stream_t stream_) {
  return mm3d_unet_topo_forward_ex(in_channels, m, num_planes, block_reps, residual, mode, training, eps, momentum, level_desc,
                                   n_points, p2v, npts, nullptr, nullptr, feats, out, params, act, act_bytes, scratch,
                                   scratch_bytes, mask, stream_, 0);
}

MM3D_API int mm3d_unet_forward(int in_channels, int m, int num_planes, int mode, int training, float eps, float momentum,
                               const int64_t* level_desc, int64_t n_points, const int32_t* p2v, const int32_t* npts,
                               const float* feats, float* out, void* const* params, void* act, size_t act_bytes,
                               void* scratch, size_t scratch_bytes, const mm3d_unet_mask* mask, mm3d_stream_t stream_) {
  return mm3d_unet_topo_forward(in_channels, m, num_planes, 1, 0, mode, training, eps, momentum, level_desc, n_points, p2v,
                                npts, feats, out, params, act, act_bytes, scratch, scratch_bytes, mask, stream_);
}

// grads: same slot order as params (running-stat slots ignored); d_feats may be NULL.
MM3D_API int mm3d_unet_topo_backward_grouped(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                             int training, const int64_t* level_desc, int64_t n_points, const int32_t* p2v,
                                             const int32_t* npts, const int32_t* vox_start, const int32_t* vox_pts,
                                             const float* d_out, float* d_feats, void* const* params, void* const* grads,
                                             void* act, size_t act_bytes, void* tmp, size_t tmp_bytes, void* scratch,
                                             size_t scratch_bytes, const mm3d_unet_mask* mask, mm3d_stream_t stream_,
                                             int flags, const mm3d_unet_groups* groups) {
  MM3D_REQUIRE(!groups || groups->groups == 1 || groups->bounds, MM3D_ERR_INVALID, "unet backward: groups without boundaries");
  MM3D_REQUIRE(level_desc, MM3D_ERR_INVALID, "unet backward: no level descriptors");
  MM3D_REQUIRE(!mask || (mask->wb && mask->d_wb && mask->ws && (n_points == 0 || (mask->s && mask->feats))), MM3D_ERR_INVALID,
               "unet backward: incomplete mask descriptor");
  MM3D_REQUIRE(!(flags & MM3D_DETERMINISTIC) || (vox_start && vox_pts), MM3D_ERR_INVALID,
               "unet backward: the deterministic mode needs the voxels' point lists (mm3d_point_csr)");
  MM3D_REQUIRE(!(flags & MM3D_DETERMINISTIC) || !mask || mask->ws_bytes >= sizeof(double) * MM3D_DET_CTAS * (in_channels + 1),
               MM3D_ERR_WORKSPACE, "unet backward: the deterministic mode's mask workspace needs %d doubles",
               MM3D_DET_CTAS * (in_channels + 1));
  Net net;
  int rc = fill_net(net, in_channels, m, num_planes, block_reps, residual, mode, level_desc, n_points, flags, groups);
  if (rc) return rc;
  const Sizes need = lay_out(net, act, tmp, scratch);
  MM3D_REQUIRE(act_bytes >= need.act, MM3D_ERR_WORKSPACE, "activation workspace too small: need %zu have %zu", need.act, act_bytes);
  MM3D_REQUIRE(tmp_bytes >= need.tmp, MM3D_ERR_WORKSPACE, "backward workspace too small: need %zu have %zu", need.tmp, tmp_bytes);
  MM3D_REQUIRE(scratch_bytes >= need.scratch, MM3D_ERR_WORKSPACE, "unet scratch too small: need %zu have %zu", need.scratch,
               scratch_bytes);
  Ctx c{&net, params, grads, (cudaStream_t)stream_, 0.f, 0.f, training, 0};
  c.side = getenv("MM3D_NO_SIDE_STREAM") ? nullptr : side_stream();
  MM3D_CUDA(cudaMemsetAsync(net.bn_ws, 0, net.bn_ws_bytes, c.stream));
  const int64_t n0 = net.lv[0].n;
  {  // One memset instead of one per layer when the gradient buffers are one contiguous block (the shipped host
     // code hands out views of one flat tensor): slot sizes follow from the network shape.
    const char *lo = nullptr, *hi = nullptr;
    size_t bytes = 0;
    bool all = true;
    for (const ConvInfo& x : net.convs) {
      const char* g0 = (const char*)grads[x.pidx];
      if (!g0) { all = false; break; }
      const size_t nb_ = sizeof(float) * (size_t)x.K * (x.pidx ? x.c_in : net.cin) * x.c_out;  // (the stem: real channels)
      if (!lo || g0 < lo) lo = g0;
      if (!hi || g0 + nb_ > hi) hi = g0 + nb_;
      bytes += nb_;
    }
    // BatchNorm gradients (2 * channels each) may sit in between: allow the span to be at most their size larger
    const size_t bn_bytes = sizeof(float) * 2 * net.bn_channels;
    if (all && lo && (size_t)(hi - lo) <= bytes + bn_bytes) {
      MM3D_CUDA(cudaMemsetAsync((void*)lo, 0, (size_t)(hi - lo), c.stream));
      c.grad_lo = lo; c.grad_hi = hi; c.wgrad_acc = 1;
    }
  }
  {  // stem weight as the kernels see it (zero-padded input channels), then every layer's dgrad weight image
    const float* w_stem_k = P(c, 0);
    if (net.cin_k != net.cin) {
      launch_pad_cols(c, w_stem_k, 27, net.cin * m, net.wp, net.cin_k * m);
      w_stem_k = net.wp;
    }
    EX(build_images(c, true, w_stem_k));
  }
  MARK("bwd start (memset, images)", -1);
  if (net.det())
    EX(mm3d_output_bwd_csr(d_out, vox_start, vox_pts, n0, m, net.d_Z, c.stream));
  else
    EX(mm3d_output_bwd(d_out, p2v, n_points, n0, m, net.d_Z, c.stream));
  MARK("output_bwd", -1);
  bn_bwd(c, net.head, 0, net.b[0].R, net.d_Z, net.d_R0, n0, m, net.s_head, 1);
  MARK("bn_bwd head", -1);
  level_bwd(c, 0, net.d_R0);
  // stem
  const float* w_stem = P(c, 0);
  float* d_w = Gp(c, 0);
  const bool need_dv = d_feats || mask;  // (the mask parameters get their gradient through the InputLayer)
  float* d_Vp = need_dv ? net.d_Vp : nullptr;
  auto input_bwd = [&](const float* d_v) {
    if (mask)
      EX(mm3d_input_masked_bwd_ex(d_v, mask->feats, mask->s, p2v, npts, n_points, net.cin, 4, mask->wb, d_feats, mask->d_wb,
                                  mask->ws, mask->ws_bytes, c.stream, net.flags));
    else
      EX(mm3d_input_bwd(d_v, p2v, npts, n_points, net.cin, 4, d_feats, c.stream));
  };
  if (net.cin_k != net.cin) {
    // (net.wp: padded at the start of this call; frozen stem weight: no gradient)
    conv_bwd(c, SMC, 0, net.Vp, net.cin_k, net.d_X0, m, net.wp, d_Vp, d_w ? net.d_wp : nullptr);
    join_side(c);  // d_wp comes from the side stream
    if (d_w) launch_pad_cols(c, net.d_wp, 27, net.cin_k * m, d_w, net.cin * m);  // slice the real channels back out
    if (need_dv) {
      launch_pad_cols(c, d_Vp, n0, net.cin_k, net.d_V, net.cin);
      input_bwd(net.d_V);
    }
  } else {
    conv_bwd(c, SMC, 0, net.Vp, net.cin, net.d_X0, m, w_stem, d_Vp, d_w);
    if (need_dv) input_bwd(d_Vp);
  }
  MARK("stem bwd + input_bwd", -1);
  join_side(c);  // everything after this call on `stream` sees the weight gradients
  MARK("join wgrad stream", -1);
  return c.rc;
}

MM3D_API int mm3d_unet_topo_backward_ex(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                        int training, const int64_t* level_desc, int64_t n_points, const int32_t* p2v,
                                        const int32_t* npts, const int32_t* vox_start, const int32_t* vox_pts,
                                        const float* d_out, float* d_feats, void* const* params, void* const* grads, void* act,
                                        size_t act_bytes, void* tmp, size_t tmp_bytes, void* scratch, size_t scratch_bytes,
                                        const mm3d_unet_mask* mask, mm3d_stream_t stream_, int flags) {
  return mm3d_unet_topo_backward_grouped(in_channels, m, num_planes, block_reps, residual, mode, training, level_desc,
                                         n_points, p2v, npts, vox_start, vox_pts, d_out, d_feats, params, grads, act,
                                         act_bytes, tmp, tmp_bytes, scratch, scratch_bytes, mask, stream_, flags, nullptr);
}

MM3D_API size_t mm3d_unet_topo_infer_bytes(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                           const int64_t* level_desc, int64_t n_points, int flags) {
  Net net;
  InferLayout IL;
  if (!level_desc || fill_net(net, in_channels, m, num_planes, block_reps, residual, mode, level_desc, n_points, flags)) return 0;
  return infer_layout(net, IL, nullptr);
}

MM3D_API int mm3d_unet_topo_infer(int in_channels, int m, int num_planes, int block_reps, int residual, int mode, float eps,
                                  const int64_t* level_desc, int64_t n_points, const int32_t* p2v, const int32_t* npts,
                                  const int32_t* vox_start, const int32_t* vox_pts, const float* feats, float* out,
                                  void* const* params, void* ws, size_t ws_bytes, const mm3d_unet_mask* mask,
                                  mm3d_stream_t stream_, int flags) {
  MM3D_REQUIRE(level_desc, MM3D_ERR_INVALID, "unet infer: no level descriptors");
  MM3D_REQUIRE(!mask || (mask->wb && (n_points == 0 || mask->s)), MM3D_ERR_INVALID, "unet infer: incomplete mask descriptor");
  MM3D_REQUIRE(!(flags & MM3D_DETERMINISTIC) || (vox_start && vox_pts), MM3D_ERR_INVALID,
               "unet infer: the deterministic mode needs the voxels' point lists (mm3d_point_csr)");
  Net net;
  int rc = fill_net(net, in_channels, m, num_planes, block_reps, residual, mode, level_desc, n_points, flags);
  if (rc) return rc;
  InferLayout IL;
  const size_t need = infer_layout(net, IL, ws);
  MM3D_REQUIRE(ws && ws_bytes >= need, MM3D_ERR_WORKSPACE, "inference workspace too small: need %zu have %zu", need, ws_bytes);
  Ctx c{&net, params, nullptr, (cudaStream_t)stream_, eps, 0.f, 0, 0};
  MARK("infer start", -1);
  const float* w_stem = input_stage(c, n_points, p2v, npts, vox_start, vox_pts, feats, mask);
  EX(build_images(c, false, w_stem));
  build_identity_plans(c);
  bn_scales(c, IL);
  MARK("pad + weight images + BatchNorm scales", -1);
  Infer f{c, IL, net};
  f.conv(SMC, 0, net.Vp, net.cin_k, m, w_stem, nullptr, f.input_of(0, net.b[0].pre[0], IL.lv[0].pre[0]));
  MARK("stem (infer)", -1);
  f.level(0);
  EX(mm3d_output_fwd(net.Z, p2v, n_points, m, out, c.stream));
  MARK("output_fwd", -1);
  return c.rc;
}

MM3D_API int mm3d_unet_topo_backward(int in_channels, int m, int num_planes, int block_reps, int residual, int mode,
                                     int training, const int64_t* level_desc, int64_t n_points, const int32_t* p2v,
                                     const int32_t* npts, const float* d_out, float* d_feats, void* const* params,
                                     void* const* grads, void* act, size_t act_bytes, void* tmp, size_t tmp_bytes,
                                     void* scratch, size_t scratch_bytes, const mm3d_unet_mask* mask,
                                     mm3d_stream_t stream_) {
  return mm3d_unet_topo_backward_ex(in_channels, m, num_planes, block_reps, residual, mode, training, level_desc, n_points,
                                    p2v, npts, nullptr, nullptr, d_out, d_feats, params, grads, act, act_bytes, tmp,
                                    tmp_bytes, scratch, scratch_bytes, mask, stream_, 0);
}

MM3D_API int mm3d_unet_backward(int in_channels, int m, int num_planes, int mode, int training,
                                const int64_t* level_desc, int64_t n_points, const int32_t* p2v, const int32_t* npts,
                                const float* d_out, float* d_feats, void* const* params, void* const* grads,
                                void* act, size_t act_bytes, void* tmp, size_t tmp_bytes, void* scratch,
                                size_t scratch_bytes, const mm3d_unet_mask* mask, mm3d_stream_t stream_) {
  return mm3d_unet_topo_backward(in_channels, m, num_planes, 1, 0, mode, training, level_desc, n_points, p2v, npts, d_out,
                                 d_feats, params, grads, act, act_bytes, tmp, tmp_bytes, scratch, scratch_bytes, mask,
                                 stream_);
}

// out[i] = in[i] rounded to TF32 (round-to-nearest, ties away); in == out allowed.  The module-by-module path uses
// it on the operands of a TF32 convolution; the executor's producers round in place of it.
MM3D_API int mm3d_round_tf32(const float* in, float* out, int64_t n, mm3d_stream_t stream_) {
  MM3D_REQUIRE(n >= 0 && (n == 0 || (in && out)), MM3D_ERR_INVALID, "round_tf32: bad arguments");
  MM3D_REQUIRE((((uintptr_t)in | (uintptr_t)out) & 15) == 0, MM3D_ERR_INVALID, "round_tf32: pointers must be 16-byte aligned");
  if (n == 0) return MM3D_OK;
  MM3D_CUDA(mm3d_launch_pdl(k_round_tf32, dim3(mm3d_grid(n / 4 + 1, 256)), dim3(256), 0, (cudaStream_t)stream_, in, out, n));
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_round_tf32");
  return MM3D_OK;
}

#ifdef MM3D_TRACE
MM3D_API void mm3d_debug_marks(int on) {
  for (Mark& m : g_marks) cudaEventDestroy(m.ev);
  g_marks.clear();
  g_marks_on = on != 0;
}
MM3D_API void mm3d_debug_dump_marks(void) {
  cudaDeviceSynchronize();
  float total = 0.f;
  for (size_t i = 1; i < g_marks.size(); ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, g_marks[i - 1].ev, g_marks[i].ev);
    total += ms;
    fprintf(stderr, "MARK %-28s L%-2d %8.1f us   (t = %8.1f)\n", g_marks[i].name, g_marks[i].level, ms * 1e3f, total * 1e3f);
  }
}
#endif

// out[0..n) = tf32(in) as float32; behind it, at float index n, bf16(in) as n BF16 elements: the operand planes of
// MM3D_MODE_BF16 (`out` holds 2 n floats like the TF32x3 planes; the BF16 plane fills the first half of the second one)
MM3D_API int mm3d_split_bf16(const float* in, float* out, int64_t n, mm3d_stream_t stream_) {
  MM3D_REQUIRE(n >= 0 && (n == 0 || (in && out)), MM3D_ERR_INVALID, "split_bf16: bad arguments");
  if (n == 0) return MM3D_OK;
  MM3D_CUDA(mm3d_launch_pdl(k_pad_cols, dim3(mm3d_grid(n, 256)), dim3(256), 0, (cudaStream_t)stream_, in, n, 1, out, 1, 3));
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_split_bf16");
  return MM3D_OK;
}

// out[0..n) = tf32(in), out[n..2n) = tf32(in - tf32(in)): the operand planes of MM3D_MODE_TF32X3
MM3D_API int mm3d_split_tf32(const float* in, float* out, int64_t n, mm3d_stream_t stream_) {
  MM3D_REQUIRE(n >= 0 && (n == 0 || (in && out)), MM3D_ERR_INVALID, "split_tf32: bad arguments");
  if (n == 0) return MM3D_OK;
  // (k_pad_cols with equal widths: a copy that writes the rounded value and the lo plane `n` floats behind it)
  MM3D_CUDA(mm3d_launch_pdl(k_pad_cols, dim3(mm3d_grid(n, 256)), dim3(256), 0, (cudaStream_t)stream_, in, n, 1, out, 1, 2));
  mm3d_count_launches(1);
  MM3D_CHECK_LAUNCH("mm3d_split_tf32");
  return MM3D_OK;
}

}  // extern "C"
