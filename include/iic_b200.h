/* iic_b200 -- C-ABI of the B200-native (sm_100a) IIC training hot path.
 *
 * This is the drop-in boundary for the hot path of xu-ji/IIC (SURVEY.md S8b).  The
 * reference has no FFI -- its "API" is a set of plain Python call signatures -- so
 * each entry point below cites the reference function (file:line under the
 * reference tree) whose device work it replaces.  The Python host side
 * (iic_b200/) mirrors those signatures and calls these symbols through ctypes.
 *
 * Conventions
 *   - plain pointers / ints / floats only; no torch types; all pointers are DEVICE
 *     pointers unless a name ends in _host.  The library never allocates
 *     caller-visible memory: outputs and workspaces are caller-allocated.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream); all
 *     work is enqueued asynchronously on it; no entry point synchronises the host.
 *   - return value: 0 on success, negative IIC_ERR_* otherwise; iic_last_error()
 *     returns a thread-local human-readable message.  Nothing throws.
 *   - activation tensors inside the network are NHWC ("pixel rows x channels",
 *     row-major [M = n*h*w][C]) in one of two storage dtypes:
 *       IIC_F32  (fp32 storage, fp32 SIMT convolutions  -- reference-precision mode)
 *       IIC_BF16 (bf16 storage, tcgen05 bf16 MMA with fp32 TMEM accumulation)
 *     The convolution entry points (iic_conv_fprop / _dgrad / _wgrad / _wgrad_workspace) additionally accept two
 *     COMPUTE modes on IIC_F32 storage (every tensor is fp32, weights packed with dst_dtype IIC_F32):
 *       IIC_TF32   tcgen05 kind::tf32 (10-bit mantissa operands, fp32 TMEM accumulation)
 *       IIC_TF32X3 the same tensor-core kernel with each operand split hi + lo in shared memory and three MMAs
 *                  per product (3xTF32): fp32-grade results (what `north_star` calls "a stated fp32 tolerance":
 *                  1e-5 relative per convolution) at ~10x the SIMT kernel's rate.
 *     Parameters, BN statistics, the heads and every loss are fp32 in all modes.
 *   - entry points are re-entrant; the only global state is a per-device cache of
 *     device properties.
 */
#ifndef IIC_B200_H_
#define IIC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IIC_OK 0
#define IIC_ERR_BAD_ARG (-1)
#define IIC_ERR_UNSUPPORTED (-2)
#define IIC_ERR_CUDA (-3)

#define IIC_F32 0
#define IIC_BF16 1
#define IIC_TF32 2   /* conv entry points only: fp32 storage, tcgen05 kind::tf32               */
#define IIC_TF32X3 3 /* conv entry points only: fp32 storage, error-compensated 3xTF32 split   */

/* phases of the joint/MI kernels (multi-GPU splits at the all-reduce of the joint) */
#define IIC_PHASE_FUSED 0    /* partial joint -> reduce -> MI -> gradients, one launch      */
#define IIC_PHASE_PARTIAL 1  /* write this rank's un-normalised joint to joint_ws and stop  */
#define IIC_PHASE_FINISH 2   /* joint_ws holds the (all-reduced) joint: MI + local gradients */

int iic_abi_version(void);
const char* iic_last_error(void);
/* number of kernels launched by this library (all host threads of the process: autograd runs backward on its own
 * threads) since the last reset */
long long iic_launch_count(int reset);
/* Kernel-variant switches of this sm_100a code base (A/B measurement and tests; not backends).  Defaults come from
 * the environment variable in brackets.  iic_set_option returns the previous value (>= 0) or IIC_ERR_BAD_ARG.
 *   "conv_halo"       [IIC_CONV_HALO=1]        halo kernel for 3x3/s1/p1 64->64 fprop+dgrad: 0 never, 1 when it pays,
 *                                              2 whenever the geometry fits
 *   "conv_halo_wgrad" [IIC_CONV_HALO_WGRAD=1]  halo kernel for the wgrad of the same layers (0 = im2col split-K kernel)
 *   "stem_quad"       [IIC_STEM_QUAD=2]        stem conv: 4 pixels x 16 channels per thread (and the fused-statistics
 *                                              entry point): 2 = channel-interleaved lanes (whole-sector stores),
 *                                              1 = 16 consecutive channels per thread; 0 = one pixel per thread
 *   "dgrad_prefetch"  [IIC_DGRAD_PREFETCH=1]   dgrad epilogues fetch the residual-gradient addend ahead of its use
 *   "bn_bwd_ctas"     [IIC_BN_BWD_CTAS=2]      CTAs per SM of the cooperative BatchNorm backward (1 = fits beside a resident conv CTA)
 *   "tc2_mt2"         [IIC_TC2_MT2=1]          128-channel fprop/dgrad: two 128-row tiles per weight k-block (0 = one)
 *   "conv_halo_store" [IIC_CONV_HALO_STORE=1]  halo fprop/dgrad: output tile staged in shared memory, one TMA store per
 *                                              work item (0 = per-thread 16-byte global stores)
 *   "stem_bwd_v2"     [IIC_STEM_BWD_V2=0]      iic_stem_bwd_fused: second version of the wgrad pass (not yet run on
 *                                              hardware)
 *   "conv_halo_stats" [IIC_CONV_HALO_STATS=1]  halo fprop: per-lane running BatchNorm sums, one warp reduction per CTA
 *                                              (not yet run on hardware)                                            */
int iic_get_option(const char* name);
int iic_set_option(const char* name, int value);

/* ---- a7/a8: clustering objective -- code/utils/cluster/IID_losses.py:6-33 (IID_loss) and
 *      :36-47 (compute_joint).
 * z, zt: [S][n][k] fp32 softmax outputs of the two views (S sub-heads, contiguous).
 * loss:  [S][2]  (loss, loss_no_lamb)                     (written unless phase==PARTIAL)
 * dz,dzt:[S][n][k] d loss / d z, d loss / d zt  (either may be NULL: no-grad callers,
 *        cluster_eval.py:281-288)
 * joint_ws: [S][k][k] fp32.  PARTIAL: out (raw sum_n z z'^T of this rank).  FINISH: in.
 *        FUSED: may be NULL.
 * joint_out: optional [S][k][k]; receives the symmetrised, normalised P (compute_joint).
 * eps: the reference passes sys.float_info.epsilon (a double); it is applied in fp32
 *      exactly as torch does when comparing / assigning into an fp32 tensor.            */
int iic_iid_loss(const float* z, const float* zt, int S, int n, int k, float lamb, double eps,
                 float* loss, float* dz, float* dzt, float* joint_ws, float* joint_out, int phase,
                 void* stream);

/* MI + analytic gradient from given (already reduced) joint matrices: the FINISH half of iic_iid_loss
 * without rows.  joint [S][k][k] raw (un-normalised) -> loss [S][2]; h_out (optional) [S][k][k] =
 * d loss / d joint.  detached_norm != 0: the normaliser carries no gradient (collapsed segmentation
 * loss, code/utils/segmentation/IID_losses.py:60).  Used with S = (2T+1)^2 for the uncollapsed loss. */
int iic_joint_mi(const float* joint, int S, int k, float lamb, double eps, int detached_norm, float* loss,
                 float* h_out, void* stream);

/* ---- a9-a11: segmentation objective -- code/utils/segmentation/IID_losses.py:14-159 and
 *      perform_affine_tf, code/utils/segmentation/transforms.py:131-143.
 * Pixel-major work layout: [n][h][w][KP] fp32 with KP = iic_seg_kp(k) (k rounded up to 4/8/16/32/48,
 * zero padded).
 *   iic_seg_prepare   x1m = x1*mask ; x2m = grid_sample(x2, affine_grid(theta))*mask
 *                     (bilinear, zeros padding, align_corners=True = torch-0.4.1 semantics);
 *                     x1,x2 NCHW (n,k,h,w); theta (n,2,3); mask (n,h,w).
 *   iic_seg_joint     joint[(2T+1)^2][k][k] : A[u][v][c][c'] = sum x1m[n,y+u-T,x+v-T,c]*x2m[n,y,x,c']
 *                     (what F.conv2d(x1^T, weight=x2^T, padding=T) evaluates, :53/:125); T = 0 gives
 *                     the plain k x k outer-product sum.  workspace: iic_seg_joint_workspace bytes.
 *   iic_seg_corr_bwd  out[n,Y,X,c] = scale * sum_{u,v,c'} H[u][v][c][c'] * in[n,Y-sgn(u-T),X-sgn(v-T),c']
 *                     (sgn=+1, in=x2m -> d x1m ; sgn=-1, in=x1m -> d x2m ; H symmetric in c,c')
 *   iic_seg_unprepare dx1 = d x1m*mask, dx2 = bilinear adjoint of d x2m*mask, back to NCHW
 *   iic_box_filter    zero-padded (2T+1)^2 box sum (collapsed loss via SURVEY.md S8 a10 identity) */
int iic_seg_kp(int k);
int iic_seg_prepare(const float* x1, const float* x2, const float* theta, const float* mask, float* x1m, float* x2m,
                    int n, int k, int h, int w, void* stream);
int iic_seg_unprepare(const float* dx1m, const float* dx2m, const float* theta, const float* mask, float* dx1,
                      float* dx2, int n, int k, int h, int w, void* stream);
/* The same with the reference's sparse random displacement (random_translation_multiple, seg transforms.py:146-166,
 * called at seg IID_losses.py:29-32 / :101-104): the resampled x2 is read at (x + tx, y + ty), zero outside the frame
 * (the caller draws (tx, ty) from numpy's global RNG exactly as the reference does). */
int iic_seg_prepare_shift(const float* x1, const float* x2, const float* theta, const float* mask, float* x1m, float* x2m,
                          int n, int k, int h, int w, int tx, int ty, void* stream);
int iic_seg_unprepare_shift(const float* dx1m, const float* dx2m, const float* theta, const float* mask, float* dx1,
                            float* dx2, int n, int k, int h, int w, int tx, int ty, void* stream);
long long iic_seg_joint_workspace(int n, int k, int T);
int iic_seg_joint(const float* x1m, const float* x2m, float* joint, void* workspace, int n, int k, int h, int w,
                  int T, void* stream);
/* The same joint on the tensor cores (tcgen05 kind::tf32, 3xTF32 operand split -> fp32-grade sums), for pixel-major inputs
 * with KP = 16 (5 <= k <= 16) and 2T+1 <= 24: the Toeplitz operand of F.conv2d(x1^T, weight=x2^T, padding=T) (:125) is read
 * straight out of one shared-memory row per displacement row.  iic_seg_joint_tc_workspace returns 0 when the geometry is
 * not supported (the caller then uses iic_seg_joint), otherwise the bytes of `workspace`. */
long long iic_seg_joint_tc_workspace(int n, int k, int h, int w, int T);
int iic_seg_joint_tc(const float* x1m, const float* x2m, float* joint, void* workspace, int n, int k, int h, int w, int T,
                     void* stream);
/* iic_seg_corr_bwd on the tensor cores (kind::tf32, round-to-nearest operands, single pass: relative error ~3e-4 of the
 * gradient scale), KP = 16, w <= 128, 2T+1 a multiple of 7 (T = 3, 10).  _workspace returns 0 if unsupported. */
long long iic_seg_corr_tc_workspace(int n, int k, int h, int w, int T);
int iic_seg_corr_tc(const float* in, const float* H, float* out, void* workspace, int n, int k, int h, int w, int T, int sgn,
                    float scale, void* stream);
int iic_seg_corr_bwd(const float* in, const float* H, float* out, int n, int k, int h, int w, int T, int sgn,
                     float scale, void* stream);
int iic_box_filter(const float* in, float* tmp, float* out, int n, int k, int h, int w, int T, void* stream);

/* ---- a1: sobel_process -- code/utils/cluster/transforms.py:47-96.
 * imgs NCHW fp32 (n, c_in, h, w) -> out NCHW fp32 (n, c_out, h, w); channel rules of
 * :50-66,:84-94 selected by include_rgb / using_ir. */
int iic_sobel(const float* imgs, float* out, int n, int c_in, int h, int w, int include_rgb,
              int using_ir, void* stream);
/* Dataloader tail + sobel_process in one pass (SURVEY S8f row 2): rgb [n,3,h,w] (uint8 when src_is_u8, else fp32 in
 * [0,1]) -> grey as custom_greyscale_to_tensor computes it (code/utils/cluster/transforms.py:12-16; PIL's integer "L"
 * formula for uint8, 0.299/0.587/0.114 for fp32) -> out [n,2,h,w] = [dx, dy] (transforms.py:69,75). */
int iic_grey_sobel(const void* rgb, int src_is_u8, float* out, int n, int h, int w, void* stream);

/* ---- layout / dtype plumbing between the reference's NCHW fp32 tensors and the internal
 *      NHWC activations (no reference counterpart: torch does this implicitly). */
int iic_nchw_to_nhwc(const float* src, void* dst, int dst_dtype, int n, int c, int h, int w, void* stream);
int iic_nhwc_to_nchw(const void* src, int src_dtype, float* dst, int n, int c, int h, int w, void* stream);
int iic_cast(const void* src, int src_dtype, void* dst, int dst_dtype, long long count, void* stream);

/* ---- convolution geometry shared by the conv entry points (nn.Conv2d, bias=False:
 *      residual.py:4-7,:53-55, net5g.py:21-23, vgg.py:25-27, net10a.py:46-47). */
typedef struct {
  int n, h, w, cin;      /* input  NHWC */
  int oh, ow, cout;      /* output NHWC */
  int kh, kw, stride, pad, dil;
} iic_conv_geom;

/* weights are repacked from torch's [cout][cin][kh][kw] fp32:
 *   kind 0 (fprop/wgrad layout): [cout][kh][kw][cin]
 *   kind 1 (dgrad layout):       [cin][kh][kw][cout]
 * dst_dtype IIC_F32 / IIC_BF16 = the storage type of the network; IIC_TF32X3 = the form the 3xTF32 fprop / dgrad take:
 * fp32, TWO planes of cout*cin*kh*kw elements, [raw w | lo = w - (w truncated to tf32)] (the weights are split once per
 * step here instead of once per tile in the convolution; the tensor core ignores the 13 low mantissa bits of the raw plane). */
int iic_pack_weight(const float* w_oihw, void* dst, int dst_dtype, int kind, int cout, int cin, int kh,
                    int kw, void* stream);
/* Every convolution weight of a trunk repacked in ONE launch (the per-step repacking of ~70 small tensors was
 * launch-latency bound).  `jobs_device` is a DEVICE array; each job is one iic_pack_weight call (all weights must
 * have fewer than 2^31 elements). */
typedef struct iic_pack_job {
  const float* w; /* torch layout [cout][cin][kh][kw] fp32 */
  void* dst;      /* kind 0: [cout][kh][kw][cin], kind 1: [cin][kh][kw][cout], in dst_dtype */
  int kind, cout, cin, kh, kw, reserved;
} iic_pack_job;
int iic_pack_weights_batched(const iic_pack_job* jobs_device, int njobs, int dst_dtype, void* stream);
/* dw_packed fp32 [cout][kh][kw][cin] -> (accumulate ? += : =) torch-layout grad [cout][cin][kh][kw] */
int iic_unpack_wgrad(const float* dw_packed, float* grad_oihw, int accumulate, int cout, int cin, int kh,
                     int kw, void* stream);

/* fprop: y[M][cout] = conv(x, w).  dtype IIC_F32 -> SIMT fp32 kernel; IIC_BF16 -> tcgen05 kind::f16;
 * IIC_TF32 / IIC_TF32X3 -> tcgen05 kind::tf32 on fp32 tensors (cin % 32 == 0, cout % 64 == 0).
 * w is the kind-0 packed weight in the storage dtype (IIC_TF32X3: the two-plane form of iic_pack_weight).  y has the
 * storage dtype. */
int iic_conv_fprop(const void* x, const void* w_packed, void* y, const iic_conv_geom* g, int dtype,
                   void* stream);
/* fprop with the BatchNorm batch statistics of y fused into the epilogue (IIC_BF16 only; otherwise
 * IIC_ERR_UNSUPPORTED and the caller uses iic_conv_fprop + iic_bn_stats).  `views` = 1 or 2: the batch is the
 * concatenation of that many equally sized views whose statistics stay separate.  stat_partial receives
 * iic_conv_fprop_stats_blocks() rows of [2][2][cout] fp32 (per-CTA column sums / sums of squares of the fp32
 * accumulators; the row layout always has two view slots, the second is zero when views == 1);
 * iic_bn_stats_from_partials(…, views = 2 (row layout), view, …) folds them (fixed order) into scale/shift,
 * mean/invstd and the running statistics of one view. */
int iic_conv_fprop_stats_blocks(const iic_conv_geom* g, int dtype);
int iic_conv_fprop_stats(const void* x, const void* w_packed, void* y, const iic_conv_geom* g, int dtype, int views,
                         float* stat_partial, void* stream);
int iic_bn_stats_from_partials(const float* stat_partial, int nblk, int views, int view, long long M, int C,
                               const float* gamma, const float* beta, float eps, float momentum, float* running_mean,
                               float* running_var, double* stats_ws, float* scale_shift, float* mean_invstd,
                               void* stream);
/* All views in one launch: stat_partial rows hold `slots` (= 2) view slots of which the first `views` are
 * folded; scale_shift / mean_invstd are [views][2*C]; the running statistics are updated view after view. */
int iic_bn_stats_from_partials_views(const float* stat_partial, int nblk, int slots, int views, long long M_per_view,
                                     int C, const float* gamma, const float* beta, float eps, float momentum,
                                     float* running_mean, float* running_var, float* scale_shift, float* mean_invstd,
                                     void* stream);
/* dgrad: dx[n,h,w,cin] = conv_transpose(dy, w) (+ addend, same shape/dtype as dx, may be NULL).
 * w is the kind-1 packed weight. */
int iic_conv_dgrad(const void* dy, const void* w_packed_t, const void* addend, void* dx,
                   const iic_conv_geom* g, int dtype, void* stream);
/* Same with an addend that only passes where its mask bit is set (bf16, stride 1, cin % 64 == 0): dx = dgrad(dy) +
 * (bit ? addend : 0); addend_mask = [pixels][cin / 8] bytes, bit j of byte b = channel 8 b + j (the layout
 * iic_bn_apply_views_mask writes).  The residual gradient of a BasicBlock, d_out * (out > 0) (residual.py:41-43 under
 * autograd), is then never materialised. */
int iic_conv_dgrad_masked(const void* dy, const void* w_packed_t, const void* addend, const unsigned char* addend_mask,
                          void* dx, const iic_conv_geom* g, int dtype, void* stream);
/* wgrad: dw_packed fp32 [cout][kh][kw][cin] = sum over pixels.  workspace: fp32, at least
 * iic_conv_wgrad_workspace(g, dtype) bytes (split-K partials; deterministic reduction). */
long long iic_conv_wgrad_workspace(const iic_conv_geom* g, int dtype);
int iic_conv_wgrad(const void* x, const void* dy, float* dw_packed, void* workspace, const iic_conv_geom* g,
                   int dtype, void* stream);
/* wgrad written straight into the torch-layout gradient [cout][cin][kh][kw] (accumulate ? += : =), i.e. iic_conv_wgrad +
 * iic_unpack_wgrad in one call; on the IIC_BF16 path the split-K fold itself writes that layout (one launch and one pass
 * over the gradient less).  workspace: iic_conv_wgrad_oihw_workspace(g, dtype) bytes. */
long long iic_conv_wgrad_oihw_workspace(const iic_conv_geom* g, int dtype);
int iic_conv_wgrad_oihw(const void* x, const void* dy, float* grad_oihw, int accumulate, void* workspace,
                        const iic_conv_geom* g, int dtype, void* stream);

/* ---- stem: first conv of ClusterNet5g (net5g.py:21-23) / 6c (vgg.py) / 10a: tiny cin
 *      (1..5), read straight from the reference's NCHW fp32 input. Direct SIMT conv.
 *      w: torch layout [cout][cin][kh][kw] fp32.  y: NHWC `dtype`. */
int iic_stem_fprop(const float* x_nchw, const float* w_oihw, void* y, const iic_conv_geom* g, int dtype,
                   void* stream);
/* The same with the BatchNorm batch statistics of y accumulated in the kernel (fp32 results, before rounding to
 * the storage type), for `views` = 1 or 2 stacked batches.  stat_partial receives
 * iic_stem_fprop_stats_blocks() rows of [2 view slots][{sum, sum of squares}][64] -- the layout of
 * iic_conv_fprop_stats, folded by iic_bn_stats_from_partials(_views).  _blocks() returns 0 when the geometry is
 * not supported (needs cout 64, stride 1, dilation 1, 3x3 or 5x5, ow % 4 == 0): use iic_stem_fprop + iic_bn_stats. */
int iic_stem_fprop_stats_blocks(const iic_conv_geom* g, int dtype, int views);
int iic_stem_fprop_stats(const float* x_nchw, const float* w_oihw, void* y, const iic_conv_geom* g, int dtype, int views,
                         float* stat_partial, void* stream);
int iic_stem_wgrad(const float* x_nchw, const void* dy, float* grad_oihw, int accumulate, void* workspace,
                   long long workspace_bytes, const iic_conv_geom* g, int dtype, void* stream);
/* Stem wgrad on tcgen05 (bf16 dy; cin*kh*kw <= 64, cout = 64, stride 1, 'same' padding): the patches of the NCHW fp32 input
 * are gathered into shared memory as the K-major operand, dy arrives by TMA as the MN-major operand, one TMEM accumulator per
 * persistent CTA, per-CTA partials in `workspace` (iic_stem_wgrad_tc_workspace bytes) folded in a fixed order into the
 * torch-layout gradient [cout][cin][kh][kw] (same contract as iic_stem_wgrad: replaces autograd's conv2d weight gradient of
 * the first trunk convolution, net5g.py:21; the patches are rounded to bf16). */
long long iic_stem_wgrad_tc_workspace(const iic_conv_geom* g);
int iic_stem_wgrad_tc(const float* x_nchw, const void* dy_bf16, float* grad_oihw, int accumulate, void* workspace,
                      const iic_conv_geom* g, void* stream);
/* Stem convolution + BatchNorm statistics partials on tcgen05 (bf16 output; cin*kh*kw <= 32, cout = 64, stride 1, 'same'
 * padding; two views only if one view is a multiple of 128 pixels): same contract as iic_stem_fprop_stats (net5g.py:21-23,
 * the first trunk convolution and the batch statistics nn.BatchNorm2d takes of its result), with the input patches and the
 * weights rounded to bf16.  _blocks() = rows of stat_partial ([blocks][2 views][{sum, sum of squares}][64]), 0 if unsupported. */
int iic_stem_fprop_stats_tc_blocks(const iic_conv_geom* g, int views);
int iic_stem_fprop_stats_tc(const float* x_nchw, const float* w_oihw, void* y_bf16, const iic_conv_geom* g, int views,
                            float* stat_partial, void* stream);
/* Whole backward of the ClusterNet5g stem, conv3x3(cin 1|2 -> 64, pad 1) -> BatchNorm -> ReLU -> MaxPool(2, 2, pool_pad)
 * (net5g.py:21-26), in two passes over (y, dpool) instead of six over y-sized tensors: the pooled gradient is routed
 * and ReLU-masked on the fly, reduced for the BatchNorm backward, and the BatchNorm input gradient is consumed by the
 * weight gradient without being stored (the network input takes no gradient).
 *   x_nchw [n][cin][h][w] fp32; y [n][h][w][64] conv output and dpool [n][oh][ow][64] in `dtype`;
 *   ss, mi [views][2*64]: per-view BatchNorm scale/shift and mean/invstd of the forward pass; views = 1 or 2 stacked
 *   batches with their own statistics; dgamma/dbeta [64] and dw_oihw [64][cin][3][3] are written or accumulated.
 * _workspace() returns the scratch bytes needed, or 0 when the geometry is not supported (then use
 * iic_bn_relu_maxpool_bwd + iic_bn_bwd_fused + iic_stem_wgrad).                                                  */
long long iic_stem_bwd_fused_workspace(const iic_conv_geom* g, int pool_pad, int views, int dtype);
int iic_stem_bwd_fused(const float* x_nchw, const void* y, const void* dpool, const float* ss, const float* mi,
                       const float* gamma, float* dgamma, float* dbeta, int bn_accumulate, float* dw_oihw,
                       int w_accumulate, const iic_conv_geom* g, int pool_pad, int views, int dtype, void* workspace,
                       long long workspace_bytes, void* stream);
/* The first two thirds of the same backward: max-pool routing, ReLU and BatchNorm backward in two passes over (y, dpool),
 * writing dy (gradient of the conv output, storage type) for iic_stem_wgrad / iic_stem_wgrad_tc; the routed gradient and the
 * BatchNorm reduce sweep never touch memory.  Same geometry conditions and workspace as iic_stem_bwd_fused. */
int iic_stem_bwd_dy(const void* y, const void* dpool, const float* scale_shift, const float* mean_invstd, const float* gamma,
                    float* dgamma, float* dbeta, int bn_accumulate, void* dy_out, const iic_conv_geom* g, int pool_pad,
                    int views, int dtype, void* workspace, long long workspace_bytes, void* stream);

/* ---- BatchNorm2d, train mode (net5g.py:24, residual.py:20,23,56, vgg.py:28-29): statistics
 *      are per forward call over all M = n*h*w rows.
 * stats ws: double[2*C] (sum, sumsq), zeroed by the call.
 * scale_shift: float[2*C]  (gamma*invstd, beta - mean*gamma*invstd)
 * mean_invstd: float[2*C]  saved for backward
 * running_mean/var: updated in place with `momentum` (unbiased var) when non-NULL.
 * When `use_running` != 0 (eval mode) no statistics are computed: scale/shift come from the
 * running buffers. */
int iic_bn_stats(const void* y, int dtype, long long M, int C, const float* gamma, const float* beta,
                 float eps, float momentum, float* running_mean, float* running_var, int use_running,
                 double* stats_ws, float* scale_shift, float* mean_invstd, void* stream);
/* out = relu?( y*scale+shift  [+ res  | + res*rscale+rshift] ) */
int iic_bn_apply(const void* y, const float* scale_shift, const void* res, const float* res_scale_shift,
                 void* out, int dtype, long long M, int C, int relu, void* stream);
/* the same over `views` stacked batches of M_per_view rows; scale_shift / res_scale_shift are [views][2*C] */
int iic_bn_apply_views(const void* y, const float* scale_shift, const void* res, const float* res_scale_shift,
                       void* out, int dtype, long long M_per_view, int C, int relu, int views, void* stream);
/* fused BN + ReLU + MaxPool2d(k=2, s=2, pad) (net5g.py:24-26; vgg.py 'M'): y (n,h,w,C) -> out (n,oh,ow,C) */
int iic_bn_relu_maxpool(const void* y, const float* scale_shift, void* out, int dtype, int n, int h, int w,
                        int C, int pad, int oh, int ow, void* stream);
/* backward of the above: g (n,h,w,C) = dP routed to the arg-max, masked by ReLU, i.e. the
 * gradient w.r.t. the BN output. */
int iic_bn_relu_maxpool_bwd(const void* y, const float* scale_shift, const void* dpool, void* g, int dtype,
                            int n, int h, int w, int C, int pad, int oh, int ow, void* stream);
/* BN backward.  g_in = dL/d(out of the BN [+res] [relu]).  ReLU mask: (act > 0) if `act` != NULL (needed when a
 * residual was added before the ReLU); else (y*scale+shift > 0) recomputed from y if `mask_scale_shift` != NULL
 * (BN directly followed by ReLU: saves reading the activation); else no mask.  Pass 1 (reduce): sums[2*C] double (sum g, sum g*yhat),
 * zeroed by the call.  Pass 2 (apply): dy = scale*(g - mean(g) - yhat*mean(g*yhat)); also
 * writes dgamma/dbeta (accumulate ? += : =) and, if g_out != NULL, the masked g
 * (gradient for the residual branch). */
int iic_bn_bwd_reduce(const void* g_in, const void* act, const float* mask_scale_shift, const void* y,
                      const float* mean_invstd, int dtype, long long M, int C, double* sums, void* stream);
int iic_bn_bwd_apply(const void* g_in, const void* act, const float* mask_scale_shift, const void* y,
                     const float* mean_invstd, const float* gamma, const double* sums, void* dy, void* g_out,
                     float* dgamma, float* dbeta, int accumulate, int dtype, long long M, int C, void* stream);
/* The same backward for `views` (1 or 2) stacked batches of M_per_view rows, each with its own statistics, in ONE
 * cooperative launch: partial sums, grid barrier, fp64 fold, grid barrier, apply over the same rows in reverse
 * order (L2 reuse).  dgamma/dbeta receive the sum over the views (the two forward calls of
 * cluster_sobel_twohead.py:320-321 share the BatchNorm parameters). */
int iic_bn_bwd_fused(const void* g_in, const void* act, const void* y, int views, const float* mean_invstd0,
                     const float* mean_invstd1, const float* mask_scale_shift0, const float* mask_scale_shift1,
                     const float* gamma, void* dy, void* g_out, float* dgamma, float* dbeta, int accumulate, int dtype,
                     long long M_per_view, int C, void* stream);
/* The ReLU of a residual block's output (residual.py:40-41) as a 1-bit mask.  iic_bn_apply_views_mask =
 * iic_bn_apply_views with relu = 1 that also writes mask_out [views * M_per_view][C / 8] bytes (bit j of a byte = channel
 * 8*c8 + j of that row is > 0); iic_bn_bwd_fused_bits = iic_bn_bwd_fused taking that mask instead of re-reading the block
 * output twice (12.25 instead of 16 bytes per element for the BatchNorm backward of bn2). */
int iic_bn_apply_views_mask(const void* y, const float* scale_shift, const void* res, const float* res_scale_shift,
                            void* out, unsigned char* mask_out, int dtype, long long M_per_view, int C, int views,
                            void* stream);
int iic_bn_bwd_fused_bits(const void* g_in, const unsigned char* mask_bits, const void* y, int views,
                          const float* mean_invstd0, const float* mean_invstd1, const float* gamma, void* dy, void* g_out,
                          float* dgamma, float* dbeta, int accumulate, int dtype, long long M_per_view, int C,
                          void* stream);

/* ---- SURVEY S8(f) row 4: evaluation -- code/utils/cluster/cluster_eval.py:46-63 (torch.argmax per sub-head),
 *      code/utils/segmentation/segmentation_eval.py:100-110 (per-pixel argmax over channels) and the
 *      `int(((flat_preds == c1) * (flat_targets == c2)).sum())` double loops of code/utils/cluster/eval_metrics.py:9-53.
 * iic_argmax_rows      z [rows][k] fp32 -> out[rows] int32 (ties: lowest index; NaN counts as the maximum, like torch)
 * iic_argmax_channels  x [n][k][hw] fp32 (NCHW) -> out[n*hw] int32
 * iic_confusion_counts counts[s][p][t] (+)= #{i < n : preds[s][i] == p, targets[i] == t, mask[i] != 0}; preds [S][n],
 *                      targets [n] int32, mask [n] bytes or NULL, counts [S][preds_k][targets_k] int64; labels outside
 *                      the ranges are ignored (the reference's loops never see them either). */
int iic_argmax_rows(const float* z, long long rows, int k, int* out, void* stream);
int iic_argmax_channels(const float* x_nchw, int n, int k, long long hw, int* out, void* stream);
int iic_confusion_counts(const int* preds, const int* targets, const unsigned char* mask, int S, long long n, int preds_k,
                         int targets_k, long long* counts, int accumulate, void* stream);

/* AvgPool2d(full extent) + flatten (net5g.py:31-39,:56): x (n,hw,C) -> feat fp32 (n,C) */
int iic_avgpool(const void* x, int dtype, float* feat, int n, int hw, int C, void* stream);
int iic_avgpool_bwd(const float* dfeat, void* dx, int dtype, int n, int hw, int C, void* stream);

/* ---- a3: sub-heads -- net5g_two_head.py:22-36 / net6c_two_head.py:31-49:
 *      S x (Linear(F -> k) + Softmax(dim=1)) on the same feature.
 * feat [n][F] fp32; w [S*k][F] fp32 (the S Linear weights stacked); b [S*k];
 * logits_ws [n][S*k] fp32 workspace; z out [S][n][k]. */
int iic_heads_fwd(const float* feat, const float* w, const float* b, float* logits_ws, float* z, int n,
                  int F, int S, int k, void* stream);
/* dz [S][n][k] -> dlogits_ws [n][S*k]; dw [S*k][F], db [S*k] (overwritten), dfeat [n][F]
 * (overwritten; may be NULL). */
int iic_heads_bwd(const float* feat, const float* w, const float* z, const float* dz, float* dlogits_ws,
                  float* dw, float* db, float* dfeat, int n, int F, int S, int k, void* stream);

/* ---- a14: semi-supervised finetuning -- code/scripts/semisup/IID_semisup_STL10.py.
 * iic_cross_entropy  nn.CrossEntropyLoss() with mean reduction (the criterion of IID_semisup_STL10.py:201, applied at
 *                    :246) and its backward, in one launch.  logits [n][k] fp32, targets [n] int64 -> loss [1] fp32
 *                    = mean_i (logsumexp(logits_i) - logits_i[t_i]) (stable log-sum-exp, fp64 sum folded in a fixed
 *                    order: deterministic) and dlogits [n][k] = (softmax(logits) - onehot(t)) / n.  A target outside
 *                    [0, k) makes the loss (and that row of dlogits) NaN; the call neither traps nor synchronises.
 * iic_linear_fwd     nn.Linear: y [n][N] = x [n][K] w^T + b (w [N][K], b [N] or NULL), fp32 (the last Linear of
 *                    SupHead5, sup_head5.py:20, and the `semisup` head of ClusterNet5gTwoHead / ClusterNet6cTwoHead,
 *                    net5g_two_head.py:22-24, net6c_two_head.py:31-33).  No softmax.
 * iic_linear_bwd     its backward: dw [N][K], db [N] (may be NULL) written (accumulate = 0) or added to (accumulate != 0);
 *                    dx [n][K] overwritten when not NULL.
 * iic_col_sum        out [cols] (=|+=) column sums of x [rows][cols] (`dtype` IIC_F32 / IIC_BF16): the bias gradient of
 *                    SupHead5's first Linear (sup_head5.py:17), whose product runs as a 1x1 convolution. */
int iic_cross_entropy(const float* logits, const long long* targets, int n, int k, float* loss, float* dlogits,
                      void* stream);
int iic_linear_fwd(const float* x, const float* w, const float* b, float* y, int n, int K, int N, void* stream);
int iic_linear_bwd(const float* x, const float* w, const float* dy, float* dw, float* db, float* dx, int accumulate,
                   int n, int K, int N, void* stream);
int iic_col_sum(const void* x, int dtype, long long rows, int cols, float* out, int accumulate, void* stream);

/* ---- a6: segmentation sub-heads -- code/archs/segmentation/net10a.py:34-59:
 *      Conv2d(C -> k, 1x1, padding=1, bias=False) -> Softmax2d -> F.interpolate(size=(H,W), bilinear,
 *      align_corners=False), one sub-head per call.
 * feat [n][hf][wf][C] NHWC (`dtype`); w [k][C] fp32; logits_ws [n*hf*wf][k]; zlow [n][hf+2][wf+2][k]
 * (saved for backward); out NCHW fp32 (n,k,H,W).
 * backward: dout NCHW (n,k,H,W) -> dw [k][C] (overwritten), dfeat [n][hf][wf][C] (`dtype`, overwritten or
 * accumulated; may be NULL).  dzlow_ws [n][hf+2][wf+2][k], dlogits_ws [n*hf*wf][k], dw_workspace of
 * iic_seg_head_workspace() bytes. */
long long iic_seg_head_workspace(int n, int hf, int wf, int C, int k);
int iic_seg_head_fwd(const void* feat, int dtype, const float* w, float* logits_ws, float* zlow, float* out, int n,
                     int hf, int wf, int C, int k, int H, int W, void* stream);
int iic_seg_head_bwd(const void* feat, int dtype, const float* w, const float* zlow, const float* dout,
                     float* dzlow_ws, float* dlogits_ws, float* dw, void* dw_workspace, void* dfeat,
                     int accumulate_dfeat, int n, int hf, int wf, int C, int k, int H, int W, void* stream);

/* ---- a12: torch.optim.Adam step (utils/cluster/general.py:8-9; defaults of
 *      cluster_sobel_twohead.py:184): one launch over a list of tensors.
 *  ptrs_host: 4*T device pointers [param, grad, exp_avg, exp_avg_sq] per tensor, sizes_host: T counts. */
int iic_adam_step(const void* const* ptrs_host, const long long* sizes_host, int T, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int step, void* stream);
/* The same with the step count read from device memory (a float scalar the caller increments on the stream before the
 * call) and the bias corrections computed on the device: the launch arguments never change, so a training step that
 * contains it can be captured once into a CUDA graph and replayed. */
int iic_adam_step_dev(const void* const* ptrs_host, const long long* sizes_host, int n_tensors, float lr, float beta1,
                      float beta2, float eps, float weight_decay, const float* step_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* IIC_B200_H_ */
