/* libosvos_b200 - C ABI of the B200-native OSVOS hot path.
 *
 * The reference (kmaninis/OSVOS-PyTorch) has no FFI of its own: its hot path is
 * Python calling torch.nn modules (SURVEY.md section 8b).  This header is the native
 * boundary introduced underneath the unchanged Python API; each entry point
 * names the reference call it replaces (file:line relative to the reference
 * repo).  The binding a maintainer adds on the reference side is the ctypes
 * stub shown in INTEGRATION.md (osvos_pytorch_b200/_native.py is that stub).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name says host;
 *   - no allocation inside: outputs and workspaces are caller-provided;
 *   - every function enqueues on `stream` and returns immediately with an
 *     OSVOS_* status (0 = ok); no exceptions cross the boundary;
 *     osvos_last_error() returns a thread-local message for the last failure;
 *   - "act" = activation tensor, NHWC, stored as split bf16: value ~= hi + lo,
 *     two planes of shape [N,H,W,C] (C a multiple of 64 for 3x3 conv inputs,
 *     16 for the side-branch gradient).  In OSVOS_FLAG_FAST mode only `hi`
 *     exists (lo pointers may be NULL) and a single tensor-core pass is issued;
 *     the default (exact) mode issues the three passes hi*hi + hi*lo + lo*hi
 *     with fp32 accumulation in TMEM.
 */
#ifndef OSVOS_B200_H_
#define OSVOS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OSVOS_B200_VERSION 100 /* major*10000 + minor*100 + patch */

#if defined(__GNUC__)
#define OSVOS_API __attribute__((visibility("default")))
#else
#define OSVOS_API
#endif

enum {
  OSVOS_OK = 0,
  OSVOS_ERR_INVALID_ARGUMENT = 1,
  OSVOS_ERR_CUDA = 2,
  OSVOS_ERR_UNSUPPORTED = 3
};

enum {
  OSVOS_FLAG_RELU = 1,       /* fwd: y = max(y, 0)            (networks/vgg_osvos.py:143) */
  OSVOS_FLAG_FAST = 2,       /* single-pass bf16 operands (hi planes only)               */
  OSVOS_FLAG_RELU_MASK = 4,  /* dgrad: dx *= (mask_hi > 0)    (autograd of :143)          */
  OSVOS_FLAG_ACCUMULATE = 8, /* add into the existing output instead of overwriting it    */
  OSVOS_FLAG_DEFER_FINISH = 16 /* osvos_conv3x3_wgrad: accumulate into a caller-zeroed workspace only; the
                                  workspace -> OIHW step is done later by osvos_wgrad_finish for many layers */
};

typedef void* osvos_stream_t; /* cudaStream_t */

OSVOS_API int osvos_version(void);
OSVOS_API const char* osvos_last_error(void);
/* Programmatic dependent launch for the kernels enqueued from now on: 1 on, 0 off, -1 = the process default
 * (environment OSVOS_PDL, off).  Returns the previous setting.  Every kernel of the library waits
 * (griddepcontrol.wait) before it first touches memory another kernel may have written, so the switch only decides
 * whether a kernel's prologue may overlap its predecessor's tail.  A captured CUDA graph keeps what it was captured with. */
OSVOS_API int osvos_set_pdl(int mode);

/* ---- weight packing ------------------------------------------------------
 * nn.Conv2d weight, OIHW fp32 (networks/vgg_osvos.py:41,142) -> split-bf16
 * K-major GEMM operand [plane(hi,lo)][tap = 3*r+s][rows][cols]:
 *   transpose_flip == 0 (forward):  rows = Cout, cols = Cin, element = w[co][ci][r][s]
 *   transpose_flip == 1 (dgrad):    rows = Cin,  cols = Cout, element = w[co][ci][2-r][2-s]
 * cols is padded up to a multiple of `col_pad` (64 or 16) with zeros.
 * Bytes needed: osvos_packed_weight_bytes(rows, cols_padded).                      */
OSVOS_API size_t osvos_packed_weight_bytes(int rows, int cols_padded);
OSVOS_API int osvos_pack_conv3x3_weights(const float* w_oihw, void* packed, int cout, int cin, int transpose_flip,
                               int col_pad, osvos_stream_t stream);

/* ---- layout conversion (test / boundary helpers) -------------------------- */
OSVOS_API int osvos_nchw_to_act(const float* x_nchw, void* act_hi, void* act_lo, int n, int c, int h, int w,
                      osvos_stream_t stream);
OSVOS_API int osvos_act_to_nchw(const void* act_hi, const void* act_lo, float* y_nchw, int n, int c, int h, int w,
                      osvos_stream_t stream);

/* ---- conv1_1: nn.Conv2d(3, 64, 3, padding=1) + ReLU ------------------------
 * Replaces stages[0][0..1] (networks/vgg_osvos.py:61,142-143).  Reads the
 * caller's NCHW fp32 frame directly (no layout pass), fp32 CUDA-core math
 * (K = 27 is bandwidth bound), writes an act [N,H,W,64].                       */
OSVOS_API int osvos_conv_first_fwd(const float* x_nchw, const float* w_oihw, const float* bias, void* y_hi, void* y_lo,
                         int n, int h, int w, int flags, osvos_stream_t stream);

/* ---- 3x3 convolution, padding 1, stride 1, as a tcgen05 implicit GEMM -------
 * Replaces every other nn.Conv2d(k=3, p=1) on the path: the 12 remaining trunk
 * convs (+ReLU, networks/vgg_osvos.py:142-143, run at :61,:66) and the four
 * side_prep convs (:41, run at :67, no ReLU); with transpose-flipped packed
 * weights it is also their data gradient (autograd of the same lines).
 *   M = N*H*W pixels (tiles of 16 rows x 8 px), N = cout, K = 9 * cin.         */
typedef struct {
  const void* x_hi;      /* act [n,h,w,cin]                                     */
  const void* x_lo;      /* NULL in FAST mode                                   */
  const void* w_packed;  /* osvos_pack_conv3x3_weights output, rows = cout      */
  const float* bias;     /* [cout] or NULL                                      */
  void* y_hi;            /* act [n,h,w,cout] or NULL                            */
  void* y_lo;            /* NULL in FAST mode / when y_hi is NULL               */
  float* y_f32;          /* optional fp32 NHWC copy of the output [n,h,w,cout]  */
  const void* mask_hi;   /* RELU_MASK: act hi plane [n,h,w,cout] of the fwd output this gradient flows into */
  /* side_prep only (cout == 16): fused 1x1 projections of the 16 features
   *   pq[px][0] = <y, proj_w[0:16]>  + proj_b[0]   score_dsn (networks/vgg_osvos.py:44,69)
   *   pq[px][1] = <y, proj_w[16:32]>               this scale's slice of fuse (:54,72)  */
  const float* proj_w;   /* [32] or NULL */
  const float* proj_b;   /* [1]  or NULL */
  float* pq;             /* [n,h,w,2] or NULL */
  /* fused MaxPool2d(2,2,ceil_mode=True) of the output (networks/vgg_osvos.py:140): act
   * [n, ceil(h/2), ceil(w/2), cout], written in addition to y (cout >= 64 only) */
  void* pool_hi;
  void* pool_lo;
  /* fused per-channel sum of the (masked) output over all pixels = bias gradient of the layer this
   * gradient belongs to; [cout] fp32, ACCUMULATED with atomics (caller zeroes); cout >= 64 only */
  float* colsum;
  int n, h, w, cin, cout;
  int flags;
  /* 0 or 64: all input channels carry data.  16 / 32 / 48: only the first k_valid channels of every 64-channel
   * chunk can be non-zero (e.g. a 16-channel operand stored padded to 64): the remaining K steps
   * are skipped - fewer tcgen05.mma, identical result. */
  int k_valid;
} osvos_conv3x3_args;
OSVOS_API int osvos_conv3x3(const osvos_conv3x3_args* args /* host */, osvos_stream_t stream);

/* ---- launch plans (tests / diagnosis) ----------------------------------------
 * What osvos_conv3x3 / osvos_conv3x3_wgrad would launch for these arguments on the current device, under the
 * current environment switches, without launching anything.  The launchers and the queries share one choice
 * function, so the answer is the schedule the call runs.  The persistent kernels deal `items` work items round-robin
 * to `grid` CTAs: CTA b runs items b, b + grid, b + 2 grid, ...                                                    */
enum { OSVOS_TAP_ROWS = 3, OSVOS_TAP_PAIRS = 5, OSVOS_TAP_NINE = 9 };  /* wgrad tap items per (m, n) block */
typedef struct {
  int block_n;       /* output channels per tile (conv) / GEMM N per item (wgrad)                              */
  int planes;        /* 2: exact split-bf16 operands, 1: FAST                                                    */
  int split_acc;     /* 1: N-concatenated split accumulator (2 MMAs per K step instead of 3)                      */
  int lean;          /* 1: the forward-only (lean) epilogue                                                     */
  int items;         /* work items: output tiles (conv), (m block, n block, tap item, pixel split) items (wgrad) */
  int grid;          /* CTAs launched                                                                          */
  int tap_mode;      /* wgrad: OSVOS_TAP_*; 0 for conv                                                          */
  int pixel_splits;  /* wgrad: pixel-range splits per tap item; 0 for conv                                      */
} osvos_launch_plan;
/* OSVOS_ERR_UNSUPPORTED when the arguments go to the side-branch kernel (cout == 2, or cout == 16 without act output). */
OSVOS_API int osvos_conv3x3_plan(const osvos_conv3x3_args* args /* host */, osvos_launch_plan* plan /* host */);

/* ---- folded side branch (inference and training) ---------------------------------------
 * side_prep has no ReLU (networks/vgg_osvos.py:67), so side_prep followed by score_dsn and this scale's slice of
 * fuse (:44,54,69,72) is ONE 3x3 convolution C -> 2:  W'[o][ci][tap] = sum_co proj_w[16 o + co] * side_w[co][ci][tap],
 * b'[o] = (o == 0 ? proj_b : 0) + sum_co proj_w[16 o + co] * side_b[co].  This writes W' in the packed operand layout
 * (osvos_packed_weight_bytes(2, cin) bytes) and b' (2 floats); osvos_conv3x3 with cout == 2, w_packed = packed,
 * bias = bias2 and pq set then produces the same pq as the cout == 16 call with projections, at 1/8 of the columns. */
OSVOS_API int osvos_fold_side_weights(const float* side_w /* [16,cin,3,3] */, const float* side_b /* [16] or NULL */,
                                      const float* proj_w /* [32] */, const float* proj_b /* [1] or NULL */, void* packed,
                                      float* bias2 /* [2] */, int cin, osvos_stream_t stream);
/* The folded side convolutions (cout == 2 calls of osvos_conv3x3) of up to four scales in ONE launch: `args` is an array
 * of `count` argument blocks, each exactly what the single call takes; results are identical.  Inference runs the four
 * scales this way after the last trunk convolution (networks/vgg_osvos.py:67,69,72 for all four stages at once). */
OSVOS_API int osvos_side_folded_multi(const osvos_conv3x3_args* args /* host array */, int count, osvos_stream_t stream);

/* The same fold for up to four scales in ONE launch (training re-folds after every optimizer step), optionally with an
 * fp32 copy of W' in [tap][o][ci] order (18 * cin floats) - the operand of the folded backward below.              */
typedef struct {
  const float* side_w;   /* [16,cin,3,3] */
  const float* side_b;   /* [16] or NULL */
  const float* proj_w;   /* [32]: score_dsn.weight | this scale's slice of fuse.weight */
  const float* proj_b;   /* [1] or NULL */
  void* packed;          /* osvos_packed_weight_bytes(2, cin) bytes */
  float* bias2;          /* [2] */
  float* folded_f32;     /* [9][2][cin] or NULL */
  int cin;
} osvos_fold_item;
OSVOS_API int osvos_fold_side_weights_multi(const osvos_fold_item* items /* host */, int count, osvos_stream_t stream);
/* Same contract on CUDA cores (fp32 FMA over hi+lo); debugging cross-check only. */
OSVOS_API int osvos_conv3x3_simt(const osvos_conv3x3_args* args /* host */, osvos_stream_t stream);

/* ---- stage 1 of the trunk as one kernel (inference) -------------------------------------
 * conv1_1 + ReLU + conv1_2 + ReLU (+ the first MaxPool2d(2,2,ceil_mode=True)): networks/vgg_osvos.py:61,140-143.
 * conv1_1 is evaluated inside conv1_2's kernel on the halo patch conv1_2 reads, so the 64-channel full-resolution map
 * between the two layers never touches memory.  Exact mode only.  Outputs: the full-resolution act (y_*), the pooled
 * act (pool_*), or both; all planes 32-byte aligned.  Same results as osvos_conv_first_fwd + osvos_conv3x3 up to the
 * fp32 summation order inside conv1_1.                                                            */
typedef struct {
  const float* x;          /* [n,3,h,w] fp32 frame (NCHW)                    */
  const float* w1;         /* conv1_1 weight [64,3,3,3] fp32 (OIHW)          */
  const float* b1;         /* conv1_1 bias [64] or NULL                      */
  const void* w2_packed;   /* conv1_2 weight, osvos_pack_conv3x3_weights(transpose_flip = 0) */
  const float* b2;         /* conv1_2 bias [64] or NULL                      */
  void* y_hi;              /* [n,h,w,64] or NULL                             */
  void* y_lo;
  void* pool_hi;           /* [n,ceil(h/2),ceil(w/2),64] or NULL             */
  void* pool_lo;
  int n, h, w;
} osvos_stage1_args;
OSVOS_API int osvos_stage1_fused(const osvos_stage1_args* args /* host */, osvos_stream_t stream);

/* ---- MaxPool2d(2, 2, ceil_mode=True) on an act (networks/vgg_osvos.py:140) --- */
OSVOS_API int osvos_maxpool2x2_fwd(const void* x_hi, const void* x_lo, void* y_hi, void* y_lo, int n, int h, int w, int c,
                         osvos_stream_t stream);

/* ---- side-branch tail ----------------------------------------------------------
 * Replaces, in one bandwidth-bound kernel, upscale_[i](score_dsn[i](.)) + center_crop
 * (networks/vgg_osvos.py:69), upscale[i] + center_crop + cat + fuse (:68,:71-72), the
 * interp_surgery bilinear taps (layers/osvos_layers.py:59-85), the crop offsets
 * (layers/osvos_layers.py:51-56) and, when `label` is given, the per-pixel terms and
 * reductions of class_balanced_cross_entropy_loss (layers/osvos_layers.py:28-41).
 *   out[k][n,0,y,x], k<4 = sum over the <=2x2 low-res taps of scale k of p_k
 *   out[4]               = sum_k (same taps of q_k) + fuse_bias
 *   sums[2k], sums[2k+1] = {sum_{y=1} (softplus(x)-x), sum_{y=0} softplus(x)} of map k,
 *   sums[10] = P = #(label >= .5), sums[11] = number of pixels N,
 *   sums[12], sums[13] = {sum_{y=1} (sigmoid(x_fused)-1), sum_{y=0} sigmoid(x_fused)} (-> d fuse.bias),
 *   sums[14] = arrival counter                         (OSVOS_TAIL_SUMS = 15 doubles, zeroed by the call)
 * and, when `losses` is given (the package's own objective: train_online.py:127, train_parent.py:143-147),
 *   losses[k] = (Nn/N * S_pos_k + P/N * S_neg_k) / divisor,  losses[5] = sum_k loss_weights[k] * losses[k]
 * so that upsample + crop + fuse + the five class-balanced BCE losses are ONE kernel.            */
#define OSVOS_TAIL_SUMS 15
typedef struct {
  const float* pq[4];      /* [n, h_k, w_k, 2], h_k = ceil-halved k+1 times          */
  const float* fuse_bias;  /* [1] */
  float* out[5];           /* each [n,1,h,w] fp32, any may be NULL                   */
  const float* label;      /* [n,1,h,w] or NULL */
  double* sums;            /* [OSVOS_TAIL_SUMS] or NULL (required with label)         */
  float* losses;           /* [6] or NULL (needs label)                               */
  float loss_weights[5];   /* weights of the five losses in losses[5]                 */
  float divisor;           /* batch size (batch_average), numel (size_average) or 1   */
  int n, h, w;
} osvos_tail_fwd_args;
OSVOS_API int osvos_tail_fwd(const osvos_tail_fwd_args* args /* host */, osvos_stream_t stream);

/* Standalone 1x1 projections of a side feature map (used when the features do
 * not come from osvos_conv3x3's fused epilogue): pq as above.                       */
OSVOS_API int osvos_side_project(const float* feat /* [n,h,w,16] */, const float* proj_w, const float* proj_b, float* pq,
                       int n, int h, int w, osvos_stream_t stream);

/* ---- class_balanced_cross_entropy_loss (layers/osvos_layers.py:19-48) -----------
 * forward: sums[0..3] = {S_pos, S_neg, P, N} (5 doubles, zeroed by the call; sums[4] is an arrival counter), loss[0] =
 * (Nn/N*S_pos + P/N*S_neg)/divisor with divisor = numel (size_average), batch
 * (batch_average) or 1.  backward: grad_in = grad_out[0] * w * (sigmoid(x) - y) / divisor
 * (grad_out == NULL means 1).                                                        */
OSVOS_API int osvos_cbce_fwd(const float* output, const float* label, size_t numel, double divisor, double* sums,
                             float* loss, osvos_stream_t stream);
OSVOS_API int osvos_cbce_bwd(const float* output, const float* label, const double* sums, const float* grad_out,
                             double divisor, size_t numel, float* grad_in, osvos_stream_t stream);

/* ======================= backward (training) entry points ======================= */

/* ---- weight gradient of a 3x3 conv (tcgen05 GEMM over the pixel axis) -----------
 * Replaces autograd's weight gradient of nn.Conv2d(k=3,p=1) (reference
 * networks/vgg_osvos.py:41,142; backward at train_online.py:141 / train_parent.py:164):
 *   dw[co][ci][r][s] = sum_px dz[px][co] * x[px + (r-1, s-1)][ci]
 * dz has `cout` channels (dz_channels == cout, a multiple of 64).  (side_prep's weight gradient does not come through
 * here: osvos_side_folded_wgrad / osvos_side_grads_finish.)
 * workspace: osvos_wgrad_workspace_bytes(dz_channels, cin) bytes, contents destroyed.  */
typedef struct {
  const void* x_hi;   /* layer input act [n,h,w,cin]        */
  const void* x_lo;
  const void* dz_hi;  /* output-gradient act [n,h,w,dz_channels] */
  const void* dz_lo;
  float* dw;          /* [cout][cin][3][3] fp32, overwritten */
  float* workspace;
  int n, h, w, cin, cout, dz_channels;
  int flags;          /* OSVOS_FLAG_FAST | OSVOS_FLAG_DEFER_FINISH (then dw may be NULL) */
} osvos_wgrad_args;
OSVOS_API size_t osvos_wgrad_workspace_bytes(int dz_channels, int cin);
OSVOS_API int osvos_conv3x3_wgrad(const osvos_wgrad_args* args /* host */, osvos_stream_t stream);
/* The launch plan of osvos_conv3x3_wgrad for these arguments (see osvos_conv3x3_plan). */
OSVOS_API int osvos_conv3x3_wgrad_plan(const osvos_wgrad_args* args /* host */, osvos_launch_plan* plan /* host */);

/* Deferred finish of up to OSVOS_WGRAD_FINISH_MAX weight gradients in ONE launch: workspace [9][a][b] -> OIHW,
 * dw = (accumulate ? dw : 0) + scale * ws.  With accumulate the destination can be the parameter's .grad itself
 * (what autograd's AccumulateGrad would do with a separate add kernel, train_online.py:141).                    */
#define OSVOS_WGRAD_FINISH_MAX 24
typedef struct {
  const float* workspace;  /* as passed to osvos_conv3x3_wgrad with OSVOS_FLAG_DEFER_FINISH */
  float* dw;               /* [cout][cin][3][3] */
  int cout, cin, dz_channels;
  int accumulate;
  float scale;
} osvos_wgrad_finish_item;
OSVOS_API int osvos_wgrad_finish(const osvos_wgrad_finish_item* items /* host */, int count, osvos_stream_t stream);

/* ---- adjoint of the tail: gradients of the five maps -> low-res dp/dq ------------
 * Backward of osvos_tail_fwd (autograd of networks/vgg_osvos.py:68-72): strided bilinear
 * DOWN-sampling of grad_out[k] (-> dpq[k][..,0]) and of grad_out[4] (-> dpq[k][..,1])
 * through the crop window.  NULL grad_out entries count as zero.                       */
typedef struct {
  const float* grad_out[5]; /* each [n,1,h,w] or NULL */
  float* dpq[4];            /* [n,h_k,w_k,2] */
  int n, h, w;
} osvos_tail_bwd_args;
OSVOS_API int osvos_tail_bwd(const osvos_tail_bwd_args* args /* host */, osvos_stream_t stream);

/* ---- backward of tail + class-balanced BCE in one launch ---------------------------
 * Autograd of `total = sum_k loss_weights[k] * class_balanced_cross_entropy_loss(out[k], label)` through
 * osvos_tail_fwd (layers/osvos_layers.py:28-46 + networks/vgg_osvos.py:68-72; the parent / online objectives of
 * train_parent.py:143-147 and train_online.py:127): dL/dlogit_k = upstream * loss_weights[k] * w * (sigmoid(x_k) - y)
 * / divisor is formed on the fly from the logit maps and the label while the bilinear adjoint gathers it - the five
 * gradient maps are never written.  `sums` is the forward call's (P, N and the fuse-bias sums are read from it).   */
typedef struct {
  const float* logits[5];   /* the five maps written by osvos_tail_fwd (NULL allowed where the weight is 0) */
  const float* label;       /* [n,1,h,w] */
  const double* sums;       /* [OSVOS_TAIL_SUMS] of the forward call */
  const float* upstream;    /* device scalar d(total) or NULL (= 1) */
  float loss_weights[5];
  float divisor;
  float* dpq[4];            /* [n,h_k,w_k,2] */
  float* fuse_bias_grad;    /* [1] or NULL */
  int n, h, w;
} osvos_tail_loss_bwd_args;
OSVOS_API int osvos_tail_loss_bwd(const osvos_tail_loss_bwd_args* args /* host */, osvos_stream_t stream);

/* out[0] = sum(x[0:n]) (fuse.bias gradient); scratch: 2 doubles (total, arrival counter).  */
OSVOS_API int osvos_sum_f32(const float* x, size_t n, double* scratch, float* out, osvos_stream_t stream);

/* ---- max-unpool + side-branch add + ReLU mask (autograd of networks/vgg_osvos.py:140,143) */
OSVOS_API int osvos_unpool_add_mask(const void* dpool_hi, const void* dpool_lo, const void* x_hi, const void* x_lo,
                                    const float* dside /* [n,h,w,c] fp32 or NULL */, void* dz_hi, void* dz_lo,
                                    float* colsum /* [c] accumulated per-channel sum of dz, or NULL */, int n,
                                    int h, int w, int c, osvos_stream_t stream);

/* ---- side branch backward in folded (rank-2) form -------------------------------------------------------------
 * Autograd of networks/vgg_osvos.py:67,69,72 (side_prep -> score_dsn / fuse slice) expressed on the folded 3x3
 * convolution C -> 2 (see osvos_fold_side_weights): the branch's backward only sees the two gradient channels
 * dpq = (dL/dp, dL/dq).
 *   osvos_side_folded_wgrad:  g[t][o][c] += sum_px dpq[px - t][o] * x[px][c]  (t = 3r + s <-> offset (r-1, s-1)),
 *                             g[18 c + o] += sum_px dpq[px][o];   g: osvos_side_folded_wgrad_floats(c) floats, PRE-ZEROED,
 *                             16-byte aligned; c a multiple of 128.
 *   osvos_side_grads_finish:  every parameter gradient of up to four scales from g, one launch:
 *                             d side_prep.weight[f][c][t] = proj[f] g[t][0][c] + proj[16+f] g[t][1][c],
 *                             d side_prep.bias[f] = proj[f] S0 + proj[16+f] S1,
 *                             d score_dsn.weight[f] = <side_w[f], g[.][0][.]> + side_b[f] S0, d score_dsn.bias = S0,
 *                             d fuse.weight slice[f] = <side_w[f], g[.][1][.]> + side_b[f] S1
 *                             (NULL outputs are skipped; accumulate: add to the destinations instead of overwriting).
 *   osvos_unpool_side_mask:   dz = ReLU'(x) * (unpool(dpool) + dX),  dX[px][c] = sum_{t,o} wfold[t][o][c] dpq[px - t][o]
 *                             - osvos_unpool_add_mask with the side gradient computed on the fly from dpq and the fp32
 *                             folded weights (osvos_fold_side_weights_multi) instead of read from an fp32 map;
 *                             dpool_hi NULL: no pooling consumer (deepest stage).                                    */
OSVOS_API size_t osvos_side_folded_wgrad_floats(int c);
OSVOS_API int osvos_side_folded_wgrad(const void* x_hi, const void* x_lo /* or NULL */, const float* dpq /* [n,h,w,2] */,
                                      float* g, int n, int h, int w, int c, osvos_stream_t stream);
/* The same for up to four scales in one launch (x_lo either set for all items or for none). */
typedef struct {
  const void* x_hi;
  const void* x_lo;
  const float* dpq;
  float* g;
  int n, h, w, c;
} osvos_side_wgrad_item;
OSVOS_API int osvos_side_folded_wgrad_multi(const osvos_side_wgrad_item* items /* host */, int count, osvos_stream_t stream);
typedef struct {
  const float* g;        /* as filled by osvos_side_folded_wgrad */
  const float* side_w;   /* [16,c,3,3] */
  const float* side_b;   /* [16] or NULL */
  const float* proj_w;   /* [32] */
  float* d_side_w;       /* [16,c,3,3] */
  float* d_side_b;       /* [16] */
  float* d_score_w;      /* [16] or NULL */
  float* d_score_b;      /* [1] or NULL */
  float* d_fuse_w;       /* [16] (this scale's slice) or NULL */
  int c;
  int accumulate;
} osvos_side_grads_item;
OSVOS_API int osvos_side_grads_finish(const osvos_side_grads_item* items /* host */, int count, osvos_stream_t stream);
OSVOS_API int osvos_unpool_side_mask(const void* dpool_hi /* or NULL */, const void* dpool_lo, const void* x_hi,
                                     const void* x_lo, const float* dpq /* [n,h,w,2] */,
                                     const float* wfold /* [9][2][c] fp32 */, void* dz_hi, void* dz_lo,
                                     float* colsum /* or NULL */, int n, int h, int w, int c, osvos_stream_t stream);

/* ---- bias gradient: out[c] = sum over pixels of an act ----------------------------- */
OSVOS_API int osvos_channel_sum(const void* act_hi, const void* act_lo, float* out, size_t npix, int c,
                                osvos_stream_t stream);

/* ---- conv1_1 backward: dw [64][3][3][3] and (optionally) dx [n,3,h,w] ---------------
 * workspace: osvos_conv_first_bwd_workspace_bytes() bytes (replicated partial sums + arrival counter; zeroed by
 * the call).                                                                                  */
OSVOS_API size_t osvos_conv_first_bwd_workspace_bytes(void);
OSVOS_API int osvos_conv_first_bwd(const float* x_nchw, const void* dz_hi, const void* dz_lo, const float* w_oihw,
                                   float* dw, float* dx_nchw /* or NULL */, void* workspace, int n, int h, int w,
                                   osvos_stream_t stream);

/* ===================== SURVEY.md 8(f) "next" rows: callers either side ===================== */

/* ---- test-time output path (train_online.py:181-187) --------------------------------
 * The reference copies the fused logits to the host, applies 1/(1+exp(-x)) in numpy and hands
 * the float map to scipy.misc.imsave, which rescales [min,max] of the frame to [0,255]
 * ("bytescale").  Here the 8-bit map is produced on the device so only H*W bytes cross PCIe.
 *   OSVOS_U8_PROB      out = floor(255*sigmoid(x) + 0.5)
 *   OSVOS_U8_BYTESCALE out = floor(clip((p - pmin) * 255/(pmax - pmin), 0, 255) + 0.5), p = sigmoid(x),
 *                      pmin/pmax over each frame (pmax == pmin -> divisor 1): the PNG the reference writes
 *   OSVOS_U8_MASK      out = x > 0 ? 255 : 0   (the thresholded mask, sigmoid(x) > 0.5)
 * logits [frames][per_frame] fp32, out [frames][per_frame] u8, minmax_ws: 2 uint32 per frame
 * (only used by BYTESCALE; zeroed by the call).                                                   */
enum { OSVOS_U8_PROB = 0, OSVOS_U8_BYTESCALE = 1, OSVOS_U8_MASK = 2 };
OSVOS_API int osvos_logits_to_u8(const float* logits, uint8_t* out, uint32_t* minmax_ws, int frames, size_t per_frame,
                                 int mode, osvos_stream_t stream);

/* ---- optimizer step (train_online.py:79-88,147; train_parent.py:87-103,170) -------------
 * torch.optim.SGD(momentum, weight_decay, dampening 0, no nesterov) over every trainable tensor in ONE launch:
 *     g' = g + wd*p ;  m = mu*m + g' ;  p = p - lr*m        (m starts at 0, so the first step gives m = g')
 * with per-tensor lr / wd / mu (the reference's parameter groups), optionally zeroing g in the same pass
 * (optimizer.zero_grad(), train_online.py:148), and - for 3x3 conv weights whose `packed_*` pointers are set -
 * re-emitting the tensor-core operand layouts of osvos_pack_conv3x3_weights (forward, col_pad = colp_fwd multiple;
 * transposed+flipped for dgrad) from the updated values, so no separate repack pass runs after the step.
 * `segments` is a DEVICE array of `count` descriptors (<= OSVOS_SGD_MAX_SEGMENTS); `work_items` of each
 * descriptor = osvos_sgd_work_items(numel, cout, cin) (host helper).  Pad columns of the packed layouts are not
 * touched (they stay zero from the initial osvos_pack_conv3x3_weights call).                           */
#define OSVOS_SGD_MAX_SEGMENTS 64
typedef struct osvos_sgd_segment {
  float* param;         /* [numel] fp32, updated in place                                         */
  float* grad;          /* [numel] fp32 (zeroed when zero_grad != 0)                              */
  float* momentum;      /* [numel] fp32 momentum buffer, updated in place                         */
  uint64_t numel;
  float lr, weight_decay, momentum_coef;
  int32_t cout, cin;    /* 3x3 conv weight [cout][cin][3][3] when packed_fwd/packed_flip are set  */
  int32_t colp_fwd;     /* padded column count of the forward layout  (multiple of its col_pad)   */
  int32_t colp_flip;    /* padded column count of the flipped layout                              */
  uint32_t work_items;  /* osvos_sgd_work_items(numel, cout, cin) when packing, (numel, 0, 0) else */
  void* packed_fwd;     /* or NULL */
  void* packed_flip;    /* or NULL */
} osvos_sgd_segment;
OSVOS_API uint32_t osvos_sgd_work_items(uint64_t numel, int cout, int cin);
OSVOS_API int osvos_sgd_step(const osvos_sgd_segment* segments /* device */, int count, uint32_t total_work_items,
                             int zero_grad, osvos_stream_t stream);

/* ---- data augmentation on the device (dataloaders/custom_transforms.py:7-54 ScaleNRotate, :87-100
 * RandomHorizontalFlip, composed flip-then-warp at train_online.py:92-94 / train_parent.py:108-110) -----
 * The reference warps every sample on the host with cv2.warpAffine(tmp, getRotationMatrix2D(center, rot, sc),
 * (w, h), flags) - INTER_CUBIC for the image, INTER_NEAREST for the 0/1 mask, BORDER_CONSTANT 0.  This entry point
 * restates OpenCV's published algorithm (cv2 is not vendored by the reference and absent from this image):
 * fixed-point source coordinates X = (rint((m1*y+m2)*1024) + delta + rint(m0*x*1024)) >> s with 1/32-pixel
 * sub-positions for cubic (delta 16, s 5) and whole pixels for nearest (delta 512, s 10); bicubic taps with
 * A = -0.75 evaluated in fp32 at the 1/32 position; taps outside the image contribute 0.
 * src/dst [n][c][h][w] fp32; inv_matrices_host: n x 6 doubles, the INVERTED 2x3 matrix (dst -> src) as
 * cv::warpAffine computes it; flips_host[n]: 1 = the source is mirrored horizontally first (cv2.flip(.., 1)).   */
enum { OSVOS_WARP_CUBIC = 0, OSVOS_WARP_NEAREST = 1 };
OSVOS_API int osvos_affine_warp(const float* src, float* dst, const double* inv_matrices_host, const int* flips_host,
                                int n, int c, int h, int w, int mode, osvos_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* OSVOS_B200_H_ */
