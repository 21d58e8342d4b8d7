/*
 * gdl_b200.h — C-ABI of the B200-native DGL training-step kernels.
 *
 * Drop-in boundary for ONE hot path of shicaiwei123/ICCV2025-GDL: the Disentangled
 * Gradient Learning step (reference main_dgl.py:69-165).  The reference has no FFI of
 * its own (it is pure Python calling torch/ATen); each entry point below therefore cites
 * the reference call site (file:line under the reference tree) whose ATen op it replaces.
 * The host side stays PyTorch: callers pass raw device pointers borrowed from torch
 * tensors plus a cudaStream_t.  Conventions:
 *   - every function returns GDL_OK (0) or a negative gdl_status; no exceptions,
 *     no hidden allocation, no hidden synchronisation, asynchronous w.r.t. the host;
 *   - all kernels are sm_100a only (tcgen05/TMEM for the convolutions); there is no
 *     CPU, cuDNN, cuBLAS or Triton fallback;
 *   - activations are NHWC bf16; parameters/gradients/optimizer state are fp32;
 *     reductions are deterministic (fixed-order partials, no float atomics);
 *   - threading / context model: the library keeps NO per-call or per-stream state, so there is no gdl_ctx object —
 *     every entry point takes all of its operands, workspaces and the stream as arguments and is re-entrant.  The
 *     only shared state is (a) the tensor-map cache (keyed by pointer + geometry, mutex-guarded) and (b) the
 *     per-kernel cudaFuncSetAttribute calls made once per process, which is why ONE process drives ONE device
 *     (torch.distributed's process-per-GPU model; gdl_init(device) checks the device).  The two scheduling hints
 *     (gdl_set_sweep, gdl_set_fused_stats_min_k) are thread-local: host threads that enqueue on different streams do
 *     not see each other's settings.
 */
#ifndef GDL_B200_H_
#define GDL_B200_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* gdl_stream_t; /* a cudaStream_t */

typedef enum {
  GDL_OK = 0,
  GDL_EINVAL = -1, /* bad shape / alignment / null pointer */
  GDL_EARCH = -2,  /* device is not sm_100 */
  GDL_ECUDA = -3,  /* CUDA runtime error; see gdl_last_error_string() */
  GDL_ENOMEM = -4  /* caller-provided workspace too small */
} gdl_status;

/* ---- library / context -------------------------------------------------------------- */
int gdl_version(void);
const char* gdl_last_error_string(void);
/* Checks the device is sm_100 and sets kernel attributes (max dynamic smem). */
int gdl_init(int device);

/* ---- convolution (reference models/backbone.py:20-28,97-100 nn.Conv2d, bias=False) --- */
typedef struct {
  int32_t N;          /* images (B for audio, B*T for visual)                         */
  int32_t Hi, Wi;     /* input spatial size                                           */
  int32_t Ci;         /* input channels AS STORED: multiple of 64, or 8 (padded stem) */
  int32_t Ho, Wo;     /* output spatial size                                          */
  int32_t Co;         /* output channels, multiple of 64                              */
  int32_t R, S;       /* filter size                                                  */
  int32_t stride, pad;
} gdl_conv_desc;

/* Length (elements) of one packed weight row: R*S*Ci rounded up to 64. */
int64_t gdl_conv_packed_k(const gdl_conv_desc* d);
/* Bytes of scratch gdl_conv_wgrad needs for its split-K partials. */
int64_t gdl_conv_wgrad_workspace_bytes(const gdl_conv_desc* d);

/* fp32 OIHW master weight [Co][ci_real][R][S] -> bf16 packed [Co][Kp] (k=(r,s,ci)) and
 * bf16 transposed [Ci][R*S*Co] (k=(r,s,co)) for dgrad (wT may be NULL). */
int gdl_conv_pack_weights(const gdl_conv_desc* d, int ci_real, const float* w_oihw,
                          void* w_packed, void* w_packed_T, gdl_stream_t s);
/* The same for many convolutions in ONE launch: table_dev is a DEVICE array of n entries sorted by `start`
 * (running sum of Co*Kp); total = sum of Co*Kp. */
typedef struct {
  const float* w; /* fp32 OIHW master */
  void* wp;       /* bf16 [Co][Kp] */
  void* wT;       /* bf16 [Ci][R*S*Co] or NULL */
  int32_t Co, Ci, ci_real, R, S, Kp;
  int64_t start;
  const float* scale; /* NULL, or fp32 [Co]: row co is multiplied by scale[co] before rounding (eval mode: the
                         BatchNorm running-statistics scale gamma/sqrt(var+eps) folded into the weights) */
} gdl_pack_entry;
int gdl_conv_pack_weights_multi(const gdl_pack_entry* table_dev, int n, int64_t total, gdl_stream_t s);
/* The same through shared-memory tiles (coalesced reads and writes), for tables whose entries ALL have
 * Ci == ci_real, Ci % 64 == 0, Co % 32 == 0 and Kp == R*S*Ci (the 19 block convolutions of a ResNet-18 encoder):
 * max_tiles = max over entries of (Co/32)*(Ci/64), max_rs = max R*S (<= 9). */
int gdl_conv_pack_weights_tiled(const gdl_pack_entry* table_dev, int n, int max_tiles, int max_rs, gdl_stream_t s);
/* y[N,Ho,Wo,Co] = conv(x[N,Hi,Wi,Ci], w).  Implicit GEMM, tcgen05 + TMEM accumulators. */
int gdl_conv_fwd(const gdl_conv_desc* d, const void* x, const void* w_packed, void* y,
                 gdl_stream_t s);
/* Eval-mode fused unit (reference valid(), main_dgl.py:168-222: model.eval() => BatchNorm2d uses its running
 * statistics, backbone.py:45-66): with the BN scale folded into w_packed (gdl_pack_entry.scale) the whole
 * conv -> BN -> (+identity) -> ReLU unit is y = [relu](conv(x, w') + bias[co] [+ res]), bias = beta - mean*scale,
 * res NULL or a bf16 tensor of y's shape.  Flat-window geometries only (3x3 s1/s2 pad 1, 1x1 pad 0, Ci % 64 == 0);
 * anything else returns GDL_EINVAL. */
int gdl_conv_fwd_bias_act(const gdl_conv_desc* d, const void* x, const void* w_packed, const float* bias,
                          const void* res, int relu, void* y, gdl_stream_t s);
/* Same, and the BatchNorm statistics of y (reference backbone.py:45,48: train-mode BN follows every conv) are
 * accumulated in the epilogue: bn_partial receives *bn_partial_rows rows of [2][Co] floats (per-warp sum and sum
 * of squares of the bf16-rounded outputs) for gdl_bn_stats_finalize.  *bn_partial_rows == 0 means the shape took
 * a path without the fused statistics (call gdl_bn_stats on y instead).  bn_partial: gdl_bn_partial_floats(). */
int gdl_conv_fwd_stats(const gdl_conv_desc* d, const void* x, const void* w_packed, void* y,
                       float* bn_partial, int* bn_partial_rows, gdl_stream_t s);
/* Fused statistics are used for convolutions with R*S*Ci >= k.  Default (k < 0): the environment variable
 * GDL_FUSED_STATS_MIN_K, else 0 = every convolution the flat-window kernels run (the per-warp shared-memory
 * transpose costs less than the separate statistics pass on every layer of the bench geometry).  Thread-local.
 * Returns the old value (negative: the default was in force). */
int gdl_set_fused_stats_min_k(int k);
/* Scheduling hint for the calling thread (no reference counterpart: the reference's kernels are cuDNN's):
 * reverse != 0 makes the following gdl_conv_fwd / gdl_conv_dgrad (flat kernels), gdl_bn_stats, gdl_bn_apply,
 * gdl_bn_bwd and gdl_bn_bwd_nores launches walk their pixel range in DESCENDING order (two-pass operations run
 * their second pass opposite to the first).  A pass that runs opposite to the pass that last touched a tensor
 * starts on the part still resident in L2.  Element-wise results are unaffected; reductions keep one fixed
 * summation order per setting (deterministic).  Returns the previous setting. */
int gdl_set_sweep(int reverse);
/* dx[N,Hi,Wi,Ci] = conv_transpose(dy, w) (+ add_src).  add_mode: 0 none, 1 add_src has the
 * shape of dx (residual gradient), 2 add_src is [N,ceil(Hi/2),ceil(Wi/2),Ci] and is added at
 * even (h,w) only (gradient of a 1x1 stride-2 downsample branch). */
int gdl_conv_dgrad(const gdl_conv_desc* d, const void* dy, const void* w_packed_T, void* dx,
                   const void* add_src, int add_mode, gdl_stream_t s);
/* dw_oihw[Co][ci_real][R][S] (fp32) = sum over pixels; deterministic split-K. */
int gdl_conv_wgrad(const gdl_conv_desc* d, int ci_real, const void* x, const void* dy,
                   float* dw_oihw, void* workspace, int64_t workspace_bytes, gdl_stream_t s);

/* ---- stem convolutions (reference models/backbone.py:97-100: Conv2d(1|3 -> 64, 7, stride 2, pad 3))
 * as a space-to-depth 4x4/s1 implicit GEMM: see csrc/conv_stem.cu.  x16 is the bf16 tensor
 * [N, Hp, Wp, 16] written by gdl_stem_layout (Hp = Ho + 3, Wp = Wo + 3). */
int gdl_stem_geometry(int H, int W, int* Ho, int* Wo, int* Hp, int* Wp);
/* src f32 [B,C,T,H,W] (C <= 4; audio: C = T = 1) -> x16; replaces backbone.py:162-164 + the cast. */
int gdl_stem_layout(const float* src, void* x16, int B, int C, int T, int H, int W, gdl_stream_t s);
/* fp32 OIHW [64][C][7][7] -> bf16 [64][256]. */
int gdl_stem_pack_weights(const float* w_oihw, void* w_packed, int C, gdl_stream_t s);
/* Same with output channel co multiplied by scale64[co] (eval mode: BatchNorm scale folded into the stem). */
int gdl_stem_pack_weights_scaled(const float* w_oihw, const float* scale64, void* w_packed, int C, gdl_stream_t s);
/* y bf16 [N,Ho,Wo,64]. */
int gdl_stem_fwd(const void* x16, const void* w_packed, void* y, int N, int H, int W, gdl_stream_t s);
/* Same, and the statistics of the following train-mode BatchNorm (reference backbone.py:104 bn1) from the epilogue:
 * bn_partial receives *bn_partial_rows rows of [2][64] floats (sum, sum of squares of the bf16-rounded outputs) for
 * gdl_bn_stats_finalize — no separate pass over the largest activation of the step. */
int gdl_stem_fwd_stats(const void* x16, const void* w_packed, void* y, int N, int H, int W, float* bn_partial,
                       int* bn_partial_rows, gdl_stream_t s);
int64_t gdl_stem_wgrad_workspace_bytes(int N, int H, int W);
/* dw fp32 OIHW [64][C][7][7] from x16 and dy bf16 [N,Ho,Wo,64]; deterministic split-K. */
int gdl_stem_wgrad(const void* x16, const void* dy, float* dw_oihw, int C, int N, int H, int W,
                   void* workspace, int64_t workspace_bytes, gdl_stream_t s);

/* ---- layout (reference models/backbone.py:162-164 permute/contiguous/view, and
 *      main_dgl.py:100 spec.unsqueeze(1).float()) ---------------------------------------- */
/* src f32 [B,C,T,H,W] -> dst bf16 [B*T,H,W,8] (channels >= C zero). */
int gdl_layout_ncthw_to_nhwc8(const float* src, void* dst, int B, int C, int T, int H, int W,
                              gdl_stream_t s);

/* ---- BatchNorm2d training mode (reference models/backbone.py:45,48,104,144) ---------- */
/* Per-channel batch statistics of x bf16 [P,C]: mean, invstd (biased var, eps), running
 * stats update (momentum, unbiased var), and the fused affine scale/shift.
 * partial: scratch of gdl_bn_partial_floats(P,C) floats. */
int64_t gdl_bn_partial_floats(int64_t P, int C);
int gdl_bn_stats(const void* x, int64_t P, int C, float* partial, const float* gamma,
                 const float* beta, float eps, float momentum, float* running_mean,
                 float* running_var, float* mean, float* invstd, float* scale, float* shift,
                 gdl_stream_t s);
/* Second half of gdl_bn_stats for partial sums produced elsewhere (gdl_conv_fwd_stats): rows x [2][C]. */
int gdl_bn_stats_finalize(const float* partial, int rows, int64_t P, int C, const float* gamma,
                          const float* beta, float eps, float momentum, float* running_mean,
                          float* running_var, float* mean, float* invstd, float* scale, float* shift,
                          gdl_stream_t s);
/* Eval mode (reference model.eval() in valid(), main_dgl.py:186): scale/shift from the running stats. */
int gdl_bn_eval_affine(const float* gamma, const float* beta, const float* running_mean,
                       const float* running_var, float eps, float* scale, float* shift, int C,
                       gdl_stream_t s);
/* y = [relu](x*scale + shift [+ res])  (BN-apply fused with ReLU backbone.py:46,57,66 and
 * the residual add backbone.py:65). */
int gdl_bn_apply(const void* x, const void* res, void* y, int64_t P, int C, const float* scale,
                 const float* shift, int relu, gdl_stream_t s);
/* Backward of y = [relu](bn(x) [+res]).  Pass 1: dz = dy*(y>0) (written to dz; dz may alias
 * dy; if !relu dz is not written and dy is used as dz), partial sums of dz and dz*xhat.
 * Then dgamma/dbeta (fp32, overwritten) and dx = gamma*invstd*(dz - dbeta/P - xhat*dgamma/P). */
int gdl_bn_bwd(const void* dy, const void* y, const void* x, void* dz, void* dx, int64_t P,
               int C, const float* gamma, const float* mean, const float* invstd,
               float* partial, float* dgamma, float* dbeta, int relu, gdl_stream_t s);

/* Same for units WITHOUT a residual input and WITH ReLU (backbone.py:44-46 conv1/bn1/relu): the mask is
 * recomputed from x (y > 0 <=> x*scale+shift > 0 with the forward's scale/shift), so y is not read and no
 * masked gradient is written: 10 B/element instead of 14. */
int gdl_bn_bwd_nores(const void* dy, const void* x, void* dx, int64_t P, int C, const float* gamma,
                     const float* mean, const float* invstd, const float* scale, const float* shift,
                     float* partial, float* dgamma, float* dbeta, gdl_stream_t s);

/* ---- stem tail fused: BN-apply + ReLU + MaxPool2d(3,2,1) (reference models/backbone.py:104-106) ----
 * Forward reads the stem conv output x [N,H,W,C] and writes the pooled map y [N,Ho,Wo,C] + 1-byte arg-max;
 * the activation relu(bn(x)) — the largest tensor of the step — is never materialised.  Backward gathers the
 * pooled gradient through the arg-max, recomputes the ReLU mask from x and does the BN backward
 * (dgamma/dbeta fp32 overwritten, dx bf16).  The forward is bit-identical to gdl_bn_apply + gdl_maxpool_fwd.
 * xmax (optional, bf16 [N,Ho,Wo,C]): the conv output at each window's arg-max, saved by the forward; with it the
 * backward forms the BN sums on the pooled grid (4x fewer elements) instead of a pass over x. */
int gdl_bn_relu_maxpool_fwd(const void* x, const float* scale, const float* shift, void* y,
                            uint8_t* argmax, void* xmax, int N, int H, int W, int C, int Ho, int Wo, gdl_stream_t s);
int gdl_bn_relu_maxpool_bwd(const void* gpool, const uint8_t* argmax, const void* xmax, const void* x, void* dx,
                            int N, int H, int W, int C, int Ho, int Wo, const float* gamma, const float* mean,
                            const float* invstd, const float* scale, const float* shift, float* partial,
                            float* dgamma, float* dbeta, gdl_stream_t s);

/* ---- MaxPool2d(3,2,1) (reference models/backbone.py:106) ------------------------------ */
int gdl_maxpool_fwd(const void* x, void* y, uint8_t* argmax, int N, int H, int W, int C, int Ho,
                    int Wo, gdl_stream_t s);
int gdl_maxpool_bwd(const void* dy, const uint8_t* argmax, void* dx, int N, int H, int W, int C,
                    int Ho, int Wo, gdl_stream_t s);

/* ---- global average pool (reference models/basic_model.py:73-82) ---------------------- */
/* x bf16 [B, G, C] (G = T*H*W pixels per sample) -> out f32 [B,C]. */
int gdl_gap_fwd(const void* x, float* out, int B, int G, int C, gdl_stream_t s);
/* dout f32 [B,C] -> dx bf16 [B,G,C] = dout/G. */
int gdl_gap_bwd(const float* dout, void* dx, int B, int G, int C, gdl_stream_t s);

/* ---- heads --------------------------------------------------------------------------- */
/* Generic Linear (reference models/fusion_modules.py nn.Linear call sites): y = x W^T + b.
 * W is [Out][In] with row stride ldw floats (so a column block of a wider matrix works). */
int gdl_linear_fwd(const float* x, const float* W, int ldw, const float* b, float* y, int B, int In,
                   int Out, gdl_stream_t s);
/* dx = dy W (if dx), dW (+)= dy^T x (row stride lddw), db (+)= sum dy (if dW / db);
 * accumulate: 0 overwrite, 1 add. */
int gdl_linear_bwd(const float* dy, const float* x, const float* W, int ldw, float* dx, float* dW,
                   int lddw, float* db, int B, int In, int Out, int accumulate, gdl_stream_t s);

/* Fused DGL head, forward + 3x softmax-CE + truncated backward in one pass over the logits
 * (reference models/fusion_modules.py:51-59 ConcatFusion_DGL / :22-30 SumFusion_DGL,
 * main_dgl.py:102-122).
 *   kind 0 = concat: Wx = fc_out.weight, Wy = Wx + D, ldw = 2D, one bias bx (by unused);
 *   kind 1 = sum   : Wx = fc_x.weight, Wy = fc_y.weight, ldw = D, biases bx, by.
 *   a,v        f32 [B,D]     pooled features
 *   logits     f32 [3,B,n]   out, out_a, out_v (reference return order basic_model.py:86)
 *   losses     f32 [3]       Lf, La, Lv = inv_batch * sum over the B local rows
 *   da,dv      f32 [B,D]     alpha*dLa/da, alpha*dLv/dv  (the encoders see ONLY these)
 *   dWx,dWy,dbx,dby          dLf/d(head params)          (the head sees ONLY Lf); row stride lddw
 *   scratch    f32 [gdl_head_scratch_floats(B,n)]
 */
int64_t gdl_head_scratch_floats(int B, int n);
int gdl_dgl_head_linear(int kind, const float* a, const float* v, const float* Wx, const float* Wy,
                        int ldw, const float* bx, const float* by, const int64_t* labels,
                        float alpha, float inv_batch, float* logits, float* losses, float* da,
                        float* dv, float* dWx, float* dWy, int lddw, float* dbx, float* dby,
                        float* scratch, int B, int D, int n, gdl_stream_t s);
/* Fused GatedFusion_DGL head (reference models/fusion_modules.py:230-250, main_dgl.py:102-122; x_gate=True):
 * hx = fc_x(a), hy = fc_y(v); out = fc_out(sigmoid(hx.detach()) * hy.detach()), out_a = fc_out(sigmoid(hx) * hx),
 * out_v = fc_out(sigmoid(hy) * hy); three CE; da = alpha*dLa/da, dv = alpha*dLv/dv through fc_out, the gates and
 * fc_x / fc_y; dWo/dbo = dLf/d(fc_out); fc_x / fc_y receive no gradient (never trained in the reference).
 * Weights [512][512] / [n][512] row-major fp32; logits f32 [3,B,n]; losses f32 [3]; D must be 512.
 * scratch f32 [gdl_gated_head_scratch_floats(B, n)]. */
int64_t gdl_gated_head_scratch_floats(int B, int n);
int gdl_dgl_head_gated(const float* a, const float* v, const float* Wx, const float* bx, const float* Wy,
                       const float* by, const float* Wo, const float* bo, const int64_t* labels, float alpha,
                       float inv_batch, float* logits, float* losses, float* da, float* dv, float* dWo, float* dbo,
                       float* scratch, int B, int D, int n, gdl_stream_t s);
/* Softmax-CE on given logits [B,n] (reference main_dgl.py:71,102-104 nn.CrossEntropyLoss):
 * loss_out[0] = loss_scale * sum_b loss_b; dlogits = grad_scale*(softmax-onehot) (may be NULL).
 * scratch f32 [B].  Used by the gated/film heads, whose layers run through gdl_linear_*. */
int gdl_softmax_ce(const float* logits, const int64_t* labels, float loss_scale, float grad_scale,
                   float* loss_out, float* dlogits, float* scratch, int B, int n, gdl_stream_t s);
/* Eval-mode head (reference valid(), main_dgl.py:168-222), one CTA per sample, from the bf16 NHWC layer-4 maps:
 *   fa bf16 [B][Ga][512] (audio, Ga = h*w), fv bf16 [B][Gv][512] (visual, Gv = T*h*w), both 16-byte aligned;
 *   global average pooling, then the three logit sets (out, out_a, out_v):
 *     kind 0 = concat: Wx = fc_out.weight, Wy = Wx + 512, ldw = 1024, bias bx (by unused);
 *     kind 1 = sum   : Wx = fc_x.weight, Wy = fc_y.weight, ldw = 512, biases bx, by;
 *     kind 2 = gated : Wx/bx = fc_x, Wy/by = fc_y (512 x 512), Wo/bo = fc_out; out = fc_out(sig(hx) hy) with
 *                      x_gate != 0, fc_out(sig(hy) hx) otherwise; out_a = fc_out(sig(hx) hx), out_v likewise;
 *     kind 3 = pooling only (the FiLM head continues with its GEMMs and gdl_eval_count);
 *   the arg-max of every row (lowest index on ties, NaN largest like torch.argmax) and, when labels != NULL,
 *   counts[h] += number of rows whose arg-max equals the label (int64 [3], device; a label < 0 never counts).
 *   a_out / v_out f32 [B][512] pooled features (may be NULL except for kind 3), logits f32 [3][B][n] (may be NULL);
 *   n <= 512. */
int gdl_eval_head(int kind, const void* fa, int Ga, const void* fv, int Gv, const float* Wx, const float* Wy,
                  int ldw, const float* bx, const float* by, const float* Wo, const float* bo, int x_gate,
                  const int64_t* labels, float* a_out, float* v_out, float* logits, int64_t* counts, int B, int n,
                  gdl_stream_t s);
/* counts[h] += #{b : argmax(logits[h][b][:]) == labels[b]} for h = 0, 1, 2; logits f32 [3][B][n]. */
int gdl_eval_count(const float* logits, const int64_t* labels, int64_t* counts, int B, int n, gdl_stream_t s);
/* Per-class report (opt-in beside gdl_eval_head / gdl_eval_count): for h = 0, 1, 2 and every row b of logits
 * f32 [3][B][n], pred = arg-max of the row (the same order as gdl_eval_head: NaN largest, ties to the lowest index)
 * and conf[h][labels[b]][pred] += 1 (int64 [3][n][n], device; rows = true class, columns = prediction).  A label < 0
 * is skipped; a label >= n adds 1 (once per row) to *out_of_range (int64, device) and writes nothing else.
 * 1 <= n <= 512, B > 0. */
int gdl_eval_confusion(const float* logits, const int64_t* labels, int64_t* conf, int64_t* out_of_range, int B, int n,
                       gdl_stream_t s);
/* Scores for average precision and top-k accuracy (opt-in, valid_report(ap=True)).  For h = 0, 1, 2 and every row b
 * of logits f32 [3][B][n]: p = softmax(logits[h][b]) in fp32 (row maximum subtracted first; fixed summation order) is
 * written class-major to store f32 [3][n][cap] at row *cursor + b, i.e. store[(h n + c) cap + *cursor + b], and the
 * label to store_labels int32 [cap] (-1 for a label outside 0..n-1).  hits[h] (int64 [3]) += the rows with a label in
 * 0..n-1 whose rank #{j : z_j > z_y} + #{j < y : z_j == z_y} (NaN largest, the arg-max order) is < k.  A row whose
 * store index is >= cap is not written; if its label is >= 0 it adds 1 to *overflow.  Then *cursor += B (a second,
 * one-thread launch), so a captured graph appends batch after batch.  1 <= n <= 512, 1 <= k <= n, B > 0,
 * 1 <= cap <= 2^28; all pointers are device pointers. */
int gdl_eval_scores(const float* logits, const int64_t* labels, int B, int n, int k, float* store,
                    int32_t* store_labels, int64_t cap, int64_t* cursor, int64_t* hits, int64_t* overflow,
                    gdl_stream_t s);
/* Per-class average precision over the N = min(*cursor, cap) rows of a gdl_eval_scores store whose label is in
 * 0..n-1: for column (h, c), AP = (1 / P_c) sum over the P_c rows i with label c of TP(>= s_i) / N(>= s_i), s_i the
 * row's score, N(>= t) the rows scoring >= t and TP(>= t) the positives among them (sklearn's
 * average_precision_score, ties included; a NaN score is the largest and ties with NaN).  Writes ap f64 [3][n] (NaN
 * for a class without rows), support int64 [n] (P_c) and *nonfinite (int64: the rows with a non-finite score in some
 * column).  Deterministic and bit-identical for any order of the rows.  Stores of more than 16384 rows sort in a
 * device workspace of gdl_eval_ap_workspace_bytes(cap, n) bytes (0 otherwise; 8-byte aligned). */
int64_t gdl_eval_ap_workspace_bytes(int64_t cap, int n);
int gdl_eval_ap(const float* store, const int32_t* store_labels, const int64_t* cursor, int64_t cap, int n, double* ap,
                int64_t* support, int64_t* nonfinite, void* workspace, int64_t workspace_bytes, gdl_stream_t s);
/* Gated-head elementwise pieces (reference models/fusion_modules.py:230-250). */
int gdl_gated_fwd(const float* hx, const float* hy, float* m_out, float* m_x, float* m_y,
                  int64_t numel, gdl_stream_t s);
int gdl_gated_bwd(const float* hx, const float* hy, const float* dm_x, const float* dm_y,
                  float* dhx, float* dhy, int64_t numel, gdl_stream_t s);

/* ---- FiLM_DGL head (reference models/fusion_modules.py:126-178: fc(512*512 -> 512) on the outer products
 * a (x) v, a (x) a, v (x) v, then fc_out).  Dense contractions on the tcgen05 flat-window kernels, operands
 * stored feature-major (see csrc/film.cu). -------------------------------------------------------------- */
/* C[M][N] bf16 = A[M][K] (row stride lda elements) * B[N][K]^T.  M % 128 == 0, N % 64 == 0, K % 64 == 0. */
int gdl_gemm_nt_bf16(const void* A, int64_t lda, const void* B, void* C, int64_t M, int N, int K,
                     gdl_stream_t s);
/* C[M][N] f32 = At[K][M]^T * Bt[K][N] (+ bias[N]); reduction over K (K % 128 == 0) with deterministic split-K.
 * M, N multiples of 128 (or M == 64).  workspace: gdl_gemm_tn_workspace_bytes(M, N, K). */
int64_t gdl_gemm_tn_workspace_bytes(int M, int N, int64_t K);
int gdl_gemm_tn_f32(const void* At, const void* Bt, const float* bias, float* C, int M, int N, int64_t K,
                    void* workspace, int64_t workspace_bytes, gdl_stream_t s);
/* Same, C += (a later K chunk of a reduction started by gdl_gemm_tn_f32; chunk order = summation order). */
int gdl_gemm_tn_f32_acc(const void* At, const void* Bt, float* C, int M, int N, int64_t K, void* workspace,
                        int64_t workspace_bytes, gdl_stream_t s);
/* Zt bf16 [D*D][ZB]: column b of variant 0 = a_b (x) v_b, variant 1 = a_b (x) a_b, variant 2 = v_b (x) v_b
 * (columns var*B + b; the rest zero).  a, v f32 [B][D]. */
int64_t gdl_film_scratch_floats(int B, int D); /* scratch of gdl_film_outer / gdl_film_contract */
int gdl_film_outer(const float* a, const float* v, void* Zt, int B, int D, int ZB, int variants, float* scratch,
                   gdl_stream_t s);
/* K-chunked form (the fused step never holds the whole 262144-row Zt): rows [f0, f0 + nf) of Zt into Zt_chunk[0 .. nf).
 * The chunk with f0 == 0 (re)builds the transposed features in scratch; run it first. */
int gdl_film_outer_chunk(const float* a, const float* v, void* Zt_chunk, int B, int D, int ZB, int variants,
                         float* scratch, int64_t f0, int64_t nf, gdl_stream_t s);
/* dst bf16 [drows][dcols], zero padded, from f32 rows [src0 (r0 rows); src1 (r1 rows)] of `cols` columns
 * (row stride ld); transpose != 0 writes dst[c][r]. */
int gdl_cast_pad_bf16(const float* src0, int r0, const float* src1, int r1, int cols, int ld, int transpose,
                      void* dst, int drows, int dcols, gdl_stream_t s);
/* G bf16 [D*D][ldg], batch row b in column c0+b: dx[b][i] = sum_j G[i*D+j]*y[b][j], dy[b][j] = sum_i G[i*D+j]*x[b][i];
 * sum_mode != 0: dx <- dx + dy (x == y), dy untouched. */
int gdl_film_contract(const void* G, int ldg, int c0, const float* x, const float* y, float* dx, float* dy,
                      int B, int D, int sum_mode, float* scratch, gdl_stream_t s);
/* K-chunked form: G_chunk holds the rows of i in [i0, i0 + ni) only (row (i - i0)*D + j).  accumulate == 0 (first
 * chunk) writes dx / dy, accumulate != 0 adds to them; rebuild_scratch != 0 re-transposes x, y into scratch. */
int gdl_film_contract_chunk(const void* G_chunk, int ldg, int c0, const float* x, const float* y, float* dx, float* dy,
                            int B, int D, int sum_mode, float* scratch, int i0, int ni, int accumulate,
                            int rebuild_scratch, gdl_stream_t s);
/* fp32 [R][Cn] <-> bf16 [Cn][R] (the feature-major shadow of fc.weight and its gradient). */
int gdl_transpose_f32_to_bf16(const float* src, void* dst, int R, int64_t Cn, gdl_stream_t s);
int gdl_transpose_bf16_to_f32(const void* src, float* dst, int R, int64_t Cn, gdl_stream_t s);
/* bf16 chunk [Cn][R] -> columns [c0, c0 + Cn) of the fp32 matrix dst [R][ldd]. */
int gdl_transpose_bf16_to_f32_window(const void* src, float* dst, int R, int64_t Cn, int64_t ldd, int64_t c0,
                                     gdl_stream_t s);

/* ---- FP32 check mode (north_star: "1e-4 with an FP32-accumulate check mode") -------------------------------
 * The encoder ops once more with fp32-STORED activations in the reference's own layout (NCHW activations, OIHW
 * weights = the nn.Parameters, no packing): CUDA-core kernels, fp64 accumulation, deterministic.  A check mode,
 * not a fallback — DGLStep(check_fp32=True) selects it explicitly so that the whole step can be compared
 * free-running with the fp32 reference (main_dgl.py:100 model(spec.unsqueeze(1).float(), image.float())).
 * d->Ci is ignored; ci_real is the true input-channel count (1 / 3 for the stems).
 * Call sites replaced: nn.Conv2d backbone.py:20-28,97-100; BatchNorm2d + ReLU (+ residual) :45-66,104-105;
 * MaxPool2d(3,2,1) :106; adaptive_avg_pool2d/3d basic_model.py:73-82; the frame fold backbone.py:162-164. */
int gdl_check_conv_fwd(const gdl_conv_desc* d, int ci_real, const float* x, const float* w_oihw, float* y,
                       gdl_stream_t s);
/* dx = conv_transpose(dy, w) (+ add, same shape as dx, may be NULL) */
int gdl_check_conv_dgrad(const gdl_conv_desc* d, int ci_real, const float* dy, const float* w_oihw,
                         const float* add, float* dx, gdl_stream_t s);
int gdl_check_conv_wgrad(const gdl_conv_desc* d, int ci_real, const float* x, const float* dy, float* dw_oihw,
                         gdl_stream_t s);
/* y = [relu](bn(x) [+ res]); training != 0: batch statistics + running-stat update, else running statistics.
 * mean / invstd f32 [C] are saved for the backward. */
int gdl_check_bn_fwd(const float* x, const float* res, float* y, int N, int C, int HW, const float* gamma,
                     const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                     float* mean, float* invstd, int relu, int training, gdl_stream_t s);
/* dz = relu ? dy*(y>0) : dy (written to dz when non-NULL: the residual branch's gradient); dgamma, dbeta, dx. */
int gdl_check_bn_bwd(const float* dy, const float* y, const float* x, float* dz, float* dx, int N, int C, int HW,
                     const float* gamma, const float* mean, const float* invstd, float* dgamma, float* dbeta,
                     int relu, gdl_stream_t s);
/* planes = N*C images of H x W; argmax = flat input index of the first maximum in scan order. */
int gdl_check_maxpool_fwd(const float* x, float* y, int32_t* argmax, int64_t planes, int H, int W, int Ho, int Wo,
                          gdl_stream_t s);
int gdl_check_maxpool_bwd(const float* dy, const int32_t* argmax, float* dx, int64_t planes, int H, int W, int Ho,
                          int Wo, gdl_stream_t s);
/* x f32 [B*T][C][HW] -> out f32 [B][C] (mean over t, hw) and its backward. */
int gdl_check_gap_fwd(const float* x, float* out, int B, int T, int C, int HW, gdl_stream_t s);
int gdl_check_gap_bwd(const float* dout, float* dx, int B, int T, int C, int HW, gdl_stream_t s);
/* src f32 [B][C][T][H][W] -> dst f32 [B*T][C][H][W]. */
int gdl_check_fold_frames(const float* src, float* dst, int B, int C, int T, int H, int W, gdl_stream_t s);

/* ---- optimizer / clipping / diagnostics (reference main_dgl.py:129-154,249) ---------- */
/* Flat fp32 gradient arena with a segment table: seg_end[nseg] (exclusive end offsets,
 * padding belongs to the preceding segment), seg_group[nseg] (0 = audio_net, 1 = visual_net,
 * 2 = fusion head) and seg_inv_numel[nseg] (1/numel of the parameter tensor).
 * stats_out f32 [4]: total L2 norm, clip coefficient min(1, max_norm/(norm+1e-6)),
 * audio  sum_p mean|g_p|*coef, visual sum_p mean|g_p|*coef  (main_dgl.py:132-143, computed on
 * the CLIPPED gradients like the reference).  scratch f32 [gdl_optim_scratch_floats()]. */
int64_t gdl_optim_scratch_floats(int64_t numel, int nseg);
int gdl_grad_stats(const float* grad, int64_t numel, const int64_t* seg_end,
                   const int32_t* seg_group, const float* seg_inv_numel, int nseg, float max_norm,
                   float* scratch, float* stats_out, gdl_stream_t s);
/* SGD-momentum with weight decay (torch.optim.SGD semantics, main_dgl.py:154,249):
 * g = grad*coef (written back, like clip_grad_norm_); g += wd*p; buf = first ? g : mu*buf+g;
 * p -= lr*buf.  coef is read from stats[1] on the device (may be NULL => 1). */
int gdl_sgd_momentum(float* param, float* grad, float* momentum_buf, int64_t numel, float lr,
                     float mu, float wd, int first_step, const float* stats, gdl_stream_t s);
/* Adam and Adagrad (torch.optim.Adam / Adagrad semantics, main_dgl.py:251-256; no amsgrad, maximize or decoupled
 * weight decay).  step_state int32 [3], device memory owned by the caller: [0] is the step count t (0 before the
 * first update, torch's state['step']), [1..2] scratch.  Each call launches a one-thread kernel that advances
 * t by one and derives the step's scalars from it in double precision, then the element kernel, so the count
 * advances on every replay of a captured graph (the *_lr_dev entries below read the lr on the device too).
 * Adam (32 bytes per element):
 *   g = grad*coef (written back); g += wd*p; m = lerp(m, g, 1-beta1); v = beta2*v + (1-beta2)*g*g;
 *   p -= (lr/(1-beta1^t)) * m / (sqrt(v)/sqrt(1-beta2^t) + eps).
 * Adagrad (24 bytes per element):
 *   g = grad*coef (written back); g += wd*p; s += g*g; p -= lr/(1+(t-1)*lr_decay) * g / (sqrt(s) + eps).
 * coef is read from stats[1] on the device (may be NULL => 1).  All arenas 16-byte aligned. */
int gdl_adam(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int32_t* step_state, int64_t numel,
             double lr, double beta1, double beta2, double eps, double wd, const float* stats, gdl_stream_t s);
int gdl_adagrad(float* param, float* grad, float* sum, int32_t* step_state, int64_t numel, double lr,
                double lr_decay, double eps, double wd, const float* stats, gdl_stream_t s);
/* The same three updates with the learning rate read from device memory (reference main_dgl.py:154
 * `optimizer.step()` under an lr scheduler): lr points to ONE float64 that the caller writes, stream-ordered, before
 * each update, so a graph captured once follows any lr schedule.  Same kernels, launches and results as the host-lr
 * entries above at the same lr: SGD casts *lr to float (as a float lr argument is rounded), Adam / Adagrad read it
 * in double in the one-thread kernel. */
int gdl_sgd_momentum_lr_dev(float* param, float* grad, float* momentum_buf, int64_t numel, const double* lr,
                            float mu, float wd, int first_step, const float* stats, gdl_stream_t s);
int gdl_adam_lr_dev(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int32_t* step_state,
                    int64_t numel, const double* lr, double beta1, double beta2, double eps, double wd,
                    const float* stats, gdl_stream_t s);
int gdl_adagrad_lr_dev(float* param, float* grad, float* sum, int32_t* step_state, int64_t numel, const double* lr,
                       double lr_decay, double eps, double wd, const float* stats, gdl_stream_t s);
/* Gradient accumulation over several replicas run one after another on one GPU (DGLStep replicas > 1):
 * dst = src (accumulate == 0, 8 bytes per element) or dst = dst + src (accumulate != 0, 12 bytes per element),
 * fp32, element-wise.  dst and src 16-byte aligned, numel > 0 (any value: a scalar tail covers numel % 4). */
int gdl_grad_accumulate(float* dst, const float* src, int64_t numel, int accumulate, gdl_stream_t s);

/* ---- visual data pipeline (reference dataset/CramedDataset.py:76-89,96-101; KSDataset.py:160-173,183-190) ---
 * RandomResizedCrop(S) | Resize((S,S)) -> RandomHorizontalFlip -> ToTensor -> Normalize for `frames` frames,
 * driven by the crop boxes / flips torchvision drew on the HOST (SURVEY.md §8f rank 2): bit-exact with
 * torchvision's PIL backend (Pillow Resample.c 8-bit two-pass bilinear, 22-bit fixed-point coefficients).
 *   store   uint8 [store_frames][Hs][Ws][3] decoded RGB frames resident in HBM (device pointer)
 *   params  int32 [frames][6] on the device: {store index, top i, left j, height h, width w, flip}
 *           (the test split's Resize((S,S)) is {idx, 0, 0, Hs, Ws, 0})
 *   mean3 / std3  HOST pointers to the three Normalize constants
 *   out     fp32 [frames/T][3][T][S][S] — the `image` tensor the reference's DataLoader yields (main_dgl.py:93)
 *   table   int32 [gdl_crop_table_ints(frames, S)] scratch for the per-frame resample coefficients
 * Frames up to 7.5x the output size (Hs, Ws <= 7.5*S).  Asynchronous, no allocation. */
int64_t gdl_crop_table_ints(int frames, int S);
int gdl_crop_resize_normalize(const uint8_t* store, int64_t store_frames, int Hs, int Ws, const int32_t* params,
                              int frames, int T, int S, const float* mean3, const float* std3, float* out,
                              int32_t* table, gdl_stream_t s);

/* ---- audio data pipeline (reference dataset/CramedDataset.py:60-66; KSDataset.py:138-150; VGGSoundDataset.py:112-122):
 * spectrogram = np.log(np.abs(librosa.stft(clip(wave, -1, 1), n_fft, hop_length)) + 1e-7), computed on the device
 * from decoded waveforms that stay resident in HBM (SURVEY.md §8f rank 2).  librosa.stft semantics: center=True,
 * periodic Hann window of n_fft samples, float64 window product and FFT, bins stored as complex64; abs / log in
 * float32.  The random draws stay on the host in the reference's order (KS/VGG: random.randint for the window start).
 *   waves     f32 [n_clips][clip_stride]   decoded mono waveforms (device)
 *   clip_len  i32 [n_clips]                valid samples per clip (device)
 *   params    i32 [B][2] (device)          {clip index, start sample}: sample i of item b is
 *                                          wave[clip][(start + i) mod clip_len] — np.tile(samples, 3)[:L] with start 0
 *                                          (CREMA-D) and the tile-to-10-s + [start : start + L] window of KS / VGGSound
 *   L         samples per item (22050*3 or 16000*5); frames = 1 + L / hop
 *   pad_mode  0 = reflect (librosa < 0.10, the era of the reference's README), 1 = zeros (librosa >= 0.10 default)
 *   out       f32 [B][1 + n_fft/2][frames]  — the `spec` tensor the reference's DataLoader yields (main_dgl.py:93)
 * n_fft a power of two in [64, 1024].  Asynchronous, no allocation. */
int gdl_log_stft(const float* waves, int64_t clip_stride, const int32_t* clip_len, const int32_t* params, int B,
                 int L, int n_fft, int hop, int pad_mode, float* out, gdl_stream_t s);

#ifdef __cplusplus
}
#endif
#endif /* GDL_B200_H_ */
