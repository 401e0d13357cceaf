/*
 * dd_b200.h -- C ABI of the B200-native six-camera scene pipeline (libdd_b200.so).
 *
 * The reference (annikabrundyn/driving-dirty) has no FFI: its hot path is PyTorch calls made
 * from LightningModule methods.  Each entry point below replaces the torch call(s) at the cited
 * reference lines (paths relative to /root/reference/src); INTEGRATION.md shows the ctypes stub
 * a maintainer adds at each site.
 *
 * Conventions
 *  - Every pointer is a DEVICE pointer owned by the caller (PyTorch's allocator); the library
 *    never allocates, frees or retains device memory.  `stream` is a cudaStream_t passed as
 *    void*; work is only enqueued on it, nothing synchronises the host.
 *  - Return value: 0 = ok, <0 = dd_status (bad argument / unsupported shape / wrong arch),
 *    >0 = cudaError_t from the launch.  dd_last_error() gives the text.  No fallbacks.
 *  - Activations inside the conv stack are NHWC ("pixel-major": [B][H][W][32 channels]), in
 *    fp32 (DD_F32) or bf16 (DD_BF16).  Weights, biases, gradients of weights, logits, losses
 *    are fp32 in torch layouts (OIHW, [out,in]).
 *  - "mosaic" = the 3 x H x 6W stitched image; "views" = the six 3 x H x W camera images of a
 *    scene in dataset order; slot j of the mosaic holds view DD_VIEW_ORDER[j] = {0,1,2,5,4,3}.
 */
#ifndef DD_B200_H
#define DD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum { DD_F32 = 0, DD_BF16 = 1 } dd_dtype;

typedef enum {
  DD_OK = 0,
  DD_ERR_BAD_ARG = -1,      /* null pointer, non-positive size */
  DD_ERR_UNSUPPORTED = -2,  /* shape/stride/dtype combination not implemented */
  DD_ERR_WORKSPACE = -3,    /* workspace too small (see dd_*_workspace_bytes) */
  DD_ERR_ALIGNMENT = -4,    /* pointer not aligned as the kernel requires */
  DD_ERR_ARCH = -5          /* device is not sm_100 */
} dd_status;

/* How a conv entry point should run: AUTO picks tcgen05 for bf16 where implemented. */
typedef enum { DD_IMPL_AUTO = 0, DD_IMPL_SIMT = 1, DD_IMPL_TCGEN05 = 2 } dd_impl;

int dd_version(void);
/* Copies the calling thread's last error text (NUL-terminated) into buf; returns its length. */
int dd_last_error(char* buf, size_t len);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
long long dd_launch_count(void);

/* ---- A1/A2: stitch ------------------------------------------------------------------------
 * roadmap_bce_v2.py:53-64 wide_stitch_six_images; autoencoder.py:53-73 six_to_one_task.
 * views [B,6,3,H,W] f32 -> mosaic [B,3,H,6W] f32.  The mask variant also writes
 * y [B,3,H,W] = mosaic[..., slot*W:(slot+1)*W] and zeroes that block of x. */
int dd_stitch_f32(const float* views, float* mosaic, int B, int H, int W, void* stream);
int dd_stitch_mask_f32(const float* views, float* x, float* y, int B, int H, int W, int slot,
                       void* stream);
/* Front-end for raw camera bytes (data_helper.py:109-114 ToTensor): views u8 [B,6,3,H,W] ->
 * mosaic f32 with value/255 (bit-identical to x.float()/255). */
int dd_stitch_u8(const uint8_t* views, float* mosaic, int B, int H, int W, void* stream);
/* Backward of the two stitches (autograd through wide_stitch_six_images / six_to_one_task):
 * dviews [B,6,3,H,W] f32 = the inverse permutation of dmosaic [B,3,H,6W].  slot = -1: dd_stitch_f32's
 * backward.  slot in [0,6): dd_stitch_mask_f32's -- the zeroed block of x passes no gradient, and
 * view DD_VIEW_ORDER[slot] takes dy [B,3,H,W], the gradient of y (dy may be NULL: zero). */
int dd_unstitch_f32(const float* dmosaic, const float* dy, float* dviews, int B, int H, int W, int slot,
                    void* stream);
/* ToTensor alone (data_helper.py:113): out[i] = float(in[i]) / 255, bit-identical, n elements of any layout. */
int dd_u8_to_f32(const uint8_t* in, float* out, long long n, void* stream);

/* ---- A3: encoder convs (components.py:19-21,41-43) ------------------------------------------
 * c1: 3->32, 3x3, pad 1, + bias + ReLU.  `in` is either the views [B,6,3,H,W] (in_flags &
 * DD_IN_VIEWS: the stitch is folded into the loads, Wm = 6W) or a mosaic / any NCHW image
 * [B,3,H,Wm]; fp32 in [0,1], or -- with DD_IN_U8, bf16 tensor-core path only -- the raw camera
 * bytes, with torchvision ToTensor's /255 (data_helper.py:109-114, roadmap_bce_v2.py:171) folded
 * into the loads, bit-identical to x.float()/255.  out: NHWC [B,H,Wm,32] of out_dtype. */
enum { DD_IN_VIEWS = 1, DD_IN_U8 = 2 };
int dd_conv_c1_fwd(const void* in, int in_flags, const float* w_oihw, const float* bias,
                   void* out, int out_dtype, int B, int H, int Wm, int impl, void* stream);
/* ReLU sign words: the ReLU mask of a1 / a2 for the input gradients of c2 / c3, 4 bytes per pixel instead of the
 * 64-byte activation.  One uint32 per pixel [B,H,W] (NHWC pixel order); bit c is 1 exactly when the stored bf16
 * activation of channel c is > 0.  `bits` must be 8-byte aligned.  The *_bits entry points run on the bf16 tensor-core
 * kernels only: fp32 or DD_IMPL_SIMT returns DD_ERR_UNSUPPORTED before anything runs.
 * dd_conv_c1_fwd_bits = dd_conv_c1_fwd (same out) that also writes out's sign words. */
int dd_conv_c1_fwd_bits(const void* in, int in_flags, const float* w_oihw, const float* bias, void* out,
                        uint32_t* bits, int out_dtype, int B, int H, int Wm, int impl, void* stream);
/* Inference front of the encoder in one kernel: a2 = relu(c2(relu(c1(x)))) (components.py:41-43), bf16 NHWC [B,H,Wm,32];
 * the first activation stays in shared memory / TMEM (halo recompute per 126-pixel x 64-row strip).  Same bits as
 * dd_conv_c1_fwd + dd_conv3x3_c32_fwd on the bf16 tensor-core path.  in / in_flags as for dd_conv_c1_fwd. */
int dd_encoder_c1c2_fused_fwd(const void* in, int in_flags, const float* w1_oihw, const float* bias1,
                              const float* w2_oihw, const float* bias2, void* a2, int B, int H, int Wm, void* stream);
/* dW [32,3,3,3], db [32] from dy = dL/d(out) ALREADY masked by out>0.  workspace: see below. */
int dd_conv_c1_wgrad(const void* in, int in_flags, const void* dy, int dtype, float* dw,
                     float* db, void* workspace, size_t ws_bytes, int B, int H, int Wm, int impl,
                     void* stream);

/* Image gradient of c1 (components.py:41, roadmap_bce_v2.py:53-64): what loss.backward() hands
 * the camera views or the mosaic.  dx[c,h,w] = sum over o, kh, kw of dy[o, h+1-kh, w+1-kw] *
 * w[o,c,kh,kw], zero outside the image; dy = dL/d(pre-activation of c1) (ReLU mask applied), NHWC
 * [B,H,Wm,32] of `dtype`, 16-byte aligned.  dx fp32: with out_flags & DD_IN_VIEWS the views
 * [B,6,3,H,Wm/6] (the inverse stitch folded into the stores), else the NCHW mosaic [B,3,H,Wm].
 * DD_IN_U8: DD_ERR_UNSUPPORTED (bytes have no gradient).  bf16 with AUTO / TCGEN05: tensor cores
 * (w read as bf16, as c1's forward reads it); fp32, or DD_IMPL_SIMT: CUDA cores, fp32 weights. */
int dd_conv_c1_dgrad(const void* dy, int dtype, const float* w_oihw, float* dx, int out_flags, int B,
                     int H, int Wm, int impl, void* stream);

/* c2 / c3: 32->32, 3x3, pad 1, stride 1 or 2, + bias + ReLU; NHWC in [B,H,W,32] ->
 * NHWC out [B,Ho,Wo,32], Ho = (H-1)/stride+1.  The bf16 tensor-core kernels read their activations
 * through TMA tensor maps built per call from the pointer and shape (nothing is cached): `in` / `dy`
 * / `x` must be 16-byte aligned and densely packed (DD_ERR_ALIGNMENT otherwise); outputs and the
 * ReLU-mask input are accessed in 32-byte pieces per pixel (64-byte pixels of a torch allocation
 * are always aligned). */
int dd_conv3x3_c32_fwd(const void* in, const float* w_oihw, const float* bias, void* out,
                       int dtype, int B, int H, int W, int stride, int impl, void* stream);
/* dx [B,H,W,32] = conv_transpose(dy, w) * (x > 0)   (x = this layer's input = previous
 * layer's post-ReLU output; pass x = NULL for no mask).  dy must already be masked. */
int dd_conv3x3_c32_dgrad(const void* dy, const float* w_oihw, const void* x, void* dx,
                         int dtype, int B, int H, int W, int stride, int impl, void* stream);
/* Sign-word forms (see dd_conv_c1_fwd_bits): the stride-1 forward also writes out's sign words; the input gradient
 * takes the mask from x's sign words (x_bits [B,H,W]) instead of x, bit-identical to passing x. */
int dd_conv3x3_c32_fwd_bits(const void* in, const float* w_oihw, const float* bias, void* out, uint32_t* bits,
                            int dtype, int B, int H, int W, int stride, int impl, void* stream);
int dd_conv3x3_c32_dgrad_bits(const void* dy, const float* w_oihw, const uint32_t* x_bits, void* dx,
                              int dtype, int B, int H, int W, int stride, int impl, void* stream);
/* dW [32,32,3,3] f32, db [32] f32 (overwritten, deterministic reduction order). */
int dd_conv3x3_c32_wgrad(const void* x, const void* dy, float* dw, float* db, void* workspace,
                         size_t ws_bytes, int dtype, int B, int H, int W, int stride, int impl,
                         void* stream);
size_t dd_conv_wgrad_workspace_bytes(void);

/* ---- A5: flatten + max_pool1d(4) over the NCHW-flat index (components.py:46-47) -------------
 * a3 NHWC [B,H,W,32] -> pooled [B, (32*H*W)/4] in the reference's feature order.
 * bwd: da3 = scatter of dpooled to the FIRST max of each window, times (a3 > 0). */
int dd_pool4_fwd(const void* a3, void* pooled, int dtype, int B, int H, int W, void* stream);
/* same, the pooled features always fp32 (a bf16 a3's maxima are exact in fp32): what Encoder.fc1 (components.py:105) reads on
 * the inference path, where no backward pass needs the bf16 copy */
int dd_pool4_fwd_f32(const void* a3, float* pooled, int dtype, int B, int H, int W, void* stream);
int dd_pool4_bwd(const void* a3, const void* dpooled, void* da3, int dtype, int B, int H, int W,
                 void* stream);

/* Layout changes at the API edge (c3_only "ssr" output, components.py:44-45; tests). */
int dd_nhwc_to_nchw_f32(const void* in, int in_dtype, float* out, int B, int C, int H, int W,
                        void* stream);
int dd_nchw_f32_to_nhwc(const float* in, void* out, int out_dtype, int B, int C, int H, int W,
                        void* stream);
/* g_masked = g * (act > 0), NHWC tensors of `dtype`, n elements. */
int dd_relu_mask(const void* g, const void* act, void* out, int dtype, long long n, void* stream);

/* ---- A6/A8: skinny linear layers (components.py:100,105; roadmap_bce_v2.py:50,75) -----------
 * y[B,N] = x[B,K] W[N,K]^T + bias.  W, bias, y, dW, db fp32; x / dx of x_dtype.  B <= 64.
 * Used for Encoder.fc1.fc1 (K = 940032), the roadmap head (N = 640000), Decoder.fc2.fc1. */
int dd_linear_fwd(const void* x, int x_dtype, const float* w, const float* bias, float* y,
                  void* workspace, size_t ws_bytes, int B, int N, long long K, int impl,
                  void* stream);
int dd_linear_dgrad(const float* dy, const float* w, void* dx, int dx_dtype, void* workspace,
                    size_t ws_bytes, int B, int N, long long K, int impl, void* stream);
int dd_linear_wgrad(const float* dy, const void* x, int x_dtype, float* dw, float* db, int B,
                    int N, long long K, int impl, void* stream);
/* Gradient accumulation over micro-batches (autograd's `.grad +=` on the wide weights between two optimizer steps, e.g.
 * Lightning's accumulate_grad_batches): accumulate = 0 is dd_linear_wgrad; accumulate = 1 writes dw = dw_old + D, where D is
 * bit for bit what dd_linear_wgrad writes for the same call -- for B > 32 too, whose 32-row chunks are summed before dw_old
 * is added, as autograd adds one finished gradient.  db (may be NULL) is always overwritten (the bias goes through autograd).
 * Errors as dd_linear_wgrad's (null pointer: DD_ERR_BAD_ARG; dw not 16-byte aligned: DD_ERR_ALIGNMENT; tcgen05 without its
 * shape or with bf16 x: DD_ERR_UNSUPPORTED), and accumulate with B > 128: DD_ERR_UNSUPPORTED. */
int dd_linear_wgrad_acc(const float* dy, const void* x, int x_dtype, float* dw, float* db, int B,
                        int N, long long K, int impl, int accumulate, void* stream);
/* The backward pass of a wide linear layer with torch.optim.Adam's update of W (roadmap_bce_v2.py:155) folded in, for world
 * size 1.  ONE pass over each weight tile: the tile of W, exp_avg and exp_avg_sq is loaded once, the input gradient dx is
 * computed from the OLD W (bit-identical to dd_linear_dgrad), the weight gradient dy^T x is formed on chip and never reaches
 * HBM, and W, exp_avg, exp_avg_sq are written back updated (24 bytes per parameter).  Same arithmetic as dd_adam_step
 * (grad_scale 1); `step` = t >= 1.  dx (x_dtype dx_dtype) may be NULL: no input gradient, and the workspace is then unused;
 * db (may be NULL) is written as by dd_linear_wgrad.  tcgen05 path only: fp32 x, B <= 32, dd_linear_tc_supported(B, N, K),
 * dy, x, W and the moments 16-byte aligned; workspace as for dd_linear_dgrad. */
int dd_linear_bwd_adam(const float* dy, const float* x, float* weight, float* exp_avg, float* exp_avg_sq, void* dx,
                       int dx_dtype, float* db, void* workspace, size_t ws_bytes, int B, int N, long long K, float lr,
                       float beta1, float beta2, float eps, float weight_decay, long long step, void* stream);
/* The last backward pass of a gradient-accumulation window with the step folded in: dd_linear_bwd_adam with the weight
 * gradient taken as dW + grad_partial, where dW is this pass's dy^T x and grad_partial fp32 [N,K] (16-byte aligned) holds
 * the sum of the window's earlier passes (dd_linear_wgrad_acc).  Bit for bit dd_linear_dgrad + dd_linear_wgrad_acc into
 * grad_partial + dd_adam_step from it; grad_partial is only read.  28 bytes per parameter (W, exp_avg, exp_avg_sq read and
 * written, grad_partial read) instead of the 40 of those three launches.  Errors as dd_linear_bwd_adam's: a null pointer,
 * B > 32 or step < 1: DD_ERR_BAD_ARG; no tensor-core path for the shape: DD_ERR_UNSUPPORTED; a pointer not 16-byte aligned:
 * DD_ERR_ALIGNMENT; workspace too small with dx: DD_ERR_WORKSPACE. */
int dd_linear_bwd_adam_acc(const float* dy, const float* x, float* weight, float* exp_avg, float* exp_avg_sq,
                           const float* grad_partial, void* dx, int dx_dtype, float* db, void* workspace, size_t ws_bytes,
                           int B, int N, long long K, float lr, float beta1, float beta2, float eps, float weight_decay,
                           long long step, void* stream);
/* The fused step that also reports the gradient's norm (FusedAdam's track_grad_norm): grad_partial NULL is
 * dd_linear_bwd_adam, non-NULL dd_linear_bwd_adam_acc, with the same results bit for bit (W, moments, dx, db), and in
 * addition *sumsq = the fp64 sum of g*g over the [N,K] gradient g that the step applies (dy^T x, or dy^T x + grad_partial),
 * each square exact in fp64 and the sum folded in a fixed order: the same bits on every run.  Only real elements count
 * (ragged N and K included).  sumsq: device, 8-byte aligned.  sumsq_ws: dd_grad_sumsq_workspace_bytes() bytes (passed as
 * sumsq_ws_bytes), zeroed by the caller ONCE (self-resetting); calls that share one must be ordered (one stream).  Errors as
 * dd_linear_bwd_adam's, plus a null sumsq / sumsq_ws: DD_ERR_BAD_ARG; sumsq misaligned: DD_ERR_ALIGNMENT; sumsq_ws too
 * small: DD_ERR_WORKSPACE. */
int dd_linear_bwd_adam_sumsq(const float* dy, const float* x, float* weight, float* exp_avg, float* exp_avg_sq,
                             const float* grad_partial, void* dx, int dx_dtype, float* db, void* workspace, size_t ws_bytes,
                             int B, int N, long long K, float lr, float beta1, float beta2, float eps, float weight_decay,
                             long long step, double* sumsq, void* sumsq_ws, size_t sumsq_ws_bytes, void* stream);
size_t dd_linear_workspace_bytes(int B, int N, long long K);
/* impl = DD_IMPL_TCGEN05 runs the weight-streaming tensor-core kernels (fp32 operands read as tf32 through
 * TMA; x must be fp32): allowed when this returns 1 (N, K multiples of 4, N*K >= 2^22).  DD_IMPL_AUTO
 * keeps the fp32 CUDA-core kernels (1e-5 parity). */
int dd_linear_tc_supported(int B, int N, long long K);

/* ---- A8-A11: sigmoid + BCE-with-logits + threat scores + binarise -----------------------------
 * roadmap_bce_v2.py:81 (sigmoid), :106 (binary_cross_entropy_with_logits, mean), :140 (.round()),
 * helper.py:74-77 (compute_ts_road_map, soft and rounded), in ONE pass over logits/target.
 * target: f32 {0,1} (target_is_u8=0) or u8/bool (1).  Optional outputs may be NULL:
 *   probs  f32 [n]  = sigmoid(logits)
 *   binary u8  [n]  = round_half_even(sigmoid(logits))  (== logits > 1.5*2^-24)
 * stats f32[4]  = {mean BCE, TS(target, probs), TS(target, binary), 0}
 * counts i64[4] = {sum target, sum binary, sum target*binary, n}
 * workspace: dd_bce_ts_workspace_bytes() bytes, zeroed by the caller ONCE (self-resetting). */
int dd_bce_ts_fwd(const float* logits, const void* target, int target_is_u8, float* probs,
                  uint8_t* binary, float* stats, long long* counts, void* workspace,
                  size_t ws_bytes, long long n, void* stream);
/* dlogits = (sigmoid(logits) - target) * (*grad_out) / n   (grad_out: device scalar or NULL=1) */
int dd_bce_bwd(const float* logits, const void* target, int target_is_u8, const float* grad_out,
               float* dlogits, long long n, void* stream);
size_t dd_bce_ts_workspace_bytes(void);
/* Standalone helper.py:74-77 on two f32 maps (any values): ts f32[1]. */
int dd_threat_score_f32(const float* a, const float* b, float* ts, void* workspace,
                        size_t ws_bytes, long long n, void* stream);

/* ---- A13/A15/A16: generic conv / transposed conv (any kernel, stride, padding, dilation) ------
 * Decoder dc1..dc4 (components.py:70-73,89-92); SpatialMappingCNN and RoadMapBoxesMergingCNN layers
 * (spatial_bb/components.py:18-26,129-139).  The descriptor states the FORWARD layer for all three
 * passes: x NHWC [B,Hi,Wi,Cin] -> y NHWC [B,Ho,Wo,Cout]; transposed = 1 for nn.ConvTranspose2d.
 * Weights fp32 in torch layout (Conv2d [Cout,Cin,kh,kw]; ConvTranspose2d [Cin,Cout,kh,kw]).
 * act: 0 none, 1 ReLU, 2 sigmoid (fused after the bias).  dgrad: dx = gather(dy, w) * (x_mask > 0),
 * x_mask may be NULL; dy must already carry this layer's own activation derivative.
 * wgrad: dw (torch layout), db (may be NULL); deterministic ordered reductions. */
typedef struct {
  int B, Cin, Cout, Hi, Wi, Ho, Wo;
  int kh, kw, sh, sw, ph, pw, dh, dw;
  int transposed;
} dd_conv_desc;
int dd_conv2d_fwd(const void* x, const float* w, const float* bias, void* y, const dd_conv_desc* d,
                  int dtype, int act, void* workspace, size_t ws_bytes, void* stream);
int dd_conv2d_dgrad(const void* dy, const float* w, const void* x_mask, void* dx,
                    const dd_conv_desc* d, int dtype, void* workspace, size_t ws_bytes, void* stream);
int dd_conv2d_wgrad(const void* x, const void* dy, float* dw, float* db, const dd_conv_desc* d,
                    int dtype, void* workspace, size_t ws_bytes, void* stream);
size_t dd_conv2d_workspace_bytes(const dd_conv_desc* d);
/* 1 when pass (0 forward, 1 input gradient, 2 weight gradient) of this layer runs on the tcgen05 implicit-GEMM kernels
 * (csrc/conv_dil_tc.cu, conv_dil_wgrad_tc.cu): bf16, stride 1, square filter of 3 or 7 taps with one dilation (1..7) /
 * padding for both axes, and (gathered, produced) channels in {(96,64), (64,32), (32,16), (32,32), (64,96), (32,64)}
 * (forward, input gradient) or {32,64,96} x {32,64} (weight gradient) once narrow tensors are zero-padded: 8 / 16
 * gathered channels to 32, and 8 produced channels to 16 (forward) or 8 / 16 to 32 (weight gradient) -- the merging
 * CNN's up_conv_1..4, rm_conv_2, out_conv and the decoder's dc1 / dc2.  Everything else (and fp32: the parity path, and
 * a sigmoid forward) runs on the CUDA-core engine. */
int dd_conv2d_tc_supported(const dd_conv_desc* d, int dtype, int pass);

/* ---- A15-A17: data movement and loss of the bounding-box model ------------------------------------
 * dd_view_extract: one camera of every scene as an NHWC image [B,H',W',3] with the rot90 / flip of
 * SpatialMappingCNN.forward (spatial_bb/components.py:34-62) folded into the indexing.
 *   mode 0 as is; 1 rot90(k=1,[2,3]); 2 rot90(k=1,[3,2]); 3 flip([2,3]).  views fp32 [B,6,3,H,W].
 * dd_nhwc_place: dir 0 copies small [B,h,w,c] into the window (oy,ox,oc) of big [B,H,W,C] (the
 *   torch.cat calls at components.py:66-73,156); dir 1 copies the window back out (their backward).
 * dd_sigmoid_bwd: out = dy * (1 - y) * y.
 * dd_bce_prob_*: F.binary_cross_entropy on probabilities, mean, logs clamped at -100
 *   (spatial_w_rm.py:131); bwd = g * (p - t) / max((1-p) p, 1e-12) / n. */
int dd_view_extract(const float* views, void* out, int out_dtype, int B, int H, int W, int view, int mode,
                    void* stream);
/* dd_view_extract_bwd: the backward of dd_view_extract.  dout NHWC [B,H',W',3] of dtype -> view
 * `view` of the fp32 views gradient dviews [B,6,3,H,W]; only that view's elements are written. */
int dd_view_extract_bwd(const void* dout, int dtype, float* dviews, int B, int H, int W, int view, int mode,
                        void* stream);
int dd_nhwc_place(void* small_, void* big, int dtype, int B, int h, int w, int c, int H, int W, int C,
                  int oy, int ox, int oc, int dir, void* stream);
int dd_sigmoid_bwd(const void* dy, const void* y, void* out, int dtype, long long n, void* stream);
int dd_bce_prob_fwd(const float* probs, const float* target, float* loss, void* workspace, size_t ws_bytes,
                    long long n, void* stream);
int dd_bce_prob_bwd(const float* probs, const float* target, const float* grad_out, float* dprobs,
                    long long n, void* stream);
size_t dd_bce_prob_workspace_bytes(void);

/* dd_boxes_to_map: the training target of the box model, boxes_to_binary_map (utils/bb_to_img.py:5-21) per scene as
 * BBSpatialRoadMap.bb_coord_to_map uses it (spatial_w_rm.py:85-95), bit for bit with the reference's Pillow fill.
 *   boxes: [total,2,4] on the device (metres; rows x / y; columns fl, fr, bl, br), float32 (boxes_f64 = 0) or float64 (1);
 *   pixel = metre * 10 + 400 in that dtype, polygon fl, fr, br, bl, filled as ImageDraw.polygon(fill=1) does.
 *   offsets: int32 [B+1] on the device, scene b owns boxes [offsets[b], offsets[b+1]).
 *   out: f32 [B,800,800] of 0./1., vertically flipped like the reference; every element is written.
 * B < 0 or a null pointer with B > 0: DD_ERR_BAD_ARG.  B == 0 enqueues nothing.  out not 16-byte aligned:
 * DD_ERR_ALIGNMENT. */
int dd_boxes_to_map(const void* boxes, int boxes_f64, const int* offsets, int B, float* out, void* stream);

/* ---- 8(f)3: bounding-box evaluation ------------------------------------------------------------------
 * compute_ats_bounding_boxes (helper.py:33-72, with compute_iou :79-83): boxes1 [n1,2,4], boxes2 [n2,2,4] fp32
 * (metres; rows x / y; columns fl, fr, bl, br) -> ats f32[1], the IoU-thresholded average threat score.
 * iou_matrix (optional, may be NULL): f32 [n1,n2], the reference's iou_matrix (0 where the extents do not overlap). */
int dd_ats_bounding_boxes(const float* boxes1, int n1, const float* boxes2, int n2, float* iou_matrix, float* ats,
                          void* stream);

/* ---- A14: mean squared error (autoencoder.py:91) ---------------------------------------------*/
int dd_mse_fwd(const float* y, const float* y_hat, float* loss, void* workspace, size_t ws_bytes,
               long long n, void* stream);
int dd_mse_bwd(const float* y, const float* y_hat, const float* grad_out, float* dy_hat,
               long long n, void* stream);

/* ---- A12 / 8(f): optimizer step ---------------------------------------------------------------
 * torch.optim.Adam(params, lr) at roadmap_bce_v2.py:155, autoencoder.py:120 (amsgrad off; weight_decay
 * is the L2 form added to the gradient).  One launch per tensor: param -= lr/(1-b1^t) * m / (sqrt(v)/
 * sqrt(1-b2^t) + eps) with m, v updated in place; `step` = t >= 1; the gradient is read as
 * grad * grad_scale.  All pointers fp32. */
int dd_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n,
                 float lr, float beta1, float beta2, float eps, float weight_decay, long long step,
                 float grad_scale, void* stream);
/* Data-parallel form (replaces Lightning ddp's gradient all-reduce + the N identical Adam updates):
 * this rank updates elements [shard_offset, shard_offset + shard_numel) of a parameter whose `world`
 * gradient / weight replicas are peer-mapped at grad_replicas[k] / param_replicas[k] (HOST arrays of
 * device pointers, index = rank).  The gradient is the SUM of the replicas times grad_scale (pass
 * 1/world for the mean); the new weights are written to every replica.  mc_grad / mc_param: NVLink
 * multicast addresses of the same buffers (both or neither; NULL = peer loads / stores).  exp_avg /
 * exp_avg_sq hold the shard only.  The caller puts a cross-rank barrier before (gradients complete)
 * and after (weights landed) on the same stream.  ctas_per_sm: 1..8 update CTAs (256 threads) per SM;
 * 1 leaves room for a persistent conv CTA beside each when the update overlaps the backward pass. */
int dd_adam_step_sharded(const void* const* grad_replicas, void* const* param_replicas,
                         const void* mc_grad, void* mc_param, int world, int rank,
                         float* exp_avg_shard, float* exp_avg_sq_shard, long long shard_offset,
                         long long shard_numel, float lr, float beta1, float beta2, float eps,
                         float weight_decay, long long step, float grad_scale, int ctas_per_sm,
                         void* stream);

/* Gradient clipping by the global L2 norm (torch.nn.utils.clip_grad_norm_(params, max_norm), Lightning's
 * gradient_clip_val), computed and applied on the device: the norm and coefficient never go to the host.
 * dd_grad_sumsq: the sum of g*g over `count` fp32 tensors given as HOST arrays ptrs[i] / numels[i]
 * (any length, 0 included, and any 4-byte alignment), in fp64, folded in a fixed order (the same bits
 * run to run).  Writes out[0] = total_norm = (float)sqrt(sum), out[1] = coef =
 * clamp(max_norm / (total_norm + 1e-6), max=1) in torch's fp32 arithmetic (NaN passes through the
 * clamp; an infinite norm gives 0) and the fp64 sum itself at out + 2.  out: device memory, 16 bytes,
 * 8-byte aligned.  max_norm: finite, >= 0.
 * workspace: dd_grad_sumsq_workspace_bytes() bytes, zeroed by the caller ONCE (self-resetting); calls
 * that share a workspace must be ordered (one stream).  Lists longer than 64 tensors take one launch
 * per 64. */
size_t dd_grad_sumsq_workspace_bytes(void);
int dd_grad_sumsq(const void* const* ptrs, const long long* numels, int count, float max_norm,
                  float* out, void* workspace, size_t ws_bytes, void* stream);
/* dd_adam_step with the gradient read as (grad * grad_scale) * (*coef), before the L2 weight-decay
 * term (the order of clip_grad_norm_ followed by torch.optim.Adam).  coef: device pointer to one
 * float, e.g. dd_grad_sumsq's out + 1.  *coef == 1 gives dd_adam_step's bits. */
int dd_adam_step_clipped(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n,
                         float lr, float beta1, float beta2, float eps, float weight_decay, long long step,
                         float grad_scale, const float* coef, void* stream);

/* Gradient norms per parameter (FusedAdam's track_grad_norm, Lightning's grad_norm), without a host round trip.
 * dd_adam_step_sharded_sumsq: dd_adam_step_sharded with the same results bit for bit, that also writes *sumsq = the fp64
 * sum of g*g over this rank's shard, g being the gradient exactly as the update consumes it (the sum of the replicas
 * in the kernel's order, times grad_scale); 0 for an empty shard.  Folded in a fixed order: the same bits on every run.
 * sumsq: device, 8-byte aligned (e.g. this rank's slot of a symmetric buffer, which the caller's closing barrier publishes
 * to the peers).  workspace: dd_grad_sumsq_workspace_bytes() bytes, zeroed ONCE (self-resetting); launches that share one
 * must be ordered.  Errors as dd_adam_step_sharded's, plus a null sumsq / workspace: DD_ERR_BAD_ARG; sumsq misaligned:
 * DD_ERR_ALIGNMENT; workspace too small: DD_ERR_WORKSPACE. */
int dd_adam_step_sharded_sumsq(const void* const* grad_replicas, void* const* param_replicas,
                               const void* mc_grad, void* mc_param, int world, int rank,
                               float* exp_avg_shard, float* exp_avg_sq_shard, long long shard_offset,
                               long long shard_numel, float lr, float beta1, float beta2, float eps,
                               float weight_decay, long long step, float grad_scale, int ctas_per_sm,
                               double* sumsq, void* workspace, size_t ws_bytes, void* stream);
/* dd_grad_sumsq_each: one fp64 sum of g*g per tensor, *outs[i] for tensor ptrs[i] / numels[i] (HOST arrays; fp32 tensors
 * of any length and any 4-byte alignment; outs[i]: device, 8-byte aligned).  Each sum is folded in a fixed order: the same
 * bits on every run.  Lists longer than 64 tensors take one launch per 64.
 * dd_grad_sumsq_each_replicas: the same for tensors of a data-parallel flat gradient bucket, whose `world` replicas are
 * peer-mapped at grad_replicas[k] (HOST array, index = rank, 16-byte aligned): tensor i is elements
 * [offsets[i], offsets[i] + numels[i]) of the bucket (offsets[i] a multiple of 4), and its gradient is the replicas' sum in
 * dd_adam_step_sharded's order for an element this rank owns (this rank's replica first, then rank+1, rank+2, ...), times
 * grad_scale -- so over this rank's shard it is exactly the gradient that rank's sharded update consumes.  The caller puts a
 * cross-rank barrier before (gradients complete) and keeps the replicas unchanged until every rank's call has finished.
 * workspace: dd_grad_sumsq_each_workspace_bytes() bytes, zeroed by the caller ONCE (self-resetting); calls that share a
 * workspace must be ordered.  Errors: a null pointer or negative length: DD_ERR_BAD_ARG; a tensor not 4-byte aligned, an
 * out not 8-byte aligned, an offset not a multiple of 4 or a replica not 16-byte aligned: DD_ERR_ALIGNMENT; world outside
 * 1..16 or rank outside the world: DD_ERR_BAD_ARG; workspace too small: DD_ERR_WORKSPACE. */
size_t dd_grad_sumsq_each_workspace_bytes(void);
int dd_grad_sumsq_each(const void* const* ptrs, const long long* numels, double* const* outs, int count,
                       void* workspace, size_t ws_bytes, void* stream);
int dd_grad_sumsq_each_replicas(const void* const* grad_replicas, int world, int rank, float grad_scale,
                                const long long* offsets, const long long* numels, double* const* outs, int count,
                                void* workspace, size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DD_B200_H */
