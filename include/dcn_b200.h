/*
 * dcn_b200.h — C ABI of libdcn_b200.so, the B200 (sm_100a) deformable-convolution engine
 * that sits below the `DeformConv2d` / `TorchDeformConv2d` module boundary of
 * x-y20/jittor-dcn.
 *
 * Everything the reference computes between "offsets are known" and "NCHW output is
 * returned" — and the autograd backward of that span — is behind these entry points:
 *
 *   reference span replaced (forward)   deform_conv.py:62-81 (+ grid_sample_wrapper :30-54)
 *                                       train.py:102-140
 *   reference span replaced (backward)  the autograd of the above, triggered at
 *                                       train.py:249 (loss.backward) / train.py:414
 *                                       (optimizer.backward)
 *
 * Beside it: multi-scale deformable attention (Deformable DETR's MSDeformAttn core), dcn_msda_forward /
 * dcn_msda_backward, DCNv3 (InternImage's core), dcn_v3_forward / dcn_v3_backward, and DCNv4, dcn_v4_forward /
 * dcn_v4_backward, below.
 *
 * The companion offset convolution (deform_conv.py:16-21,58 / train.py:80-85,98) stays a
 * framework convolution: its output is the `offset` argument here and `grad_offset` is
 * handed back to it.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the name
 *     says host; the caller owns every buffer including the workspace;
 *   - every function returns a DcnStatus (0 = OK, negative = error) and never throws;
 *     dcn_last_error() returns a thread-local human readable message for the last failure;
 *   - all work is enqueued on the caller's stream (`stream` is a cudaStream_t passed as
 *     void*; NULL = legacy default stream); nothing synchronises the device;
 *   - tensors are dense, contiguous, 16-byte aligned, NCHW, float32 (DCN_OPERAND_FP32) —
 *     see DcnShape.operand for the bf16 storage mode.
 */
#ifndef DCN_B200_H_
#define DCN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* every entry point below is exported; everything else in the library is hidden */
#if defined(__GNUC__)
#define DCN_API __attribute__((visibility("default")))
#else
#define DCN_API
#endif

#define DCN_B200_VERSION 100 /* major*10000 + minor*100 + patch */

typedef enum DcnStatus {
  DCN_OK = 0,
  DCN_ERR_BAD_SHAPE = -1,      /* non-positive dims, empty output, index space > 2^31 */
  DCN_ERR_NULL_POINTER = -2,   /* a required pointer is NULL */
  DCN_ERR_MISALIGNED = -3,     /* a pointer is not 16-byte aligned */
  DCN_ERR_WORKSPACE = -4,      /* workspace smaller than dcn_workspace_bytes() */
  DCN_ERR_CUDA = -5,           /* a CUDA runtime call failed (see dcn_last_error) */
  DCN_ERR_UNSUPPORTED = -6,    /* combination of variant / operand / flags not available */
  DCN_ERR_NCCL = -7            /* NCCL could not be loaded or a collective failed */
} DcnStatus;

/* Which of the reference's two (mathematically different) operators to reproduce. */
enum {
  /* deform_conv.py:56-81 — coordinates normalised by (W_out-1,H_out-1) (:34-38), columns
   * ordered (n, c) (:72-73). */
  DCN_VARIANT_JITTOR = 0,
  /* train.py:95-140 — coordinates normalised by (W_in-1,H_in-1) (:111-112), columns are the
   * memory-reinterpreting reshape of the [B,C,Ho,Wo,N] sample tensor (:129-131). */
  DCN_VARIANT_TORCH = 1,
  /* Not in the reference (SURVEY.md 8f.3): standard deformable convolution v1 as in
   * torchvision.ops.deform_conv2d / mmcv (one offset group, dilation 1; with a mask through
   * dcn_forward_modulated / dcn_backward_modulated = DCNv2): sampling point
   * (h*s - p + ki + dy, w*s - p + kj + dx), offsets interleaved (dy, dx) per tap, columns ordered
   * (c, tap).  Same kernels, different coordinate generator; torchvision is its oracle. */
  DCN_VARIANT_DCNV1 = 2
};

/* Storage / arithmetic mode of the dense contraction. */
enum {
  /* x, weight, out, grads: float32.  Tensor-core path uses a 3-term bf16 split
   * (hi*hi + hi*lo + lo*hi, fp32 accumulate; |err| ~ 5e-6 relative). */
  DCN_OPERAND_FP32 = 0,
  /* x, weight, grad_out stored as bfloat16; out, all gradients float32; fp32 accumulate. */
  DCN_OPERAND_BF16 = 1
};

/* DcnShape.flags */
enum {
  DCN_FLAG_ACCUM_GRAD_X = 1 << 0,  /* dcn_backward adds into grad_x instead of overwriting */
  DCN_FLAG_FORCE_SIMT = 1 << 1,    /* use the generic CUDA-core kernels even when the
                                      tcgen05 path supports the shape (A/B testing) */
  DCN_FLAG_NO_GRAD_X = 1 << 2,     /* dcn_backward: skip grad_x (first layer of a net) */
  DCN_FLAG_RELU_OUT = 1 << 3,      /* fused post-op epilogue (SURVEY 8f.2; train.py:167-170): dcn_forward / dcn_layer_forward
                                      store max(acc + bias, 0).  With eval-mode BatchNorm folded into weight / bias
                                      by the caller (scale_o = gamma_o / sqrt(var_o + eps); weight_o *= scale_o,
                                      bias_o = (bias_o - mean_o) * scale_o + beta_o) this is relu(bn(conv(x))) in the
                                      producing kernel.  The backward entry points take grad_out with respect to
                                      the PRE-activation sum: the caller masks it with out > 0 (the Python autograd
                                      nodes do); the flag itself is ignored there */
  DCN_FLAG_GRAD_X_FRAMED = 1 << 6, /* dcn_backward / dcn_layer_backward (tensor path): grad_x is NOT [B,C,H,W] but the framed
                                      channels-last accumulator itself — [B][(H+3) x (W+2)][C] floats in the layer's
                                      staging layout (dcn_staged_input_bytes) — overwritten; the post-op of the producer
                                      layer reads it in that layout (dcn_bn_relu_backward_staged).  dcn_backward,
                                      dcn_backward_modulated and dcn_layer_backward* return DCN_ERR_UNSUPPORTED, before
                                      any CUDA call, for this flag together with DCN_FLAG_ACCUM_GRAD_X, and for a
                                      shape / operand / flags whose data gradient does not run on the tensor path
                                      (dcn_path_name(s, DCN_PHASE_BACKWARD) other than "umma", or the generic fp32
                                      data-gradient kernel inside it) */
  DCN_FLAG_XT_STAGED = 1 << 4      /* the workspace is the very buffer a preceding call of this library for the
                                      same shape / operand was given (dcn_offset_conv_forward, dcn_forward or
                                      dcn_layer_forward; sized for the largest phase used) and nothing has written
                                      to it since, so its head still holds the staged copy of x: skip re-staging.
                                      Honoured by dcn_forward, dcn_backward, dcn_offset_conv_forward and
                                      dcn_layer_backward.  Meaningful on the tensor path (dcn_path_name == "umma") and on
                                      the materialised-sample path ("gemm": the sampling plan and the samples are kept
                                      as well); ignored otherwise */
};

/* Problem description.  Constructor arguments of the reference modules
 * (deform_conv.py:7-14, train.py:71-78) plus the input extent. */
typedef struct DcnShape {
  int32_t B, C, O;     /* batch, in_channels, out_channels */
  int32_t H, W;        /* input height / width */
  int32_t kh, kw;      /* kernel_size  (N = kh*kw taps) */
  int32_t sh, sw;      /* stride   — only enters through H_out/W_out (SURVEY A.1) */
  int32_t ph, pw;      /* padding  — idem */
  int32_t variant;     /* DCN_VARIANT_* */
  int32_t operand;     /* DCN_OPERAND_* */
  int32_t flags;       /* DCN_FLAG_* */
} DcnShape;

/* phases for dcn_workspace_bytes / dcn_path_name */
enum {
  DCN_PHASE_FORWARD = 0, DCN_PHASE_BACKWARD = 1, DCN_PHASE_CORNERS = 2,
  /* whole layer = companion offset convolution + DCN span (dcn_layer_forward / dcn_layer_backward); dcn_path_name
   * answers "umma" when the layer calls are available for the shape, "unsupported" otherwise (the caller then keeps
   * the offset conv on its framework and uses dcn_forward / dcn_backward) */
  DCN_PHASE_LAYER_FORWARD = 3, DCN_PHASE_LAYER_BACKWARD = 4,
  /* whole MODULATED layer (dcn_*_modulated layer calls below: 3N-channel offset-and-mask conv + DCNv2 span); "umma"
   * or "unsupported" as for the two phases above */
  DCN_PHASE_LAYER_FORWARD_MODULATED = 5, DCN_PHASE_LAYER_BACKWARD_MODULATED = 6
};

/* ---- introspection ---------------------------------------------------------------- */
DCN_API int dcn_version(void);
DCN_API const char* dcn_last_error(void);
DCN_API const char* dcn_status_string(int status);
/* H_out / W_out exactly as the offset conv produces them (deform_conv.py:34-35). */
DCN_API int dcn_output_hw(const DcnShape* s, int32_t* h_out, int32_t* w_out);
/* Bytes of caller-owned scratch the given phase needs (16-byte aligned). */
DCN_API size_t dcn_workspace_bytes(const DcnShape* s, int phase);
/* Name of the kernel family dcn_forward/dcn_backward will pick for this shape
 * ("umma" = fused tcgen05 implicit GEMM; "gemm" = Torch column layout whose gcd(Ho*Wo, C) is not a multiple of 16:
 * samples materialised once, contractions as plain cuBLAS GEMMs; "simt" = generic CUDA-core kernels). */
DCN_API const char* dcn_path_name(const DcnShape* s, int phase);
/* Number of kernel launches issued by this library (all threads of the process) since the
 * last reset (bench.py's gpu_launches). */
DCN_API uint64_t dcn_launch_count(void);
DCN_API void dcn_launch_count_reset(void);
/* Per-kernel timing for bench.py's roofline: between begin and end every kernel this
 * library launches (from any thread) is bracketed by CUDA events on its own stream.
 * dcn_profile_end synchronises those events and writes one line per kernel name:
 * "<name> <launches> <total_ms>\n" (NUL terminated, truncated to cap). */
DCN_API int dcn_profile_begin(void);
DCN_API int dcn_profile_end(char* out, size_t cap);

/* ---- the hot path ------------------------------------------------------------------ */

/* Forward: replaces deform_conv.py:62-81 / train.py:102-140.
 *   x       [B,C,H,W]            offset [B,2N,Ho,Wo]  (planar: channels 0..N-1 "x", N..2N-1 "y")
 *   weight  [O,C,kh,kw]          bias   [O] or NULL
 *   out     [B,O,Ho,Wo]                                                                   */
DCN_API int dcn_forward(const DcnShape* s, const void* x, const void* offset, const void* weight,
                const void* bias, void* out, void* workspace, size_t workspace_bytes,
                void* stream);

/* Backward: replaces the autograd of the same span (train.py:249, train.py:414).
 *   grad_out    [B,O,Ho,Wo]
 *   grad_x      [B,C,H,W]      (overwritten, or accumulated with DCN_FLAG_ACCUM_GRAD_X;
 *                               may be NULL with DCN_FLAG_NO_GRAD_X)
 *   grad_offset [B,2N,Ho,Wo]   grad_weight [O,C,kh,kw]   grad_bias [O] or NULL            */
DCN_API int dcn_backward(const DcnShape* s, const void* x, const void* offset, const void* weight,
                 const void* grad_out, void* grad_x, void* grad_offset, void* grad_weight,
                 void* grad_bias, void* workspace, size_t workspace_bytes, void* stream);

/* ---- modulated deformable convolution (DCNv2: torchvision.ops.deform_conv2d(..., mask=), mmcv's
 * ModulatedDeformConv2d) ------------------------------------------------------------------------------------------
 * DCN_VARIANT_DCNV1 sampling, every sample scaled by a per-(tap, output pixel) mask value:
 *   out[b,o,p]       = bias[o] + sum_{c,n} W[o,c,n] * m[b,n,p] * bil(x[b,c], sample(n,p))
 *   grad_mask[b,n,p] = sum_c gA[b,c,n,p] * bil(x[b,c], sample(n,p))   (gA = W^T grad_out; the UNmasked sample)
 * grad_x, grad_offset and grad_weight are those of dcn_backward with every sample (and its corner weights) scaled by m.
 *   mask        [B,N,Ho,Wo]  float32 in both operand modes, channel n = ki*kw + kj (torchvision's tap order); any
 *                            value is allowed (no range or sigmoid is applied)
 *   grad_mask   [B,N,Ho,Wo]  float32, overwritten; a sample with no corner inside the image gets 0
 * Both are required and 16-byte aligned.  Every other argument, flag, workspace size (dcn_workspace_bytes with
 * DCN_PHASE_FORWARD / DCN_PHASE_BACKWARD) and kernel family (dcn_path_name) is exactly that of dcn_forward /
 * dcn_backward: the mask needs no extra workspace and never moves a shape off the tensor path.
 * variant != DCN_VARIANT_DCNV1: DCN_ERR_UNSUPPORTED. */
DCN_API int dcn_forward_modulated(const DcnShape* s, const void* x, const void* offset, const void* mask,
                                  const void* weight, const void* bias, void* out,
                                  void* workspace, size_t workspace_bytes, void* stream);
DCN_API int dcn_backward_modulated(const DcnShape* s, const void* x, const void* offset, const void* mask,
                                   const void* weight, const void* grad_out, void* grad_x, void* grad_offset,
                                   void* grad_mask, void* grad_weight, void* grad_bias,
                                   void* workspace, size_t workspace_bytes, void* stream);

/* ---- the whole layer: companion offset convolution + DCN span (SURVEY 8f.1) ------------------------------------
 * The offset conv (deform_conv.py:16-21,58 / train.py:80-85,98: C -> 2N channels, same kernel / stride / padding) runs
 * as a "plain" mode of the same tcgen05 kernels: a regular convolution is the DCNv1 sampling with all offsets zero,
 * i.e. ONE exact pixel per (pixel, tap) instead of four weighted corners.  x is staged once for offset conv, DCN
 * forward and the whole backward; in the backward pass grad_offset never leaves the workspace and the offset conv's
 * data gradient accumulates into the same channels-last grad_x buffer as the DCN data gradient (one transposition
 * at the end).  fp32 operands; shapes: dcn_path_name(s, DCN_PHASE_LAYER_*) == "umma".
 *   offset_weight [2N,C,kh,kw]   offset_bias [2N] or NULL   offset [B,2N,Ho,Wo] (written by the forward pass and
 *   handed back to the backward pass: it is the saved activation)
 * dcn_offset_conv_forward alone computes `offset` (stages x unless DCN_FLAG_XT_STAGED); a following
 * dcn_forward with DCN_FLAG_XT_STAGED on the same workspace reuses the staged copy. */
DCN_API int dcn_offset_conv_forward(const DcnShape* s, const void* x, const void* offset_weight, const void* offset_bias,
                            void* offset, void* workspace, size_t workspace_bytes, void* stream);
DCN_API int dcn_layer_forward(const DcnShape* s, const void* x, const void* offset_weight, const void* offset_bias,
                      const void* weight, const void* bias, void* offset, void* out, void* workspace,
                      size_t workspace_bytes, void* stream);
/* grad_x may be NULL with DCN_FLAG_NO_GRAD_X; grad_offset_bias / grad_bias may be NULL. */
DCN_API int dcn_layer_backward(const DcnShape* s, const void* x, const void* offset, const void* offset_weight,
                       const void* weight, const void* grad_out, void* grad_x, void* grad_offset_weight,
                       void* grad_offset_bias, void* grad_weight, void* grad_bias, void* workspace,
                       size_t workspace_bytes, void* stream);

/* ---- the whole modulated layer (DCNv2): mmcv's ModulatedDeformConv2dPack / mmdet's DCNv2 backbone layers --------
 * That layer owns a conv_offset with 3N outputs (same kernel / stride / padding, bias): channels [0, 2N) are the
 * offsets (torchvision's interleaved (dy, dx) per tap, as dcn_forward_modulated reads them), channels [2N, 3N) one
 * mask logit per tap, and mask = sigmoid(logit).  Here that conv runs on the engine's own convolution kernels, its
 * epilogue writes `offset` and `mask` directly (no [B, 3N, Ho, Wo] tensor), and the modulated DCN span follows on the
 * same staged copy of x.  The backward pass packs the conv's output gradient [grad_offset ; grad_mask * m * (1 - m)]
 * inside the workspace, runs the conv's data gradient into the same channels-last grad_x accumulator as the DCN data
 * gradient (one transposition at the end) and returns the conv's parameter gradients.
 * DCN_VARIANT_DCNV1 and fp32 operands only (anything else: DCN_ERR_UNSUPPORTED); shapes: dcn_path_name(s,
 * DCN_PHASE_LAYER_*_MODULATED) == "umma", workspace: dcn_workspace_bytes with the same phases.  DCN_FLAG_NO_GRAD_X and
 * DCN_FLAG_XT_STAGED behave as in dcn_layer_*: one buffer of the larger phase size passed to both calls stages x once.
 *   offset_weight [3N,C,kh,kw]   offset_bias [3N] or NULL
 *   offset [B,2N,Ho,Wo] = conv channels [0,2N)   mask [B,N,Ho,Wo] = sigmoid(conv channels [2N,3N)) (bias added first)
 * offset and mask are written by the forward pass and handed back to the backward pass (the saved activations).
 *   grad_offset_weight [3N,C,kh,kw]   grad_offset_bias [3N] or NULL   grad_x may be NULL with DCN_FLAG_NO_GRAD_X */
DCN_API int dcn_offset_conv_forward_modulated(const DcnShape* s, const void* x, const void* offset_weight,
                                              const void* offset_bias, void* offset, void* mask, void* workspace,
                                              size_t workspace_bytes, void* stream);
DCN_API int dcn_layer_forward_modulated(const DcnShape* s, const void* x, const void* offset_weight,
                                        const void* offset_bias, const void* weight, const void* bias, void* offset,
                                        void* mask, void* out, void* workspace, size_t workspace_bytes, void* stream);
DCN_API int dcn_layer_backward_modulated(const DcnShape* s, const void* x, const void* offset, const void* mask,
                                         const void* offset_weight, const void* weight, const void* grad_out,
                                         void* grad_x, void* grad_offset_weight, void* grad_offset_bias,
                                         void* grad_weight, void* grad_bias, void* workspace, size_t workspace_bytes,
                                         void* stream);

/* ---- chained inference: channels-last activations between consecutive engine layers (SURVEY 8f.2) ----------------
 * dcn_layer_forward_chained is dcn_layer_forward whose epilogue writes the output DIRECTLY as the staged input of the
 * consumer layer: the framed channels-last copy at the head of `consumer_workspace` (the layout dcn_layer_forward /
 * dcn_forward would build from an NCHW tensor: [B][(Ho+3) x (Wo+2)][O] inside an all-zero frame, channels permuted
 * for a Torch-layout consumer).  The consumer is then called with DCN_FLAG_XT_STAGED on that workspace (its `x`
 * argument is not read), so no activation crosses the layer boundary in NCHW and no staging pass runs between the
 * layers.  With DCN_FLAG_RELU_OUT and eval-mode BatchNorm folded into weight / bias this chains the whole
 * relu(bn(conv(x))) stages of train.py:167-170.  Forward only (inference); fp32; both layers on the tensor path;
 * consumer->C == s->O, consumer->H / W == this layer's output extent, O <= 256.
 * The consumer's frame must be zero: dcn_staged_input_clear once after allocating its workspace is enough (the
 * chained epilogue only ever writes interior pixels).  dcn_staged_input_bytes = size of that staged copy. */
DCN_API size_t dcn_staged_input_bytes(const DcnShape* s);
DCN_API int dcn_staged_input_clear(const DcnShape* s, void* workspace, void* stream);
DCN_API int dcn_layer_forward_chained(const DcnShape* s, const DcnShape* consumer, const void* x,
                                      const void* offset_weight, const void* offset_bias, const void* weight,
                                      const void* bias, void* offset, void* consumer_workspace, void* workspace,
                                      size_t workspace_bytes, void* stream);

/* ---- training: channels-last hand-over between a layer's post-op and the next layer (SURVEY 8f.2) -----------------
 * dcn_bn_relu_forward_staged = dcn_bn_relu_forward whose normalise + ReLU pass writes its result DIRECTLY as the staged
 * input of the consumer layer (the framed channels-last copy at the head of `consumer_workspace`, frame zeroed here) —
 * the consumer then runs with DCN_FLAG_XT_STAGED; x [B,C,H,W] is the producer layer's NCHW output with
 * B, C, H, W = consumer->B, C, H, W.  dcn_bn_relu_backward_staged takes the gradient in the same layout — the
 * consumer's grad_x written with DCN_FLAG_GRAD_X_FRAMED — and returns grad_x [B,C,H,W] for the producer layer.
 * Per layer boundary two passes over the activation disappear in each direction (bn_apply + staging transposition ->
 * one kernel; un-staging transposition + bn_bwd_apply -> one kernel).  fp32; consumer on the tensor path.
 * saved / workspace as for dcn_bn_relu_forward. */
DCN_API int dcn_bn_relu_forward_staged(const DcnShape* consumer, int training, const void* x, const void* gamma,
                                       const void* beta, void* running_mean, void* running_var, float momentum, float eps,
                                       void* consumer_workspace, void* saved, void* workspace, size_t workspace_bytes,
                                       void* stream);
DCN_API int dcn_bn_relu_backward_staged(const DcnShape* consumer, int training, const void* x, const void* grad_staged,
                                        const void* saved, void* grad_x, void* grad_gamma, void* grad_beta,
                                        void* workspace, size_t workspace_bytes, void* stream);

/* Sampling geometry only (bit-exactness probe): for every (b, n, h, w)
 *   y0,x0 [B,N,Ho,Wo] int32   floor'ed row / column of the north-west corner
 *   w4    [B,N,Ho,Wo,4] f32   corner weights nw, ne, sw, se (unmasked)                     */
DCN_API int dcn_debug_corners(const DcnShape* s, const void* offset, int32_t* y0, int32_t* x0,
                      float* w4, void* stream);

/* ---- DeformRoIPool / DeformPSRoIPool (SURVEY 8f.4; deform_conv.py:83-157, 160-241) ----------------------------------
 * Only the pooled 1 x 1 case exists: both reference modules sum over the bin axis and then reshape [num_rois, C] to
 * [num_rois, C, pooled_h, pooled_w] (:137-157, :236-241), which is only defined for one bin.  Semantics as written in
 * the reference, including the clamp-then-subtract corner weights (:125-131):
 *   features [B,C,H,W] f32   rois [R,5] f32 = (batch index, x1, y1, x2, y2)
 *   offsets  [R,2] f32 = (x, y) of the single bin  (DeformRoIPool: offsets[:, 0, 0:2], scaled by roi_w / roi_h;
 *                         DeformPSRoIPool: offsets[:, 0:2], scaled by roi_w / roi_h * trans_std, skipped if no_trans)
 *   out      [R,C] f32 (the caller views it as [R,C,1,1])
 * Backward: grad_features [B,C,H,W] is zeroed and accumulated (may be NULL), grad_offsets [R,2] (may be NULL); rois
 * receive no gradient. */
enum { DCN_ROI_POOL = 0, DCN_PSROI_POOL = 1 };
DCN_API int dcn_roi_pool_forward(int kind, int B, int C, int H, int W, int R, const void* features, const void* rois,
                                 const void* offsets, float spatial_scale, float trans_std, int no_trans, void* out,
                                 void* stream);
DCN_API int dcn_roi_pool_backward(int kind, int B, int C, int H, int W, int R, const void* features, const void* rois,
                                  const void* offsets, float spatial_scale, float trans_std, int no_trans,
                                  const void* grad_out, void* grad_features, void* grad_offsets, void* stream);

/* ---- multi-scale deformable attention (Deformable DETR's MSDeformAttn core; mmcv's MultiScaleDeformableAttnFunction) ----
 *   out[b, q, m*D + d] = sum_{l,p} a[b,q,m,l,p] * bilinear(value_l[b, :, :, m, d], x*W_l - 0.5, y*H_l - 0.5)
 * with (x, y) = sampling_locations[b,q,m,l,p] normalised to [0, 1] (any value allowed) and corners outside level l
 * reading 0: F.grid_sample(bilinear, zeros, align_corners=False) on 2*loc - 1.  Tokens of `value` are level-major,
 * row-major inside a level (S = sum_l H_l*W_l).  The softmax of the weights happens outside; any value is allowed.
 *   value [B,S,M,D] f32   spatial_shapes [L,2] int64 = (H_l, W_l)   level_start_index [L] int64
 *   sampling_locations [B,Q,M,L,P,2] f32   attention_weights [B,Q,M,L,P] f32   out [B,Q,M*D] f32
 * spatial_shapes and level_start_index are DEVICE pointers and are read by the kernels only (no host synchronisation:
 * the calls can be captured in a CUDA graph); a level that does not fit [0, S) reads as empty and no corner outside
 * [0, S) is ever addressed.  Every pointer is 16-byte aligned.  No workspace.
 * Limits (anything else: DCN_ERR_UNSUPPORTED, or DCN_ERR_BAD_SHAPE for non-positive extents and index spaces):
 *   D in {16, 32, 64, 128, 256};  1 <= L <= 16;  1 <= P <= 32;  B*Q*M <= 2^31 - 1;  flags == 0.
 * Backward: grad_value [B,S,M,D] is zeroed and accumulated with atomics (its summation order is not deterministic);
 * grad_sampling_locations and grad_attention_weights are each written by one plain store per element, bit-identical
 * across runs.  Each of the three may be NULL (not computed); spatial_shapes / level_start_index get no gradient. */
typedef struct DcnMsdaShape {
  int32_t B, S, Q, M, D, L, P; /* batch, value tokens, queries, heads, channels per head, levels, points */
  int32_t flags;               /* must be 0 (reserved) */
} DcnMsdaShape;

DCN_API int dcn_msda_forward(const DcnMsdaShape* s, const void* value, const int64_t* spatial_shapes,
                             const int64_t* level_start_index, const void* sampling_locations,
                             const void* attention_weights, void* out, void* stream);
DCN_API int dcn_msda_backward(const DcnMsdaShape* s, const void* value, const int64_t* spatial_shapes,
                              const int64_t* level_start_index, const void* sampling_locations,
                              const void* attention_weights, const void* grad_out, void* grad_value,
                              void* grad_sampling_locations, void* grad_attention_weights, void* stream);

/* ---- DCNv3 (InternImage's ops_dcnv3 core: DCNv3Function / dcnv3_core_pytorch), float32, channels-last ---------------
 *   out[n, ho, wo, g*Gc + c] = sum_p m[n, ho, wo, g*P + p] * bilinear(input[n, :, :, g*Gc + c], y_p, x_p)
 * P = kh*kw points in x-major order: p = i*kh + j with kernel column i < kw and kernel row j < kh (for a square kernel
 * the transpose of torchvision's tap order).  Offsets are (dx, dy) per point: offset[n, ho, wo, 2*(g*P + p)] and
 * [... + 1].  With hw = (dw*(kw-1)) / 2, hh = (dh*(kh-1)) / 2 (rounded down) and os = offset_scale, in unpadded pixel
 * coordinates, evaluated in fp32 in this order:
 *   x_p = (hw - pw + wo*sw) - hw*os + (i*dw + dx)*os        y_p = (hh - ph + ho*sh) - hh*os + (j*dh + dy)*os
 * so os scales the dilation grid as well as the offsets.  Corners outside [0, H) x [0, W) read 0 (grid_sample, bilinear,
 * zeros, align_corners=False on the zero-padded input); a NaN coordinate contributes 0.
 *   Ho = (H + 2*ph - (dh*(kh-1) + 1)) / sh + 1 (rounded down), Wo likewise
 *   input [N,H,W,G*Gc] f32   offset [N,Ho,Wo,G*P*2] f32   mask [N,Ho,Wo,G*P] f32   out [N,Ho,Wo,G*Gc] f32
 * DCN_V3_FLAG_SOFTMAX_MASK: `mask` holds logits and m is their softmax over the P points of each (n, ho, wo, g)
 * (InternImage's module applies that softmax right before the core); grad_mask is then the logits' gradient.
 * Every pointer is 16-byte aligned.  No workspace and no host synchronisation: the calls can be captured in a CUDA graph.
 * Checked before any CUDA call, in this order:
 *   DCN_ERR_BAD_SHAPE     N, H, W, G, Gc, kh, kw < 1;  strides or dilations < 1;  paddings < 0;  Ho or Wo < 1;
 *                         N*Ho*Wo*G or N*H*W above 2^31 - 1
 *   DCN_ERR_NULL_POINTER / DCN_ERR_MISALIGNED   per pointer
 *   DCN_ERR_UNSUPPORTED   Gc not in {16, 32, 64, 128, 256};  P > 32;  a flag other than DCN_V3_FLAG_SOFTMAX_MASK
 * Backward: grad_input [N,H,W,G*Gc] is zeroed (cudaMemsetAsync) and accumulated with atomics (its summation order is not
 * deterministic); grad_offset and grad_mask are each written by one plain store per element, bit-identical across runs.
 * grad_offset = m*os*(sum_c g*dbil/dx, sum_c g*dbil/dy); grad_mask = sum_c g*bil, or with the softmax flag
 * m_p*(gamma_p - sum_q m_q*gamma_q) with gamma = sum_c g*bil.  Each of the three may be NULL (not computed).
 * InternImage's remove_center (the centre point dropped from the kernel) is not supported here; DCNv4 below has it. */
enum { DCN_V3_FLAG_SOFTMAX_MASK = 1 };

typedef struct DcnV3Shape {
  int32_t N, H, W, G, Gc;  /* batch, input extent, groups, channels per group (C = G*Gc) */
  int32_t kh, kw, sh, sw, ph, pw, dh, dw; /* kernel, stride, padding, dilation */
  int32_t flags;           /* DCN_V3_FLAG_* */
} DcnV3Shape;

DCN_API int dcn_v3_forward(const DcnV3Shape* s, float offset_scale, const void* input, const void* offset,
                           const void* mask, void* out, void* stream);
DCN_API int dcn_v3_backward(const DcnV3Shape* s, float offset_scale, const void* input, const void* offset,
                            const void* mask, const void* grad_out, void* grad_input, void* grad_offset,
                            void* grad_mask, void* stream);

/* ---- DCNv4 (the DCNv4 repository's DCNv4Function core), float32, channels-last --------------------------------------
 * DCNv3's operator and coordinate chain (above) with three changes:
 *   - no softmax: the mask is used as given;
 *   - offsets and mask packed into one tensor offset_mask [N, Ho, Wo, Cm], Cm = ceil(3*G*K / 8)*8.  Group g owns
 *     floats [g*3K, g*3K + 3K) of each pixel row: first 2K offsets as interleaved (dx, dy) per point, then K mask
 *     values.  Columns [3*G*K, Cm) are padding: never read (NaN there reaches no output);
 *   - DCN_V4_FLAG_REMOVE_CENTER drops the centre point of an odd kernel: K = kh*kw - 1 instead of kh*kw, and point
 *     k < K of a group is grid point p = k + (k >= c), c = (kw/2)*kh + kh/2, i.e. kernel column i = p / kh, row
 *     j = p % kh of DCNv3's x-major order (without the flag K = kh*kw and p = k).
 *   x_p = (hw - pw + wo*sw) - hw*os + (i*dw + dx)*os        y_p = (hh - ph + ho*sh) - hh*os + (j*dh + dy)*os
 *   input [N,H,W,G*Gc] f32   offset_mask [N,Ho,Wo,Cm] f32   out [N,Ho,Wo,G*Gc] f32
 * Every pointer is 16-byte aligned.  No workspace and no host synchronisation: the calls can be captured in a CUDA graph.
 * Checked before any CUDA call, in DCNv3's order and with its status codes, and in addition:
 *   DCN_ERR_BAD_SHAPE     K = 0 (a 1 x 1 kernel with remove_center);  Cm above 2^31 - 1
 *   DCN_ERR_UNSUPPORTED   Gc not in {16, 32, 64, 128, 256};  remove_center with an even kh or kw;  a flag other than
 *                         DCN_V4_FLAG_REMOVE_CENTER (DCN_V3_FLAG_SOFTMAX_MASK included).  K has no upper limit.
 * Backward: grad_input [N,H,W,G*Gc] is zeroed (cudaMemsetAsync) and accumulated with atomics (its summation order is not
 * deterministic).  grad_offset_mask [N,Ho,Wo,Cm] has offset_mask's layout: each non-padding element is written by one
 * plain store, bit-identical across runs, and the padding columns hold +0.0.  With g the incoming gradient and m the
 * point's mask value, per point:  (d dx, d dy) = m*os*(sum_c g*dbil/dx, sum_c g*dbil/dy);  d m = sum_c g*bil.
 * grad_input and grad_offset_mask may each be NULL (not computed). */
enum { DCN_V4_FLAG_REMOVE_CENTER = 2 };

DCN_API int dcn_v4_forward(const DcnV3Shape* s, float offset_scale, const void* input, const void* offset_mask,
                           void* out, void* stream);
DCN_API int dcn_v4_backward(const DcnV3Shape* s, float offset_scale, const void* input, const void* offset_mask,
                            const void* grad_out, void* grad_input, void* grad_offset_mask, void* stream);

/* ---- producer of the first DCN layer's input (train.py:145,166 / 307,328: conv1 = Conv2d(1, 16, 3, 1, 1)) ------------
 * A 3 x 3, stride 1, padding 1 convolution with Cin <= 4 input channels and O in {16, 32} outputs, float32 NCHW,
 * W % 4 == 0 (anything else: DCN_ERR_UNSUPPORTED, the caller keeps the framework's conv).  The framework's kernels for
 * this layer were 4.7 ms of the 24 ms detector step at batch 1024; these are two streaming kernels at the HBM floor.
 *   x [B,Cin,H,W]   weight [O,Cin,3,3]   bias [O] or NULL   out [B,O,H,W]
 * Backward: grad_weight [O,Cin,3,3] and grad_bias [O] are overwritten; there is no input gradient (network input). */
DCN_API int dcn_stem_conv_forward(int B, int Cin, int O, int H, int W, const void* x, const void* weight,
                                  const void* bias, void* out, void* stream);
DCN_API int dcn_stem_conv_backward(int B, int Cin, int O, int H, int W, const void* x, const void* grad_out,
                                   void* grad_weight, void* grad_bias, void* stream);

/* ---- post-op: BatchNorm2d + ReLU (SURVEY 8f.2) ------------------------------------------
 * Replaces `relu(bn(x))` after every DeformConv2d layer of the reference's detector (modules
 * train.py:146-159 / 311-322, call sites train.py:167-170 / 329-332): nn.BatchNorm2d semantics
 * (biased batch variance normalises, unbiased variance updates running_var, momentum as in torch)
 * with the ReLU fused on both sides.  NCHW float32, HW = H*W.  Every channel is split over many
 * CTAs (the framework kernels run one CTA per channel).
 *   gamma, beta   [C] or NULL (= 1, 0)      running_mean/var [C], updated in training mode, read in
 *   saved         4*C floats, written by the forward pass and handed to the backward pass       eval mode
 *   workspace     dcn_bn_workspace_bytes(C) bytes of caller-owned scratch                          */
DCN_API size_t dcn_bn_workspace_bytes(int32_t C);
DCN_API int dcn_bn_relu_forward(int32_t B, int32_t C, int32_t HW, int32_t training, const void* x,
                        const void* gamma, const void* beta, void* running_mean, void* running_var,
                        float momentum, float eps, void* y, void* saved, void* workspace,
                        size_t workspace_bytes, void* stream);
/* grad_x may be NULL (first layer); grad_gamma / grad_beta [C] or NULL. */
DCN_API int dcn_bn_relu_backward(int32_t B, int32_t C, int32_t HW, int32_t training, const void* x,
                         const void* grad_y, const void* saved, void* grad_x, void* grad_gamma,
                         void* grad_beta, void* workspace, size_t workspace_bytes, void* stream);

/* ---- data-parallel helpers (one process per GPU; NCCL over NVLink) --------------------
 * NCCL is dlopen'ed on first use; the core library has no link-time dependency on it.   */
DCN_API int dcn_comm_unique_id(void* out128_host);                     /* 128-byte ncclUniqueId  */
DCN_API int dcn_comm_init(int rank, int world, const void* unique_id128_host, void** comm);
/* buf[i] = scale * sum_over_ranks(buf[i]), in place, float32 */
DCN_API int dcn_allreduce_sum_f32(void* comm, void* buf, size_t count, float scale, void* stream);
DCN_API int dcn_comm_destroy(void* comm);

/* ---- the same all-reduce as ONE kernel over NVLink peer memory (csrc/dcn_p2p.cu) ----------------------------
 * For the gradient bucket of SURVEY.md 8(e) (1.74 MB: pure latency) every rank publishes its bucket in a buffer the
 * peers have mapped through CUDA IPC and sums all `world` copies itself, in rank order (bit-identical results on
 * every rank).  No NCCL, no host synchronisation; the exchange is sequenced by an epoch counter in device memory
 * that the kernel advances itself, so the call can be captured in a CUDA graph and replayed.
 *   dcn_p2p_create        allocates the published buffers (room for max_floats) on the current device
 *   dcn_p2p_local_handle  writes dcn_p2p_handle_bytes() bytes (a cudaIpcMemHandle_t) to host memory; the caller
 *                         gathers the handles of all ranks (any host-side transport), rank order, and passes the
 *                         concatenation to dcn_p2p_connect
 *   dcn_p2p_allreduce_sum_f32  buf[i] = scale * sum_ranks buf[i], in place; buf 16-byte aligned and readable /
 *                         writable up to the next multiple of 4 floats; every rank must call with the same count */
DCN_API size_t dcn_p2p_handle_bytes(void);
DCN_API int dcn_p2p_create(int rank, int world, size_t max_floats, void** comm);
DCN_API int dcn_p2p_local_handle(void* comm, void* out_handle_host);
DCN_API int dcn_p2p_connect(void* comm, const void* all_handles_host);
DCN_API int dcn_p2p_allreduce_sum_f32(void* comm, void* buf, size_t count, float scale, void* stream);
DCN_API int dcn_p2p_destroy(void* comm);

#ifdef __cplusplus
}
#endif
#endif /* DCN_B200_H_ */
