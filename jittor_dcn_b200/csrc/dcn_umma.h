// dcn_umma.h — interface of the tcgen05 / TMEM kernel family (dcn_umma_*.cu).
#pragma once
#include "dcn_common.cuh"

namespace dcn {

// Does the tensor-core path cover this problem?  (channel / output counts must tile the
// UMMA shapes; everything else goes to the generic kernels in dcn_simt.cu.)
bool umma_supported(const Geo& g, int operand, int phase);
size_t umma_workspace_bytes(const Geo& g, int operand, int phase);

// mask [B, N, Ho, Wo] (DCNv1 only; nullptr = unmodulated) scales every sample; gmask [B, N, Ho, Wo] receives its
// gradient (overwritten; required with a mask)
int umma_forward(const Geo& g, int operand, int flags, const void* x, const float* off,
                 const void* wt, const float* bias, void* out, void* workspace, cudaStream_t st,
                 const float* mask = nullptr);
int umma_backward(const Geo& g, int operand, int flags, const void* x, const float* off,
                  const void* wt, const void* gout, float* gx, float* goff, float* gw, float* gb,
                  void* workspace, cudaStream_t st, const float* mask = nullptr, float* gmask = nullptr);
// Does umma_backward run the data gradient of this problem on the tensor path (rather than the generic fp32 kernel)?
// Only that kernel writes grad_x in the framed channels-last layout (DCN_FLAG_GRAD_X_FRAMED).
bool umma_bwd_data_on_tensor_path(const Geo& g, int operand);

// ---- whole layer (companion offset conv as a PLAIN problem + DCN span), fp32 operands.  n_out: the conv's output
// channels, 2N, or 3N for the modulated layer (mmcv's ModulatedDeformConv2dPack: offsets, then one mask logit per tap)
bool umma_offset_conv_fwd_supported(const Geo& g, int n_out);
size_t umma_offset_conv_fwd_workspace(const Geo& g, int n_out);
// mask_out != nullptr: the modulated layer's conv (woff [3N, C, kh, kw], boff [3N]): offset_out [B, 2N, Ho, Wo] =
// channels [0, 2N), mask_out [B, N, Ho, Wo] = sigmoid(channels [2N, 3N)); needs umma_offset_conv_fwd_supported(g, 3N)
int umma_offset_conv_forward(const Geo& g, const void* x, const float* woff, const float* boff, float* offset_out,
                             void* workspace, cudaStream_t st, bool stage_x, float* mask_out = nullptr);
bool umma_layer_bwd_supported(const Geo& g, int n_out);
size_t umma_layer_bwd_workspace(const Geo& g, int n_out);
// mask != nullptr: the modulated layer (off / mask: what the forward wrote; gwoff [3N, C, kh, kw], gboff [3N] or null)
int umma_layer_backward(const Geo& g, int flags, const void* x, const float* off, const float* mask, const float* woff,
                        const void* wt, const void* gout, float* gx, float* gwoff, float* gboff, float* gw, float* gb,
                        void* workspace, size_t workspace_bytes, cudaStream_t st);

}  // namespace dcn
