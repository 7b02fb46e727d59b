// dcn_umma_bwd.cu — backward pass on the tensor path: orchestration.
//
//   grad_x, grad_offset   dcn_umma_bwd_data.cu: tcgen05 GEMM gA = gout * Wm whose TMEM accumulator is
//                 consumed in place by the bilinear col2im scatter (red.global.add.f32 into a
//                 channels-last grad copy) and the warp-shuffle coordinate-gradient reduction
//                 (both column layouts; shapes it cannot tile use dcn_simt.cu:bwd_data_kernel).
//   grad_weight   Torch layout, O <= 128 (bf16 operands: O <= 256): FUSED into the kernel above — its scatter warps already
//                 hold every sample's four corner values, so they also emit the blended sample as
//                 a bf16 hi/lo operand and a second TMEM accumulator set collects gW = gout^T * S:
//                 the whole backward touches x once.  Otherwise dcn_umma_fwd.cu (MODE_WGRAD):
//                 S re-sampled by the forward's plan / gather warps; nothing is materialised.
//   grad_bias     column sums of gout (dcn_simt.cu:bias_grad_kernel).
#include <cstdlib>
#include <type_traits>

#include "dcn_umma.h"
#include "dcn_umma_common.cuh"

namespace dcn {

bool umma_wgrad_supported(const Geo& g, int operand);
size_t umma_xt_bytes(const Geo& g, int operand);
int umma_wgrad_any(const Geo& g, int operand, const void* xt, const float* off, const void* gout, float* gw,
                   uint8_t* gtiles, cudaStream_t st, const float* mask = nullptr);
size_t umma_wgrad_gtile_bytes(const Geo& g, int operand);
bool umma_bwd_data_supported(const Geo& g, int operand);
size_t umma_bwd_data_wtile_bytes(const Geo& g, int operand);
bool umma_bwd_data_fuses_wgrad(const Geo& g, int operand);
int umma_bwd_data_any(const Geo& g, int operand, const void* xt, float* gxt, const float* off, const void* wt,
                      const void* gout, float* goff, float* gw, uint8_t* wtiles, uint8_t* gtiles,
                      cudaStream_t st, float* gb_fused = nullptr, const float* mask = nullptr,
                      float* gmask = nullptr);
size_t umma_bwd_data_gtile_bytes(const Geo& g, int operand);
bool o_groups(const Geo& g, int* size);
Geo o_group_geo(const Geo& g, int o0, int size);

static size_t plan_bytes(const Geo& g) { return align_up(sizeof(Tap) * (size_t)g.B * g.P, 1024); }

bool umma_bwd_supported(const Geo& g, int operand) {
  if (!umma_wgrad_supported(g, operand)) return false;
  // the generic data-gradient kernel is fp32 only: bf16 needs the tensor-path one
  return operand == DCN_OPERAND_FP32 || umma_bwd_data_supported(g, operand);
}

// shifted-view convolution kernels (dcn_conv.cu): preferred when they cover the shape
bool conv_offset_bwd_supported(const Geo& g, int O);
size_t conv_offset_wtile_bytes(const Geo& g, int O);
int conv_offset_backward(const Geo& g, int O, const float* xt, float* gxt, const float* goff, const float* woff,
                         float* gwoff, uint8_t* wtiles, cudaStream_t st);

// ---- companion offset convolution (PLAIN problem) inside the layer's backward pass ---------------------------------
// n_out = the conv's output channels (2N; 3N for the modulated layer's offset-and-mask conv)
static bool plain_bwd_ok(const Geo& g, int n_out) {
  Tiling t;
  if (!make_tiling(g, &t)) return false;
  if (conv_offset_bwd_supported(g, n_out)) return true;
  const Geo gp = plain_geo(g, t, false, n_out);
  return umma_bwd_data_supported(gp, DCN_OPERAND_FP32) && umma_bwd_data_fuses_wgrad(gp, DCN_OPERAND_FP32);
}

// decided on the largest output-channel group, which sizes every scratch region of umma_backward_any
bool umma_bwd_data_on_tensor_path(const Geo& g, int operand) {
  int gsize;
  if (!o_groups(g, &gsize)) return false;
  return operand != DCN_OPERAND_FP32 || umma_bwd_data_supported(o_group_geo(g, 0, gsize), operand);
}

// Whole-layer backward (DCN span + offset conv) on the tensor path: fp32 operands, one output-channel group or more,
// data gradient on the tcgen05 kernel (so that the channels-last grad_x accumulator exists for both passes).
bool umma_layer_bwd_supported(const Geo& g, int n_out) {
  int gsize;
  if (!o_groups(g, &gsize)) return false;
  const Geo g0 = o_group_geo(g, 0, gsize);
  return umma_bwd_supported(g0, DCN_OPERAND_FP32) && umma_bwd_data_supported(g0, DCN_OPERAND_FP32) &&
         plain_bwd_ok(g, n_out);
}

// The modulated layer's conv output gradient, per image b: g3[b] = [goff[b] (2N planes) ; gmask[b] * m * (1 - m)
// (N planes)], m = mask[b] = sigmoid(logit): the derivative of the sigmoid the forward epilogue applied.  Units of 4
// floats when a plane is a multiple of 4 long (then every segment boundary is too), else single floats.
template <int V>
__global__ void __launch_bounds__(256) pack_offset_mask_grad_kernel(size_t per_b, size_t n_off, size_t total,
                                                                    const float* __restrict__ goff,
                                                                    const float* __restrict__ gmask,
                                                                    const float* __restrict__ mask,
                                                                    float* __restrict__ g3) {
  using T = typename std::conditional<V == 4, float4, float>::type;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t b = i / per_b, r = i - b * per_b;
    T v;
    if (r < n_off) {
      v = __ldg(reinterpret_cast<const T*>(goff) + b * n_off + r);
    } else {
      const size_t k = b * (per_b - n_off) + (r - n_off);
      const T gm = __ldg(reinterpret_cast<const T*>(gmask) + k), m = __ldg(reinterpret_cast<const T*>(mask) + k);
      if constexpr (V == 4)
        v = make_float4(gm.x * (m.x * (1.f - m.x)), gm.y * (m.y * (1.f - m.y)), gm.z * (m.z * (1.f - m.z)),
                        gm.w * (m.w * (1.f - m.w)));
      else
        v = gm * (m * (1.f - m));
    }
    reinterpret_cast<T*>(g3)[i] = v;
  }
}

static int launch_pack_offset_mask_grad(const Geo& g, const float* goff, const float* gmask, const float* mask,
                                        float* g3, cudaStream_t st) {
  const int v = g.HW % 4 == 0 ? 4 : 1;
  const size_t per_b = (size_t)3 * g.N * g.HW / v, n_off = (size_t)2 * g.N * g.HW / v, total = per_b * g.B;
  const int grid = (int)(total / 256 + 1 < 148 * 16 ? total / 256 + 1 : 148 * 16);
  KernelScope scope("pack_offset_mask_grad_kernel", st);
  if (v == 4) pack_offset_mask_grad_kernel<4><<<grid, 256, 0, st>>>(per_b, n_off, total, goff, gmask, mask, g3);
  else pack_offset_mask_grad_kernel<1><<<grid, 256, 0, st>>>(per_b, n_off, total, goff, gmask, mask, g3);
  DCN_KERNEL_CHECK("pack_offset_mask_grad_kernel");
  return DCN_OK;
}

static size_t goff_bytes(const Geo& g) { return align_up(sizeof(float) * (size_t)g.B * 2 * g.N * g.HW, 1024); }
static size_t planes_bytes(const Geo& g, int ch) { return align_up(sizeof(float) * (size_t)g.B * ch * g.HW, 1024); }

// [xt][rest as umma_bwd_workspace, its tile regions sized for the larger of the two passes][grad_offset], and for the
// modulated layer (n_out = 3N) then [grad_mask][g3]
size_t umma_layer_bwd_workspace(const Geo& g, int n_out) {
  int gsize;
  if (!o_groups(g, &gsize)) return 0;
  const Geo g0 = o_group_geo(g, 0, gsize);
  Tiling t;
  if (!make_tiling(g, &t)) return 0;
  const Geo gp = plain_geo(g, t, false, n_out);
  const size_t tiles_dcn = umma_bwd_data_wtile_bytes(g0, DCN_OPERAND_FP32) + umma_bwd_data_gtile_bytes(g0, DCN_OPERAND_FP32);
  const size_t tiles_conv = conv_offset_bwd_supported(g, n_out) ? conv_offset_wtile_bytes(g, n_out) :
      umma_bwd_data_wtile_bytes(gp, DCN_OPERAND_FP32) + umma_bwd_data_gtile_bytes(gp, DCN_OPERAND_FP32);
  const size_t a = umma_xt_bytes(g, DCN_OPERAND_FP32) + (tiles_dcn > tiles_conv ? tiles_dcn : tiles_conv);
  const size_t c = umma_wgrad_gtile_bytes(g0, DCN_OPERAND_FP32);
  const size_t tail = goff_bytes(g) + (n_out == 2 * g.N ? 0 : planes_bytes(g, g.N) + planes_bytes(g, n_out));
  return umma_xt_bytes(g, DCN_OPERAND_FP32) + (a > c ? a : c) + tail;
}

size_t umma_bwd_workspace(const Geo& g, int operand) {
  // [xt] then either [gxt | Wm^T tiles | grad_out tiles] (tensor-path data gradient) or [sampling plan]
  // (generic); the unfused weight-gradient pass runs last and re-uses that region for its own staged
  // grad_out tiles
  const size_t a = umma_xt_bytes(g, DCN_OPERAND_FP32) + umma_bwd_data_wtile_bytes(g, operand) +
                   umma_bwd_data_gtile_bytes(g, operand);
  const size_t b = operand == DCN_OPERAND_FP32 ? plan_bytes(g) : 0;
  const size_t c = umma_wgrad_gtile_bytes(g, operand);
  const size_t m = a > b ? a : b;
  return umma_xt_bytes(g, operand) + (m > c ? m : c);
}

// g is the whole layer; the kernels run per output-channel group (dcn_umma_host.cu) — one group unless
// O > 256.  grad_x (via gxt) and grad_offset accumulate over the groups.
// woff != nullptr: whole-layer backward — the companion offset convolution's backward runs as a PLAIN pass between the
// DCN data gradient and the final transposition: grad_offset (goff) is its grad_out, its data gradient accumulates
// into the SAME channels-last grad_x buffer, gwoff / gboff receive its parameter gradients.
// mask != nullptr: modulated DCNv1 (DCNv2); gmask [B, N, Ho, Wo] is zeroed next to grad_offset and, like it, accumulates
// over the output-channel groups.  Every branch below passes the mask on: fused data + weight gradient, tensor-path
// data gradient + unfused weight gradient, generic data gradient + tensor-path weight gradient.
// woff and g3 != nullptr: the modulated whole layer, whose conv has 3N outputs (offsets, then mask logits).  Its output
// gradient g3 [B, 3N, Ho, Wo] = [grad_offset ; grad_mask * m * (1 - m)] is packed after the DCN data gradient and
// drives the conv's backward (shifted-view or warp-MMA kernels).
int umma_backward_any(const Geo& g, int operand, int flags, const void* xv, const float* off, const void* wtv,
                      const void* goutv, float* gx, float* goff, float* gw, float* gb, void* workspace,
                      cudaStream_t st, const float* woff, float* gwoff, float* gboff, const float* mask,
                      float* gmask, float* g3) {
  int gsize;
  if (!o_groups(g, &gsize)) {
    set_error("umma backward: O = %d cannot be split into groups", g.O);
    return DCN_ERR_UNSUPPORTED;
  }
  const Geo g0 = o_group_geo(g, 0, gsize);  // the largest group: sizes every scratch region
  const size_t esz = operand == DCN_OPERAND_BF16 ? 2 : 4;
  const void* x = xv;
  void* xt = workspace;
  uint8_t* rest = (uint8_t*)workspace + umma_xt_bytes(g, operand);
  Tiling t;
  if (!make_tiling(g, &t)) {
    set_error("umma backward: shape not tileable");
    return DCN_ERR_UNSUPPORTED;
  }
  int rc;
  // DCN_FLAG_XT_STAGED: the head of the workspace still holds the staged copy of x that dcn_forward
  // wrote for this very shape / operand (same layout in both phases) — skip the transpose
  if (!(flags & DCN_FLAG_XT_STAGED) && (rc = launch_nchw_to_nhwc(g, t, x, xt, operand, st))) return rc;
  const bool want_gx = !(flags & DCN_FLAG_NO_GRAD_X) && gx != nullptr;
  bool all_fused = true;
  const bool data_on_umma = umma_bwd_data_on_tensor_path(g, operand);
  if (data_on_umma) {
    // DCN_FLAG_GRAD_X_FRAMED: grad_x IS the framed channels-last accumulator (the producer-side post-op reads it in
    // that layout, dcn_bn_relu_backward_staged): scatter straight into the caller's buffer, no transposition at the end
    const bool gx_framed = (flags & DCN_FLAG_GRAD_X_FRAMED) != 0;
    float* gxt = gx_framed ? gx : (float*)rest;
    uint8_t* wtiles = rest + umma_xt_bytes(g, DCN_OPERAND_FP32);
    uint8_t* gtiles = wtiles + umma_bwd_data_wtile_bytes(g0, operand);
    if (want_gx) DCN_CUDA_TRY(cudaMemsetAsync(gxt, 0, sizeof(float) * (size_t)g.B * xt_image_stride(g), st));
    DCN_CUDA_TRY(cudaMemsetAsync(goff, 0, sizeof(float) * (size_t)g.B * 2 * g.N * g.HW, st));
    if (mask) DCN_CUDA_TRY(cudaMemsetAsync(gmask, 0, sizeof(float) * (size_t)g.B * g.N * g.HW, st));
    // Torch layout: the staging pass of grad_out sums grad_bias on its way (every element passes through it once)
    const bool gb_rides = gb != nullptr && g.variant == DCN_VARIANT_TORCH;
    if (gb_rides) DCN_CUDA_TRY(cudaMemsetAsync(gb, 0, sizeof(float) * (size_t)g.O, st));
    for (int o0 = 0; o0 < g.O; o0 += gsize) {
      const Geo gc = o_group_geo(g, o0, gsize);
      const bool fused = umma_bwd_data_fuses_wgrad(gc, operand);  // one pass over the samples yields gW as well
      all_fused = all_fused && fused;
      float* gwc = gw + (size_t)o0 * g.K;
      if (fused) DCN_CUDA_TRY(cudaMemsetAsync(gwc, 0, sizeof(float) * (size_t)gc.O * g.K, st));
      if ((rc = umma_bwd_data_any(gc, operand, xt, want_gx ? gxt : nullptr, off,
                                  (const uint8_t*)wtv + (size_t)o0 * g.K * esz,
                                  (const uint8_t*)goutv + (size_t)o0 * g.HW * esz, goff, gwc, wtiles, gtiles, st,
                                  gb_rides ? gb + o0 : nullptr, mask, gmask)))
        return rc;
    }
    if (woff) {
      // the conv's output count and output gradient: 2N and goff, or 3N and g3 = [goff ; gmask * m * (1 - m)]
      const int n_out = g3 ? 3 * g.N : 2 * g.N;
      const float* gconv = goff;
      if (g3) {
        if (!mask || !plain_bwd_ok(g, n_out)) {
          set_error("modulated layer backward: the offset-and-mask conv of this shape has no backward kernel");
          return DCN_ERR_UNSUPPORTED;
        }
        if ((rc = launch_pack_offset_mask_grad(g, goff, gmask, mask, g3, st))) return rc;
        gconv = g3;
      }
      const Geo gp = plain_geo(g, t, false, n_out);
      uint8_t* wtiles2 = rest + umma_xt_bytes(g, DCN_OPERAND_FP32);
      if (conv_offset_bwd_supported(g, n_out)) {
        if ((rc = conv_offset_backward(g, n_out, (const float*)xt, want_gx ? gxt : nullptr, gconv, woff, gwoff, wtiles2,
                                       st)))
          return rc;
      } else {
        // plain mode of the fused data-gradient kernel (stride 2 at 64+ channels: the shifted-view data gradient
        // would need four parity accumulators of 64 columns, more than TMEM holds double-buffered)
        uint8_t* gtiles2 = wtiles2 + umma_bwd_data_wtile_bytes(gp, DCN_OPERAND_FP32);
        DCN_CUDA_TRY(cudaMemsetAsync(gwoff, 0, sizeof(float) * (size_t)gp.O * g.K, st));
        if ((rc = umma_bwd_data_any(gp, DCN_OPERAND_FP32, xt, want_gx ? gxt : nullptr, nullptr, woff, gconv, nullptr,
                                    gwoff, wtiles2, gtiles2, st)))
          return rc;
      }
      if ((rc = launch_bias_grad(gp, gconv, DCN_OPERAND_FP32, gboff, st))) return rc;
    }
    if (want_gx && !gx_framed && (rc = launch_nhwc_to_nchw_add(g, t, gxt, gx, (flags & DCN_FLAG_ACCUM_GRAD_X) ? 1 : 0, st)))
      return rc;
    if (!gb_rides && (rc = launch_bias_grad(g, goutv, operand, gb, st))) return rc;
    if (all_fused) return DCN_OK;
  } else {
    if (woff) {
      set_error("layer backward: the data gradient of this shape does not run on the tensor path");
      return DCN_ERR_UNSUPPORTED;
    }
    all_fused = false;
    Tap* plan = (Tap*)rest;
    if ((rc = launch_plan(g, off, plan, st))) return rc;
    if ((rc = simt_backward(g, flags, (const float*)x, plan, (const float*)wtv, (const float*)goutv, gx, goff, gw,
                            gb, st, SIMT_BWD_DATA | SIMT_BWD_BIAS, mask, gmask)))
      return rc;
  }
  // everything that lived in `rest` (gxt, tiles, plan) is dead by now: the unfused weight-gradient
  // pass of the remaining groups stages its grad_out tiles there
  for (int o0 = 0; o0 < g.O; o0 += gsize) {
    const Geo gc = o_group_geo(g, o0, gsize);
    if (data_on_umma && umma_bwd_data_fuses_wgrad(gc, operand)) continue;
    if ((rc = umma_wgrad_any(gc, operand, xt, off, (const uint8_t*)goutv + (size_t)o0 * g.HW * esz,
                             gw + (size_t)o0 * g.K, rest, st, mask)))
      return rc;
  }
  return DCN_OK;
}

}  // namespace dcn

namespace dcn {

// Whole-layer backward: see umma_backward_any.  The internal grad_offset buffer, and with a mask the grad_mask and
// packed 3N-channel conv gradient buffers after it, sit at the tail of the workspace (umma_layer_bwd_workspace).
int umma_layer_backward(const Geo& g, int flags, const void* x, const float* off, const float* mask, const float* woff,
                        const void* wt, const void* gout, float* gx, float* gwoff, float* gboff, float* gw, float* gb,
                        void* workspace, size_t workspace_bytes, cudaStream_t st) {
  uint8_t* tail = (uint8_t*)workspace + workspace_bytes;
  float *g3 = nullptr, *gmask = nullptr;
  if (mask) {
    g3 = (float*)(tail -= planes_bytes(g, 3 * g.N));
    gmask = (float*)(tail -= planes_bytes(g, g.N));
  }
  float* goff = (float*)(tail - goff_bytes(g));
  return umma_backward_any(g, DCN_OPERAND_FP32, flags, x, off, wt, gout, gx, goff, gw, gb, workspace, st, woff, gwoff,
                           gboff, mask, gmask, g3);
}

}  // namespace dcn
