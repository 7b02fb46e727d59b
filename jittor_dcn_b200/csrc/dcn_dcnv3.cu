// dcn_dcnv3.cu — DCNv3 (InternImage's ops_dcnv3 core: dcnv3_core_pytorch / dcnv3_im2col_cuda.cuh), float32,
// channels-last:
//   out[n, ho, wo, g*Gc + c] = sum_p m[n, ho, wo, g*P + p] * bilinear(input[n, :, :, g*Gc + c], y_p, x_p)
// with P = kh*kw points in x-major order (p = i*kh + j: kernel column i, kernel row j), offsets (dx, dy) at
// offset[n, ho, wo, 2*(g*P + p)] and, in unpadded pixel coordinates (os = offset_scale, hw / hh = half the dilated
// kernel extent, rounded down),
//   x_p = (hw - pw + wo*sw) - hw*os + (i*dw + dx)*os,   y_p = (hh - ph + ho*sh) - hh*os + (j*dh + dy)*os
// evaluated in this order in fp32, as the original does.  Corners outside the image read 0 (grid_sample, bilinear,
// zeros padding, align_corners=False on the zero-padded input).  With DCN_V3_FLAG_SOFTMAX_MASK `mask` holds logits and
// m is their softmax over the P points of each (n, ho, wo, g): the forward takes max and sum by group shuffles before
// the samples, the backward returns the logits' gradient.
//
// This is the gather core of dcn_gather.cuh with one level: item (n, ho, wo, g) <-> (b, q, m) of multi-scale
// deformable attention with S = H*W tokens, Q = Ho*Wo queries, M = G heads of D = Gc channels; the location gradient
// is scaled by m*os.
#include <cuda_runtime.h>

#include "dcn_gather.cuh"

namespace dcn {

namespace dcnv3 {

using gather::kThreads;
using gather::Smp;

struct Args {
  // the gather core's fields (dcn_gather.cuh)
  const float* value;  // input [N, H, W, G*Gc]
  const float* loc;    // offset [N, Ho, Wo, G*P*2]
  const float* attn;   // mask [N, Ho, Wo, G*P]
  const float* gout;   // [N, Ho, Wo, G*Gc]          backward
  float* out;          // [N, Ho, Wo, G*Gc]          forward
  float* gvalue;       // like input, or null        backward
  float* gloc;         // like offset, or null       backward
  float* gattn;        // like mask, or null         backward
  int B, S, Q, M, D, L, P;  // N, H*W, Ho*Wo, G, Gc, 1, kh*kw
  // the coordinate generator
  int H, W, Wo, kh, sh, sw, dh, dw;
  int p0x, p0y;  // hw - pw, hh - ph: the unscaled part of the kernel centre at (ho, wo) = (0, 0)
  int hw, hh;
  float os;
};

template <bool SOFTMAX>
struct Source {
  using Args = dcnv3::Args;
  struct Item {
    float x0, y0;   // (hw - pw + wo*sw) - hw*os, (hh - ph + ho*sh) - hh*os
    float mx, inv;  // softmax: max of the item's logits and 1 / sum exp(logit - max)
  };
  static constexpr bool kSoftmax = SOFTMAX;
  const Args& a;

  template <int G>
  __device__ __forceinline__ Item begin(int item, int j, const float* attnp) const {
    Item it;
    const int q = (item / a.M) % a.Q;
    const int ho = q / a.Wo, wo = q - ho * a.Wo;
    it.x0 = (float)(a.p0x + wo * a.sw) - (float)a.hw * a.os;
    it.y0 = (float)(a.p0y + ho * a.sh) - (float)a.hh * a.os;
    it.mx = 0.f;
    it.inv = 1.f;
    if constexpr (SOFTMAX) {  // the whole group is here (clamped items included): lane j reads logits j, j + G, ...
      float mx = -INFINITY;
      for (int s = j; s < a.P; s += G) mx = fmaxf(mx, attnp[s]);
      mx = gather::group_max<G>(mx);
      float sum = 0.f;
      for (int s = j; s < a.P; s += G) sum += expf(attnp[s] - mx);
      it.mx = mx;
      it.inv = 1.f / gather::group_sum<G>(sum);
    }
    return it;
  }

  __device__ __forceinline__ Smp sample(const Item& it, const float* locp, const float* attnp, int s) const {
    const float2 d = *reinterpret_cast<const float2*>(locp + 2 * s);  // (dx, dy)
    const int i = s / a.kh, jr = s - i * a.kh;                        // kernel column, kernel row
    Smp r = gather::empty_sample();
    r.a = SOFTMAX ? expf(attnp[s] - it.mx) * it.inv : attnp[s];
    r.W = a.W;
    const float x = it.x0 + ((float)(i * a.dw) + d.x) * a.os;
    const float y = it.y0 + ((float)(jr * a.dh) + d.y) * a.os;
    gather::locate(r, x, y, a.H, a.W, 0, a.S);
    return r;
  }

  __device__ __forceinline__ float2 loc_scale(const Smp& own, int) const {
    return make_float2(own.a * a.os, own.a * a.os);
  }
};

template <int G, int V, bool SOFTMAX>
__global__ void __launch_bounds__(kThreads) dcnv3_fwd_kernel(const Args a) {
  gather::fwd_body<G, V>(Source<SOFTMAX>{a});
}

template <int G, int V, bool SOFTMAX>
__global__ void __launch_bounds__(kThreads) dcnv3_bwd_kernel(const Args a) {
  gather::bwd_body<G, V>(Source<SOFTMAX>{a});
}

template <int G, int V, bool SOFTMAX>
static int launch(const Args& a, bool backward, cudaStream_t st) {
  const long long threads = (long long)a.B * a.Q * a.M * G;
  const unsigned blocks = (unsigned)((threads + kThreads - 1) / kThreads);
  if (!backward) {
    KernelScope scope("dcnv3_fwd_kernel", st);
    dcnv3_fwd_kernel<G, V, SOFTMAX><<<blocks, kThreads, 0, st>>>(a);
    DCN_KERNEL_CHECK("dcnv3_fwd_kernel");
  } else {
    KernelScope scope("dcnv3_bwd_kernel", st);
    dcnv3_bwd_kernel<G, V, SOFTMAX><<<blocks, kThreads, 0, st>>>(a);
    DCN_KERNEL_CHECK("dcnv3_bwd_kernel");
  }
  return DCN_OK;
}

template <bool SOFTMAX>
static int dispatch_gc(const Args& a, bool backward, cudaStream_t st) {
  switch (a.D) {
    case 16: return launch<4, 1, SOFTMAX>(a, backward, st);
    case 32: return launch<8, 1, SOFTMAX>(a, backward, st);
    case 64: return launch<16, 1, SOFTMAX>(a, backward, st);
    case 128: return launch<32, 1, SOFTMAX>(a, backward, st);
    case 256: return launch<32, 2, SOFTMAX>(a, backward, st);
    default: set_error("dcnv3: Gc = %d is not supported", a.D); return DCN_ERR_UNSUPPORTED;
  }
}

static int dispatch(const Args& a, bool softmax, bool backward, cudaStream_t st) {
  return softmax ? dispatch_gc<true>(a, backward, st) : dispatch_gc<false>(a, backward, st);
}

static Args make_args(const DcnV3Shape& s, int Ho, int Wo, float offset_scale, const float* input,
                      const float* offset, const float* mask) {
  Args a{};
  a.value = input; a.loc = offset; a.attn = mask;
  a.B = s.N; a.S = s.H * s.W; a.Q = Ho * Wo; a.M = s.G; a.D = s.Gc; a.L = 1; a.P = s.kh * s.kw;
  a.H = s.H; a.W = s.W; a.Wo = Wo; a.kh = s.kh; a.sh = s.sh; a.sw = s.sw; a.dh = s.dh; a.dw = s.dw;
  a.hw = (s.dw * (s.kw - 1)) >> 1;
  a.hh = (s.dh * (s.kh - 1)) >> 1;
  a.p0x = a.hw - s.pw;
  a.p0y = a.hh - s.ph;
  a.os = offset_scale;
  return a;
}

}  // namespace dcnv3

// The C entry points (dcn_api.cu) validate the shape and every pointer, and compute the output extent Ho x Wo, before
// these run.
int dcnv3_forward(const DcnV3Shape& s, int Ho, int Wo, float offset_scale, const float* input, const float* offset,
                  const float* mask, float* out, cudaStream_t st) {
  dcnv3::Args a = dcnv3::make_args(s, Ho, Wo, offset_scale, input, offset, mask);
  a.out = out;
  return dcnv3::dispatch(a, s.flags & DCN_V3_FLAG_SOFTMAX_MASK, false, st);
}

int dcnv3_backward(const DcnV3Shape& s, int Ho, int Wo, float offset_scale, const float* input, const float* offset,
                   const float* mask, const float* gout, float* ginput, float* goffset, float* gmask, cudaStream_t st) {
  if (!ginput && !goffset && !gmask) return DCN_OK;
  if (ginput) DCN_CUDA_TRY(cudaMemsetAsync(ginput, 0, sizeof(float) * (size_t)s.N * s.H * s.W * s.G * s.Gc, st));
  dcnv3::Args a = dcnv3::make_args(s, Ho, Wo, offset_scale, input, offset, mask);
  a.gout = gout; a.gvalue = ginput; a.gloc = goffset; a.gattn = gmask;
  return dcnv3::dispatch(a, s.flags & DCN_V3_FLAG_SOFTMAX_MASK, true, st);
}

}  // namespace dcn
