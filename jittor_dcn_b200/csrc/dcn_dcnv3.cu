// dcn_dcnv3.cu — DCNv3 (InternImage's ops_dcnv3 core: dcnv3_core_pytorch / dcnv3_im2col_cuda.cuh), channels-last,
// on float32, bfloat16 or float16 operands (float32 arithmetic throughout; see dcn_gather.cuh):
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
//
// DCNv4 (dcnv4_*_kernel) is the same chain with three changes: no softmax; offsets and mask packed into one tensor
// offset_mask [N, Ho, Wo, Cm], Cm = ceil(3*G*K / 8)*8, where group g owns elements [g*3K, g*3K + 3K) of a pixel's row
// (2K interleaved (dx, dy), then K mask values; columns [3*G*K, Cm) are padding, never read, written +0.0 in the
// gradient); and remove_center, which drops the centre point c = (kw/2)*kh + kh/2 of an odd kernel, so that sample
// s < K = kh*kw - 1 is grid point s + (s >= c).  A group's row starts only element-aligned (3K elements per group),
// so it is read and its gradient written one element at a time (PackedRows).
#include <type_traits>

#include <cuda_runtime.h>

#include "dcn_gather.cuh"

namespace dcn {

// DCNv4: elements per pixel row of offset_mask, Cm = ceil(3*G*K / 8)*8 with K = kh*kw - remove_center
long long dcnv4_row_floats(const DcnV3Shape& s) {
  const long long K = (long long)s.kh * s.kw - ((s.flags & DCN_V4_FLAG_REMOVE_CENTER) ? 1 : 0);
  return (3LL * s.G * K + 7) / 8 * 8;
}

namespace dcnv3 {

using gather::kThreads;
using gather::Smp;

// T: the storage type of every tensor but gvalue (float, __nv_bfloat16 or __half); gvalue is float (dcn_gather.cuh)
template <class T>
struct Args {
  // the gather core's fields (dcn_gather.cuh)
  const T* value;  // input [N, H, W, G*Gc]
  const T* loc;    // offset [N, Ho, Wo, G*P*2]
  const T* attn;   // mask [N, Ho, Wo, G*P]
  const T* gout;   // [N, Ho, Wo, G*Gc]          backward
  T* out;          // [N, Ho, Wo, G*Gc]          forward
  float* gvalue;   // like input, or null        backward
  T* gloc;         // like offset, or null       backward
  T* gattn;        // like mask, or null         backward
  int B, S, Q, M, D, L, P;  // N, H*W, Ho*Wo, G, Gc, 1, kh*kw (DCNv4: K)
  // the coordinate generator
  int H, W, Wo, kh, sh, sw, dh, dw;
  int p0x, p0y;  // hw - pw, hh - ph: the unscaled part of the kernel centre at (ho, wo) = (0, 0)
  int hw, hh;
  float os;
  // DCNv4 (PACKED): Cm = elements per pixel row of offset_mask; samples s >= center take grid point s + 1 (center = the
  // centre point with remove_center, else P: none)
  int Cm, center;
};

// Src::Rows of DCNv4's packed offset_mask (loc = offset_mask, gloc = gattn = grad_offset_mask): item (pixel, g) owns
// the 3P elements at pixel*Cm + g*3P, (dx, dy) of sample s at 2s, 2s + 1 and its mask at 2P + s.
struct PackedRows {
  template <class T>
  static __device__ __forceinline__ size_t at(const Args<T>& a, int item) {
    return (size_t)(item / a.M) * a.Cm + (size_t)(item % a.M) * 3 * a.P;
  }
  template <class T>
  static __device__ __forceinline__ const T* loc_row(const Args<T>& a, int item, int) { return a.loc + at(a, item); }
  template <class T>
  static __device__ __forceinline__ const T* attn_row(const Args<T>& a, int item, int) {
    return a.loc + at(a, item) + 2 * a.P;
  }
  template <class T>
  static __device__ __forceinline__ size_t grad_slot(const Args<T>& a, int item, int, int) { return at(a, item); }
  template <class T>
  static __device__ __forceinline__ void store_gattn(const Args<T>& a, size_t row, int s, float v) {
    gather::st1(a.gattn + row + 2 * a.P + s, v);
  }
  template <class T>
  static __device__ __forceinline__ void store_gloc(const Args<T>& a, size_t row, int s, float2 v) {
    T* p = a.gloc + row + 2 * s;
    gather::st1(p, v.x);
    gather::st1(p + 1, v.y);
  }
  // the padding columns of a pixel's row: +0.0, written by the group of its last item
  template <int G, class T>
  static __device__ __forceinline__ void end_grad(const Args<T>& a, int item, int j, bool live) {
    if (!a.gloc || !live || item % a.M != a.M - 1) return;
    const int used = a.M * 3 * a.P;
    T* p = a.gloc + (size_t)(item / a.M) * a.Cm + used;
    for (int c = j; c < a.Cm - used; c += G) gather::st1(p + c, 0.f);
  }
};

template <class T, bool SOFTMAX, bool PACKED = false>
struct Source {
  static_assert(!(SOFTMAX && PACKED), "DCNv4 has no softmax");
  using Args = dcnv3::Args<T>;
  using Rows = std::conditional_t<PACKED, PackedRows, gather::DenseRows>;
  struct Item {
    float x0, y0;   // (hw - pw + wo*sw) - hw*os, (hh - ph + ho*sh) - hh*os
    float mx, inv;  // softmax: max of the item's logits and 1 / sum exp(logit - max)
  };
  static constexpr bool kSoftmax = SOFTMAX;
  const Args& a;

  template <int G>
  __device__ __forceinline__ Item begin(int item, int j, const T* attnp) const {
    Item it;
    const int q = (item / a.M) % a.Q;
    const int ho = q / a.Wo, wo = q - ho * a.Wo;
    it.x0 = (float)(a.p0x + wo * a.sw) - (float)a.hw * a.os;
    it.y0 = (float)(a.p0y + ho * a.sh) - (float)a.hh * a.os;
    it.mx = 0.f;
    it.inv = 1.f;
    if constexpr (SOFTMAX) {  // the whole group is here (clamped items included): lane j reads logits j, j + G, ...
      float mx = -INFINITY;
      for (int s = j; s < a.P; s += G) mx = fmaxf(mx, gather::ld1(attnp + s));
      mx = gather::group_max<G>(mx);
      float sum = 0.f;
      for (int s = j; s < a.P; s += G) sum += expf(gather::ld1(attnp + s) - mx);
      it.mx = mx;
      it.inv = 1.f / gather::group_sum<G>(sum);
    }
    return it;
  }

  __device__ __forceinline__ Smp sample(const Item& it, const T* locp, const T* attnp, int s) const {
    float2 d;  // (dx, dy)
    int p = s;  // grid point
    if constexpr (PACKED) {
      d = make_float2(gather::ld1(locp + 2 * s), gather::ld1(locp + 2 * s + 1));
      p += s >= a.center;
    } else {
      d = gather::ld2(locp + 2 * s);
    }
    const int i = p / a.kh, jr = p - i * a.kh;  // kernel column, kernel row
    Smp r = gather::empty_sample();
    r.a = SOFTMAX ? expf(gather::ld1(attnp + s) - it.mx) * it.inv : gather::ld1(attnp + s);
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

// Forward on half types with V = 1: 6 blocks per SM (<= 40 registers), which they reach without spills.  Left to
// itself, ptxas aims the bf16 / fp16 Gc = 128 forward at full occupancy (32 registers) and spills there.  The float
// kernels keep the bound they always had.
template <class T, int V>
constexpr int kFwdMinBlocks = std::is_same_v<T, float> || V > 1 ? 0 : 6;

template <class T, int G, int V, bool SOFTMAX>
__global__ void __launch_bounds__(kThreads, kFwdMinBlocks<T, V>) dcnv3_fwd_kernel(const Args<T> a) {
  gather::fwd_body<G, V>(Source<T, SOFTMAX>{a});
}

template <class T, int G, int V, bool SOFTMAX>
__global__ void __launch_bounds__(kThreads) dcnv3_bwd_kernel(const Args<T> a) {
  gather::bwd_body<G, V>(Source<T, SOFTMAX>{a});
}

template <class T, int G, int V>
__global__ void __launch_bounds__(kThreads, kFwdMinBlocks<T, V>) dcnv4_fwd_kernel(const Args<T> a) {
  gather::fwd_body<G, V>(Source<T, false, true>{a});
}

template <class T, int G, int V>
__global__ void __launch_bounds__(kThreads) dcnv4_bwd_kernel(const Args<T> a) {
  gather::bwd_body<G, V>(Source<T, false, true>{a});
}

enum class Op { v3, v3_softmax, v4 };

// KernelScope names: [DCNv3 / DCNv4][forward / backward][float / bf16 / fp16]
static const char* const kNames[2][2][3] = {
    {{"dcnv3_fwd_kernel", "dcnv3_fwd_kernel_bf16", "dcnv3_fwd_kernel_f16"},
     {"dcnv3_bwd_kernel", "dcnv3_bwd_kernel_bf16", "dcnv3_bwd_kernel_f16"}},
    {{"dcnv4_fwd_kernel", "dcnv4_fwd_kernel_bf16", "dcnv4_fwd_kernel_f16"},
     {"dcnv4_bwd_kernel", "dcnv4_bwd_kernel_bf16", "dcnv4_bwd_kernel_f16"}}};

template <int G, int V, Op OP, class T>
static int launch(const Args<T>& a, bool backward, cudaStream_t st) {
  constexpr bool SOFTMAX = OP == Op::v3_softmax;
  constexpr int type = std::is_same_v<T, float> ? 0 : std::is_same_v<T, __nv_bfloat16> ? 1 : 2;
  const long long threads = (long long)a.B * a.Q * a.M * G;
  const unsigned blocks = (unsigned)((threads + kThreads - 1) / kThreads);
  const char* name = kNames[OP == Op::v4][backward][type];
  KernelScope scope(name, st);
  if constexpr (OP == Op::v4) {
    if (!backward) dcnv4_fwd_kernel<T, G, V><<<blocks, kThreads, 0, st>>>(a);
    else dcnv4_bwd_kernel<T, G, V><<<blocks, kThreads, 0, st>>>(a);
  } else {
    if (!backward) dcnv3_fwd_kernel<T, G, V, SOFTMAX><<<blocks, kThreads, 0, st>>>(a);
    else dcnv3_bwd_kernel<T, G, V, SOFTMAX><<<blocks, kThreads, 0, st>>>(a);
  }
  DCN_KERNEL_CHECK(name);
  return DCN_OK;
}

template <Op OP, class T>
static int dispatch_gc(const Args<T>& a, bool backward, cudaStream_t st) {
  switch (a.D) {
    case 16: return launch<4, 1, OP>(a, backward, st);
    case 32: return launch<8, 1, OP>(a, backward, st);
    case 64: return launch<16, 1, OP>(a, backward, st);
    case 128: return launch<32, 1, OP>(a, backward, st);
    case 256: return launch<32, 2, OP>(a, backward, st);
    default: set_error("dcnv3: Gc = %d is not supported", a.D); return DCN_ERR_UNSUPPORTED;
  }
}

template <class T>
static int dispatch(const Args<T>& a, bool softmax, bool backward, cudaStream_t st) {
  return softmax ? dispatch_gc<Op::v3_softmax>(a, backward, st) : dispatch_gc<Op::v3>(a, backward, st);
}

// f(T{}) with T the storage type of a DCN_OPERAND_* value (checked by the caller)
template <class F>
static int with_operand(int operand, F&& f) {
  if (operand == DCN_OPERAND_BF16) return f(__nv_bfloat16{});
  if (operand == DCN_OPERAND_FP16) return f(__half{});
  return f(float{});
}

template <class T>
static Args<T> make_args(const DcnV3Shape& s, int Ho, int Wo, float offset_scale, const void* input,
                         const void* offset, const void* mask) {
  Args<T> a{};
  a.value = (const T*)input; a.loc = (const T*)offset; a.attn = (const T*)mask;
  a.B = s.N; a.S = s.H * s.W; a.Q = Ho * Wo; a.M = s.G; a.D = s.Gc; a.L = 1; a.P = s.kh * s.kw;
  a.H = s.H; a.W = s.W; a.Wo = Wo; a.kh = s.kh; a.sh = s.sh; a.sw = s.sw; a.dh = s.dh; a.dw = s.dw;
  a.hw = (s.dw * (s.kw - 1)) >> 1;
  a.hh = (s.dh * (s.kh - 1)) >> 1;
  a.p0x = a.hw - s.pw;
  a.p0y = a.hh - s.ph;
  a.os = offset_scale;
  a.center = a.P;
  return a;
}

// DCNv4: P = K points per group, loc = offset_mask
template <class T>
static Args<T> make_args_v4(const DcnV3Shape& s, int Ho, int Wo, float offset_scale, const void* input,
                            const void* offset_mask) {
  Args<T> a = make_args<T>(s, Ho, Wo, offset_scale, input, offset_mask, offset_mask);
  const bool rc = s.flags & DCN_V4_FLAG_REMOVE_CENTER;
  a.P -= rc;
  a.center = rc ? (s.kw / 2) * s.kh + s.kh / 2 : a.P;
  a.Cm = (int)dcnv4_row_floats(s);  // < 2^31 (dcn_api.cu)
  return a;
}

}  // namespace dcnv3

// The C entry points (dcn_api.cu) validate the shape, the operand and every pointer, and compute the output extent
// Ho x Wo, before these run.  Every tensor is of the operand's type except ginput, which is float.
int dcnv3_forward(const DcnV3Shape& s, int operand, int Ho, int Wo, float offset_scale, const void* input,
                  const void* offset, const void* mask, void* out, cudaStream_t st) {
  return dcnv3::with_operand(operand, [&](auto t) {
    using T = decltype(t);
    dcnv3::Args<T> a = dcnv3::make_args<T>(s, Ho, Wo, offset_scale, input, offset, mask);
    a.out = (T*)out;
    return dcnv3::dispatch(a, s.flags & DCN_V3_FLAG_SOFTMAX_MASK, false, st);
  });
}

int dcnv3_backward(const DcnV3Shape& s, int operand, int Ho, int Wo, float offset_scale, const void* input,
                   const void* offset, const void* mask, const void* gout, float* ginput, void* goffset, void* gmask,
                   cudaStream_t st) {
  if (!ginput && !goffset && !gmask) return DCN_OK;
  if (ginput) DCN_CUDA_TRY(cudaMemsetAsync(ginput, 0, sizeof(float) * (size_t)s.N * s.H * s.W * s.G * s.Gc, st));
  return dcnv3::with_operand(operand, [&](auto t) {
    using T = decltype(t);
    dcnv3::Args<T> a = dcnv3::make_args<T>(s, Ho, Wo, offset_scale, input, offset, mask);
    a.gout = (const T*)gout; a.gvalue = ginput; a.gloc = (T*)goffset; a.gattn = (T*)gmask;
    return dcnv3::dispatch(a, s.flags & DCN_V3_FLAG_SOFTMAX_MASK, true, st);
  });
}

int dcnv4_forward(const DcnV3Shape& s, int operand, int Ho, int Wo, float offset_scale, const void* input,
                  const void* offset_mask, void* out, cudaStream_t st) {
  return dcnv3::with_operand(operand, [&](auto t) {
    using T = decltype(t);
    dcnv3::Args<T> a = dcnv3::make_args_v4<T>(s, Ho, Wo, offset_scale, input, offset_mask);
    a.out = (T*)out;
    return dcnv3::dispatch_gc<dcnv3::Op::v4>(a, false, st);
  });
}

int dcnv4_backward(const DcnV3Shape& s, int operand, int Ho, int Wo, float offset_scale, const void* input,
                   const void* offset_mask, const void* gout, float* ginput, void* goffset_mask, cudaStream_t st) {
  if (!ginput && !goffset_mask) return DCN_OK;
  if (ginput) DCN_CUDA_TRY(cudaMemsetAsync(ginput, 0, sizeof(float) * (size_t)s.N * s.H * s.W * s.G * s.Gc, st));
  return dcnv3::with_operand(operand, [&](auto t) {
    using T = decltype(t);
    dcnv3::Args<T> a = dcnv3::make_args_v4<T>(s, Ho, Wo, offset_scale, input, offset_mask);
    a.gout = (const T*)gout; a.gvalue = ginput; a.gloc = (T*)goffset_mask; a.gattn = (T*)goffset_mask;
    return dcnv3::dispatch_gc<dcnv3::Op::v4>(a, true, st);
  });
}

}  // namespace dcn
