// dcn_msda.cu — multi-scale deformable attention (Deformable DETR's MSDeformAttn core; mmcv's
// MultiScaleDeformableAttnFunction), float32:
//   out[b, q, m*D + d] = sum_{l,p} a[b,q,m,l,p] * bilinear(value_l[b, :, :, m, d], x*W_l - 0.5, y*H_l - 0.5)
// with (x, y) = sampling_locations[b,q,m,l,p] and corners outside level l reading 0 (grid_sample, zeros padding,
// align_corners=False, on 2*loc - 1).
//
// The kernels are the gather core of dcn_gather.cuh (one group of min(D/4, 32) lanes per (b, q, m), in-place float4
// corner loads, red.global.add.v4.f32 into grad_value, butterfly reduce-scatter and plain stores for the two
// coordinate-side gradients) with the sample source below: lane j reads location and weight of sample s0 + j
// (consecutive addresses across the group) and maps it into its level; the location gradient is scaled by a*W_l, a*H_l.
// spatial_shapes / level_start_index stay in device memory (no host synchronisation): each block copies them to
// shared memory, a level that cannot address `value` is treated as empty, and every corner's token index is checked
// against [0, S) before an address is formed.  That check is part of the release build: it validates input.
#include <cuda_runtime.h>

#include "dcn_gather.cuh"

namespace dcn {

namespace msda {

using gather::kThreads;
using gather::Smp;
constexpr int kMaxLevels = 16;

struct Args {
  const float* value;     // [B, S, M, D]
  const int64_t* shapes;  // [L, 2] = (H_l, W_l)
  const int64_t* starts;  // [L]
  const float* loc;       // [B, Q, M, L, P, 2]
  const float* attn;      // [B, Q, M, L, P]
  const float* gout;      // [B, Q, M*D]            backward
  float* out;             // [B, Q, M*D]            forward
  float* gvalue;          // [B, S, M, D] or null   backward
  float* gloc;            // like loc, or null      backward
  float* gattn;           // like attn, or null     backward
  int B, S, Q, M, D, L, P;
};

struct Level {
  int H, W, start;
};

__device__ __forceinline__ void load_levels(const Args& a, Level* lv) {
  for (int l = threadIdx.x; l < a.L; l += blockDim.x) {
    const long long H = a.shapes[2 * l], W = a.shapes[2 * l + 1], st = a.starts[l];
    const bool ok = H > 0 && W > 0 && H <= a.S && W <= a.S && st >= 0 && st < a.S;
    lv[l] = ok ? Level{(int)H, (int)W, (int)st} : Level{0, 0, 0};
  }
  __syncthreads();
}

// The gather core's sample source (dcn_gather.cuh): normalised locations on the levels of the block's level table.
struct Source {
  using Args = msda::Args;
  using Rows = gather::DenseRows;
  struct Item {};
  static constexpr bool kSoftmax = false;
  const Args& a;
  const Level* lv;

  template <int G>
  __device__ __forceinline__ Item begin(int, int, const float*) const { return Item{}; }

  __device__ __forceinline__ Smp sample(Item, const float* locp, const float* attnp, int s) const {
    const Level v = lv[s / a.P];
    const float2 xy = *reinterpret_cast<const float2*>(locp + 2 * s);
    Smp r = gather::empty_sample();
    r.a = attnp[s];
    r.W = v.W;
    gather::locate(r, fmaf(xy.x, (float)v.W, -0.5f), fmaf(xy.y, (float)v.H, -0.5f), v.H, v.W, v.start, a.S);
    return r;
  }

  __device__ __forceinline__ float2 loc_scale(const Smp& own, int s) const {
    const Level v = lv[s / a.P];
    return make_float2(own.a * (float)v.W, own.a * (float)v.H);
  }
};

template <int G, int V>
__global__ void __launch_bounds__(kThreads) msda_fwd_kernel(const Args a) {
  __shared__ Level lv[kMaxLevels];
  load_levels(a, lv);
  gather::fwd_body<G, V>(Source{a, lv});
}

template <int G, int V>
__global__ void __launch_bounds__(kThreads) msda_bwd_kernel(const Args a) {
  __shared__ Level lv[kMaxLevels];
  load_levels(a, lv);
  gather::bwd_body<G, V>(Source{a, lv});
}

template <int G, int V>
static int launch(const Args& a, bool backward, cudaStream_t st) {
  const long long threads = (long long)a.B * a.Q * a.M * G;
  const unsigned blocks = (unsigned)((threads + kThreads - 1) / kThreads);
  if (!backward) {
    KernelScope scope("msda_fwd_kernel", st);
    msda_fwd_kernel<G, V><<<blocks, kThreads, 0, st>>>(a);
    DCN_KERNEL_CHECK("msda_fwd_kernel");
  } else {
    KernelScope scope("msda_bwd_kernel", st);
    msda_bwd_kernel<G, V><<<blocks, kThreads, 0, st>>>(a);
    DCN_KERNEL_CHECK("msda_bwd_kernel");
  }
  return DCN_OK;
}

static int dispatch(const Args& a, bool backward, cudaStream_t st) {
  switch (a.D) {
    case 16: return launch<4, 1>(a, backward, st);
    case 32: return launch<8, 1>(a, backward, st);
    case 64: return launch<16, 1>(a, backward, st);
    case 128: return launch<32, 1>(a, backward, st);
    case 256: return launch<32, 2>(a, backward, st);
    default: set_error("msda: D = %d is not supported", a.D); return DCN_ERR_UNSUPPORTED;
  }
}

static Args make_args(const DcnMsdaShape& s, const float* value, const int64_t* shapes, const int64_t* starts,
                      const float* loc, const float* attn) {
  Args a{};
  a.value = value; a.shapes = shapes; a.starts = starts; a.loc = loc; a.attn = attn;
  a.B = s.B; a.S = s.S; a.Q = s.Q; a.M = s.M; a.D = s.D; a.L = s.L; a.P = s.P;
  return a;
}

}  // namespace msda

// The C entry points (dcn_api.cu) validate the shape and every pointer before these run.
int msda_forward(const DcnMsdaShape& s, const float* value, const int64_t* shapes, const int64_t* starts,
                 const float* loc, const float* attn, float* out, cudaStream_t st) {
  msda::Args a = msda::make_args(s, value, shapes, starts, loc, attn);
  a.out = out;
  return msda::dispatch(a, false, st);
}

int msda_backward(const DcnMsdaShape& s, const float* value, const int64_t* shapes, const int64_t* starts,
                  const float* loc, const float* attn, const float* gout, float* gvalue, float* gloc, float* gattn,
                  cudaStream_t st) {
  if (!gvalue && !gloc && !gattn) return DCN_OK;
  if (gvalue) DCN_CUDA_TRY(cudaMemsetAsync(gvalue, 0, sizeof(float) * (size_t)s.B * s.S * s.M * s.D, st));
  msda::Args a = msda::make_args(s, value, shapes, starts, loc, attn);
  a.gout = gout; a.gvalue = gvalue; a.gloc = gloc; a.gattn = gattn;
  return msda::dispatch(a, true, st);
}

}  // namespace dcn
