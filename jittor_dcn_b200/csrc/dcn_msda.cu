// dcn_msda.cu — multi-scale deformable attention (Deformable DETR's MSDeformAttn core; mmcv's
// MultiScaleDeformableAttnFunction), float32:
//   out[b, q, m*D + d] = sum_{l,p} a[b,q,m,l,p] * bilinear(value_l[b, :, :, m, d], x*W_l - 0.5, y*H_l - 0.5)
// with (x, y) = sampling_locations[b,q,m,l,p] and corners outside level l reading 0 (grid_sample, zeros padding,
// align_corners=False, on 2*loc - 1).
//
// Mapping: a group of G = min(D/4, 32) lanes owns one item (b, q, m) and its D contiguous channels, V = D/(4G) float4
// per lane.  One corner of one head is 4*D contiguous bytes (one 128-byte line at D = 32), so every corner is read in
// place with one float4 load per lane; whether a corner is inside its level is the same for the whole group.
//   forward   the L*P samples of an item are cut into rounds of G: lane j reads location and weight of sample
//             s0 + j (consecutive addresses across the group), runs the coordinate chain once, and hands the result
//             to the group by shuffle.  `out` is written once, coalesced; no atomics.
//   backward  the same mapping with rounds of K = min(G, 8) samples.  Per sample and lane: grad_value[corner] +=
//             a*w_k*g (red.global.add.v4.f32, corners inside the level only) and three partials over the lane's
//             channels, sum g*bil (-> grad_attention_weights) and sum g*dbil/dx, sum g*dbil/dy (-> grad_sampling_
//             locations, scaled by a*W_l, a*H_l).  The 3K partials of a round are reduced over the group with the
//             butterfly reduce-scatter of dcn_umma_bwd_data.cu, after which lane j holds the totals of sample s0 + j —
//             the sample whose chain it computed — and writes its three gradient elements with plain stores.  Those
//             two gradients are therefore deterministic; only grad_value depends on the order of the atomics.
// spatial_shapes / level_start_index stay in device memory (no host synchronisation): each block copies them to
// shared memory, a level that cannot address `value` is treated as empty, and every corner's token index is checked
// against [0, S) before an address is formed.  That check is part of the release build: it validates input.
#include <cuda_runtime.h>

#include "dcn_common.cuh"

namespace dcn {

namespace msda {

constexpr int kThreads = 256;
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

// One sampling point after the coordinate chain.  mask bit k: corner k (NW, NE, SW, SE) lies inside the level and its
// token index inside [0, S).  base = token of the NW corner (meaningful only when mask != 0).
struct Smp {
  int base, W;
  unsigned mask;
  float fx, fy, a;
};

__device__ __forceinline__ void load_levels(const Args& a, Level* lv) {
  for (int l = threadIdx.x; l < a.L; l += blockDim.x) {
    const long long H = a.shapes[2 * l], W = a.shapes[2 * l + 1], st = a.starts[l];
    const bool ok = H > 0 && W > 0 && H <= a.S && W <= a.S && st >= 0 && st < a.S;
    lv[l] = ok ? Level{(int)H, (int)W, (int)st} : Level{0, 0, 0};
  }
  __syncthreads();
}

__device__ __forceinline__ Smp empty_sample() { return Smp{0, 0, 0u, 0.f, 0.f, 0.f}; }

__device__ __forceinline__ Smp make_sample(const Args& a, const Level* lv, const float* locp, const float* attnp,
                                           int s) {
  const Level v = lv[s / a.P];
  const float2 xy = *reinterpret_cast<const float2*>(locp + 2 * s);
  Smp r = empty_sample();
  r.a = attnp[s];
  r.W = v.W;
  const float x = fmaf(xy.x, (float)v.W, -0.5f), y = fmaf(xy.y, (float)v.H, -0.5f);
  const float xf = floorf(x), yf = floorf(y);
  const int x0 = sat_int(xf), y0 = sat_int(yf);
  const long long base = (long long)v.start + (long long)y0 * v.W + x0;
  unsigned m = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int dy = k >> 1, dx = k & 1;
    const long long t = base + (long long)dy * v.W + dx;
    if ((unsigned)(y0 + dy) < (unsigned)v.H && (unsigned)(x0 + dx) < (unsigned)v.W && t >= 0 && t < a.S) m |= 1u << k;
  }
  if (m) {  // otherwise the sample reads nothing and contributes nothing (fractions of a NaN location stay out)
    r.mask = m;
    r.base = (int)base;  // >= (valid corner) - W - 1 > -2^31
    r.fx = x - xf;
    r.fy = y - yf;
  }
  return r;
}

template <int G>
__device__ __forceinline__ Smp bcast(const Smp& s, int k) {
  Smp r;
  r.base = __shfl_sync(0xffffffffu, s.base, k, G);
  r.W = __shfl_sync(0xffffffffu, s.W, k, G);
  r.mask = __shfl_sync(0xffffffffu, s.mask, k, G);
  r.fx = __shfl_sync(0xffffffffu, s.fx, k, G);
  r.fy = __shfl_sync(0xffffffffu, s.fy, k, G);
  r.a = __shfl_sync(0xffffffffu, s.a, k, G);
  return r;
}

__device__ __forceinline__ float4 axpy4(float w, float4 x, float4 y) {
  return make_float4(fmaf(w, x.x, y.x), fmaf(w, x.y, y.y), fmaf(w, x.z, y.z), fmaf(w, x.w, y.w));
}

__device__ __forceinline__ float dot4(float4 a, float4 b) { return fmaf(a.w, b.w, fmaf(a.z, b.z, fmaf(a.y, b.y, a.x * b.x))); }

// token offset of corner k relative to the NW corner
__device__ __forceinline__ int corner_delta(int k, int W) { return (k >> 1) * W + (k & 1); }

template <int G, int V>
__global__ void __launch_bounds__(kThreads) msda_fwd_kernel(const Args a) {
  __shared__ Level lv[kMaxLevels];
  load_levels(a, lv);
  const long long n_items = (long long)a.B * a.Q * a.M;
  const long long item_l = ((long long)blockIdx.x * kThreads + threadIdx.x) / G;
  const bool live = item_l < n_items;
  const int item = (int)(live ? item_l : n_items - 1);  // clamped: address arithmetic only
  const int j = threadIdx.x & (G - 1);
  const int LP = a.L * a.P;
  const int m = item % a.M, b = item / (a.Q * a.M);
  const float* locp = a.loc + (size_t)item * LP * 2;
  const float* attnp = a.attn + (size_t)item * LP;
  const size_t row = (size_t)a.M * a.D;  // floats per token
  const float* vb = a.value + ((size_t)b * a.S * a.M + m) * a.D + 4 * j;
  float4 acc[V];
#pragma unroll
  for (int v = 0; v < V; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int s0 = 0; s0 < LP; s0 += G) {
    Smp own = empty_sample();
    if (live && s0 + j < LP) own = make_sample(a, lv, locp, attnp, s0 + j);
    const int kn = min(G, LP - s0);  // warp-uniform
#pragma unroll
    for (int k = 0; k < G; ++k) {
      if (k >= kn) break;
      const Smp sm = bcast<G>(own, k);
      if (!sm.mask) continue;  // uniform within the group
      const float ex = 1.f - sm.fx, ey = 1.f - sm.fy;
      const float w[4] = {ey * ex, ey * sm.fx, sm.fy * ex, sm.fy * sm.fx};
#pragma unroll
      for (int v = 0; v < V; ++v) {
        float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (!(sm.mask & (1u << c))) continue;
          const int t = sm.base + corner_delta(c, sm.W);
          DCN_DEV_ASSERT(t >= 0 && t < a.S && 4 * j + 4 * G * v < a.D);
          val = axpy4(w[c], __ldg(reinterpret_cast<const float4*>(vb + (size_t)t * row + 4 * G * v)), val);
        }
        acc[v] = axpy4(sm.a, val, acc[v]);
      }
    }
  }
  if (!live) return;
#pragma unroll
  for (int v = 0; v < V; ++v)
    *reinterpret_cast<float4*>(a.out + (size_t)item * a.D + 4 * j + 4 * G * v) = acc[v];
}

template <int G, int V>
__global__ void __launch_bounds__(kThreads) msda_bwd_kernel(const Args a) {
  constexpr int K = G < 8 ? G : 8;  // samples per round = partials per lane and kind
  __shared__ Level lv[kMaxLevels];
  load_levels(a, lv);
  const long long n_items = (long long)a.B * a.Q * a.M;
  const long long item_l = ((long long)blockIdx.x * kThreads + threadIdx.x) / G;
  const bool live = item_l < n_items;
  const int item = (int)(live ? item_l : n_items - 1);
  const int j = threadIdx.x & (G - 1);
  const int LP = a.L * a.P;
  const int m = item % a.M, b = item / (a.Q * a.M);
  const float* locp = a.loc + (size_t)item * LP * 2;
  const float* attnp = a.attn + (size_t)item * LP;
  const size_t row = (size_t)a.M * a.D;
  const size_t vofs = ((size_t)b * a.S * a.M + m) * a.D + 4 * j;
  const float* vb = a.value + vofs;
  float* gvb = a.gvalue ? a.gvalue + vofs : nullptr;
  const bool coord = a.gloc || a.gattn;
  float4 g[V];
#pragma unroll
  for (int v = 0; v < V; ++v)
    g[v] = live ? __ldg(reinterpret_cast<const float4*>(a.gout + (size_t)item * a.D + 4 * j + 4 * G * v))
                : make_float4(0.f, 0.f, 0.f, 0.f);
  for (int s0 = 0; s0 < LP; s0 += K) {
    Smp own = empty_sample();
    if (live && j < K && s0 + j < LP) own = make_sample(a, lv, locp, attnp, s0 + j);
    float pa[K], px[K], py[K];  // sum g*bil, sum g*dbil/dx, sum g*dbil/dy over this lane's channels
#pragma unroll
    for (int k = 0; k < K; ++k) {
      pa[k] = px[k] = py[k] = 0.f;
      const Smp sm = bcast<G>(own, k);  // samples past L*P come from an empty owner
      if (!sm.mask) continue;
      const float ex = 1.f - sm.fx, ey = 1.f - sm.fy;
      const float w[4] = {ey * ex, ey * sm.fx, sm.fy * ex, sm.fy * sm.fx};
#pragma unroll
      for (int v = 0; v < V; ++v) {
        float4 c[4];
#pragma unroll
        for (int cn = 0; cn < 4; ++cn) {
          c[cn] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (!(sm.mask & (1u << cn))) continue;
          const int t = sm.base + corner_delta(cn, sm.W);
          DCN_DEV_ASSERT(t >= 0 && t < a.S && 4 * j + 4 * G * v < a.D);
          const size_t o = (size_t)t * row + 4 * G * v;
          if (gvb) {
            const float aw = sm.a * w[cn];
            atomicAdd(reinterpret_cast<float4*>(gvb + o), make_float4(aw * g[v].x, aw * g[v].y, aw * g[v].z, aw * g[v].w));
          }
          if (coord) c[cn] = __ldg(reinterpret_cast<const float4*>(vb + o));
        }
        if (coord) {
          float4 bil = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int cn = 0; cn < 4; ++cn) bil = axpy4(w[cn], c[cn], bil);
          // d bil / dx = ey*(ne - nw) + fy*(se - sw);  d bil / dy = ex*(sw - nw) + fx*(se - ne)
          const float4 dx = make_float4(ey * (c[1].x - c[0].x) + sm.fy * (c[3].x - c[2].x),
                                        ey * (c[1].y - c[0].y) + sm.fy * (c[3].y - c[2].y),
                                        ey * (c[1].z - c[0].z) + sm.fy * (c[3].z - c[2].z),
                                        ey * (c[1].w - c[0].w) + sm.fy * (c[3].w - c[2].w));
          const float4 dy = make_float4(ex * (c[2].x - c[0].x) + sm.fx * (c[3].x - c[1].x),
                                        ex * (c[2].y - c[0].y) + sm.fx * (c[3].y - c[1].y),
                                        ex * (c[2].z - c[0].z) + sm.fx * (c[3].z - c[1].z),
                                        ex * (c[2].w - c[0].w) + sm.fx * (c[3].w - c[1].w));
          pa[k] += dot4(g[v], bil);
          px[k] += dot4(g[v], dx);
          py[k] += dot4(g[v], dy);
        }
      }
    }
    if (!coord) continue;
    // lanes of the group that are K or more apart hold different channels of the same K samples: plain sum
#pragma unroll
    for (int s = G / 2; s >= K; s >>= 1) {
#pragma unroll
      for (int k = 0; k < K; ++k) {
        pa[k] += __shfl_xor_sync(0xffffffffu, pa[k], s);
        px[k] += __shfl_xor_sync(0xffffffffu, px[k], s);
        py[k] += __shfl_xor_sync(0xffffffffu, py[k], s);
      }
    }
    // butterfly reduce-scatter over the remaining K lanes: afterwards lane j holds the totals of sample s0 + (j % K)
#pragma unroll
    for (int s = K / 2, n = K / 2; s >= 1; s >>= 1, n >>= 1) {
      const bool up = (j & s) != 0;
#pragma unroll
      for (int k = 0; k < n; ++k) {
        const float sa = up ? pa[k] : pa[k + n], sx = up ? px[k] : px[k + n], sy = up ? py[k] : py[k + n];
        const float ka = up ? pa[k + n] : pa[k], kx = up ? px[k + n] : px[k], ky = up ? py[k + n] : py[k];
        pa[k] = ka + __shfl_xor_sync(0xffffffffu, sa, s);
        px[k] = kx + __shfl_xor_sync(0xffffffffu, sx, s);
        py[k] = ky + __shfl_xor_sync(0xffffffffu, sy, s);
      }
    }
    const int s = s0 + j;
    if (live && j < K && s < LP) {  // the owner of sample s: one plain store per gradient element
      const size_t o = (size_t)item * LP + s;
      if (a.gattn) a.gattn[o] = pa[0];
      if (a.gloc) {
        const Level v = lv[s / a.P];
        *reinterpret_cast<float2*>(a.gloc + 2 * o) = make_float2(own.a * (float)v.W * px[0], own.a * (float)v.H * py[0]);
      }
    }
  }
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
