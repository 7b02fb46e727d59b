// dcn_gather.cuh — the depthwise bilinear gather core shared by multi-scale deformable attention (dcn_msda.cu),
// DCNv3 and DCNv4 (dcn_dcnv3.cu).  All compute, per item (batch, query, head) with its D contiguous channels of `value`,
//   out[item, d] = sum_s a_s * bilinear(value[b, :, m, d], y_s, x_s)
// with corners outside the image reading 0.  Only where the samples come from differs; a sample source supplies it:
//   Src::Args        tensors and extents.  Fields the core reads: value, loc, attn, gout, out, gvalue, gloc, gattn
//                    and B, S, Q, M, D, L, P — value [B, S, M, D] (S tokens of M heads of D channels), items
//                    B*Q*M, L*P samples per item, loc [items, L*P, 2], attn [items, L*P], out / gout [items, D].
//   Src::Rows        where an item's per-sample data lives: loc_row / attn_row (the pointers handed to sample()),
//                    grad_slot, store_gattn / store_gloc (where the three gradient elements of sample s go: the
//                    slot is computed once, each store adds what it needs) and end_grad<G> (anything
//                    else of the item's coordinate-side gradient).  DenseRows below is the layout just described;
//                    DCNv4's packed offset_mask row is the other one (dcn_dcnv3.cu).
//   Src::Item        per-item state, made once per item by begin<G>(item, j, attnp) with the whole group present.
//   sample(it, locp, attnp, s)   the coordinate chain of sample s -> Smp (corner mask, NW token, fractions, weight).
//   loc_scale(own, s)            (dx/dloc_x, dy/dloc_y) times the sample's weight: the factors of the two partials
//                                sum g*dbil/dx, sum g*dbil/dy in the location gradient.
//   kSoftmax         attn holds logits; the weight of sample s is softmax over the item's L*P logits.  The backward
//                    then writes the logits' gradient m_s*(gamma_s - sum_q m_q*gamma_q), gamma = sum g*bil.
// Mapping: a group of G = min(D/4, 32) lanes owns one item, V = D/(4G) float4 per lane; one corner of one head is 4*D
// contiguous bytes, read in place with one float4 per lane; whether a corner is inside is the same for the group.
//   forward   the samples are cut into rounds of G: lane j runs the chain of sample s0 + j and hands the result to
//             the group by shuffle.  `out` is written once, coalesced; no atomics.
//   backward  rounds of K = min(G, 8) samples.  Per sample and lane: gvalue[corner] += a*w_k*g (red.global.add.v4.f32,
//             corners inside only) and three partials over the lane's channels, sum g*bil, sum g*dbil/dx,
//             sum g*dbil/dy.  The 3K partials of a round are reduced over the group with the butterfly reduce-scatter
//             of dcn_umma_bwd_data.cu, after which lane j holds the totals of sample s0 + j — the sample whose chain it
//             computed — and writes its gradient elements with plain stores.  The two coordinate-side gradients are
//             therefore deterministic; only gvalue depends on the order of the atomics.
#pragma once
#include <cuda_runtime.h>

#include "dcn_common.cuh"

namespace dcn {

namespace gather {

constexpr int kThreads = 256;

// One sampling point after the coordinate chain.  mask bit k: corner k (NW, NE, SW, SE) lies inside the image and its
// token index inside [0, S).  base = token of the NW corner (meaningful only when mask != 0).
struct Smp {
  int base, W;
  unsigned mask;
  float fx, fy, a;
};

__device__ __forceinline__ Smp empty_sample() { return Smp{0, 0, 0u, 0.f, 0.f, 0.f}; }

// Src::Rows of the dense layout: loc [items, L*P, 2] with one float2 per sample, attn [items, L*P], gradients alike.
struct DenseRows {
  template <class A>
  static __device__ __forceinline__ const float* loc_row(const A& a, int item, int LP) {
    return a.loc + (size_t)item * LP * 2;
  }
  template <class A>
  static __device__ __forceinline__ const float* attn_row(const A& a, int item, int LP) {
    return a.attn + (size_t)item * LP;
  }
  template <class A>
  static __device__ __forceinline__ size_t grad_slot(const A&, int item, int LP, int s) {
    return (size_t)item * LP + s;
  }
  template <class A>
  static __device__ __forceinline__ void store_gattn(const A& a, size_t o, int, float v) {
    a.gattn[o] = v;
  }
  template <class A>
  static __device__ __forceinline__ void store_gloc(const A& a, size_t o, int, float2 v) {
    *reinterpret_cast<float2*>(a.gloc + 2 * o) = v;
  }
  template <int G, class A>
  static __device__ __forceinline__ void end_grad(const A&, int, int, bool) {}
};

// Corner mask, NW token and fractions of pixel coordinate (x, y) in an H x W image whose first token is `start`;
// corners are also checked against [0, S).  A NaN coordinate saturates low (sat_int) and reads nothing.
__device__ __forceinline__ void locate(Smp& r, float x, float y, int H, int W, long long start, int S) {
  const float xf = floorf(x), yf = floorf(y);
  const int x0 = sat_int(xf), y0 = sat_int(yf);
  const long long base = start + (long long)y0 * W + x0;
  unsigned m = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int dy = k >> 1, dx = k & 1;
    const long long t = base + (long long)dy * W + dx;
    if ((unsigned)(y0 + dy) < (unsigned)H && (unsigned)(x0 + dx) < (unsigned)W && t >= 0 && t < S) m |= 1u << k;
  }
  if (m) {  // otherwise the sample reads nothing and contributes nothing (fractions of a NaN location stay out)
    r.mask = m;
    r.base = (int)base;  // >= (valid corner) - W - 1 > -2^31
    r.fx = x - xf;
    r.fy = y - yf;
  }
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

// Sum over the G lanes of a group (every lane ends with the same bits: the butterfly adds the same pairs everywhere).
template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int s = G / 2; s >= 1; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
  return v;
}

template <int G>
__device__ __forceinline__ float group_max(float v) {
#pragma unroll
  for (int s = G / 2; s >= 1; s >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, s));
  return v;
}

template <int G, int V, class Src>
__device__ __forceinline__ void fwd_body(const Src& src) {
  const typename Src::Args& a = src.a;
  const long long n_items = (long long)a.B * a.Q * a.M;
  const long long item_l = ((long long)blockIdx.x * kThreads + threadIdx.x) / G;
  const bool live = item_l < n_items;
  const int item = (int)(live ? item_l : n_items - 1);  // clamped: address arithmetic only
  const int j = threadIdx.x & (G - 1);
  const int LP = a.L * a.P;
  const int m = item % a.M, b = item / (a.Q * a.M);
  using Rows = typename Src::Rows;
  const float* locp = Rows::loc_row(a, item, LP);
  const float* attnp = Rows::attn_row(a, item, LP);
  const typename Src::Item it = src.template begin<G>(item, j, attnp);
  const size_t row = (size_t)a.M * a.D;  // floats per token
  const float* vb = a.value + ((size_t)b * a.S * a.M + m) * a.D + 4 * j;
  float4 acc[V];
#pragma unroll
  for (int v = 0; v < V; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int s0 = 0; s0 < LP; s0 += G) {
    Smp own = empty_sample();
    if (live && s0 + j < LP) own = src.sample(it, locp, attnp, s0 + j);
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

template <int G, int V, class Src>
__device__ __forceinline__ void bwd_body(const Src& src) {
  constexpr int K = G < 8 ? G : 8;  // samples per round = partials per lane and kind
  // softmax: rounds an owner lane keeps (m_s, gamma_s) for; the sources with kSoftmax have L*P <= 32
  constexpr int R = Src::kSoftmax ? 32 / K : 1;
  const typename Src::Args& a = src.a;
  const long long n_items = (long long)a.B * a.Q * a.M;
  const long long item_l = ((long long)blockIdx.x * kThreads + threadIdx.x) / G;
  const bool live = item_l < n_items;
  const int item = (int)(live ? item_l : n_items - 1);
  const int j = threadIdx.x & (G - 1);
  const int LP = a.L * a.P;
  const int m = item % a.M, b = item / (a.Q * a.M);
  using Rows = typename Src::Rows;
  const float* locp = Rows::loc_row(a, item, LP);
  const float* attnp = Rows::attn_row(a, item, LP);
  const typename Src::Item it = src.template begin<G>(item, j, attnp);
  const size_t row = (size_t)a.M * a.D;
  const size_t vofs = ((size_t)b * a.S * a.M + m) * a.D + 4 * j;
  const float* vb = a.value + vofs;
  float* gvb = a.gvalue ? a.gvalue + vofs : nullptr;
  const bool coord = a.gloc || a.gattn;
  float keep_m[R], keep_g[R];
#pragma unroll
  for (int r = 0; r < R; ++r) keep_m[r] = keep_g[r] = 0.f;
  float4 g[V];
#pragma unroll
  for (int v = 0; v < V; ++v)
    g[v] = live ? __ldg(reinterpret_cast<const float4*>(a.gout + (size_t)item * a.D + 4 * j + 4 * G * v))
                : make_float4(0.f, 0.f, 0.f, 0.f);
  for (int s0 = 0; s0 < LP; s0 += K) {
    Smp own = empty_sample();
    if (live && j < K && s0 + j < LP) own = src.sample(it, locp, attnp, s0 + j);
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
      const size_t o = Rows::grad_slot(a, item, LP, s);
      if constexpr (Src::kSoftmax) {  // the logit gradient needs every gamma of the item: kept, written below
#pragma unroll
        for (int r = 0; r < R; ++r)
          if (r * K == s0) keep_m[r] = own.a, keep_g[r] = pa[0];
      } else {
        if (a.gattn) Rows::store_gattn(a, o, s, pa[0]);
      }
      if (a.gloc) {
        const float2 sc = src.loc_scale(own, s);
        Rows::store_gloc(a, o, s, make_float2(sc.x * px[0], sc.y * py[0]));
      }
    }
  }
  Rows::template end_grad<G>(a, item, j, live);
  if constexpr (Src::kSoftmax) {
    if (!a.gattn) return;
    // sum_q m_q*gamma_q over the item: each owner lane adds its samples in round order, then the group
    float t = 0.f;
#pragma unroll
    for (int r = 0; r < R; ++r) t = fmaf(keep_m[r], keep_g[r], t);
    t = group_sum<G>(t);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int s = r * K + j;
      if (live && j < K && s < LP) Rows::store_gattn(a, Rows::grad_slot(a, item, LP, s), s, keep_m[r] * (keep_g[r] - t));
    }
  }
}

}  // namespace gather

}  // namespace dcn
