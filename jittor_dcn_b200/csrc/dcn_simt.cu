// dcn_simt.cu — generic CUDA-core kernels: every shape, both variants, float32.
//
// These are the shape-agnostic path of the engine (odd channel counts, tiny layers, 1x1
// taps, ...) and the A/B reference for the tcgen05 kernels (DCN_FLAG_FORCE_SIMT).  All of
// them are implicit GEMMs: the column matrix the reference materialises
// (deform_conv.py:72-73 / train.py:129-131) is produced tile by tile from the sampling plan
// and never touches HBM.
//
//   plan_kernel          deform_conv.py:62-68,34-39 / train.py:102-113 + grid_sample geometry
//   fwd_kernel           sampling (:47-52 / :121-127) + GEMM (:74-76 / :133-134) + bias
//   bwd_data_kernel      gA = g * Wm, bilinear col2im scatter (red.global.add.f32) and the
//                        coordinate-gradient reduction                (autograd, A.4)
//   bwd_weight_kernel    gW = g^T * A with A re-sampled                (autograd, A.4)
//   bias_grad / offset_scale kernels
//
// MOD instantiations (modulated DCNv1 = DCNv2, pixel-row column order): every sample is scaled by
// mask[b, n, p] ([B, N, Ho, Wo], the same [b][n][p] order as the plan of that layout), and
// bwd_data_kernel also writes grad_mask[b, n, p] = sum_c gA * (unmasked sample).
#include <cuda_bf16.h>

#include "dcn_common.cuh"

namespace dcn {

// ------------------------------------------------------------------------------ plan
template <int VARIANT>
__device__ __forceinline__ size_t plan_index(const Geo& g, int b, int n, int p) {
  return VARIANT == DCN_VARIANT_TORCH ? ((size_t)b * g.HW + p) * g.N + n
                                      : ((size_t)b * g.N + n) * g.HW + p;
}

template <int VARIANT>
__global__ void __launch_bounds__(256) plan_kernel(Geo g, const float* __restrict__ off,
                                                   Tap* __restrict__ plan) {
  const int total = g.N * g.HW;  // per batch element
  const int b = blockIdx.y;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int n = i / g.HW, p = i - n * g.HW;
    const float* ob = off + (size_t)b * 2 * g.N * g.HW;
    const float ox = __ldg(ob + (size_t)off_row_ch(g, n) * g.HW + p);
    const float oy = __ldg(ob + (size_t)off_col_ch(g, n) * g.HW + p);
    const int h = p / g.Wo, w = p - h * g.Wo;
    plan[plan_index<VARIANT>(g, b, n, p)] = tap_of(g, h, w, n, ox, oy);
  }
}

int launch_plan(const Geo& g, const float* off, Tap* plan, cudaStream_t st) {
  const int total = g.N * g.HW;
  dim3 grid((unsigned)min((total + 255) / 256, 4096), g.B);
  KernelScope scope("plan_kernel", st);
  if (g.variant == DCN_VARIANT_TORCH)
    plan_kernel<DCN_VARIANT_TORCH><<<grid, 256, 0, st>>>(g, off, plan);
  else
    plan_kernel<DCN_VARIANT_JITTOR><<<grid, 256, 0, st>>>(g, off, plan);
  DCN_KERNEL_CHECK("plan_kernel");
  return DCN_OK;
}

__global__ void __launch_bounds__(256) corners_kernel(Geo g, const float* __restrict__ off,
                                                      int32_t* __restrict__ y0,
                                                      int32_t* __restrict__ x0,
                                                      float* __restrict__ w4) {
  const int total = g.N * g.HW;
  const int b = blockIdx.y;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int n = i / g.HW, p = i - n * g.HW;
    const float* ob = off + (size_t)b * 2 * g.N * g.HW;
    const int h = p / g.Wo, w = p - h * g.Wo;
    Tap t = tap_of(g, h, w, n, ob[(size_t)off_row_ch(g, n) * g.HW + p], ob[(size_t)off_col_ch(g, n) * g.HW + p]);
    float cw[4];
    corner_weights(t, cw);
    const size_t o = (size_t)b * total + i;
    y0[o] = t.y0;
    x0[o] = t.x0;
    reinterpret_cast<float4*>(w4)[o] = make_float4(cw[0], cw[1], cw[2], cw[3]);
  }
}

int launch_corners(const Geo& g, const float* off, int32_t* y0, int32_t* x0, float* w4,
                   cudaStream_t st) {
  const int total = g.N * g.HW;
  dim3 grid((unsigned)min((total + 255) / 256, 4096), g.B);
  corners_kernel<<<grid, 256, 0, st>>>(g, off, y0, x0, w4);
  DCN_KERNEL_CHECK("corners_kernel");
  return DCN_OK;
}

// ------------------------------------------------------------------------- sampling
// zero-padded bilinear sample of one channel plane (grid_sample semantics)
__device__ __forceinline__ float sample_plane(const float* __restrict__ xp, int H, int W,
                                              const Tap& t) {
  float cw[4];
  corner_weights(t, cw);
  const unsigned m = corner_mask(t, H, W);
  const float* base = xp + (ptrdiff_t)t.y0 * W + t.x0;
  float acc = 0.f;
  if (m & 1u) acc = __ldg(base) * cw[0];
  if (m & 2u) acc += __ldg(base + 1) * cw[1];
  if (m & 4u) acc += __ldg(base + W) * cw[2];
  if (m & 8u) acc += __ldg(base + W + 1) * cw[3];
  return acc;
}

template <int VARIANT>
__device__ __forceinline__ float sample_a(const Geo& g, const float* __restrict__ xb,
                                          const Tap* __restrict__ planb, int r, int j) {
  int c, q;
  col_map<VARIANT>(g, r, j, c, q);
  Tap t;
  if (VARIANT == DCN_VARIANT_TORCH) {
    t = planb[q];
  } else {
    const int p = q / g.N, n = q - p * g.N;
    t = planb[(size_t)n * g.HW + p];
  }
  return sample_plane(xb + (size_t)c * g.H * g.W, g.H, g.W, t);
}

// --------------------------------------------------------------------------- forward
// out[b, o, r] = sum_j A_b[r, j] * Wm[o, j] + bias[o]
// tile 64 rows x 64 outputs, BK = 16, 256 threads, 4x4 micro-tile per thread.
constexpr int TM = 64, TN = 64, TK = 16;

template <int VARIANT, bool MOD = false>
__global__ void __launch_bounds__(256) fwd_kernel(Geo g, const float* __restrict__ x,
                                                  const Tap* __restrict__ plan,
                                                  const float* __restrict__ wt,
                                                  const float* __restrict__ bias,
                                                  float* __restrict__ out,
                                                  const float* __restrict__ mask) {
  static_assert(!MOD || VARIANT != DCN_VARIANT_TORCH, "modulation exists for the DCNv1 (pixel-row) order only");
  __shared__ float As[TK][TM + 4];
  __shared__ float Bs[TK][TN + 4];
  const int b = blockIdx.z, r0 = blockIdx.x * TM, o0 = blockIdx.y * TN;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;  // tx -> rows, ty -> outputs
  const float* xb = x + (size_t)b * g.C * g.H * g.W;
  const Tap* planb = plan + (size_t)b * g.P;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < g.K; k0 += TK) {
// A tile: 64 x 16 samples, 4 per thread
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int rr, kk;
      if (VARIANT == DCN_VARIANT_TORCH) {  // lanes along k (consecutive samples q)
        kk = tid & 15;
        rr = (tid >> 4) + 16 * i;
      } else {  // lanes along rows (consecutive pixels)
        rr = tid & 63;
        kk = (tid >> 6) + 4 * i;
      }
      float v = 0.f;
      if (r0 + rr < g.HW && k0 + kk < g.K) {
        v = sample_a<VARIANT>(g, xb, planb, r0 + rr, k0 + kk);
        if (MOD) {
          const size_t mi = ((size_t)b * g.N + (k0 + kk) / g.C) * g.HW + r0 + rr;
          DCN_DEV_ASSERT(mi < (size_t)g.B * g.N * g.HW);
          v = __ldg(mask + mi) * v;
        }
      }
      As[kk][rr] = v;
    }
// B tile: Wm[o0..o0+63, k0..k0+15]
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int kk = tid & 15, oo = (tid >> 4) + 16 * i;
      float v = 0.f;
      if (o0 + oo < g.O && k0 + kk < g.K) v = __ldg(wt + wt_index(g, o0 + oo, k0 + kk));
      Bs[kk][oo] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < TK; ++kk) {
      float a[4], w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][tx * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) w[j] = Bs[kk][ty * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int o = o0 + ty * 4 + j;
    if (o >= g.O) continue;
    const float bv = bias ? __ldg(bias + o) : 0.f;
    float* orow = out + ((size_t)b * g.O + o) * g.HW;
    const int r = r0 + tx * 4;
    float v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[i] = acc[i][j] + bv;
      if (g.relu_out) v[i] = fmaxf(v[i], 0.f);   // DCN_FLAG_RELU_OUT
    }
    if (r + 3 < g.HW && (g.HW & 3) == 0) {
      *reinterpret_cast<float4*>(orow + r) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (r + i < g.HW) orow[r + i] = v[i];
    }
  }
}

int simt_forward(const Geo& g, const float* x, const Tap* plan, const float* wt, const float* bias,
                 float* out, cudaStream_t st, const float* mask) {
  dim3 grid((g.HW + TM - 1) / TM, (g.O + TN - 1) / TN, g.B);
  KernelScope scope("fwd_kernel", st);
  if (mask)
    fwd_kernel<DCN_VARIANT_JITTOR, true><<<grid, 256, 0, st>>>(g, x, plan, wt, bias, out, mask);
  else if (g.variant == DCN_VARIANT_TORCH)
    fwd_kernel<DCN_VARIANT_TORCH><<<grid, 256, 0, st>>>(g, x, plan, wt, bias, out, nullptr);
  else
    fwd_kernel<DCN_VARIANT_JITTOR><<<grid, 256, 0, st>>>(g, x, plan, wt, bias, out, nullptr);
  DCN_KERNEL_CHECK("fwd_kernel");
  return DCN_OK;
}

// -------------------------------------------------------------------- backward: data
// gA[r, j] = sum_o g[r, o] * Wm[o, j]; then per element (c, q):
//   grad_x[c, corner] += w_corner * gA            (zero-padded bilinear col2im, atomics)
//   g_ix[q] += gA * ((v_ne - v_nw)(1-fy) + (v_se - v_sw) fy)
//   g_iy[q] += gA * ((v_sw - v_nw)(1-fx) + (v_se - v_ne) fx)
// g_iy is accumulated raw into grad_offset channel n, g_ix into channel N+n (the "x"
// offset moves the ROW because the reference hands grid_sample [norm_y, norm_x]);
// offset_scale_kernel applies the chain-rule factors afterwards.
template <int VARIANT, bool MOD = false>
__global__ void __launch_bounds__(256) bwd_data_kernel(Geo g, int want_gx,
                                                       const float* __restrict__ x,
                                                       const Tap* __restrict__ plan,
                                                       const float* __restrict__ wt,
                                                       const float* __restrict__ gout,
                                                       float* __restrict__ gx,
                                                       float* __restrict__ goff,
                                                       const float* __restrict__ mask,
                                                       float* __restrict__ gmask) {
  static_assert(!MOD || VARIANT != DCN_VARIANT_TORCH, "modulation exists for the DCNv1 (pixel-row) order only");
  __shared__ float Gs[TK][TM + 4];  // g[r, o]   (o along TK)
  __shared__ float Ws[TK][TN + 4];  // Wm[o, j]
  const int b = blockIdx.z, r0 = blockIdx.x * TM, j0 = blockIdx.y * TN;
  const int tid = threadIdx.x;
  // rows fastest across lanes for Jittor (a thread owns 4 consecutive c of one pixel),
  // columns fastest for Torch (a thread owns 4 consecutive samples q of one channel)
  const int tx = tid & 15, ty = tid >> 4;
  const float* gob = gout + (size_t)b * g.O * g.HW;
  float acc[4][4] = {};  // [row i][col jj]
  for (int o0 = 0; o0 < g.O; o0 += TK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int rr = tid & 63, oo = (tid >> 6) + 4 * i;
      float v = 0.f;
      if (r0 + rr < g.HW && o0 + oo < g.O) v = __ldg(gob + (size_t)(o0 + oo) * g.HW + r0 + rr);
      Gs[oo][rr] = v;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int jj = tid & 63, oo = (tid >> 6) + 4 * i;
      float v = 0.f;
      if (j0 + jj < g.K && o0 + oo < g.O) v = __ldg(wt + wt_index(g, o0 + oo, j0 + jj));
      Ws[oo][jj] = v;
    }
    __syncthreads();
#pragma unroll
    for (int oo = 0; oo < TK; ++oo) {
      float a[4], w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = Gs[oo][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) w[j] = Ws[oo][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
    }
    __syncthreads();
  }
  // epilogue: scatter + coordinate gradient
  const float* xb = x + (size_t)b * g.C * g.H * g.W;
  float* gxb = gx + (size_t)b * g.C * g.H * g.W;
  const Tap* planb = plan + (size_t)b * g.P;
  float* goffb = goff + (size_t)b * 2 * g.N * g.HW;
  int q_prev = -1;
  float six = 0.f, siy = 0.f;
  float smk = 0.f;  // MOD: sum of gA * (unmasked sample) of sampling point q_prev
  auto flush = [&]() {
    if (q_prev >= 0 && (six != 0.f || siy != 0.f)) {
      const int p = q_prev / g.N, n = q_prev - p * g.N;
      atomicAdd(goffb + (size_t)off_row_ch(g, n) * g.HW + p, siy);
      atomicAdd(goffb + (size_t)off_col_ch(g, n) * g.HW + p, six);
    }
    six = siy = 0.f;
    if constexpr (MOD) {
      if (q_prev >= 0 && smk != 0.f) {
        const int p = q_prev / g.N, n = q_prev - p * g.N;
        const size_t mi = ((size_t)b * g.N + n) * g.HW + p;
        DCN_DEV_ASSERT(mi < (size_t)g.B * g.N * g.HW);
        atomicAdd(gmask + mi, smk);
      }
      smk = 0.f;
    }
  };
  // MOD: gA of sampling point q scaled by its mask value
  auto modulated = [&](float ga, int q) {
    const int p = q / g.N, n = q - p * g.N;
    const size_t mi = ((size_t)b * g.N + n) * g.HW + p;
    DCN_DEV_ASSERT(mi < (size_t)g.B * g.N * g.HW);
    return __ldg(mask + mi) * ga;
  };
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = r0 + ty * 4 + i;
    if (r >= g.HW) continue;
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const int j = j0 + tx * 4 + jj;
      if (j >= g.K) continue;
      int c, q;
      col_map<VARIANT>(g, r, j, c, q);
      if (q != q_prev) {
        flush();
        q_prev = q;
      }
      Tap t;
      if (VARIANT == DCN_VARIANT_TORCH) {
        t = planb[q];
      } else {
        const int p = q / g.N, n = q - p * g.N;
        t = planb[(size_t)n * g.HW + p];
      }
      const unsigned m = corner_mask(t, g.H, g.W);
      if (!m) continue;
      float cw[4];
      corner_weights(t, cw);
      const float gs = MOD ? modulated(acc[i][jj], q) : acc[i][jj];
      const ptrdiff_t base = (ptrdiff_t)c * g.H * g.W + (ptrdiff_t)t.y0 * g.W + t.x0;
      const float v0 = (m & 1u) ? __ldg(xb + base) : 0.f;
      const float v1 = (m & 2u) ? __ldg(xb + base + 1) : 0.f;
      const float v2 = (m & 4u) ? __ldg(xb + base + g.W) : 0.f;
      const float v3 = (m & 8u) ? __ldg(xb + base + g.W + 1) : 0.f;
      if (want_gx) {
        if (m & 1u) atomicAdd(gxb + base, gs * cw[0]);
        if (m & 2u) atomicAdd(gxb + base + 1, gs * cw[1]);
        if (m & 4u) atomicAdd(gxb + base + g.W, gs * cw[2]);
        if (m & 8u) atomicAdd(gxb + base + g.W + 1, gs * cw[3]);
      }
      six += gs * ((v1 - v0) * (1.f - t.fy) + (v3 - v2) * t.fy);
      siy += gs * ((v2 - v0) * (1.f - t.fx) + (v3 - v1) * t.fx);
      if constexpr (MOD) smk += acc[i][jj] * (v0 * cw[0] + v1 * cw[1] + v2 * cw[2] + v3 * cw[3]);
    }
  }
  flush();
}

// grad_offset[b, n] = g_iy * sy * 2 / Dx ;  grad_offset[b, N+n] = g_ix * sx * 2 / Dy
// (autograd order of train.py:111-113 -> GridSampler.h:27-36)
__global__ void __launch_bounds__(256) offset_scale_kernel(Geo g, float* __restrict__ goff) {
  const size_t per_b = (size_t)2 * g.N * g.HW, total = per_b * g.B;
  const size_t half = (size_t)g.N * g.HW;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (size_t)gridDim.x * blockDim.x) {
    const bool is_x = (i % per_b) < half;
    const float v = goff[i];
    goff[i] = is_x ? v * g.sy * 2.0f / g.Dx : v * g.sx * 2.0f / g.Dy;
  }
}

// ------------------------------------------------------------------ backward: weight
// gW[o, j] = sum_{b, r} g_b[r, o] * A_b[r, j]; the (b, r) range is split over gridDim.z
// and partial tiles are reduced with red.global.add.f32 into a zeroed gW.
template <int VARIANT, bool MOD = false>
__global__ void __launch_bounds__(256) bwd_weight_kernel(Geo g, int chunks_per_split,
                                                         const float* __restrict__ x,
                                                         const Tap* __restrict__ plan,
                                                         const float* __restrict__ gout,
                                                         float* __restrict__ gw,
                                                         const float* __restrict__ mask) {
  static_assert(!MOD || VARIANT != DCN_VARIANT_TORCH, "modulation exists for the DCNv1 (pixel-row) order only");
  __shared__ float Gs[TK][TM + 4];  // g[r, o]  (r along TK)
  __shared__ float As[TK][TN + 4];  // A[r, j]
  const int o0 = blockIdx.x * TM, j0 = blockIdx.y * TN;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;  // tx -> j, ty -> o
  const int chunks_per_b = (g.HW + TK - 1) / TK;
  const int total_chunks = chunks_per_b * g.B;
  const int c_begin = blockIdx.z * chunks_per_split;
  const int c_end = min(total_chunks, c_begin + chunks_per_split);
  float acc[4][4] = {};  // [o i][j jj]
  for (int ch = c_begin; ch < c_end; ++ch) {
    const int b = ch / chunks_per_b, r0 = (ch - b * chunks_per_b) * TK;
    const float* gob = gout + (size_t)b * g.O * g.HW;
    const float* xb = x + (size_t)b * g.C * g.H * g.W;
    const Tap* planb = plan + (size_t)b * g.P;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int rr = tid & 15, oo = (tid >> 4) + 16 * i;
      float v = 0.f;
      if (r0 + rr < g.HW && o0 + oo < g.O) v = __ldg(gob + (size_t)(o0 + oo) * g.HW + r0 + rr);
      Gs[rr][oo] = v;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int rr, jj;
      if (VARIANT == DCN_VARIANT_TORCH) {  // lanes along j (consecutive samples q)
        jj = tid & 63;
        rr = (tid >> 6) + 4 * i;
      } else {  // lanes along rows (consecutive pixels)
        rr = tid & 15;
        jj = (tid >> 4) + 16 * i;
      }
      float v = 0.f;
      if (r0 + rr < g.HW && j0 + jj < g.K) {
        v = sample_a<VARIANT>(g, xb, planb, r0 + rr, j0 + jj);
        if (MOD) {
          const size_t mi = ((size_t)b * g.N + (j0 + jj) / g.C) * g.HW + r0 + rr;
          DCN_DEV_ASSERT(mi < (size_t)g.B * g.N * g.HW);
          v = __ldg(mask + mi) * v;
        }
      }
      As[rr][jj] = v;
    }
    __syncthreads();
#pragma unroll
    for (int rr = 0; rr < TK; ++rr) {
      float a[4], w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = Gs[rr][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) w[j] = As[rr][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int o = o0 + ty * 4 + i;
    if (o >= g.O) continue;
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const int j = j0 + tx * 4 + jj;
      if (j < g.K) atomicAdd(gw + wt_index(g, o, j), acc[i][jj]);
    }
  }
}

// grad_bias[o] = sum_{b, r} gout[b, o, r]: one block per (o, batch slice), float4 streaming
// reads, block reduction, one red.global.add per block into a zeroed grad_bias.
template <typename T>
__global__ void __launch_bounds__(256) bias_grad_kernel(Geo g, int b_per_block, const T* __restrict__ gout,
                                                        float* __restrict__ gb) {
  const int o = blockIdx.x, b0 = blockIdx.y * b_per_block, b1 = min(g.B, b0 + b_per_block);
  float s = 0.f;
  // 4 elements per load: one float4, or 4 bfloat16 in 8 bytes
  const bool vec = (g.HW & 3) == 0;
  // the (batch element, pixel) pairs of this block's slice are walked as ONE flat index space, so that small
  // planes (8 x 8 pixels in the detector's last layer) keep all 256 threads busy
  const int per_b = vec ? (g.HW >> 2) : g.HW, total = (b1 - b0) * per_b;
  const size_t b_stride = (size_t)g.O * g.HW;
  const T* base = gout + ((size_t)b0 * g.O + o) * g.HW;
  for (int i = threadIdx.x; i < total; i += blockDim.x) {
    const int b = i / per_b, r = i - b * per_b;
    if (vec && sizeof(T) == 4) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(base + (size_t)b * b_stride) + r);
      s += (v.x + v.y) + (v.z + v.w);
    } else if (vec) {
      const uint2 v = __ldg(reinterpret_cast<const uint2*>(base + (size_t)b * b_stride) + r);
      s += (__uint_as_float(v.x << 16) + __uint_as_float(v.x & 0xffff0000u)) +
           (__uint_as_float(v.y << 16) + __uint_as_float(v.y & 0xffff0000u));
    } else {
      s += (float)base[(size_t)b * b_stride + r];
    }
  }
  __shared__ float red[8];
  for (int d = 16; d; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 8) {
    s = red[threadIdx.x];
    for (int d = 4; d; d >>= 1) s += __shfl_xor_sync(0xffu, s, d);
    if (threadIdx.x == 0) atomicAdd(gb + o, s);
  }
}

// grad_bias (may be null) from float or bfloat16 grad_out
int launch_bias_grad(const Geo& g, const void* gout, int operand, float* gb, cudaStream_t st) {
  if (!gb) return DCN_OK;
  DCN_CUDA_TRY(cudaMemsetAsync(gb, 0, sizeof(float) * (size_t)g.O, st));
  // enough blocks to stream gout at full bandwidth: ~8 per SM
  int slices = max(1, min(g.B, (148 * 8 + g.O - 1) / g.O));
  const int bpb = (g.B + slices - 1) / slices;
  slices = (g.B + bpb - 1) / bpb;
  KernelScope scope("bias_grad_kernel", st);
  if (operand == DCN_OPERAND_BF16)
    bias_grad_kernel<__nv_bfloat16><<<dim3(g.O, slices), 256, 0, st>>>(g, bpb, (const __nv_bfloat16*)gout, gb);
  else
    bias_grad_kernel<float><<<dim3(g.O, slices), 256, 0, st>>>(g, bpb, (const float*)gout, gb);
  DCN_KERNEL_CHECK("bias_grad_kernel");
  return DCN_OK;
}

// bf16 storage mode on the generic kernels: the bfloat16 operands are widened (exactly) into fp32
// scratch copies and the fp32 kernels run on those.  n must be even (every tensor here is).
__global__ void __launch_bounds__(256) widen_bf16_kernel(const __nv_bfloat162* __restrict__ src,
                                                         float2* __restrict__ dst, size_t n2) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (size_t)gridDim.x * blockDim.x)
    dst[i] = __bfloat1622float2(src[i]);
}

int launch_widen_bf16(const void* src, float* dst, size_t n, cudaStream_t st) {
  if (n & 1) {
    set_error("widen_bf16: odd element count %zu", n);
    return DCN_ERR_UNSUPPORTED;
  }
  const size_t n2 = n / 2;
  KernelScope scope("widen_bf16_kernel", st);
  widen_bf16_kernel<<<(unsigned)min((n2 + 255) / 256, (size_t)148 * 16), 256, 0, st>>>(
      (const __nv_bfloat162*)src, (float2*)dst, n2);
  DCN_KERNEL_CHECK("widen_bf16_kernel");
  return DCN_OK;
}

int launch_offset_scale(const Geo& g, float* goff, cudaStream_t st) {
  if (g.variant == DCN_VARIANT_DCNV1) return DCN_OK;  // coordinates are pixels already: factor 1
  const size_t total = (size_t)g.B * 2 * g.N * g.HW;
  KernelScope scope("offset_scale_kernel", st);
  offset_scale_kernel<<<(unsigned)min((total + 255) / 256, (size_t)8192), 256, 0, st>>>(g, goff);
  DCN_KERNEL_CHECK("offset_scale_kernel");
  return DCN_OK;
}

int simt_backward(const Geo& g, int flags, const float* x, const Tap* plan, const float* wt,
                  const float* gout, float* gx, float* goff, float* gw, float* gb,
                  cudaStream_t st, int parts, const float* mask, float* gmask) {
  const bool want_gx = !(flags & DCN_FLAG_NO_GRAD_X) && gx != nullptr;
  if (parts & SIMT_BWD_DATA) {
    if (want_gx && !(flags & DCN_FLAG_ACCUM_GRAD_X))
      DCN_CUDA_TRY(cudaMemsetAsync(gx, 0, sizeof(float) * (size_t)g.B * g.C * g.H * g.W, st));
    DCN_CUDA_TRY(cudaMemsetAsync(goff, 0, sizeof(float) * (size_t)g.B * 2 * g.N * g.HW, st));
    if (mask) DCN_CUDA_TRY(cudaMemsetAsync(gmask, 0, sizeof(float) * (size_t)g.B * g.N * g.HW, st));
  }
  if (parts & SIMT_BWD_WEIGHT) DCN_CUDA_TRY(cudaMemsetAsync(gw, 0, sizeof(float) * (size_t)g.O * g.K, st));
  if (parts & SIMT_BWD_DATA) {
    dim3 grid((g.HW + TM - 1) / TM, (g.K + TN - 1) / TN, g.B);
    {
      KernelScope scope("bwd_data_kernel", st);
      if (mask)
        bwd_data_kernel<DCN_VARIANT_JITTOR, true><<<grid, 256, 0, st>>>(g, want_gx, x, plan, wt, gout, gx, goff,
                                                                         mask, gmask);
      else if (g.variant == DCN_VARIANT_TORCH)
          bwd_data_kernel<DCN_VARIANT_TORCH><<<grid, 256, 0, st>>>(g, want_gx, x, plan, wt, gout, gx, goff, nullptr,
                                                                   nullptr);
      else
        bwd_data_kernel<DCN_VARIANT_JITTOR><<<grid, 256, 0, st>>>(g, want_gx, x, plan, wt, gout, gx, goff, nullptr,
                                                                  nullptr);
    }
    DCN_KERNEL_CHECK("bwd_data_kernel");
    int rc = launch_offset_scale(g, goff, st);
    if (rc) return rc;
  }
  if (parts & SIMT_BWD_WEIGHT) {
    const int tiles = ((g.O + TM - 1) / TM) * ((g.K + TN - 1) / TN);
    const int chunks = ((g.HW + TK - 1) / TK) * g.B;
    int splits = max(1, min(chunks, (148 * 8 + tiles - 1) / tiles));
    const int cps = (chunks + splits - 1) / splits;
    splits = (chunks + cps - 1) / cps;
    dim3 grid((g.O + TM - 1) / TM, (g.K + TN - 1) / TN, splits);
    KernelScope scope("bwd_weight_kernel", st);
    if (mask)
      bwd_weight_kernel<DCN_VARIANT_JITTOR, true><<<grid, 256, 0, st>>>(g, cps, x, plan, gout, gw, mask);
    else if (g.variant == DCN_VARIANT_TORCH)
      bwd_weight_kernel<DCN_VARIANT_TORCH><<<grid, 256, 0, st>>>(g, cps, x, plan, gout, gw, nullptr);
    else
      bwd_weight_kernel<DCN_VARIANT_JITTOR><<<grid, 256, 0, st>>>(g, cps, x, plan, gout, gw, nullptr);
    DCN_KERNEL_CHECK("bwd_weight_kernel");
  }
  if (gb && (parts & SIMT_BWD_BIAS)) {
    int rc = launch_bias_grad(g, gout, DCN_OPERAND_FP32, gb, st);
    if (rc) return rc;
  }
  return DCN_OK;
}

}  // namespace dcn

// in-place scale used by dcn_allreduce_sum_f32 (mean over ranks)
namespace dcn {
__global__ void __launch_bounds__(256) scale_kernel(float* __restrict__ buf, size_t count, float s) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count;
       i += (size_t)gridDim.x * blockDim.x)
    buf[i] *= s;
}
int scale_f32(float* buf, size_t count, float scale, cudaStream_t st) {
  if (!count) return DCN_OK;
  scale_kernel<<<(unsigned)min((count + 255) / 256, (size_t)1184), 256, 0, st>>>(buf, count, scale);
  DCN_KERNEL_CHECK("scale_kernel");
  return DCN_OK;
}
}  // namespace dcn
