// dcn_conv_small.cu — the companion offset convolution (deform_conv.py:16-21,58; train.py:80-85,98) for layers the
// shifted-view tcgen05 kernels of dcn_conv.cu do not take: fewer than 64 input channels (the detector's 16- and
// 32-channel layers, where a K step of one pixel's channels leaves 3/4 or 1/2 of a 128-byte operand row empty), and the
// forward pass of other channel counts that are a multiple of 16 but not of 64.
//
// These layers are small GEMMs with tiny N (2N = 18 outputs) on a lot of pixels: HBM-bound by far (conv2 of the
// detector at batch 1024: 21.7 GFLOP over 1.4 GB).  The plain mode of the DCN kernels ran them at 1.2 ms forward and
// 1.8 ms backward because it pays the sampling machinery (plan entries, four-corner blends) for integer taps.  Here
// they are warp-level tensor-core kernels — mma.sync.m16n8k16 bf16 with the same hi/lo 3-term split as everywhere else
// (fp32-class result), operands converted in registers straight from the framed channels-last copy of x, no operand
// staging in shared memory, no barriers in the main loops:
//   forward   D[pixel, o]      = sum_{tap, c} x[pixel @ tap, c] * W[o, c, tap]        warp = 32 output pixels
//   dgrad     E[pixel, tap, c] = sum_o goff[pixel, o] * W[o, c, tap], red.global.add.v4 into the framed channels-last
//             gradient accumulator the DCN data gradient also adds into            warp = 16 output pixels
//   wgrad     gW[c, o | tap]  += sum_pixel x[pixel @ tap, c] * goff[pixel, o]         block = (kernel row, 16 channels),
//             accumulators live in registers over each warp's whole pixel stream (next chunk's loads issued before the
//             current one is converted), shared-memory block reduction, one atomicAdd per block and entry
// Measured on detector conv2 (batch 1024): 0.375 / 0.66 / 0.45 ms — forward and data gradient at 58 % of the HBM copy
// peak (profiles/r2_ncu_conv_small.txt); HMMA.16816 issues every 8 cycles per sub-partition (tools/hmma_probe.cu), far
// above what N = 18 needs.  The backward pair is used below 64 channels only: at 64 / 128 channels the plain mode of the
// fused DCN backward kernel is faster (dcn_conv.cu:conv_offset_bwd_supported).
// 3 x 3 kernels, padding 1, stride 1 or 2, C % 16 == 0, 2N <= 32.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>

#include "dcn_common.cuh"
#include "dcn_umma.cuh"
#include "dcn_umma_common.cuh"

namespace dcn {

namespace cs {

constexpr int kThreads = 256;

struct Params {
  int B, C, O, H, W, Ho, Wo, HoWo, s;
  int pitch;            // pixels per framed row (W + 2)
  size_t img_stride;    // floats per framed image
  int perm_G, perm_Cs;  // staged channel cs <-> original channel (cs % G) * Cs + cs / G (Torch layout), 0 = identity
  int KS;               // 16-channel K steps per tap (forward) = channel m-tiles (wgrad)
  int KO;               // 16-output K steps (dgrad)
  int chunks;           // pixel chunks per image: 32 (forward) or 16 (dgrad, wgrad) pixels
  FastDiv div_chunks, div_wo;
  const float* xt;
  const float* bias;
  const float* goff;
  float* out;
  float* gxt;
  float* gw;
  const uint2* wfrag;
};

__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], const uint2 b) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b.x), "r"(b.y));
}

// element offset of framed pixel (row ho * s + kh, column wo * s + kw), channel 0 — padding 1 cancels the frame
__device__ __forceinline__ int pix_off(const Params& P, int q) {
  uint32_t ho, wo;
  P.div_wo.divmod((uint32_t)q, ho, wo);
  return ((int)ho * P.s * P.pitch + (int)wo * P.s) * P.C;
}

// ---- weight fragments -----------------------------------------------------------------------------------------------
// The MMA does not care which channel sits in which K slot / N column as long as both operands (or the epilogue) agree,
// so the slots are dealt such that every thread reads or adds 16 contiguous bytes:
// forward: [(tap * KS + ks) * NT + nt][hi | lo][lane] = B fragment of W[o = nt * 8 + g][cs][tap], K slots (2t, 2t + 1,
//          2t + 8, 2t + 9) of step ks <-> staged channels ks * 16 + 4t + (0, 1, 2, 3): A is ONE float4 per row
// dgrad:   [(tap * C / 8 + ct) * KO + ks][hi | lo][lane] = B fragment of W[o = ks * 16 + 2t (+1, +8, +9)][cs][tap], column
//          2t' + j of n-tile ct = 2p + h <-> staged channel p * 16 + 4t' + 2h + j: the two accumulators of a tile pair
//          are one float4 of the gradient
__global__ void __launch_bounds__(256) wfrag_kernel(Params P, int dgrad, int NT, const float* __restrict__ w,
                                                    uint2* __restrict__ frag) {
  const int nfr = dgrad ? 9 * (P.C / 8) * P.KO : 9 * P.KS * NT;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < nfr * 32; i += gridDim.x * 256) {
    const int lane = i & 31, f = i >> 5, g = lane >> 2, t = lane & 3;
    float v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int kk = 2 * t + (e & 1) + (e >> 1) * 8;  // K index inside the step
      int o, csn, tap;
      if (dgrad) {
        const int ks = f % P.KO, nt = f / P.KO;
        const int ct = nt % (P.C / 8);
        tap = nt / (P.C / 8);
        csn = (ct >> 1) * 16 + 4 * (g >> 1) + 2 * (ct & 1) + (g & 1);
        o = ks * 16 + kk;
      } else {
        const int nt = f % NT, r = f / NT;
        tap = r / P.KS;
        csn = (r % P.KS) * 16 + 4 * t + e;
        o = nt * 8 + g;
      }
      const int c = P.perm_G ? (csn % P.perm_G) * P.perm_Cs + csn / P.perm_G : csn;
      v[e] = o < P.O ? w[((size_t)o * P.C + c) * 9 + tap] : 0.f;
    }
    uint2 hi, lo;
    ptx::split_pair(v[0], v[1], hi.x, lo.x);
    ptx::split_pair(v[2], v[3], hi.y, lo.y);
    frag[(size_t)f * 64 + lane] = hi;
    frag[(size_t)f * 64 + 32 + lane] = lo;
  }
}

// ---- forward --------------------------------------------------------------------------------------------------------
// MASK: the modulated layer's 3N-channel conv: outputs [0, 2N) go to out [B, 2N, Ho*Wo], outputs [2N, 3N) to
// mask [B, N, Ho*Wo] as sigmoid(acc + bias); a trailing argument, the unmodulated parameter layout does not move
template <int NT, bool MASK = false>
__global__ void __launch_bounds__(kThreads) fwd_kernel(Params P, float* mask = nullptr) {
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int warps = gridDim.x * (kThreads / 32);
  const int units = P.B * P.chunks;
  for (int u = blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); u < units; u += warps) {
    uint32_t b, ch;
    P.div_chunks.divmod((uint32_t)u, b, ch);
    const int q0 = (int)ch * 32;
    int roff[2][2];  // element offsets of rows g / g + 8 of the two m-tiles (clamped: out-of-range rows are not stored)
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int h = 0; h < 2; ++h) roff[mt][h] = pix_off(P, min(q0 + mt * 16 + h * 8 + g, P.HoWo - 1)) + 4 * t;
    const float* xb = P.xt + (size_t)b * P.img_stride;
    float acc[2][NT][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.f;
    const uint2* wf = P.wfrag + lane;
    for (int tap = 0; tap < 9; ++tap) {
      const int kh = tap / 3, kw = tap - kh * 3;
      const float* xtap = xb + (kh * P.pitch + kw) * P.C;
      for (int ks = 0; ks < P.KS; ++ks) {
        uint32_t ahi[2][4], alo[2][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          // rows g / g + 8: channels ks * 16 + 4t .. + 3 = K slots 2t, 2t + 1 | 2t + 8, 2t + 9
          DCN_DEV_ASSERT((size_t)((kh * P.pitch + kw) * P.C + max(roff[mt][0], roff[mt][1]) + ks * 16 + 4) <= P.img_stride);
          const float4 v0 = __ldg(reinterpret_cast<const float4*>(xtap + roff[mt][0] + ks * 16));
          const float4 v1 = __ldg(reinterpret_cast<const float4*>(xtap + roff[mt][1] + ks * 16));
          ptx::split_pair(v0.x, v0.y, ahi[mt][0], alo[mt][0]);
          ptx::split_pair(v1.x, v1.y, ahi[mt][1], alo[mt][1]);
          ptx::split_pair(v0.z, v0.w, ahi[mt][2], alo[mt][2]);
          ptx::split_pair(v1.z, v1.w, ahi[mt][3], alo[mt][3]);
        }
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
          const uint2 bh = __ldg(wf), bl = __ldg(wf + 32);
          wf += 64;
#pragma unroll
          for (int mt = 0; mt < 2; ++mt) {
            mma16816(acc[mt][nt], alo[mt], bh);
            mma16816(acc[mt][nt], ahi[mt], bl);
            mma16816(acc[mt][nt], ahi[mt], bh);
          }
        }
      }
    }
    // offsets [B, O, Ho*Wo]: thread holds pixels g / g + 8, outputs nt * 8 + 2t (+1)
    if constexpr (MASK) {
      const int n_off = P.O / 3 * 2;
      float* ob = P.out + (size_t)b * n_off * P.HoWo;
      float* mb = mask + (size_t)b * (P.O - n_off) * P.HoWo;
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int o = nt * 8 + 2 * t + j;
          if (o >= P.O) continue;
          const float bv = P.bias ? P.bias[o] : 0.f;
#pragma unroll
          for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int q = q0 + mt * 16 + h * 8 + g;
              if (q >= P.HoWo) continue;
              const float z = acc[mt][nt][h * 2 + j] + bv;
              if (o < n_off) ob[(size_t)o * P.HoWo + q] = z;
              else mb[(size_t)(o - n_off) * P.HoWo + q] = 1.f / (1.f + expf(-z));
            }
        }
      }
      continue;
    }
    float* ob = P.out + (size_t)b * P.O * P.HoWo;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int o = nt * 8 + 2 * t + j;
        if (o >= P.O) continue;
        const float bv = P.bias ? P.bias[o] : 0.f;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int q = q0 + mt * 16 + h * 8 + g;
            if (q < P.HoWo) ob[(size_t)o * P.HoWo + q] = acc[mt][nt][h * 2 + j] + bv;
          }
      }
    }
  }
}

// ---- data gradient: scatter form ------------------------------------------------------------------------------------
template <int KO>
__global__ void __launch_bounds__(kThreads) dgrad_kernel(Params P) {
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int warps = gridDim.x * (kThreads / 32);
  const int units = P.B * P.chunks;
  const int CT = P.C / 8;
  for (int u = blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); u < units; u += warps) {
    uint32_t b, ch;
    P.div_chunks.divmod((uint32_t)u, b, ch);
    const int q0 = (int)ch * 16;
    const int qa = q0 + g, qb = q0 + g + 8;
    const bool oka = qa < P.HoWo, okb = qb < P.HoWo;
    // A = goff[pixel, o]: rows = pixels g / g + 8, K = outputs 2t, 2t + 1, 2t + 8, 2t + 9 of the step
    const float* gb = P.goff + (size_t)b * P.O * P.HoWo;
    uint32_t ahi[KO][4], alo[KO][4];
#pragma unroll
    for (int ks = 0; ks < KO; ++ks) {
      float v[2][4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int o = ks * 16 + 2 * t + (e & 1) + (e >> 1) * 8;
        const bool oo = o < P.O;
        v[0][e] = (oo && oka) ? __ldg(gb + (size_t)o * P.HoWo + qa) : 0.f;
        v[1][e] = (oo && okb) ? __ldg(gb + (size_t)o * P.HoWo + qb) : 0.f;
      }
      ptx::split_pair(v[0][0], v[0][1], ahi[ks][0], alo[ks][0]);
      ptx::split_pair(v[1][0], v[1][1], ahi[ks][1], alo[ks][1]);
      ptx::split_pair(v[0][2], v[0][3], ahi[ks][2], alo[ks][2]);
      ptx::split_pair(v[1][2], v[1][3], ahi[ks][3], alo[ks][3]);
    }
    float* ga = P.gxt + (size_t)b * P.img_stride + pix_off(P, min(qa, P.HoWo - 1)) + 4 * t;
    float* gbp = P.gxt + (size_t)b * P.img_stride + pix_off(P, min(qb, P.HoWo - 1)) + 4 * t;
    const uint2* wf = P.wfrag + lane;
    for (int tap = 0; tap < 9; ++tap) {
      const int kh = tap / 3, kw = tap - kh * 3;
      const int toff = (kh * P.pitch + kw) * P.C;
      for (int cp = 0; cp < CT / 2; ++cp) {  // n-tile pair = 16 staged channels, 4 per thread
        float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
          for (int ks = 0; ks < KO; ++ks) {
            const uint2 bh = __ldg(wf), bl = __ldg(wf + 32);
            wf += 64;
            mma16816(acc[h], alo[ks], bh);
            mma16816(acc[h], ahi[ks], bl);
            mma16816(acc[h], ahi[ks], bh);
          }
        DCN_DEV_ASSERT((size_t)(pix_off(P, min(qb, P.HoWo - 1)) + 4 * t + toff + cp * 16 + 4) <= P.img_stride);
        if (oka)
          atomicAdd(reinterpret_cast<float4*>(ga + toff + cp * 16), make_float4(acc[0][0], acc[0][1], acc[1][0], acc[1][1]));
        if (okb)
          atomicAdd(reinterpret_cast<float4*>(gbp + toff + cp * 16), make_float4(acc[0][2], acc[0][3], acc[1][2], acc[1][3]));
      }
    }
  }
}

// ---- weight gradient ------------------------------------------------------------------------------------------------
// warp role = (kernel row kh, channel m-tile mt); the warps of one role share the pixel chunks round-robin.  The loads of
// the NEXT chunk are issued before the current one is converted and multiplied (both operands stream from HBM and nothing
// else hides that latency: 105 registers of accumulators and fragments leave four warps per scheduler).
constexpr int kWgradThreads = 128;

template <int NT>
struct WgradRaw {
  float4 b[NT];     // goff[o = nt * 8 + g][pixels q0 + 4t .. + 3]
  float2 a[3][4];   // x[pixel e @ (kh, kw)][channels mt * 16 + 2g, + 1]
};

template <int NT>
__device__ __forceinline__ void wgrad_load(const Params& P, int u, int kh, int mt, int g, int t, WgradRaw<NT>& r) {
  uint32_t b, ch;
  P.div_chunks.divmod((uint32_t)u, b, ch);
  const int q0 = (int)ch * 16 + 4 * t;  // K slots 2t, 2t + 1, 2t + 8, 2t + 9 <-> pixels q0 .. q0 + 3 (both operands)
  const float* gb = P.goff + (size_t)b * P.O * P.HoWo + q0;
  // row g <-> staged channel mt * 16 + 2g, row g + 8 <-> channel mt * 16 + 2g + 1: one float2 per pixel and tap; pixels
  // past the end read a valid pixel (their goff is zero)
  const float* xb = P.xt + (size_t)b * P.img_stride + kh * P.pitch * P.C + mt * 16 + 2 * g;
  if ((P.Wo & 3) == 0) {
    // the thread's four pixels are in the image together or not at all, lie in one output row and every plane of goff
    // is 16-byte aligned: one float4 per plane, one row / column split per thread
    const bool in = q0 < P.HoWo;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const int o = nt * 8 + g;
      r.b[nt] = (in && o < P.O) ? __ldg(reinterpret_cast<const float4*>(gb + (size_t)o * P.HoWo))
                                : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const float* xp = xb + pix_off(P, in ? q0 : 0);
    const int step = P.s * P.C;
    DCN_DEV_ASSERT((size_t)(kh * P.pitch * P.C + mt * 16 + 2 * g + pix_off(P, in ? q0 : 0) + 3 * step + 2 * P.C + 2) <= P.img_stride);
#pragma unroll
    for (int e = 0; e < 4; ++e)
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) r.a[kw][e] = __ldg(reinterpret_cast<const float2*>(xp + e * step + kw * P.C));
    return;
  }
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    const int o = nt * 8 + g;
    float v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) v[e] = (o < P.O && q0 + e < P.HoWo) ? __ldg(gb + (size_t)o * P.HoWo + e) : 0.f;
    r.b[nt] = make_float4(v[0], v[1], v[2], v[3]);
  }
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float* xp = xb + pix_off(P, min(q0 + e, P.HoWo - 1));
#pragma unroll
    for (int kw = 0; kw < 3; ++kw) r.a[kw][e] = __ldg(reinterpret_cast<const float2*>(xp + kw * P.C));
  }
}

template <int NT>
__global__ void __launch_bounds__(kWgradThreads) wgrad_kernel(Params P) {
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  // the role is uniform over the block (its four warps are four streams of it): one shared-memory reduction and one
  // atomicAdd per block and entry at the end.  gridDim.x is a multiple of the role count.
  constexpr int kWarps = kWgradThreads / 32;
  const int roles = 3 * P.KS;
  const int warp = threadIdx.x >> 5;
  const int role = blockIdx.x % roles;
  const int nstreams = gridDim.x / roles * kWarps, stream = blockIdx.x / roles * kWarps + warp;
  const int kh = role % 3, mt = role / 3;
  const int units = P.B * P.chunks;
  float acc[3][NT][4];
#pragma unroll
  for (int kw = 0; kw < 3; ++kw)
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[kw][nt][e] = 0.f;
  WgradRaw<NT> cur, nxt;
  if (stream < units) wgrad_load<NT>(P, stream, kh, mt, g, t, cur);
  for (int u = stream; u < units; u += nstreams) {
    if (u + nstreams < units) wgrad_load<NT>(P, u + nstreams, kh, mt, g, t, nxt);
    uint2 bhi[NT], blo[NT];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      ptx::split_pair(cur.b[nt].x, cur.b[nt].y, bhi[nt].x, blo[nt].x);
      ptx::split_pair(cur.b[nt].z, cur.b[nt].w, bhi[nt].y, blo[nt].y);
    }
#pragma unroll
    for (int kw = 0; kw < 3; ++kw) {
      uint32_t ahi[4], alo[4], H[4], L[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) ptx::split_pair(cur.a[kw][e].x, cur.a[kw][e].y, H[e], L[e]);   // (ch 2g | ch 2g + 1) of pixel e
      // a0,a1: row g, K slots 2t, 2t + 1 (pixels 0, 1); a2,a3: row g + 8, same pixels; a4..a7: pixels 2, 3 — the
      // (channel pair) x (pixel pair) transposition is two PRMTs per register pair
      ahi[0] = __byte_perm(H[0], H[1], 0x5410); ahi[1] = __byte_perm(H[0], H[1], 0x7632);
      ahi[2] = __byte_perm(H[2], H[3], 0x5410); ahi[3] = __byte_perm(H[2], H[3], 0x7632);
      alo[0] = __byte_perm(L[0], L[1], 0x5410); alo[1] = __byte_perm(L[0], L[1], 0x7632);
      alo[2] = __byte_perm(L[2], L[3], 0x5410); alo[3] = __byte_perm(L[2], L[3], 0x7632);
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        mma16816(acc[kw][nt], alo, bhi[nt]);
        mma16816(acc[kw][nt], ahi, blo[nt]);
        mma16816(acc[kw][nt], ahi, bhi[nt]);
      }
    }
    cur = nxt;
  }
  // block reduction: warps 1..3 park their accumulators in shared memory, warp 0 adds them up
  __shared__ float red[kWarps - 1][3 * NT * 4][32];
  if (warp > 0) {
#pragma unroll
    for (int kw = 0; kw < 3; ++kw)
#pragma unroll
      for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) red[warp - 1][(kw * NT + nt) * 4 + e][lane] = acc[kw][nt][e];
  }
  __syncthreads();
  if (warp > 0) return;
  // D rows g / g + 8 = staged channels mt * 16 + 2g / + 1, columns = outputs nt * 8 + 2t (+1)
  int crow[2];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int csn = mt * 16 + 2 * g + h;
    crow[h] = P.perm_G ? (csn % P.perm_G) * P.perm_Cs + csn / P.perm_G : csn;
  }
#pragma unroll
  for (int kw = 0; kw < 3; ++kw)
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int o = nt * 8 + 2 * t + (e & 1);
        if (o >= P.O) continue;
        float v = acc[kw][nt][e];
#pragma unroll
        for (int w2 = 0; w2 < kWarps - 1; ++w2) v += red[w2][(kw * NT + nt) * 4 + e][lane];
        atomicAdd(P.gw + ((size_t)o * P.C + crow[e >> 1]) * 9 + kh * 3 + kw, v);
      }
}

}  // namespace cs

// ---------------------------------------------------------------------------- host side
// O = output channels of the conv: 2N (offsets) or 3N (offsets and mask logits of the modulated layer)
static bool small_params(const Geo& g, cs::Params* Pp, int O) {
  cs::Params& P = *Pp;
  memset(&P, 0, sizeof(P));
  if (g.N != 9 || g.kw != 3 || g.sh != g.sw || g.ph != 1 || g.pw != 1) return false;
  if (g.sh != 1 && g.sh != 2) return false;
  if (g.C % 16 != 0 || g.C > 512 || O > 32) return false;
  // every read stays inside the framed copy (rows 0 .. H + 2, columns 0 .. W + 1)
  if ((g.Ho - 1) * g.sh + 2 > g.H + 2 || (g.Wo - 1) * g.sw + 2 > g.W + 1) return false;
  if ((long long)xt_image_stride(g) >= (1LL << 30)) return false;
  if ((long long)g.B * ((g.HW + 15) / 16) > 0x7fffffffLL) return false;
  Tiling t;
  if (!make_tiling(g, &t)) return false;
  if (g.variant == DCN_VARIANT_TORCH) {
    P.perm_G = t.G;
    P.perm_Cs = t.Cs;
  }
  P.B = g.B; P.C = g.C; P.O = O; P.H = g.H; P.W = g.W; P.Ho = g.Ho; P.Wo = g.Wo; P.HoWo = g.HW; P.s = g.sh;
  P.pitch = g.W + 2;
  P.img_stride = xt_image_stride(g);
  P.KS = g.C / 16;
  P.KO = (O + 15) / 16;
  P.div_wo = FastDiv::make(g.Wo);
  return true;
}

bool conv_small_supported(const Geo& g, int O) {
  cs::Params P;
  return small_params(g, &P, O);
}

// fragment scratch: the forward and the data-gradient pass run one after the other and share it
size_t conv_small_wfrag_bytes(const Geo& g, int O) {
  cs::Params P;
  if (!small_params(g, &P, O)) return 0;
  const int NT = (P.O + 7) / 8;
  const size_t f = (size_t)9 * P.KS * NT, d = (size_t)9 * (P.C / 8) * P.KO;
  return align_up((f > d ? f : d) * 64 * sizeof(uint2), 1024);
}

static int small_wfrag(const cs::Params& P, int dgrad, int NT, const float* w, uint2* frag, cudaStream_t st) {
  const int nfr = dgrad ? 9 * (P.C / 8) * P.KO : 9 * P.KS * NT;
  KernelScope scope("conv_small_wfrag_kernel", st);
  cs::wfrag_kernel<<<std::min((nfr * 32 + 255) / 256, 1024), 256, 0, st>>>(P, dgrad, NT, w, frag);
  DCN_KERNEL_CHECK("conv_small_wfrag_kernel");
  return DCN_OK;
}

// mask_out != nullptr: O = 3N, outputs [2N, 3N) go to mask_out through the sigmoid
int conv_small_forward(const Geo& g, int O, const float* xt, const float* woff, const float* boff, float* offset_out,
                       uint8_t* wfrag, cudaStream_t st, float* mask_out) {
  cs::Params P;
  if (!small_params(g, &P, O)) {
    set_error("offset conv (warp-MMA kernel): shape not supported");
    return DCN_ERR_UNSUPPORTED;
  }
  const int NT = (P.O + 7) / 8;
  int rc;
  if ((rc = small_wfrag(P, 0, NT, woff, (uint2*)wfrag, st))) return rc;
  P.xt = xt;
  P.bias = boff;
  P.out = offset_out;
  P.wfrag = (const uint2*)wfrag;
  P.chunks = (P.HoWo + 31) / 32;
  P.div_chunks = FastDiv::make(P.chunks);
  const long long units = (long long)P.B * P.chunks;
  const int grid = (int)std::min<long long>((units + 7) / 8, (long long)num_sms() * 8);
  if (mask_out) {
    KernelScope scope("conv_small_mask_fwd_kernel", st);
    if (NT == 4) cs::fwd_kernel<4, true><<<grid, cs::kThreads, 0, st>>>(P, mask_out);
    else if (NT == 3) cs::fwd_kernel<3, true><<<grid, cs::kThreads, 0, st>>>(P, mask_out);
    else if (NT == 2) cs::fwd_kernel<2, true><<<grid, cs::kThreads, 0, st>>>(P, mask_out);
    else cs::fwd_kernel<1, true><<<grid, cs::kThreads, 0, st>>>(P, mask_out);
    DCN_KERNEL_CHECK("conv_small_mask_fwd_kernel");
    return DCN_OK;
  }
  KernelScope scope("conv_small_fwd_kernel", st);
  switch (NT) {
    case 1: cs::fwd_kernel<1><<<grid, cs::kThreads, 0, st>>>(P); break;
    case 2: cs::fwd_kernel<2><<<grid, cs::kThreads, 0, st>>>(P); break;
    case 3: cs::fwd_kernel<3><<<grid, cs::kThreads, 0, st>>>(P); break;
    default: cs::fwd_kernel<4><<<grid, cs::kThreads, 0, st>>>(P); break;
  }
  DCN_KERNEL_CHECK("conv_small_fwd_kernel");
  return DCN_OK;
}

// gxt += data gradient (gxt may be null), gwoff = weight gradient (zeroed here)
int conv_small_backward(const Geo& g, int O, const float* xt, float* gxt, const float* goff, const float* woff,
                        float* gwoff, uint8_t* wfrag, cudaStream_t st) {
  cs::Params P;
  if (!small_params(g, &P, O)) {
    set_error("offset conv backward (warp-MMA kernel): shape not supported");
    return DCN_ERR_UNSUPPORTED;
  }
  const int NT = (P.O + 7) / 8;
  const int sms = num_sms();
  int rc;
  P.xt = xt;
  P.goff = goff;
  P.chunks = (P.HoWo + 15) / 16;
  P.div_chunks = FastDiv::make(P.chunks);
  const long long units = (long long)P.B * P.chunks;
  if (gxt) {
    if ((rc = small_wfrag(P, 1, NT, woff, (uint2*)wfrag, st))) return rc;
    P.gxt = gxt;
    P.wfrag = (const uint2*)wfrag;
    const int grid = (int)std::min<long long>((units + 7) / 8, (long long)sms * 8);
    KernelScope scope("conv_small_dgrad_kernel", st);
    if (P.KO == 1) cs::dgrad_kernel<1><<<grid, cs::kThreads, 0, st>>>(P);
    else cs::dgrad_kernel<2><<<grid, cs::kThreads, 0, st>>>(P);
    DCN_KERNEL_CHECK("conv_small_dgrad_kernel");
  }
  DCN_CUDA_TRY(cudaMemsetAsync(gwoff, 0, sizeof(float) * (size_t)P.O * P.C * 9, st));
  P.gw = gwoff;
  {
    // blocks = roles x groups of four streams: enough to fill the machine (four blocks per SM by registers), at least
    // 16 chunks per stream
    const int roles = 3 * P.KS;
    const int wpb = cs::kWgradThreads / 32;
    long long groups = std::max<long long>(1, (long long)sms * 4 / roles);
    groups = std::max<long long>(1, std::min<long long>(groups, units / (16 * wpb)));
    const int grid = (int)(groups * roles);
    KernelScope scope("conv_small_wgrad_kernel", st);
    switch (NT) {
      case 1: cs::wgrad_kernel<1><<<grid, cs::kWgradThreads, 0, st>>>(P); break;
      case 2: cs::wgrad_kernel<2><<<grid, cs::kWgradThreads, 0, st>>>(P); break;
      case 3: cs::wgrad_kernel<3><<<grid, cs::kWgradThreads, 0, st>>>(P); break;
      default: cs::wgrad_kernel<4><<<grid, cs::kWgradThreads, 0, st>>>(P); break;
    }
    DCN_KERNEL_CHECK("conv_small_wgrad_kernel");
  }
  return DCN_OK;
}

}  // namespace dcn
