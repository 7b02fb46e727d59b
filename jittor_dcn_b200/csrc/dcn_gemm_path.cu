// dcn_gemm_path.cu — Torch column layout (train.py:129-131) at shapes the fused tensor path cannot tile:
// gcd(Ho*Wo, C) not a multiple of 16 (ResNet-50 C5: gcd(196, 512) = 4).
//
// The raw reshape of train.py:129-131 hands GEMM row r, column j the flat sample f = r*K + j of the (c, h, w, n)-ordered
// sample tensor S[b, c, q], q = pixel*N + tap.  Only gcd(Ho*Wo, C) rows share their sampling points, so with a small
// gcd the fused kernels (which amortise one bilinear footprint over 16 .. 64 channels of a tile) have nothing to
// amortise over and these layers ran on the generic CUDA-core kernels: 23 ms per C5 layer, 69 of the 98 ms of the
// configs[3] stack.  But exactly these layers are SMALL in samples (B*C*P = 115 M for C5: 231 MB in bf16), so here the
// reference's own structure is affordable: materialise S once — sampled point by point with all channels vectorised
// from the channels-last framed copy, written transposed —, and the three contractions are PLAIN GEMMs over views of it:
//   forward       out_b[O, HW]  = Wm[O, K] * A_b^T,            A_b = S_b viewed as [HW, K]          (train.py:133-134)
//   data gradient gS_b[HW, K]   = gout_b^T[HW, O] * Wm[O, K]   -> scatter kernel (bilinear col2im + coordinate gradient)
//   weight grad   gW[O, K]      = goutT[O, B*HW] * A[B*HW, K]
// Plain library GEMMs go to cuBLAS (dlopen'ed like NCCL: no link-time dependency; inside a PyTorch process this binds
// to the libcublas.so.12 torch already loaded).  Every GEMM is bf16 x bf16 -> fp32 accumulate.  fp32 operands: three
// GEMMs over (hi, lo) bfloat16 splits (see gemm_path_forward); bf16 operands: one GEMM, S and gS stored in bf16 (one
// rounding of each sample, as the tensor path).
#include <cublas_v2.h>
#include <cuda_bf16.h>
#include <dlfcn.h>

#include <mutex>

#include "dcn_umma.cuh"
#include "dcn_umma_common.cuh"

namespace dcn {

size_t umma_xt_bytes(const Geo& g, int operand);

namespace gp {

// ---------------------------------------------------------------------------- cuBLAS through dlopen
struct CublasApi {
  void* handle = nullptr;
  cublasStatus_t (*Create)(cublasHandle_t*) = nullptr;
  cublasStatus_t (*SetStream)(cublasHandle_t, cudaStream_t) = nullptr;
  cublasStatus_t (*SetWorkspace)(cublasHandle_t, void*, size_t) = nullptr;
  cublasStatus_t (*GemmEx)(cublasHandle_t, cublasOperation_t, cublasOperation_t, int, int, int, const void*, const void*,
                           cudaDataType, int, const void*, cudaDataType, int, const void*, void*, cudaDataType, int,
                           cublasComputeType_t, cublasGemmAlgo_t) = nullptr;
  cublasStatus_t (*GemmStridedBatchedEx)(cublasHandle_t, cublasOperation_t, cublasOperation_t, int, int, int, const void*,
                                         const void*, cudaDataType, int, long long, const void*, cudaDataType, int,
                                         long long, const void*, void*, cudaDataType, int, long long, int,
                                         cublasComputeType_t, cublasGemmAlgo_t) = nullptr;
};
static CublasApi g_api;
static std::once_flag g_once;
static std::mutex g_mu, g_use_mu;
static cublasHandle_t g_handles[64] = {};

static bool load_cublas() {
  std::call_once(g_once, [] {
    for (const char* n : {"libcublas.so.12", "libcublas.so"}) {
      g_api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (g_api.handle) break;
    }
    if (!g_api.handle) return;
    g_api.Create = (decltype(g_api.Create))dlsym(g_api.handle, "cublasCreate_v2");
    g_api.SetStream = (decltype(g_api.SetStream))dlsym(g_api.handle, "cublasSetStream_v2");
    g_api.SetWorkspace = (decltype(g_api.SetWorkspace))dlsym(g_api.handle, "cublasSetWorkspace_v2");
    g_api.GemmEx = (decltype(g_api.GemmEx))dlsym(g_api.handle, "cublasGemmEx");
    g_api.GemmStridedBatchedEx = (decltype(g_api.GemmStridedBatchedEx))dlsym(g_api.handle, "cublasGemmStridedBatchedEx");
  });
  const bool ok = g_api.handle && g_api.Create && g_api.SetStream && g_api.GemmEx && g_api.GemmStridedBatchedEx;
  if (!ok) set_error("cuBLAS (libcublas.so.12) could not be loaded: %s", dlerror());
  return ok;
}

// one handle per device, created on first use and kept (cuBLAS handles are expensive)
static cublasHandle_t handle_for_current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) return nullptr;
  std::lock_guard<std::mutex> lock(g_mu);
  if (!g_handles[dev] && g_api.Create(&g_handles[dev]) != CUBLAS_STATUS_SUCCESS) g_handles[dev] = nullptr;
  return g_handles[dev];
}

constexpr size_t kCublasWs = 32u << 20;   // caller-owned cuBLAS workspace (keeps the calls capturable in CUDA graphs)

// ---------------------------------------------------------------------------- kernels
constexpr int kQT = 32, kCT = 128;   // block tile: 32 sampling points x 128 channels

template <typename T>
__device__ __forceinline__ float ldf(const T* p) { return (float)__ldg(p); }
template <>
__device__ __forceinline__ float ldf<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat162float(*p);
}

struct Corner {
  int base;        // element offset (channel 0) of the north-west corner inside the framed image
  float w[4];      // nw, ne, sw, se — zero when no corner lies inside the image
  float fx, fy;
  int inside;
};
__device__ __forceinline__ Corner corner_of(const Geo& g, const Tap& tp) {
  Corner c;
  bool inside;
  c.base = xt_corner_base(g, tp.y0, tp.x0, inside);
  c.inside = inside ? 1 : 0;
  c.fx = tp.fx;
  c.fy = tp.fy;
  c.w[0] = c.w[1] = c.w[2] = c.w[3] = 0.f;
  if (inside) corner_weights(tp, c.w);
  return c;
}

// S[b, c, q] = bilinear sample of channel c at sampling point q (deform_conv.py:47-52 / train.py:121-127).
// Block = 32 points of one image; loop over 128-channel tiles: warps gather point by point (lane = channel: 128-byte
// coalesced corner reads), the tile is transposed through shared memory and written with lane = point.
// fp32 operands (T = float): S is written as TWO bfloat16 matrices, hi = bf16(v) into S and lo = bf16(v - hi) into S_lo,
// for the three-term tensor-core GEMMs (see gemm_path_forward); bf16 operands: S only
template <typename T>
__global__ void __launch_bounds__(256) sample_kernel(Geo g, const T* __restrict__ xt, const Tap* __restrict__ plan,
                                                     __nv_bfloat16* __restrict__ S, __nv_bfloat16* __restrict__ S_lo) {
  __shared__ float tile[kQT][kCT + 1];
  const int b = blockIdx.y, q0 = blockIdx.x * kQT;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const T* img = xt + (size_t)b * xt_image_stride(g);
  const int pitch = xt_row_pitch(g);
  Corner cs[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int q = q0 + warp + 8 * i;
    Tap tp = {0, 0, 0.f, 0.f};
    tp.y0 = tp.x0 = -100;
    if (q < g.P) tp = plan[(size_t)b * g.P + q];
    cs[i] = corner_of(g, tp);
  }
  for (int c0 = 0; c0 < g.C; c0 += kCT) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const T* p = img + cs[i].base;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int c = c0 + k * 32 + lane;
        float v = 0.f;
        if (c < g.C) {
          const float v0 = ldf(p + c), v1 = ldf(p + g.C + c), v2 = ldf(p + pitch + c), v3 = ldf(p + pitch + g.C + c);
          v = fmaf(v3, cs[i].w[3], fmaf(v2, cs[i].w[2], fmaf(v1, cs[i].w[1], v0 * cs[i].w[0])));
        }
        tile[warp + 8 * i][k * 32 + lane] = v;
      }
    }
    __syncthreads();
    const int q = q0 + lane;
#pragma unroll
    for (int j = 0; j < kCT / 8; ++j) {
      const int cl = warp + 8 * j, c = c0 + cl;
      if (c < g.C && q < g.P) {
        const size_t idx = ((size_t)b * g.C + c) * g.P + q;
        if constexpr (sizeof(T) == 4) {
          __nv_bfloat16 hi, lo;
          ptx::split_bf16(tile[lane][cl], hi, lo);
          S[idx] = hi;
          S_lo[idx] = lo;
        } else {
          S[idx] = (T)tile[lane][cl];
        }
      }
    }
    __syncthreads();
  }
}

// Backward of the sampling: gS[b, c, q] -> grad_x (red.global.add into the framed channels-last accumulator, 128-byte
// coalesced) and grad_offset.  Every sampling point belongs to exactly one warp, which accumulates its coordinate
// gradient over all channel tiles and writes grad_offset with plain stores.
// (launch bounds: the fully unrolled version took 142 registers = ONE block per SM, 12 % occupancy, and sat in
// long-scoreboard stalls on the corner loads: 1.53 ms for a C5 layer)
template <typename T>
__global__ void __launch_bounds__(256, 4) scatter_kernel(Geo g, const T* __restrict__ xt, const Tap* __restrict__ plan,
                                                      const T* __restrict__ gS, float* __restrict__ gxt,
                                                      float* __restrict__ goff, float scale_iy, float scale_ix) {
  __shared__ float tile[kQT][kCT + 1];
  const int b = blockIdx.y, q0 = blockIdx.x * kQT;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const T* img = xt + (size_t)b * xt_image_stride(g);
  float* gimg = gxt ? gxt + (size_t)b * xt_image_stride(g) : nullptr;
  const int pitch = xt_row_pitch(g);
  Corner cs[4];
  float gix[4], giy[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int q = q0 + warp + 8 * i;
    Tap tp = {0, 0, 0.f, 0.f};
    tp.y0 = tp.x0 = -100;
    if (q < g.P) tp = plan[(size_t)b * g.P + q];
    cs[i] = corner_of(g, tp);
    gix[i] = giy[i] = 0.f;
  }
  for (int c0 = 0; c0 < g.C; c0 += kCT) {
    const int q = q0 + lane;
#pragma unroll
    for (int j = 0; j < kCT / 8; ++j) {
      const int cl = warp + 8 * j, c = c0 + cl;
      tile[lane][cl] = (c < g.C && q < g.P) ? ldf(gS + ((size_t)b * g.C + c) * g.P + q) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (!cs[i].inside) continue;   // warp-uniform: no corner inside the image, nothing flows back
      const T* p = img + cs[i].base;
      const float ex = 1.0f - cs[i].fx, sy = 1.0f - cs[i].fy;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int c = c0 + k * 32 + lane;
        if (c >= g.C) continue;
        const float gs = tile[warp + 8 * i][k * 32 + lane];
        if (gimg) {
          float* gp = gimg + cs[i].base + c;
          atomicAdd(gp, gs * cs[i].w[0]);
          atomicAdd(gp + g.C, gs * cs[i].w[1]);
          atomicAdd(gp + pitch, gs * cs[i].w[2]);
          atomicAdd(gp + pitch + g.C, gs * cs[i].w[3]);
        }
        const float v0 = ldf(p + c), v1 = ldf(p + g.C + c), v2 = ldf(p + pitch + c), v3 = ldf(p + pitch + g.C + c);
        gix[i] += gs * ((v1 - v0) * sy + (v3 - v2) * cs[i].fy);
        giy[i] += gs * ((v2 - v0) * ex + (v3 - v1) * cs[i].fx);
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float a = gix[i], c = giy[i];
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      c += __shfl_xor_sync(0xffffffffu, c, o);
    }
    const int q = q0 + warp + 8 * i;
    if (lane == 0 && q < g.P) {
      const int p = q / g.N, n = q - p * g.N;
      float* ob = goff + (size_t)b * 2 * g.N * g.HW;
      // grad_offset[row-moving channel] = g_iy * scale_iy, [column-moving channel] = g_ix * scale_ix
      // (autograd of the coordinate normalisation; dcn_umma_bwd_data.cu)
      ob[(size_t)off_row_ch(g, n) * g.HW + p] = c * scale_iy;
      ob[(size_t)off_col_ch(g, n) * g.HW + p] = a * scale_ix;
    }
  }
}

// out[b, o, :] = bias[o] (the GEMM then accumulates with beta = 1)
__global__ void __launch_bounds__(256) bias_fill_kernel(int B, int O, int Oimg, int HW, const float* __restrict__ bias,
                                                        float* __restrict__ out) {
  const size_t total = (size_t)B * O * HW;
  for (size_t i = blockIdx.x * 256ull + threadIdx.x; i < total; i += (size_t)gridDim.x * 256) {
    const int p = (int)(i % HW);
    const size_t bo = i / HW;
    const int o = (int)(bo % O), b = (int)(bo / O);
    out[((size_t)b * Oimg + o) * HW + p] = bias ? bias[o] : 0.f;
  }
}

// DCN_FLAG_RELU_OUT: out[b, o, :] = max(out[b, o, :], 0) once the GEMMs have accumulated onto the bias
__global__ void __launch_bounds__(256) relu_kernel(int B, int O, int Oimg, int HW, float* __restrict__ out) {
  const size_t total = (size_t)B * O * HW;
  for (size_t i = blockIdx.x * 256ull + threadIdx.x; i < total; i += (size_t)gridDim.x * 256) {
    const int p = (int)(i % HW);
    const size_t bo = i / HW;
    const int o = (int)(bo % O), b = (int)(bo / O);
    float* v = out + ((size_t)b * Oimg + o) * HW + p;
    *v = fmaxf(*v, 0.f);
  }
}

// goutT[o, b*HW + p] = gout[b, o, p]: rows of HW elements re-ordered (o, b)  (bf16 operands)
__global__ void __launch_bounds__(256) gout_rows_kernel(int B, int O, int Oimg, int HW,
                                                        const __nv_bfloat16* __restrict__ gout,
                                                        __nv_bfloat16* __restrict__ goutT) {
  const int o = blockIdx.x, b = blockIdx.y;
  const __nv_bfloat16* src = gout + ((size_t)b * Oimg + o) * HW;
  __nv_bfloat16* dst = goutT + ((size_t)o * B + b) * HW;
  for (int p = threadIdx.x; p < HW; p += 256) dst[p] = src[p];
}

// fp32 -> (hi, lo) bfloat16 pair, flat (the weight matrix)
__global__ void __launch_bounds__(256) split_flat_kernel(size_t n, const float* __restrict__ src,
                                                         __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  for (size_t i = blockIdx.x * 256ull + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) {
    __nv_bfloat16 h, l;
    ptx::split_bf16(src[i], h, l);
    hi[i] = h;
    lo[i] = l;
  }
}

// grad_out [B, Oimg, HW] fp32 -> hi / lo bfloat16 in BOTH orders the backward GEMMs read: compact [b][o][p] (data
// gradient) and [o][b][p] (weight gradient); one read of grad_out
__global__ void __launch_bounds__(256) gout_split_kernel(int B, int O, int Oimg, int HW, const float* __restrict__ gout,
                                                         __nv_bfloat16* __restrict__ g_hi, __nv_bfloat16* __restrict__ g_lo,
                                                         __nv_bfloat16* __restrict__ gT_hi,
                                                         __nv_bfloat16* __restrict__ gT_lo) {
  const int o = blockIdx.x, b = blockIdx.y;
  const float* src = gout + ((size_t)b * Oimg + o) * HW;
  const size_t d = ((size_t)b * O + o) * HW, dT = ((size_t)o * B + b) * HW;
  for (int p = threadIdx.x; p < HW; p += 256) {
    __nv_bfloat16 h, l;
    ptx::split_bf16(src[p], h, l);
    g_hi[d + p] = h;
    g_lo[d + p] = l;
    gT_hi[dT + p] = h;
    gT_lo[dT + p] = l;
  }
}

}  // namespace gp

// ---------------------------------------------------------------------------- host side
static size_t gp_esz(int operand) { return operand == DCN_OPERAND_BF16 ? 2 : 4; }
static size_t gp_plan_bytes(const Geo& g) { return align_up(sizeof(Tap) * (size_t)g.B * g.P, 1024); }
static size_t gp_S_bytes(const Geo& g, int operand) { return align_up(gp_esz(operand) * (size_t)g.B * g.C * g.P, 1024); }

bool gemm_path_supported(const Geo& g, int operand) {
  if (g.variant != DCN_VARIANT_TORCH || g.plain) return false;
  if (operand != DCN_OPERAND_FP32 && operand != DCN_OPERAND_BF16) return false;
  if (g.C % 4 || (operand == DCN_OPERAND_BF16 && g.C % 8)) return false;     // framed staging copy: 16-byte pixels
  if (g.C < 32 || g.O < 32 || g.K < 256) return false;                        // too small to be worth three GEMMs
  if (gp_S_bytes(g, operand) > (2ull << 30)) return false;                    // the materialised samples stay small
  if ((long long)g.B * g.HW > 0x7fffffffLL || (long long)g.C * g.P > 0x7fffffffLL) return false;
  return true;
}

// fp32 operands on tensor cores: every operand of the three GEMMs as a (hi, lo) bfloat16 pair, every product as
// lo*hi + hi*lo + hi*hi with fp32 accumulation (the split of the tcgen05 kernels; relative error ~5e-6).  The true-fp32
// cuBLAS GEMMs took 2.5 ms each for a C5 layer (47 TFLOP/s) against 0.5 ms for one bf16 GEMM.
static size_t gp_W_bytes(const Geo& g, int operand) {
  return operand == DCN_OPERAND_FP32 ? align_up(4 * (size_t)g.O * g.K, 1024) : 0;
}
static size_t gp_gout_bytes(const Geo& g, int operand) {
  return align_up(gp_esz(operand) * (size_t)g.B * g.O * g.HW, 1024);
}

// forward: [xt][plan][S][W hi|lo][cuBLAS workspace]; backward: [xt][plan][S][gS][gxt][goutT][gout hi|lo][W hi|lo][cuBLAS
// workspace] — S and goutT hold (hi | lo) halves for fp32 operands (same bytes as the fp32 matrix)
size_t gemm_path_workspace(const Geo& g, int operand, int phase) {
  size_t b = umma_xt_bytes(g, operand) + gp_plan_bytes(g) + gp_S_bytes(g, operand) + gp_W_bytes(g, operand) + gp::kCublasWs;
  if (phase == DCN_PHASE_BACKWARD)
    b += gp_S_bytes(g, operand) + umma_xt_bytes(g, DCN_OPERAND_FP32) + gp_gout_bytes(g, operand) +
         (operand == DCN_OPERAND_FP32 ? gp_gout_bytes(g, operand) : 0);
  return b;
}

static int gp_cublas_fail(cublasStatus_t st, const char* what) {
  set_error("cuBLAS error %d at %s", (int)st, what);
  return DCN_ERR_CUDA;
}

// stage x (identity channel order), plan, sample
// staged = DCN_FLAG_XT_STAGED: the head of the workspace ([xt][plan][S], the same prefix in both phases) still holds
// what the forward pass of this very call pair wrote — nothing to redo
static int gp_stage_and_sample(const Geo& g, int operand, const void* x, const float* off, uint8_t* ws, cudaStream_t st,
                               void** xt_out, Tap** plan_out, void** S_out, bool staged = false) {
  void* xt = ws;
  Tap* plan = (Tap*)(ws + umma_xt_bytes(g, operand));
  void* S = (uint8_t*)plan + gp_plan_bytes(g);
  *xt_out = xt;
  *plan_out = plan;
  *S_out = S;
  if (staged) return DCN_OK;
  Tiling t;
  memset(&t, 0, sizeof(t));
  t.variant = DCN_VARIANT_JITTOR;   // identity channel order in the staged copy
  t.G = t.Cs = 1;
  int rc;
  if ((rc = launch_nchw_to_nhwc(g, t, x, xt, operand, st))) return rc;
  if ((rc = launch_plan(g, off, plan, st))) return rc;
  const dim3 grid((unsigned)((g.P + gp::kQT - 1) / gp::kQT), (unsigned)g.B);
  {
    KernelScope scope("gemm_sample_kernel", st);
    if (operand == DCN_OPERAND_BF16)
      gp::sample_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(g, (const __nv_bfloat16*)xt, plan, (__nv_bfloat16*)S, nullptr);
    else
      gp::sample_kernel<float><<<grid, 256, 0, st>>>(g, (const float*)xt, plan, (__nv_bfloat16*)S,
                                                     (__nv_bfloat16*)S + (size_t)g.B * g.C * g.P);
    DCN_KERNEL_CHECK("gemm_sample_kernel");
  }
  return DCN_OK;
}

int gemm_path_forward(const Geo& g, int operand, const void* x, const float* off, const void* wt, const float* bias,
                      float* out, void* workspace, cudaStream_t st) {
  if (!gp::load_cublas()) return DCN_ERR_UNSUPPORTED;
  cublasHandle_t h = gp::handle_for_current_device();
  if (!h) return gp_cublas_fail(CUBLAS_STATUS_NOT_INITIALIZED, "cublasCreate");
  uint8_t* ws = (uint8_t*)workspace;
  void *xt, *S;
  Tap* plan;
  int rc;
  if ((rc = gp_stage_and_sample(g, operand, x, off, ws, st, &xt, &plan, &S))) return rc;
  uint8_t* whl = (uint8_t*)S + gp_S_bytes(g, operand);
  uint8_t* cws = whl + gp_W_bytes(g, operand);
  const bool split = operand == DCN_OPERAND_FP32;
  {
    KernelScope scope("gemm_bias_fill_kernel", st);
    gp::bias_fill_kernel<<<1024, 256, 0, st>>>(g.B, g.O, g.Oimg, g.HW, bias, out);
    DCN_KERNEL_CHECK("gemm_bias_fill_kernel");
  }
  const size_t nS = (size_t)g.B * g.C * g.P, nW = (size_t)g.O * g.K;
  __nv_bfloat16 *w_hi = (__nv_bfloat16*)whl, *w_lo = w_hi + nW;
  if (split) {
    KernelScope scope("gemm_split_kernel", st);
    gp::split_flat_kernel<<<256, 256, 0, st>>>(nW, (const float*)wt, w_hi, w_lo);
    DCN_KERNEL_CHECK("gemm_split_kernel");
  }
  const float one = 1.f;
  cublasStatus_t cs;
  std::lock_guard<std::mutex> use(gp::g_use_mu);   // a cuBLAS handle must not be driven by two host threads at once
  if ((cs = gp::g_api.SetStream(h, st)) != CUBLAS_STATUS_SUCCESS) return gp_cublas_fail(cs, "cublasSetStream");
  if (gp::g_api.SetWorkspace) gp::g_api.SetWorkspace(h, cws, gp::kCublasWs);
  {
    // row-major out_b[O, HW] += Wm[O, K] * A_b^T  <=>  column-major C'[HW, O] = op_T(A'[K, HW]) * B'[K, O]
    KernelScope scope("cublas_gemm_fwd", st);
    auto gemm = [&](const void* Sm, const void* Wm) {
      count_launch();
      return gp::g_api.GemmStridedBatchedEx(h, CUBLAS_OP_T, CUBLAS_OP_N, g.HW, g.O, g.K, &one, Sm, CUDA_R_16BF, g.K,
                                            (long long)g.C * g.P, Wm, CUDA_R_16BF, g.K, 0, &one, out, CUDA_R_32F, g.HW,
                                            (long long)g.Oimg * g.HW, g.B, CUBLAS_COMPUTE_32F, CUBLAS_GEMM_DEFAULT);
    };
    if (split) {
      const __nv_bfloat16 *s_hi = (const __nv_bfloat16*)S, *s_lo = s_hi + nS;
      if ((cs = gemm(s_lo, w_hi)) == CUBLAS_STATUS_SUCCESS && (cs = gemm(s_hi, w_lo)) == CUBLAS_STATUS_SUCCESS)
        cs = gemm(s_hi, w_hi);
    } else {
      cs = gemm(S, wt);
    }
  }
  if (cs != CUBLAS_STATUS_SUCCESS) return gp_cublas_fail(cs, "cublasGemmStridedBatchedEx(forward)");
  if (g.relu_out) {
    KernelScope scope("gemm_relu_kernel", st);
    gp::relu_kernel<<<1024, 256, 0, st>>>(g.B, g.O, g.Oimg, g.HW, out);
    DCN_KERNEL_CHECK("gemm_relu_kernel");
  }
  return DCN_OK;
}

int gemm_path_backward(const Geo& g, int operand, int flags, const void* x, const float* off, const void* wt,
                       const void* gout, float* gx, float* goff, float* gw, float* gb, void* workspace, cudaStream_t st) {
  if (!gp::load_cublas()) return DCN_ERR_UNSUPPORTED;
  cublasHandle_t h = gp::handle_for_current_device();
  if (!h) return gp_cublas_fail(CUBLAS_STATUS_NOT_INITIALIZED, "cublasCreate");
  uint8_t* ws = (uint8_t*)workspace;
  void *xt, *S;
  Tap* plan;
  int rc;
  if ((rc = gp_stage_and_sample(g, operand, x, off, ws, st, &xt, &plan, &S, (flags & DCN_FLAG_XT_STAGED) != 0))) return rc;
  uint8_t* gS = (uint8_t*)S + gp_S_bytes(g, operand);
  float* gxt = (float*)(gS + gp_S_bytes(g, operand));
  uint8_t* goutT = (uint8_t*)gxt + umma_xt_bytes(g, DCN_OPERAND_FP32);
  const bool split = operand == DCN_OPERAND_FP32;
  uint8_t* ghl = goutT + gp_gout_bytes(g, operand);                       // split mode: compact grad_out, hi | lo
  uint8_t* whl = ghl + (split ? gp_gout_bytes(g, operand) : 0);
  uint8_t* cws = whl + gp_W_bytes(g, operand);
  const bool want_gx = !(flags & DCN_FLAG_NO_GRAD_X) && gx != nullptr;
  const cudaDataType dt_gs = operand == DCN_OPERAND_BF16 ? CUDA_R_16BF : CUDA_R_32F;   // gS feeds the scatter kernel
  const float one = 1.f, zero = 0.f;
  const size_t nS = (size_t)g.B * g.C * g.P, nW = (size_t)g.O * g.K, nG = (size_t)g.B * g.O * g.HW;
  __nv_bfloat16 *w_hi = (__nv_bfloat16*)whl, *w_lo = w_hi + nW;
  __nv_bfloat16 *g_hi = (__nv_bfloat16*)ghl, *g_lo = g_hi + nG;
  __nv_bfloat16 *gT_hi = (__nv_bfloat16*)goutT, *gT_lo = gT_hi + nG;
  const __nv_bfloat16 *s_hi = (const __nv_bfloat16*)S, *s_lo = s_hi + nS;
  if (split) {
    KernelScope scope("gemm_split_kernel", st);
    gp::split_flat_kernel<<<256, 256, 0, st>>>(nW, (const float*)wt, w_hi, w_lo);
    gp::gout_split_kernel<<<dim3((unsigned)g.O, (unsigned)g.B), 256, 0, st>>>(g.B, g.O, g.Oimg, g.HW, (const float*)gout,
                                                                               g_hi, g_lo, gT_hi, gT_lo);
    count_launch();
    DCN_KERNEL_CHECK("gemm_split_kernel");
  }
  cublasStatus_t cs;
  std::lock_guard<std::mutex> use(gp::g_use_mu);   // see gemm_path_forward
  if ((cs = gp::g_api.SetStream(h, st)) != CUBLAS_STATUS_SUCCESS) return gp_cublas_fail(cs, "cublasSetStream");
  if (gp::g_api.SetWorkspace) gp::g_api.SetWorkspace(h, cws, gp::kCublasWs);
  // row-major gS_b[HW, K] = gout_b^T[HW, O] * Wm[O, K]  <=>  column-major C'[K, HW] = B'[K, O] * op_T(gout'[HW, O])
  {
    KernelScope scope("cublas_gemm_bwd_data", st);
    auto gemm = [&](const void* Wm, const void* Gm, long long gstride, const float* beta) {
      count_launch();
      return gp::g_api.GemmStridedBatchedEx(h, CUBLAS_OP_N, CUBLAS_OP_T, g.K, g.HW, g.O, &one, Wm, CUDA_R_16BF, g.K, 0, Gm,
                                            CUDA_R_16BF, g.HW, gstride, beta, gS, dt_gs, g.K, (long long)g.C * g.P, g.B,
                                            CUBLAS_COMPUTE_32F, CUBLAS_GEMM_DEFAULT);
    };
    if (split) {
      const long long gs = (long long)g.O * g.HW;
      if ((cs = gemm(w_lo, g_hi, gs, &zero)) == CUBLAS_STATUS_SUCCESS &&
          (cs = gemm(w_hi, g_lo, gs, &one)) == CUBLAS_STATUS_SUCCESS)
        cs = gemm(w_hi, g_hi, gs, &one);
    } else {
      cs = gemm(wt, gout, (long long)g.Oimg * g.HW, &zero);
    }
    if (cs != CUBLAS_STATUS_SUCCESS) return gp_cublas_fail(cs, "cublasGemmStridedBatchedEx(data gradient)");
  }
  if (want_gx) DCN_CUDA_TRY(cudaMemsetAsync(gxt, 0, sizeof(float) * (size_t)g.B * xt_image_stride(g), st));
  {
    const dim3 grid((unsigned)((g.P + gp::kQT - 1) / gp::kQT), (unsigned)g.B);
    const float scale_iy = g.sy * 2.0f / g.Dx, scale_ix = g.sx * 2.0f / g.Dy;
    KernelScope scope("gemm_scatter_kernel", st);
    if (operand == DCN_OPERAND_BF16)
      gp::scatter_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(g, (const __nv_bfloat16*)xt, plan, (const __nv_bfloat16*)gS,
                                                              want_gx ? gxt : nullptr, goff, scale_iy, scale_ix);
    else
      gp::scatter_kernel<float><<<grid, 256, 0, st>>>(g, (const float*)xt, plan, (const float*)gS, want_gx ? gxt : nullptr,
                                                      goff, scale_iy, scale_ix);
    DCN_KERNEL_CHECK("gemm_scatter_kernel");
  }
  if (want_gx) {
    Tiling t;
    memset(&t, 0, sizeof(t));
    t.variant = DCN_VARIANT_JITTOR;
    t.G = t.Cs = 1;
    if ((rc = launch_nhwc_to_nchw_add(g, t, gxt, gx, (flags & DCN_FLAG_ACCUM_GRAD_X) ? 1 : 0, st))) return rc;
  }
  // weight gradient: row-major gW[O, K] = goutT[O, B*HW] * A[B*HW, K]  <=>  column-major C'[K, O] = A'[K, BHW] * G'[BHW, O]
  if (!split) {
    KernelScope scope("gemm_gout_rows_kernel", st);
    gp::gout_rows_kernel<<<dim3((unsigned)g.O, (unsigned)g.B), 256, 0, st>>>(g.B, g.O, g.Oimg, g.HW,
                                                                             (const __nv_bfloat16*)gout,
                                                                             (__nv_bfloat16*)goutT);
    DCN_KERNEL_CHECK("gemm_gout_rows_kernel");
  }
  {
    KernelScope scope("cublas_gemm_bwd_weight", st);
    const int bhw = g.B * g.HW;
    auto gemm = [&](const void* Sm, const void* Gm, const float* beta) {
      count_launch();
      return gp::g_api.GemmEx(h, CUBLAS_OP_N, CUBLAS_OP_N, g.K, g.O, bhw, &one, Sm, CUDA_R_16BF, g.K, Gm, CUDA_R_16BF, bhw,
                              beta, gw, CUDA_R_32F, g.K, CUBLAS_COMPUTE_32F, CUBLAS_GEMM_DEFAULT);
    };
    if (split) {
      if ((cs = gemm(s_lo, gT_hi, &zero)) == CUBLAS_STATUS_SUCCESS && (cs = gemm(s_hi, gT_lo, &one)) == CUBLAS_STATUS_SUCCESS)
        cs = gemm(s_hi, gT_hi, &one);
    } else {
      cs = gemm(S, goutT, &zero);
    }
    if (cs != CUBLAS_STATUS_SUCCESS) return gp_cublas_fail(cs, "cublasGemmEx(weight gradient)");
  }
  if (gb && (rc = launch_bias_grad(g, gout, operand, gb, st))) return rc;
  return DCN_OK;
}

}  // namespace dcn
