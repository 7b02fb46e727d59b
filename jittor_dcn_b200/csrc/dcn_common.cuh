// dcn_common.cuh — shared geometry, the bit-exact coordinate chain and launch bookkeeping.
//
// Reference semantics implemented here (SURVEY.md Appendix A):
//   coordinates  deform_conv.py:62-68,34-39 / train.py:102-113
//   un-normalise + corners  grid_sample(bilinear, zeros, align_corners=True),
//                deform_conv.py:47-52 / train.py:121-127
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/dcn_b200.h"

// Debug build (python -m jittor_dcn_b200.build --debug -> libdcn_b200_dbg.so, selected with DCN_B200_LIB=dbg):
// compute-sanitizer is closed on the GPU pool, so the kernels carry their own checks — bounds on every global address
// the gather / scatter / epilogue code forms from plan entries, and at kernel exit the agreement of the step counts of
// all roles that hand stages to each other through mbarriers (a role that ran one step more or less than its partner
// would not necessarily hang).  A failed check prints its location and traps; the release build compiles them away.
#ifdef DCN_DEBUG_CHECKS
#include <cstdio>
#define DCN_DEV_ASSERT(cond)                                                                                  \
  do {                                                                                                        \
    if (!(cond)) {                                                                                            \
      printf("DCN_DEV_ASSERT failed: %s  at %s:%d  block %d thread %d\n", #cond, __FILE__, __LINE__, (int)blockIdx.x, \
             (int)threadIdx.x);                                                                               \
      __trap();                                                                                               \
    }                                                                                                         \
  } while (0)
#define DCN_DBG_ONLY(...) __VA_ARGS__
#else
#define DCN_DEV_ASSERT(cond) do { } while (0)
#define DCN_DBG_ONLY(...)
#endif

namespace dcn {

// Device-side problem geometry (passed by value to every kernel).
struct Geo {
  int B, C, O, H, W;
  int Oimg;     // channels per image of out / grad_out IN MEMORY (== O unless this Geo describes a
                // group of O output channels of a wider layer: dcn_umma_host.cu splits O > 256)
  int N;        // taps = kh*kw
  int Ho, Wo;   // output extent
  int HW;       // Ho*Wo   rows of the GEMM per batch element
  int K;        // C*N     contraction length
  int P;        // HW*N    samples per (b, c) plane
  int variant;  // DCN_VARIANT_*
  float Dx, Dy; // normalisation divisors            (:37-38 / :111-112)
  float sx, sy; // (W-1)/2, (H-1)/2                  (GridSampler.h:27-36)
  // DCNv1 coordinate mode needs the conv geometry itself
  int kw, sh, sw, ph, pw;
  // Offset channel that moves the ROW (iy) / COLUMN (ix) coordinate of tap n: n*mul + add.
  //   reference: row <- channel n ("x" offset: the sample is transposed), column <- channel N + n
  //   DCNv1    : row <- channel 2n (dy),                                   column <- channel 2n + 1 (dx)
  int row_mul, row_add, col_mul, col_add;
  // PLAIN problems (the companion offset convolution, deform_conv.py:16-21,58 / train.py:80-85,98, on the tensor
  // kernels): a regular convolution = DCNv1 coordinates with all offsets zero, i.e. ONE exact pixel per (pixel, tap)
  // instead of four weighted corners; no offset tensor is read.  plain_geo() builds such a Geo; o_valid = 2N real
  // output channels inside the padded O the forward accumulators need.
  int plain, o_valid;
  // channel permutation of the staged copy the plain problem shares with its Torch-layout DCN layer (0 = none):
  // staged channel c' holds image channel (c' % perm_G) * perm_Cs + c' / perm_G  (dcn_umma_prep.cu)
  int perm_G, perm_Cs;
  // DCN_FLAG_RELU_OUT: the forward epilogues store max(acc + bias, 0) (SURVEY 8f.2: with eval-mode BatchNorm folded
  // into weight / bias by the caller this is the whole relu(bn(conv(x))) post-op of train.py:167-170 in the epilogue)
  int relu_out;
  // Chained inference (dcn_layer_forward_chained, SURVEY 8f.2): the forward epilogue writes `out` directly as the
  // framed channels-last staging copy of the CONSUMER layer — [B][(Ho + 3) x (Wo + 2)][O], pixel (h, w) at frame
  // position (h + 1, w + 1), channel o at out_G ? (o % out_Cs) * out_G + o / out_Cs : o (the consumer's Torch-layout
  // permutation) — so that the consumer runs with DCN_FLAG_XT_STAGED and no activation crosses a layer boundary in NCHW
  int out_framed, out_G, out_Cs;
};

__host__ __device__ __forceinline__ int off_row_ch(const Geo& g, int n) { return n * g.row_mul + g.row_add; }
__host__ __device__ __forceinline__ int off_col_ch(const Geo& g, int n) { return n * g.col_mul + g.col_add; }

// Flat index into weight[O, C, kh, kw] of GEMM column j of output o.  The tile kernels order the
// columns of every non-Torch layout (tap, channel): j = n*C + c.
//   Jittor layout (deform_conv.py:72-74): column n*C + c multiplies flat weight element j itself;
//   DCNv1: column (c, n) of the (c, tap)-ordered weight, i.e. element c*N + n.
__host__ __device__ __forceinline__ size_t wt_index(const Geo& g, int o, int j) {
  if (g.variant == DCN_VARIANT_DCNV1) {
    const int n = j / g.C;
    int c = j - n * g.C;
    if (g.perm_G) c = (c % g.perm_G) * g.perm_Cs + c / g.perm_G;
    return (size_t)o * g.K + (size_t)c * g.N + n;
  }
  return (size_t)o * g.K + j;
}

// One sampling point: north-west corner + fractions.  16 bytes, the "plan" entry.
struct __align__(16) Tap {
  int y0, x0;
  float fx, fy;
};

__host__ inline int make_geo(const DcnShape* s, Geo* g) {
  if (!s) return DCN_ERR_NULL_POINTER;
  if (s->B <= 0 || s->C <= 0 || s->O <= 0 || s->H <= 0 || s->W <= 0 || s->kh <= 0 || s->kw <= 0 ||
      s->sh <= 0 || s->sw <= 0 || s->ph < 0 || s->pw < 0)
    return DCN_ERR_BAD_SHAPE;
  if (s->H + 2 * s->ph < s->kh || s->W + 2 * s->pw < s->kw) return DCN_ERR_BAD_SHAPE;
  if (s->variant != DCN_VARIANT_JITTOR && s->variant != DCN_VARIANT_TORCH && s->variant != DCN_VARIANT_DCNV1)
    return DCN_ERR_BAD_SHAPE;
  g->B = s->B; g->C = s->C; g->O = s->O; g->H = s->H; g->W = s->W;
  g->Oimg = s->O;
  g->plain = 0;
  g->o_valid = s->O;
  g->perm_G = g->perm_Cs = 0;
  g->relu_out = (s->flags & DCN_FLAG_RELU_OUT) ? 1 : 0;
  g->out_framed = g->out_G = g->out_Cs = 0;
  g->N = s->kh * s->kw;
  g->Ho = (s->H + 2 * s->ph - s->kh) / s->sh + 1;
  g->Wo = (s->W + 2 * s->pw - s->kw) / s->sw + 1;
  g->HW = g->Ho * g->Wo;
  g->variant = s->variant;
  // index spaces that the kernels keep in 32-bit registers
  const long long lim = 0x7fffffffLL;
  if ((long long)g->C * g->N > lim || (long long)g->HW * g->C * g->N > lim ||
      (long long)g->C * g->H * g->W > lim || (long long)g->O * g->C * g->N > lim ||
      (long long)g->B * g->HW * g->N > lim || (long long)g->O * g->HW > lim)
    return DCN_ERR_BAD_SHAPE;
  g->K = g->C * g->N;
  g->P = g->HW * g->N;
  if (s->variant == DCN_VARIANT_TORCH) {
    g->Dx = (float)(s->W - 1);
    g->Dy = (float)(s->H - 1);
  } else {
    g->Dx = (float)(g->Wo - 1);
    g->Dy = (float)(g->Ho - 1);
  }
  g->sx = (float)(s->W - 1) / 2.0f;
  g->sy = (float)(s->H - 1) / 2.0f;
  g->kw = s->kw; g->sh = s->sh; g->sw = s->sw; g->ph = s->ph; g->pw = s->pw;
  if (s->variant == DCN_VARIANT_DCNV1) {
    g->row_mul = 2; g->row_add = 0; g->col_mul = 2; g->col_add = 1;
  } else {
    g->row_mul = 1; g->row_add = 0; g->col_mul = 1; g->col_add = g->N;
  }
  return DCN_OK;
}

// float -> int that is total: NaN and anything below -2^30 saturate low.
__device__ __forceinline__ int sat_int(float v) {
  if (!(v > -1073741824.0f)) return -1073741824;
  if (v > 1073741824.0f) return 1073741824;
  return (int)v;
}

// The reference's float32 op chain, one IEEE rounding per op, no FMA contraction
// (the _rn intrinsics are never fused by nvcc).  Bit-exact with the CPU reference:
// torch CPU evaluates `tensor / python_int` as a true IEEE divide (SURVEY.md A.3).
// off_x = the offset that ends up moving the ROW (channel off_row_ch(n)), off_y the COLUMN one.
__device__ __forceinline__ Tap tap_of(const Geo& g, int h, int w, int n, float off_x, float off_y) {
  if (g.variant == DCN_VARIANT_DCNV1) {
    // torchvision deform_conv2d: y = (h*sh - ph + ki) + dy ; x = (w*sw - pw + kj) + dx, no round trip
    const int ki = n / g.kw, kj = n - ki * g.kw;
    const float iy = __fadd_rn((float)(h * g.sh - g.ph + ki), off_x);
    const float ix = __fadd_rn((float)(w * g.sw - g.pw + kj), off_y);
    const float xf = floorf(ix), yf = floorf(iy);
    Tap t;
    t.fx = __fsub_rn(ix, xf);
    t.fy = __fsub_rn(iy, yf);
    t.x0 = sat_int(xf);
    t.y0 = sat_int(yf);
    return t;
  }
  float loc_x = __fadd_rn((float)w, off_x);
  float loc_y = __fadd_rn((float)h, off_y);
  float nx = __fsub_rn(__fmul_rn(__fdiv_rn(loc_x, g.Dx), 2.0f), 1.0f);
  float ny = __fsub_rn(__fmul_rn(__fdiv_rn(loc_y, g.Dy), 2.0f), 1.0f);
  // grid = [norm_y, norm_x]; grid_sample takes slot 0 as the WIDTH coordinate.
  float ix = __fmul_rn(__fadd_rn(ny, 1.0f), g.sx);
  float iy = __fmul_rn(__fadd_rn(nx, 1.0f), g.sy);
  float xf = floorf(ix), yf = floorf(iy);
  Tap t;
  t.fx = __fsub_rn(ix, xf);
  t.fy = __fsub_rn(iy, yf);
  t.x0 = sat_int(xf);
  t.y0 = sat_int(yf);
  return t;
}

// Corner weights nw, ne, sw, se exactly as the reference forms them
// (s = 1-fy, e = 1-fx; nw = s*e, ne = s*fx, sw = fy*e, se = fy*fx).
__device__ __forceinline__ void corner_weights(const Tap& t, float w[4]) {
  float e = __fsub_rn(1.0f, t.fx), s = __fsub_rn(1.0f, t.fy);
  w[0] = __fmul_rn(s, e);
  w[1] = __fmul_rn(s, t.fx);
  w[2] = __fmul_rn(t.fy, e);
  w[3] = __fmul_rn(t.fy, t.fx);
}

// Validity of the four corners (zero padding): bit k set <=> corner k inside the image.
__device__ __forceinline__ unsigned corner_mask(const Tap& t, int H, int W) {
  bool y0 = (unsigned)t.y0 < (unsigned)H, y1 = (unsigned)(t.y0 + 1) < (unsigned)H;
  bool x0 = (unsigned)t.x0 < (unsigned)W, x1 = (unsigned)(t.x0 + 1) < (unsigned)W;
  return (y0 && x0 ? 1u : 0u) | (y0 && x1 ? 2u : 0u) | (y1 && x0 ? 4u : 0u) | (y1 && x1 ? 8u : 0u);
}

// (GEMM row r within a batch element, GEMM column j) -> (channel c, sample q = p*N + n)
//   Jittor  A[(h,w), n*C + c]                      deform_conv.py:72-73
//   Torch   A[r, j] = S_b.flat[r*K + j], (c,h,w,n) train.py:129-131
template <int VARIANT>
__device__ __forceinline__ void col_map(const Geo& g, int r, int j, int& c, int& q) {
  if (VARIANT == DCN_VARIANT_TORCH) {
    int f = r * g.K + j;  // < HW*K, checked < 2^31 in make_geo
    c = f / g.P;
    q = f - c * g.P;
  } else {
    int n = j / g.C;
    c = j - n * g.C;
    q = r * g.N + n;
  }
}

// ---- host-side bookkeeping ---------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
void count_launch(int n = 1);

#define DCN_CUDA_TRY(expr)                                        \
  do {                                                            \
    cudaError_t _e = (expr);                                      \
    if (_e != cudaSuccess) return ::dcn::cuda_fail(_e, #expr);    \
  } while (0)

#define DCN_KERNEL_CHECK(name)                                    \
  do {                                                            \
    ::dcn::count_launch();                                        \
    cudaError_t _e = cudaGetLastError();                          \
    if (_e != cudaSuccess) return ::dcn::cuda_fail(_e, name);     \
  } while (0)

// Optional per-kernel timing (dcn_profile_begin/end): CUDA events recorded on the launching
// stream right before and after a kernel.  Zero cost when profiling is off.
void profile_mark(const char* name, cudaStream_t st, bool begin);
struct KernelScope {
  const char* name;
  cudaStream_t st;
  KernelScope(const char* n, cudaStream_t s) : name(n), st(s) { profile_mark(name, st, true); }
  ~KernelScope() { profile_mark(name, st, false); }
};

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---- kernel families (each returns a DcnStatus) --------------------------------------
// plan: Tap per (b, q); stored in q-order [b][p][n] (Torch) or tap-major [b][n][p] (Jittor)
int launch_plan(const Geo& g, const float* off, Tap* plan, cudaStream_t st);
int launch_corners(const Geo& g, const float* off, int32_t* y0, int32_t* x0, float* w4, cudaStream_t st);
// mask / gmask [B, N, Ho, Wo] (DCNv1 only; nullptr = unmodulated): modulated sampling and its gradient
int simt_forward(const Geo& g, const float* x, const Tap* plan, const float* wt, const float* bias,
                 float* out, cudaStream_t st, const float* mask = nullptr);
int launch_offset_scale(const Geo& g, float* goff, cudaStream_t st);
int launch_bias_grad(const Geo& g, const void* gout, int operand, float* gb, cudaStream_t st);
int launch_widen_bf16(const void* src, float* dst, size_t n, cudaStream_t st);
enum { SIMT_BWD_DATA = 1, SIMT_BWD_WEIGHT = 2, SIMT_BWD_BIAS = 4, SIMT_BWD_ALL = 7 };
int simt_backward(const Geo& g, int flags, const float* x, const Tap* plan, const float* wt,
                  const float* gout, float* gx, float* goff, float* gw, float* gb, cudaStream_t st,
                  int parts = SIMT_BWD_ALL, const float* mask = nullptr, float* gmask = nullptr);

}  // namespace dcn
