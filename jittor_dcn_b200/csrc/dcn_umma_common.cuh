// dcn_umma_common.cuh — pieces shared by the tcgen05 forward / backward kernels:
// fast integer division, the tile decomposition of both column layouts, the channels-last
// staging of x and the pre-tiled bf16 hi/lo weight images.
#pragma once
#include "dcn_common.cuh"
#include "dcn_umma.cuh"

namespace dcn {

// dynamic shared memory one block may opt in to on sm_100
constexpr size_t kSmemBudget = 227 * 1024;

// SMs of the current device (148 on a B200) for the grids of the persistent kernels
__host__ inline int num_sms() {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return sms;
}

// n / d for 0 <= n < 2^31 by multiply-high (d >= 1), exact.
struct FastDiv {
  uint32_t d, mul, shr;
  __host__ static FastDiv make(uint32_t d) {
    FastDiv f;
    f.d = d;
    if (d == 1) {
      f.mul = 0;
      f.shr = 0;
      return f;
    }
    uint32_t l = 0;
    while ((1ull << l) < d) ++l;  // ceil(log2 d)
    f.shr = l - 1;
    f.mul = (uint32_t)(((1ull << (32 + l - 1)) + d - 1) / d);  // ceil(2^(32+l-1) / d), fits for n < 2^31
    return f;
  }
  __device__ __forceinline__ uint32_t div(uint32_t n) const {
    return d == 1 ? n : (__umulhi(n, mul) >> shr);
  }
  __device__ __forceinline__ void divmod(uint32_t n, uint32_t& q, uint32_t& r) const {
    q = div(n);
    r = n - q * d;
  }
};

// How the GEMM rows of one variant are grouped into 128-row UMMA tiles.
//
// Jittor (deform_conv.py:72-73): row = pixel.  Tile = 128 consecutive pixels of one image;
//   K-block kb covers columns j in [64kb, 64kb+64) = taps n in [n0, n0+T), channels within.
//
// Torch (train.py:129-131): row r, column j <-> flat sample index f = r*K + j of the
//   (c,h,w,n)-ordered sample tensor.  With G = gcd(HW, C), R = HW/G, Cs = C/G the rows
//   {r0 + i*R : i < G} ("class" r0) share their sampling points q(r0, j) = (r0*K + j) mod P and
//   differ only in the channel c = cbase(r0, j) + i*Cs.  A tile takes Gt channels of Rt
//   consecutive classes so that every bilinear footprint is fetched once per Gt channels:
//   row m of the tile = quad*(4*Rt) + inst*4 + chq  <->  class instance `inst`, i = 4*quad + chq.
//   The staging copy of x is channel-permuted (c -> (c % Cs)*G + c / Cs) so that those Gt
//   channels are contiguous.
struct Tiling {
  int variant;
  int KB;          // K blocks of 64
  int num_tiles;
  // torch
  int G, R, Cs, Gt, Rt, chunks, num_inst;
  FastDiv divR, divChunks, divP, divN, divWo, divC;
  // jittor
  int pix_blocks, taps_per_kb;
};

__host__ inline int gcd_int(int a, int b) {
  while (b) {
    int t = a % b;
    a = b;
    b = t;
  }
  return a;
}

__host__ inline bool make_tiling(const Geo& g, Tiling* t) {
  t->variant = g.variant;
  t->KB = (g.K + 63) / 64;
  t->divP = FastDiv::make(g.P);
  t->divN = FastDiv::make(g.N);
  t->divWo = FastDiv::make(g.Wo);
  t->divC = FastDiv::make(g.C);
  t->G = t->R = t->Cs = t->Gt = t->Rt = t->chunks = t->num_inst = 1;
  t->divR = FastDiv::make(1);
  t->divChunks = FastDiv::make(1);
  t->pix_blocks = t->taps_per_kb = 1;
  if (g.C % 4) return false;
  if (g.variant == DCN_VARIANT_TORCH) {
    t->G = gcd_int(g.HW, g.C);
    if (t->G % 16) return false;
    t->R = g.HW / t->G;
    t->Cs = g.C / t->G;
    t->Gt = (t->G % 64 == 0) ? 64 : ((t->G % 32 == 0) ? 32 : 16);
    t->Rt = 128 / t->Gt;
    t->chunks = t->G / t->Gt;
    long long inst = (long long)g.B * t->chunks * t->R;
    if (inst > 0x7fffffffLL) return false;
    t->num_inst = (int)inst;
    t->num_tiles = (int)((inst + t->Rt - 1) / t->Rt);
    t->divR = FastDiv::make(t->R);
    t->divChunks = FastDiv::make(t->chunks);
  } else {
    if (!(g.C % 64 == 0 || g.C == 32 || g.C == 16)) return false;
    t->pix_blocks = (g.HW + 127) / 128;
    t->taps_per_kb = g.C >= 64 ? 1 : 64 / g.C;
    t->num_tiles = g.B * t->pix_blocks;
  }
  return true;
}

struct TileRowInfo {  // what a Torch-layout tile row needs
  int b, r0, chunk, valid;
};

// T: Tiling, or a kernel parameter block that carries its num_inst, divR and divChunks
template <class T>
__device__ __forceinline__ TileRowInfo decode_inst(const T& t, int inst) {
  TileRowInfo ri;
  ri.valid = inst < t.num_inst;
  uint32_t bc, r0, b, ch;
  t.divR.divmod((uint32_t)(ri.valid ? inst : 0), bc, r0);
  t.divChunks.divmod(bc, b, ch);
  ri.b = (int)b;
  ri.r0 = (int)r0;
  ri.chunk = (int)ch;
  return ri;
}

// channel permutation of the channels-last staging copy
__host__ __device__ inline int perm_channel(int c, int variant, int G, int Cs) {
  return variant == DCN_VARIANT_TORCH ? (c % Cs) * G + c / Cs : c;
}

// Channels-last staging copy with an all-zero frame: [B][(H + 3) x (W + 2)][C].  Image pixel (y, x)
// lives at frame position (y + 1, x + 1); frame rows 0, H + 1, H + 2 and frame columns 0, W + 1
// are zero.  Every sample with at least one corner inside the image has its top-left corner
// (y0, x0) in [-1, H-1] x [-1, W-1], so its four corners are base + {0, C, pitch, pitch + C} with
// NO validity test: zero padding is reading the frame, and gradient scattered into the frame is
// discarded.  The 2 x 2 block at frame position (H + 1, 0) is frame only: it stands in for samples
// with no corner inside the image (and for padding rows / columns of a tile), so a foreign,
// possibly non-finite value is never multiplied by a zero weight.
__host__ __device__ inline int xt_row_pitch(const Geo& g) { return (g.W + 2) * g.C; }  // elements
__host__ __device__ inline size_t xt_image_stride(const Geo& g) { return (size_t)(g.H + 3) * (g.W + 2) * g.C; }
__host__ __device__ inline int xt_null_base(const Geo& g) { return (g.H + 1) * (g.W + 2) * g.C; }
// element offset (channel 0) of the top-left corner of a sample; inside = some corner is in the image
__device__ __forceinline__ int xt_corner_base(const Geo& g, int y0, int x0, bool& inside) {
  inside = (unsigned)(y0 + 1) <= (unsigned)g.H && (unsigned)(x0 + 1) <= (unsigned)g.W;
  return inside ? ((y0 + 1) * (g.W + 2) + (x0 + 1)) * g.C : xt_null_base(g);
}

// PLAIN problems (regular convolution, Geo::plain — the companion offset conv): tap (ki, kj) of output pixel (h, w)
// reads image pixel (h*sh - ph + ki, w*sw - pw + kj) = frame position (+1, +1).  Anything inside the framed copy is
// either the pixel or the zero border (= zero padding; gradient that lands there is discarded); positions outside
// the frame (padding > 1) use the frame-only block with weight 0.
__device__ __forceinline__ int plain_base(const Geo& g, int h, int w, int n, bool& inside) {
  const int ki = n / g.kw, kj = n - ki * g.kw;
  const int fy = h * g.sh - g.ph + ki + 1, fx = w * g.sw - g.pw + kj + 1;
  inside = (unsigned)fy <= (unsigned)(g.H + 2) && (unsigned)fx <= (unsigned)(g.W + 1);
  return inside ? (fy * (g.W + 2) + fx) * g.C : xt_null_base(g);
}

// The plain Geo of a DCN layer's companion offset convolution (deform_conv.py:16-21 / train.py:80-85): same input,
// kernel, stride and padding, 2N output channels, columns ordered (tap, staged channel) like the DCNv1 layout, weight
// element (o, c, ki, kj) with c un-permuted when the staged copy follows the Torch layout's channel permutation.
// pad_o: round O up to 16 accumulator columns (forward kernel); the real count stays in o_valid / Oimg.
// n_out: output channels, 0 = 2N (the modulated layer's offset-and-mask conv has 3N)
__host__ inline Geo plain_geo(const Geo& g, const Tiling& layer_tiling, bool pad_o, int n_out = 0) {
  const int O = n_out ? n_out : 2 * g.N;
  Geo p = g;
  p.variant = DCN_VARIANT_DCNV1;
  p.plain = 1;
  p.relu_out = 0;
  p.out_framed = p.out_G = p.out_Cs = 0;
  p.o_valid = O;
  p.Oimg = O;
  p.O = pad_o ? (O + 15) / 16 * 16 : O;
  p.perm_G = p.perm_Cs = 0;
  if (g.variant == DCN_VARIANT_TORCH) {
    p.perm_G = layer_tiling.G;
    p.perm_Cs = layer_tiling.Cs;
  }
  p.row_mul = 2; p.row_add = 0; p.col_mul = 2; p.col_add = 1;
  return p;
}

// Plan entry as the forward gather warps consume it (32 bytes in shared memory): the four
// corners' element offsets inside image b of the framed copy and their weights.
struct __align__(16) PlanEntry {
  int off[4];   // nw, ne, sw, se
  float w[4];
};

// x / xt: float (DCN_OPERAND_FP32) or bfloat16 (DCN_OPERAND_BF16)
// (the frame is re-zeroed on every call: the workspace belongs to the caller)
int launch_nchw_to_nhwc(const Geo& g, const Tiling& t, const void* x, void* xt, int operand, cudaStream_t st);
int launch_xt_frame_zero(const Geo& g, float* xt, cudaStream_t st);
int launch_nhwc_to_nchw_add(const Geo& g, const Tiling& t, const float* gxt, float* gx, int accumulate,
                            cudaStream_t st);
// weight images for the forward GEMM: per K block [hi: O x 64 K-major SW128][lo: same]
int launch_weight_tiles_fwd(const Geo& g, const Tiling& t, const void* wt, uint8_t* tiles, int operand,
                            cudaStream_t st);

}  // namespace dcn
