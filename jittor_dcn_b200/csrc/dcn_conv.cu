// dcn_conv.cu — the companion offset convolution (deform_conv.py:16-21,58 / train.py:80-85,98) and its autograd as
// "shifted-view" implicit GEMMs on the 5th-gen tensor cores.
//
// A regular k x k convolution reads, for tap (ki, kj), the SAME input pixels as every other tap — only shifted.  The
// plain mode of the DCN kernels (dcn_umma_fwd.cu, PLAIN) ignored that: it gathered and converted every pixel once
// per tap (9x), and the cfg2 offset conv ran instruction-bound at 2.46 ms forward / 4.4 ms backward.  Here a row of
// input pixels is converted to bf16 hi/lo ONCE per K step into a 128B-swizzled shared-memory image whose rows are
// pixels, and the kw taps of that row are kw tcgen05 descriptors into the same image, start address moved by
// (kj / stride) * 128 bytes: the tensor core applies the 128-byte swizzle to the final address bits, so a start that
// is not 1024-byte aligned addresses "row m + shift" exactly (tools/shift_probe.cu, profiles/r2_shift_probe.txt:
// K-major A and MN-major operand, shifts 0..9, descriptor base-offset field 0).  Stride 2 splits the row into an
// even- and an odd-column image.
//
//   MODE_FWD    offset[b, o, h, w]   = bias[o] + sum_{ki,kj,c} x[b, c, h*s-p+ki, w*s-p+kj] * W[o, c, ki, kj]
//               A = image of input row (h*s-p+ki) (rows = pixels, K = 64-channel slab), B = W tap image [o][c]
//   MODE_DGRAD  gxt[b, y, x, c]     += sum_{ki,kj,o} goff[b, o, (y+p-ki)/s, (x+p-kj)/s] * W[o, c, ki, kj]
//               A = image of a grad_offset row (rows = pixels, K = o, zero halo), B = W tap image [c][o];
//               stride 2: the four output parities (y+p, x+p) mod 2 are four accumulators, every tap feeds one
//               of them; the result is ADDED to the channels-last grad_x accumulator of the DCN backward (red.v4)
//   MODE_WGRAD  gW[o, c, ki, kj]     = sum_{b,h,w} goff[b, o, h, w] * x[b, c, h*s-p+ki, w*s-p+kj]
//               A = the forward's image read MN-major (M = channels, K = pixels), B = grad_offset tile [o][pixels]
//
// A tile is `rpt` consecutive rows of the output grid x up to Wt columns; GEMM row m = hr * Wseg + w (Wseg =
// 128 / rpt), so narrow images pack several rows into the 128 tensor-core rows.  Rows of an image that no valid
// output reads hold stale (finite: everything is zero-initialised) data and only ever meet zero operands or feed
// accumulator rows that are not stored.
//
// Warp roles (960 threads, 1 CTA / SM, persistent): warps 0-3 epilogue, 4 MMA issuer, 5 bulk loader (weight tap
// images), 6-29 conversion (global -> bf16 hi/lo -> swizzled shared memory; all loads of a K step are issued before
// the first conversion).  fp32 parity as in the DCN kernels: hi*hi + hi*lo + lo*hi, fp32 accumulation in TMEM.
#include <cstring>

#include "dcn_umma.h"
#include "dcn_umma_common.cuh"

namespace dcn {

using namespace ptx;

namespace cv {

enum { MODE_FWD = 0, MODE_DGRAD = 1, MODE_WGRAD = 2 };

constexpr int kEpiWarps = 4, kConvWarps = 24;
constexpr int kMmaWarp = kEpiWarps, kLoadWarp = kEpiWarps + 1, kFirstConvWarp = kEpiWarps + 2;
constexpr int kThreads = (kFirstConvWarp + kConvWarps) * 32;  // 960
constexpr int kConvThreads = kConvWarps * 32;
constexpr uint32_t kImgRows = 136;                 // 128 GEMM rows + shifted views (<= 2 rows) rounded to 8
constexpr uint32_t kImg = kImgRows * 128;          // one bf16 image: 17408 B = 17 * 1024
constexpr int kMaxItems = 3;                       // conversion items per thread and K step (x image)
constexpr int kMaxStages = 3;
constexpr int kSlab = 64;                          // channels of one K slab of the x image (FWD / WGRAD): one 128 B row

struct Params {
  // the convolution: x[B, C, H, W] -> [B, O, Ho, Wo], kernel kh x kw, stride s, padding p (both axes)
  int B, C, O, H, W, Ho, Wo, kh, kw, s, p;
  int perm_G, perm_Cs;        // channel permutation of the staged copy (Torch layout), 0 = none
  // tile grid: FWD / WGRAD = the conv output grid; DGRAD = the grad_x grid (stride 1) or its half-resolution
  // (Y, X) = (frame row / 2, frame column / 2) grid (stride 2)
  int GR, GC;                 // rows / columns of the tile grid
  int Wseg, rpt, Wt;          // GEMM row m = hr * Wseg + w; rpt = 128 / Wseg rows per tile, Wt <= Wseg valid columns
  int ncolseg, nrowt;         // column segments per row, row tiles per image
  int nchunks_n;              // DGRAD: 64-channel chunks of C handled as separate tiles
  int num_tiles;
  int nslab;                  // FWD: C / kSlab
  int nk4;                    // K = 16 steps per image: kSlab / 16 (FWD), ceil(O / 16) (DGRAD)
  int Nn;                     // MMA N: o_pad (FWD, WGRAD), channels per chunk (DGRAD)
  int nph;                    // phase images per stage: s (FWD / WGRAD), 1 (DGRAD)
  int ncols_in;               // input columns one image row holds, all phases together
  int ne0;                    // entries of phase 0 (phase 1 holds ncols_in - ne0)
  int stages;
  int w_res;                  // weight tap images of ALL K steps resident in shared memory (loaded once), else streamed
  uint32_t w_res_bytes;
  uint32_t w_tile;            // bytes of ONE weight tap image (hi or lo): Nn * 128
  uint32_t stage_bytes;       // nph * 2 * kImg + (FWD / DGRAD: kw * 2 * w_tile)
  uint32_t tmem_cols;
  FastDiv div_cols, div_rowt, div_colseg, div_nch;
  // tensors
  const float* xt;            // framed channels-last x (FWD, WGRAD)
  float* gxt;                 // framed channels-last grad_x accumulator (DGRAD)
  const float* goff;          // [B, O, Ho, Wo] (DGRAD, WGRAD)
  float* out;                 // [B, O, Ho, Wo] (FWD)
  const float* bias;
  float* gw;                  // [O, C, kh, kw] (WGRAD), zeroed
  const uint8_t* wtiles;      // FWD: [slab][ki][kj][hi|lo][Nn x 128 B]; DGRAD: [chunk][ki][kj][hi|lo][Nn x 128 B]
  size_t img_stride;          // elements per framed image
  int pitch;                  // elements per frame row
  // WGRAD: CTA = (slab, chunk of tiles)
  int w_nchunks;
};

struct TileInfo {
  int b, r0, c0, nch;
};
__device__ __forceinline__ TileInfo decode_tile(const Params& P, int tile) {
  TileInfo ti;
  uint32_t q, r;
  P.div_nch.divmod((uint32_t)tile, q, r);
  ti.nch = (int)r;
  uint32_t q2, cs;
  P.div_colseg.divmod(q, q2, cs);
  uint32_t b, rt;
  P.div_rowt.divmod(q2, b, rt);
  ti.b = (int)b;
  ti.r0 = (int)rt * P.rpt;
  ti.c0 = (int)cs * P.Wt;
  return ti;
}

// DGRAD tap tables.  stride 1: source row = y + p - ki, view shift = kw - 1 - kj (image column e <-> source column
// c0 + e + p - (kw - 1)), one accumulator.  stride 2 (k = 3, p = 1 only): frame row fy = 2Y + py; ki = 1 feeds py = 1
// from grad row Y, ki = 0 / 2 feed py = 0 from rows Y / Y - 1; columns alike (image column e <-> source column
// c0 + e - 1, view shift 1 + dX).
__device__ __forceinline__ int dgrad_row_off(const Params& P, int ki) {
  return P.s == 1 ? P.p - ki : (ki == 2 ? -1 : 0);
}
__device__ __forceinline__ int dgrad_shift(const Params& P, int kj) {
  return P.s == 1 ? P.kw - 1 - kj : (kj == 2 ? 0 : 1);
}
__device__ __forceinline__ int dgrad_acc(const Params& P, int ki, int kj) {
  return P.s == 1 ? 0 : ((ki == 1 ? 2 : 0) + (kj == 1 ? 1 : 0));
}

// MASK (MODE_FWD only): the modulated layer's 3N-channel conv (mmcv's ModulatedDeformConv2dPack.conv_offset): channels
// [0, 2N) go to out [B, 2N, Ho, Wo], channels [2N, 3N) to mask [B, N, Ho, Wo] as sigmoid(acc + bias).  The pointer is a
// trailing argument so that the parameter layout of the unmodulated instantiations does not move.
template <int MODE, bool MASK = false>
__global__ void __launch_bounds__(kThreads, 1) conv_kernel(const __grid_constant__ Params P, float* mask = nullptr) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  // carve-up: [stages x (phase images hi|lo, weight tap images)] [WGRAD: 2 grad tiles (2 K blocks x hi|lo x 4 KB)]
  uint8_t* stage_base = smem;
  uint8_t* gbuf_base = smem + (size_t)P.stages * P.stage_bytes;
  constexpr uint32_t kGBlk = 32 * 128;                 // one K block of the grad tile: 32 rows (o) x 64 pixels
  constexpr uint32_t kGBuf = 2 * 2 * kGBlk;            // [K block][hi|lo]
  uint8_t* wres_base = gbuf_base + (MODE == MODE_WGRAD ? 2 * kGBuf : 0);
  uint64_t* bars = reinterpret_cast<uint64_t*>(wres_base + (P.w_res ? P.w_res_bytes : 0u));
  uint64_t* full = bars;                     // [kMaxStages]
  uint64_t* empty = bars + kMaxStages;       // [kMaxStages]
  uint64_t* tfull = bars + 2 * kMaxStages;   // [2]
  uint64_t* tempty = tfull + 2;              // [2]
  uint64_t* gfull = tempty + 2;              // [2] WGRAD grad tile
  uint64_t* gempty = gfull + 2;              // [2]
  uint64_t* wfull = gempty + 2;              // [1] resident weight images loaded
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wfull + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool wstream = MODE != MODE_WGRAD && !P.w_res;   // weight tap images arrive by bulk copy, once per K step
  if (tid == 0) {
    for (int s = 0; s < P.stages; ++s) {
      mbar_init(&full[s], kConvWarps + (wstream ? 1 : 0));
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], kEpiWarps);
      mbar_init(&gfull[a], kConvWarps);
      mbar_init(&gempty[a], 1);
    }
    mbar_init(wfull, 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(P.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // every operand byte starts finite: image rows / K columns that are never converted meet zero operands or feed
  // accumulator rows that are not stored, but 0 * NaN would still poison a sum
  {
    const uint32_t total = (uint32_t)P.stages * P.stage_bytes + (MODE == MODE_WGRAD ? 2 * kGBuf : 0);
    for (uint32_t i = tid * 16; i < total; i += kThreads * 16) *reinterpret_cast<uint4*>(smem + i) = make_uint4(0, 0, 0, 0);
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // tiles of this CTA; WGRAD: a fixed K slab for a chunk of the tiles
  int tile0 = blockIdx.x, tile_step = gridDim.x, slab0 = 0;
  if (MODE == MODE_WGRAD) {
    slab0 = blockIdx.x % P.nslab;
    tile0 = blockIdx.x / P.nslab;
    tile_step = P.w_nchunks;
  }
  const int ksteps = MODE == MODE_FWD ? P.nslab * P.kh : P.kh;   // K steps per tile
  const uint32_t img_pair = 2 * kImg;                            // hi | lo of one phase
  const uint32_t w_off = (uint32_t)P.nph * img_pair;             // weight tap images inside a stage

  if (warp < kEpiWarps) {
    // ================================================================ epilogue
    const int m = warp * 32 + lane;
    const int hr = m / P.Wseg, wl = m - hr * P.Wseg;
    if constexpr (MODE == MODE_FWD && MASK) {
      const int n_off = P.O / 3 * 2;   // offset channels; the remaining P.O / 3 are mask logits
      const size_t plane = (size_t)P.Ho * P.Wo;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = tile0; tile < P.num_tiles; tile += tile_step) {
        const TileInfo ti = decode_tile(P, tile);
        const int r = ti.r0 + hr, c = ti.c0 + wl;
        const bool valid = r < P.GR && wl < P.Wt && c < P.GC;
        float* dst = P.out + (size_t)ti.b * n_off * plane + (size_t)r * P.Wo + c;
        float* mdst = mask + (size_t)ti.b * (P.O - n_off) * plane + (size_t)r * P.Wo + c;
        mbar_wait_relaxed(&tfull[acc], acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(acc * 2 * P.Nn);
        for (int c0 = 0; c0 < P.Nn; c0 += 16) {
          float v[16], w[16];
          tmem_ld16(taddr + c0, v);
          tmem_ld16(taddr + P.Nn + c0, w);   // the hi*lo half
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] += w[i];
          if (valid) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int o = c0 + i;
              if (o >= P.O) break;
              const float z = v[i] + (P.bias ? __ldg(P.bias + o) : 0.f);
              if (o < n_off) dst[(size_t)o * plane] = z;
              else mdst[(size_t)(o - n_off) * plane] = 1.f / (1.f + expf(-z));
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[acc]);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    } else if constexpr (MODE == MODE_FWD) {
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = tile0; tile < P.num_tiles; tile += tile_step) {
        const TileInfo ti = decode_tile(P, tile);
        const int r = ti.r0 + hr, c = ti.c0 + wl;
        const bool valid = r < P.GR && wl < P.Wt && c < P.GC;
        float* dst = P.out + (size_t)ti.b * P.O * P.Ho * P.Wo + (size_t)r * P.Wo + c;
        mbar_wait_relaxed(&tfull[acc], acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(acc * 2 * P.Nn);
        for (int c0 = 0; c0 < P.Nn; c0 += 16) {
          float v[16], w[16];
          tmem_ld16(taddr + c0, v);
          tmem_ld16(taddr + P.Nn + c0, w);   // the hi*lo half
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] += w[i];
          if (valid) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              if (c0 + i >= P.O) break;
              const float bv = P.bias ? __ldg(P.bias + c0 + i) : 0.f;
              DCN_DEV_ASSERT((size_t)(dst - P.out) + (size_t)(c0 + i) * P.Ho * P.Wo < (size_t)P.B * P.O * P.Ho * P.Wo);
              dst[(size_t)(c0 + i) * P.Ho * P.Wo] = v[i] + bv;
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[acc]);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    } else if constexpr (MODE == MODE_DGRAD) {
      int acc = 0;
      uint32_t acc_phase = 0;
      const int nacc = P.s == 1 ? 1 : 4;
      for (int tile = tile0; tile < P.num_tiles; tile += tile_step) {
        const TileInfo ti = decode_tile(P, tile);
        float* img = P.gxt + (size_t)ti.b * P.img_stride + ti.nch * 64;
        mbar_wait_relaxed(&tfull[acc], acc_phase);
        tc_fence_after();
        for (int a = 0; a < nacc; ++a) {
          // frame position of this lane's pixel for accumulator a
          int fy, fx;
          bool valid = wl < P.Wt;
          if (P.s == 1) {
            fy = ti.r0 + hr + 1;
            fx = ti.c0 + wl + 1;
            valid = valid && ti.r0 + hr < P.H && ti.c0 + wl < P.W;
          } else {
            fy = 2 * (ti.r0 + hr) + (a >> 1);
            fx = 2 * (ti.c0 + wl) + (a & 1);
            valid = valid && fy >= 1 && fy <= P.H && fx >= 1 && fx <= P.W;
          }
          float* dst = img + ((size_t)fy * (P.W + 2) + fx) * P.C;
          DCN_DEV_ASSERT(!valid || (size_t)(dst - P.gxt) + P.Nn <= (size_t)P.B * P.img_stride);
          const uint32_t taddr =
              tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)((acc * nacc + a) * 2 * P.Nn);
          for (int c0 = 0; c0 < P.Nn; c0 += 16) {
            float v[16], w[16];
            tmem_ld16(taddr + c0, v);
            tmem_ld16(taddr + P.Nn + c0, w);   // the hi*lo half
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] += w[i];
            if (valid) {
#pragma unroll
              for (int i = 0; i < 16; i += 4)
                atomicAdd(reinterpret_cast<float4*>(dst + c0 + i), make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]));
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[acc]);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    } else {
      // WGRAD: one-shot epilogue.  TMEM lane = staged channel of the slab, columns = (tap, o)
      mbar_wait_relaxed(&tfull[0], 0);
      tc_fence_after();
      const int cs = slab0 * kSlab + m;   // staged channel
      int c_real = cs;
      if (P.perm_G) c_real = (cs % P.perm_G) * P.perm_Cs + cs / P.perm_G;
      const int ntaps = P.kh * P.kw;
      for (int t = 0; t < ntaps; ++t) {
        const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(t * P.Nn);
        for (int c0 = 0; c0 < P.Nn; c0 += 16) {
          float v[16];
          tmem_ld16(taddr + c0, v);
          if (m < kSlab) {
#pragma unroll
            for (int i = 0; i < 16; ++i)
              if (c0 + i < P.O) atomicAdd(P.gw + ((size_t)(c0 + i) * P.C + c_real) * ntaps + t, v[i]);
          }
        }
      }
      tc_fence_before();
    }
  } else if (warp == kMmaWarp) {
    // ================================================================ MMA issuer
    // The whole warp runs this (uniform) loop and elect.sync picks the issuing lane per instruction (see
    // dcn_umma.cuh:elect_one).  One thread issues ~100 small MMAs (N = 16 .. 64) per tile, so ITS instruction stream is the critical path: the
    // first version rebuilt four 64-bit descriptors per K = 16 step (~40 dependent integer instructions per 3 MMAs) and
    // the tensor pipe sat at 12 %.  A descriptor's address field is its low 14 bits (address >> 4; 18-bit shared
    // addresses cannot carry into the next field), so every descriptor here is ONE 64-bit add onto a per-stage base,
    // and the loops have constant bounds (guards instead of runtime trip counts) so that they unroll.
    {
      int s = 0;
      uint32_t phase = 0;
      const uint64_t desc0 = make_sdesc_sw128(smem_u32(stage_base), 16, 1024);   // K-major, 8-row groups 1024 B apart
      const uint32_t stage16 = P.stage_bytes >> 4, wt16 = P.w_tile >> 4;
      constexpr uint32_t kImg16 = kImg >> 4, kPair16 = (2 * kImg) >> 4;
      if constexpr (MODE != MODE_WGRAD) {
        const uint32_t idesc = make_idesc_bf16(128, P.Nn, false, false), idesc2 = make_idesc_bf16(128, 2 * P.Nn, false, false);
        const int nacc = (MODE == MODE_DGRAD && P.s == 2) ? 4 : 1;
        int acc = 0;
        uint32_t acc_phase = 0;
        const uint64_t wres0 = make_sdesc_sw128(smem_u32(wres_base), 16, 1024);
        if (P.w_res && tile0 < P.num_tiles) {
          mbar_wait_relaxed(wfull, 0, 32);
          tc_fence_after();
        }
        for (int tile = tile0; tile < P.num_tiles; tile += tile_step) {
          const int nch = MODE == MODE_DGRAD ? decode_tile(P, tile).nch : 0;
          mbar_wait_relaxed(&tempty[acc], acc_phase ^ 1, 32);
          tc_fence_after();
          uint32_t started = 0;   // accumulators that already hold a partial sum
          for (int ks = 0; ks < ksteps; ++ks) {
            const int ki = MODE == MODE_FWD ? ks % P.kh : ks;
            mbar_wait_relaxed(&full[s], phase, 20);
            tc_fence_after();
            const uint64_t ad = desc0 + (uint64_t)((uint32_t)s * stage16);
            // streamed: the K step's kw tap images sit behind the phase images of the stage; resident: image
            // ((group * kh + ki) * kw + kj) of the resident region, group = K slab (FWD) / channel chunk (DGRAD)
            const uint64_t wd = P.w_res ? wres0 + (uint64_t)((uint32_t)((MODE == MODE_FWD ? ks : nch * P.kh + ks) * P.kw) * 2u * wt16)
                                        : ad + (w_off >> 4);
#pragma unroll
            for (int kq = 0; kq < 3; ++kq) {
              if (kq >= P.kw) break;
              // stride-2 DGRAD: taps 0 and 2 feed the same parity accumulator; switching the accumulator between
              // consecutive MMAs costs ~120 cycles (tools/mma_rate_probe.cu), so they go back to back
              const int kj = (MODE == MODE_DGRAD && P.s == 2) ? (kq == 0 ? 0 : (kq == 1 ? 2 : 1)) : kq;
              int ph, shift, a;
              if (MODE == MODE_FWD) {
                ph = kj % P.s;
                shift = kj / P.s;
                a = 0;
              } else {
                ph = 0;
                shift = dgrad_shift(P, kj);
                a = dgrad_acc(P, ki, kj);
              }
              const uint64_t a_hi = ad + (uint64_t)((uint32_t)ph * kPair16 + (uint32_t)shift * 8u);
              const uint64_t b_hi = wd + (uint64_t)((uint32_t)kj * 2u * wt16);
              const uint32_t d_tmem = tmem_base + (uint32_t)((acc * nacc + a) * 2 * P.Nn);
              const uint32_t st0 = (started >> a) & 1u;
              // two MMAs per K = 16 step instead of three: the tap's [W_hi ; W_lo] images are contiguous, i.e. ONE
              // K-major operand of 2 * Nn rows, so x_hi meets both in one instruction (accumulator columns [0, Nn) =
              // hi*hi, [Nn, 2Nn) = hi*lo; the epilogue adds the halves); x_lo * W_hi then goes into the first half.
              // An MMA of this shape costs 64 cycles for any N <= 128 (tools/mma_rate_probe.cu), so N is free.
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4) {
                if (k4 >= P.nk4) break;
                const uint64_t dah = a_hi + 2u * k4, dbh = b_hi + 2u * k4;
                if (elect_one()) {
                  umma_bf16(d_tmem, dah, dbh, idesc2, k4 ? 1u : st0);
                  umma_bf16(d_tmem, dah + kImg16, dbh, idesc, 1u);
                }
              }
              started |= 1u << a;
            }
            if (elect_one()) {
              umma_commit(&empty[s]);
              if (ks == ksteps - 1) umma_commit(&tfull[acc]);
            }
            __syncwarp();
            if (++s == P.stages) {
              s = 0;
              phase ^= 1;
            }
          }
          acc ^= 1;
          if (acc == 0) acc_phase ^= 1;
        }
      } else {
        // D[c, (tap, o)] += sum_px X_tap[px, c] * G[px, o]: A = the x image read MN-major (M = 64 channels = one
        // 128-byte row; the second 64-row atom of the M = 128 shape points at the lo image — finite, rows ignored),
        // K = image rows; B = grad tile [o][64 px] K-major, two K blocks of 64 pixels
        const uint32_t idesc = make_idesc_bf16(128, P.Nn, true, false);
        const uint64_t xdesc0 = make_sdesc_sw128(smem_u32(stage_base), kImg, 1024);
        const uint64_t gdesc0 = make_sdesc_sw128(smem_u32(gbuf_base), 16, 1024);
        constexpr uint32_t kGBlk16 = kGBlk >> 4, kGBuf16 = kGBuf >> 4;
        int gb = 0;
        uint32_t gphase = 0;
        bool first_tile = true;
        for (int tile = tile0; tile < P.num_tiles; tile += tile_step) {
          mbar_wait_relaxed(&gfull[gb], gphase, 20);
          const uint64_t gd = gdesc0 + (uint64_t)((uint32_t)gb * kGBuf16);
          for (int ki = 0; ki < P.kh; ++ki) {
            mbar_wait_relaxed(&full[s], phase, 20);
            tc_fence_after();
            const uint64_t xd = xdesc0 + (uint64_t)((uint32_t)s * stage16);
            // one accumulator per tap; all MMAs of a tap back to back (switching the accumulator between consecutive
            // MMAs costs ~120 cycles, tools/mma_rate_probe.cu)
#pragma unroll
            for (int kj = 0; kj < 3; ++kj) {
              if (kj >= P.kw) break;
              const uint64_t x0 = xd + (uint64_t)((uint32_t)(kj % P.s) * kPair16 + (uint32_t)(kj / P.s) * 8u);
              const uint32_t d_tmem = tmem_base + (uint32_t)((ki * P.kw + kj) * P.Nn);
#pragma unroll
              for (int k8 = 0; k8 < 8; ++k8) {   // 8 steps of 16 pixels
                const uint64_t g_hi = gd + (uint64_t)((uint32_t)(k8 >> 2) * 2u * kGBlk16 + (uint32_t)(k8 & 3) * 2u);
                const uint64_t x_hi = x0 + (uint64_t)((uint32_t)k8 * 128u);
                if (elect_one()) {
                  umma_bf16(d_tmem, x_hi, g_hi, idesc, (first_tile && k8 == 0) ? 0u : 1u);
                  umma_bf16(d_tmem, x_hi, g_hi + kGBlk16, idesc, 1u);
                  umma_bf16(d_tmem, x_hi + kImg16, g_hi, idesc, 1u);
                }
              }
            }
            if (elect_one()) umma_commit(&empty[s]);
            __syncwarp();
            if (++s == P.stages) {
              s = 0;
              phase ^= 1;
            }
          }
          if (elect_one()) umma_commit(&gempty[gb]);
          __syncwarp();
          first_tile = false;
          gb ^= 1;
          if (gb == 0) gphase ^= 1;
        }
        if (elect_one()) umma_commit(&tfull[0]);
        __syncwarp();
      }
    }
  } else if (warp == kLoadWarp) {
    // ================================================================ weight tap images (bulk copies)
    if (P.w_res && MODE != MODE_WGRAD && lane == 0 && tile0 < P.num_tiles) {
      mbar_arrive_expect_tx(wfull, P.w_res_bytes);
      for (uint32_t o = 0; o < P.w_res_bytes; o += 32768u) {
        const uint32_t n = P.w_res_bytes - o < 32768u ? P.w_res_bytes - o : 32768u;
        bulk_g2s(wres_base + o, P.wtiles + o, n, wfull);
      }
    }
    if (wstream && lane == 0) {
      int s = 0;
      uint32_t phase = 0;
      const uint32_t bytes = (uint32_t)P.kw * 2u * P.w_tile;
      for (int tile = tile0; tile < P.num_tiles; tile += tile_step) {
        const int nch = MODE == MODE_DGRAD ? decode_tile(P, tile).nch : 0;
        for (int ks = 0; ks < ksteps; ++ks) {
          // FWD: ks = slab * kh + ki; DGRAD: (chunk, ki)
          const size_t idx = MODE == MODE_FWD ? (size_t)ks : (size_t)nch * P.kh + ks;
          mbar_wait_relaxed(&empty[s], phase ^ 1);
          mbar_arrive_expect_tx(&full[s], bytes);
          bulk_g2s(stage_base + (size_t)s * P.stage_bytes + w_off, P.wtiles + idx * bytes, bytes, &full[s]);
          if (++s == P.stages) {
            s = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else {
    // ================================================================ conversion warps
    // Software pipeline over the flattened (tile, K step) sequence: the global loads of step i + 1 are issued before
    // step i is converted (two register sets, used alternately), so a warp always has a K step of loads in flight and
    // the DRAM / L2 latency is paid once, not once per step (the first version issued and consumed the loads of a
    // step back to back: 2.5 us per K step on cfg2).
    const int ct = tid - kFirstConvWarp * 32;   // 0 .. kConvThreads - 1
    int s = 0;
    uint32_t phase = 0;
    struct Step {
      int tile, ks;
      TileInfo ti;
    };
    auto advance = [&](Step& q) {
      if (++q.ks == ksteps) {
        q.ks = 0;
        q.tile += tile_step;
        if (q.tile < P.num_tiles) q.ti = decode_tile(P, q.tile);
      }
    };
    auto publish = [&]() {
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[s]);
      if (++s == P.stages) {
        s = 0;
        phase ^= 1;
      }
    };
    Step cur;
    cur.tile = tile0;
    cur.ks = 0;
    cur.ti = decode_tile(P, tile0 < P.num_tiles ? tile0 : 0);
    if constexpr (MODE != MODE_DGRAD) {
      // x image: items = (row hr, input column j, 4-channel quad); the decomposition does not depend on the tile.
      // packed item: bits 0..16 byte offset inside the stage, 17..24 column j, 25..27 row hr, 28 live
      constexpr int q4 = kSlab / 4, q4_sh = 4;                // 16 quads of 4 channels per pixel
      const int n_items = P.rpt * P.ncols_in * q4;
      uint32_t src_off[kMaxItems], item[kMaxItems];
#pragma unroll
      for (int i = 0; i < kMaxItems; ++i) {
        const int idx = ct + i * kConvThreads;
        src_off[i] = item[i] = 0;
        if (idx < n_items) {
          const int cq = idx & (q4 - 1), t = idx >> q4_sh;
          uint32_t hr, pp;
          P.div_cols.divmod((uint32_t)t, hr, pp);
          // phase-major column order: pp < ne0 -> phase 0 entry pp, else phase 1 entry pp - ne0
          const int ph = (int)pp >= P.ne0 ? 1 : 0, e = (int)pp - ph * P.ne0, j = e * P.nph + ph;
          src_off[i] = (uint32_t)(((int)hr * P.s * (P.W + 2) + j) * P.C + cq * 4);
          item[i] = ((uint32_t)ph * img_pair + kmajor_sw128_off((int)hr * P.Wseg + e, cq * 4)) | ((uint32_t)j << 17) |
                    (hr << 25) | (1u << 28);
        }
      }
      auto issue = [&](const Step& q, float4 (&v)[kMaxItems], uint32_t& ok) {
        const int slab = MODE == MODE_FWD ? q.ks / P.kh : slab0, ki = MODE == MODE_FWD ? q.ks % P.kh : q.ks;
        const int fy0 = q.ti.r0 * P.s + ki + 1 - P.p, fx0 = q.ti.c0 * P.s + 1 - P.p;
        const float* base = P.xt + (size_t)q.ti.b * P.img_stride + ((size_t)fy0 * (P.W + 2) + fx0) * P.C + slab * kSlab;
        ok = 0;
#pragma unroll
        for (int i = 0; i < kMaxItems; ++i) {
          const int hr = (int)((item[i] >> 25) & 7u), j = (int)((item[i] >> 17) & 0xffu);
          const bool oki = (item[i] >> 28) && q.ti.r0 + hr < P.GR && fy0 + hr * P.s <= P.H + 2 && fx0 + j <= P.W + 1;
          v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (oki) {
            DCN_DEV_ASSERT(base >= P.xt && (size_t)(base - P.xt) + src_off[i] + 4 <= (size_t)P.B * P.img_stride);
            v[i] = __ldg(reinterpret_cast<const float4*>(base + src_off[i]));
            ok |= 1u << i;
          }
        }
      };
      int gb = 0;
      uint32_t gphase = 0;
      auto convert = [&](const Step& q, const float4 (&v)[kMaxItems], uint32_t ok) {
        if constexpr (MODE == MODE_WGRAD) {
          if (q.ks == 0) {
            // the tile's grad_offset operand [o][pixels]: items = (o, group of 8 pixels)
            mbar_wait(&gempty[gb], gphase ^ 1);
            uint8_t* gbuf = gbuf_base + (size_t)gb * kGBuf;
            const float* gsrc = P.goff + (size_t)q.ti.b * P.O * P.Ho * P.Wo;
            for (int it = ct; it < P.O * 16; it += kConvThreads) {
              const int pg = it & 15, o = it >> 4, px = pg * 8;
              const int hr = px / P.Wseg, wl = px - hr * P.Wseg;
              const int r = q.ti.r0 + hr;
              float g8[8];
#pragma unroll
              for (int u = 0; u < 8; ++u) {
                const int c = q.ti.c0 + wl + u;
                g8[u] = (r < P.Ho && wl + u < P.Wt && c < P.Wo) ? __ldg(gsrc + ((size_t)o * P.Ho + r) * P.Wo + c) : 0.f;
              }
              uint4 hi, lo;
              split_pair(g8[0], g8[1], hi.x, lo.x);
              split_pair(g8[2], g8[3], hi.y, lo.y);
              split_pair(g8[4], g8[5], hi.z, lo.z);
              split_pair(g8[6], g8[7], hi.w, lo.w);
              uint8_t* d = gbuf + (size_t)(px >> 6) * 2 * kGBlk + kmajor_sw128_off(o, px & 63);
              *reinterpret_cast<uint4*>(d) = hi;
              *reinterpret_cast<uint4*>(d + kGBlk) = lo;
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&gfull[gb]);
            gb ^= 1;
            if (gb == 0) gphase ^= 1;
          }
        }
        mbar_wait(&empty[s], phase ^ 1);
        uint8_t* st = stage_base + (size_t)s * P.stage_bytes;
#pragma unroll
        for (int i = 0; i < kMaxItems; ++i) {
          if (!((ok >> i) & 1u)) continue;
          uint2 hi, lo;
          split_pair(v[i].x, v[i].y, hi.x, lo.x);
          split_pair(v[i].z, v[i].w, hi.y, lo.y);
          uint8_t* d = st + (item[i] & 0x1ffffu);
          *reinterpret_cast<uint2*>(d) = hi;
          *reinterpret_cast<uint2*>(d + kImg) = lo;
        }
        publish();
      };
      float4 va[kMaxItems], vb[kMaxItems];
      uint32_t oka = 0, okb = 0;
      if (cur.tile < P.num_tiles) issue(cur, va, oka);
      while (cur.tile < P.num_tiles) {
        Step nxt = cur;
        advance(nxt);
        const bool nv = nxt.tile < P.num_tiles;
        if (nv) issue(nxt, vb, okb);
        convert(cur, va, oka);
        if (!nv) break;
        Step nn = nxt;
        advance(nn);
        if (nn.tile < P.num_tiles) issue(nn, va, oka);
        convert(nxt, vb, okb);
        cur = nn;
      }
    } else {
      // DGRAD image: rows = (hr, column e) of the grad_offset grid with a zero halo, K = o.  Items = (hr, e, group of
      // 8 o); lanes run along e: coalesced plane reads, conflict-free 16-byte stores.
      const int ne = P.ncols_in, ngrp = P.nk4 * 2;           // 8-o groups that the MMAs read
      const int n_items = P.rpt * ne * ngrp;
      const int col_off = P.s == 1 ? P.p - (P.kw - 1) : -1;  // image column e <-> source column c0 + e + col_off
      constexpr int kDI = 2;                                 // items per thread (host checks)
      uint32_t item[kDI];                                    // bits 0..16 byte offset, 17..24 e, 25..27 hr, 28..29 og, 30 live
#pragma unroll
      for (int i = 0; i < kDI; ++i) {
        const int it = ct + i * kConvThreads;
        item[i] = 0;
        if (it < n_items) {
          uint32_t t, e;
          P.div_cols.divmod((uint32_t)it, t, e);
          const uint32_t og = t % (uint32_t)ngrp, hr = t / (uint32_t)ngrp;
          item[i] = kmajor_sw128_off((int)hr * P.Wseg + (int)e, (int)og * 8) | (e << 17) | (hr << 25) | (og << 28) | (1u << 30);
        }
      }
      auto issue = [&](const Step& q, float (&v)[kDI][8]) {
        const float* gsrc = P.goff + (size_t)q.ti.b * P.O * P.Ho * P.Wo;
        const int roff = dgrad_row_off(P, q.ks);
#pragma unroll
        for (int i = 0; i < kDI; ++i) {
          const int e = (int)((item[i] >> 17) & 0xffu), hr = (int)((item[i] >> 25) & 7u), og = (int)((item[i] >> 28) & 3u);
          const int r = q.ti.r0 + hr + roff, c = q.ti.c0 + e + col_off;
          const bool in = (item[i] >> 30) && r >= 0 && r < P.Ho && c >= 0 && c < P.Wo;
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int o = og * 8 + u;
            v[i][u] = (in && o < P.O) ? __ldg(gsrc + ((size_t)o * P.Ho + r) * P.Wo + c) : 0.f;
          }
        }
      };
      auto convert = [&](const float (&v)[kDI][8]) {
        mbar_wait(&empty[s], phase ^ 1);
        uint8_t* st = stage_base + (size_t)s * P.stage_bytes;
#pragma unroll
        for (int i = 0; i < kDI; ++i) {
          if (!(item[i] >> 30)) continue;
          uint4 hi, lo;
          split_pair(v[i][0], v[i][1], hi.x, lo.x);
          split_pair(v[i][2], v[i][3], hi.y, lo.y);
          split_pair(v[i][4], v[i][5], hi.z, lo.z);
          split_pair(v[i][6], v[i][7], hi.w, lo.w);
          uint8_t* d = st + (item[i] & 0x1ffffu);
          *reinterpret_cast<uint4*>(d) = hi;
          *reinterpret_cast<uint4*>(d + kImg) = lo;
        }
        publish();
      };
      float va[kDI][8], vb[kDI][8];
      if (cur.tile < P.num_tiles) issue(cur, va);
      while (cur.tile < P.num_tiles) {
        Step nxt = cur;
        advance(nxt);
        const bool nv = nxt.tile < P.num_tiles;
        if (nv) issue(nxt, vb);
        convert(va);
        if (!nv) break;
        Step nn = nxt;
        advance(nn);
        if (nn.tile < P.num_tiles) issue(nn, va);
        convert(vb);
        cur = nn;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(P.tmem_cols) : "memory");
  }
}

// weight tap images.  FWD: [slab][ki][kj][hi|lo] of [Nn rows o][64 staged channels of the slab];
// DGRAD: [chunk][ki][kj][hi|lo] of [Nn rows = staged channels of the chunk][64 k = o].  K-major, 128B swizzle.
__global__ void __launch_bounds__(256) conv_weight_tiles_kernel(Params P, int dgrad, const float* __restrict__ w,
                                                               uint8_t* __restrict__ tiles) {
  const int ntaps = P.kh * P.kw;
  const int groups = dgrad ? P.nchunks_n : P.nslab;
  const int total = groups * ntaps * P.Nn * 64;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < total; i += gridDim.x * 256) {
    const int k = i & 63, row = (i >> 6) % P.Nn, t = (i / (64 * P.Nn)) % ntaps, grp = i / (64 * P.Nn * ntaps);
    const int cs = grp * 64 + (dgrad ? row : k), o = dgrad ? k : row;
    float v = 0.f;
    if (o < P.O) {
      int c = cs;
      if (P.perm_G) c = (cs % P.perm_G) * P.perm_Cs + cs / P.perm_G;
      v = w[((size_t)o * P.C + c) * ntaps + t];
    }
    __nv_bfloat16 hi, lo;
    split_bf16(v, hi, lo);
    uint8_t* base = tiles + ((size_t)(grp * ntaps + t) * 2) * P.w_tile + kmajor_sw128_off(row, k);
    *reinterpret_cast<__nv_bfloat16*>(base) = hi;
    *reinterpret_cast<__nv_bfloat16*>(base + P.w_tile) = lo;
  }
}

}  // namespace cv

// ---------------------------------------------------------------------------- host side
static uint32_t conv_pow2_cols(int cols) {
  uint32_t c = 32;
  while ((int)c < cols) c <<= 1;
  return c;
}

// g = the DCN layer (its companion conv: same input, kernel, stride, padding; O outputs: 2N, or 3N for the modulated
// layer's offset-and-mask conv)
static bool conv_params(const Geo& g, int mode, cv::Params* Pp, int O) {
  cv::Params& P = *Pp;
  memset(&P, 0, sizeof(P));
  const int kh = g.N / g.kw;
  if (kh * g.kw != g.N || g.sh != g.sw || g.ph != g.pw) return false;
  if (g.sh != 1 && g.sh != 2) return false;
  if (g.ph > 1 || kh > 3 || g.kw > 3) return false;
  // K of one MMA row is the channels of ONE pixel: with fewer than 64 channels the per-tile MMA count (fixed: taps x
  // 16-column steps x hi/lo terms) dominates and the plain mode of the DCN kernels, which packs (tap, channel) pairs
  // into its K blocks, is faster (measured on the detector's 16- and 32-channel layers: backward 6.6 vs 2.8 ms).  Those
  // layers run on the warp-MMA kernels of dcn_conv_small.cu instead (conv_offset_*_supported below).
  if (g.C % 64 != 0) return false;
  if (O > 32) return false;
  // every read stays inside the framed copy
  if ((g.Ho - 1) * g.sh + kh - g.ph > g.H + 2 || (g.Wo - 1) * g.sw + g.kw - g.pw > g.W + 1) return false;
  if (mode == cv::MODE_DGRAD && g.sh == 2 && !(kh == 3 && g.kw == 3 && g.ph == 1)) return false;
  if ((long long)xt_image_stride(g) >= (1LL << 30)) return false;
  P.B = g.B; P.C = g.C; P.O = O; P.H = g.H; P.W = g.W; P.Ho = g.Ho; P.Wo = g.Wo;
  P.kh = kh; P.kw = g.kw; P.s = g.sh; P.p = g.ph;
  Tiling t;
  if (!make_tiling(g, &t)) return false;
  if (g.variant == DCN_VARIANT_TORCH) {
    P.perm_G = t.G;
    P.perm_Cs = t.Cs;
  }
  P.img_stride = xt_image_stride(g);
  P.pitch = xt_row_pitch(g);
  int extra;  // image entries a row needs beyond its Wt outputs
  if (mode == cv::MODE_DGRAD) {
    if (P.s == 1) {
      P.GR = g.H;
      P.GC = g.W;
      extra = P.kw - 1;
    } else {
      P.GR = g.H / 2 + 1;
      P.GC = g.W / 2 + 1;
      extra = 1;
    }
    P.nph = 1;
  } else {
    P.GR = g.Ho;
    P.GC = g.Wo;
    extra = (P.kw - 1) / P.s;
    P.nph = P.s;
  }
  // rows per tile: the largest power of two such that a row segment (valid columns + the shifted views) fits;
  // a single row may use the two spare image rows
  P.Wseg = 128;
  for (int ws = 16; ws < 128; ws <<= 1)
    if (P.GC + extra <= ws) {
      P.Wseg = ws;
      break;
    }
  P.rpt = 128 / P.Wseg;
  P.Wt = P.rpt == 1 ? (P.GC < 128 ? P.GC : 128) : P.GC;
  if (P.rpt == 1 && P.Wt + extra > (int)cv::kImgRows) return false;
  P.ncolseg = (P.GC + P.Wt - 1) / P.Wt;
  P.nrowt = (P.GR + P.rpt - 1) / P.rpt;
  if (mode == cv::MODE_DGRAD) {
    P.ncols_in = P.Wt + extra;
    P.ne0 = P.ncols_in;
    P.nslab = 1;
    P.nk4 = (O + 15) / 16;
    P.Nn = 64;
    P.nchunks_n = g.C / 64;
  } else {
    P.ncols_in = (P.Wt - 1) * P.s + P.kw;
    P.ne0 = (P.ncols_in + P.s - 1) / P.s;
    P.nslab = g.C / cv::kSlab;
    P.nk4 = cv::kSlab / 16;
    P.Nn = (O + 15) / 16 * 16;
    P.nchunks_n = 1;
  }
  const long long tiles = (long long)g.B * P.nrowt * P.ncolseg * P.nchunks_n;
  if (tiles > 0x7fffffffLL) return false;
  P.num_tiles = (int)tiles;
  P.div_rowt = FastDiv::make(P.nrowt);
  P.div_colseg = FastDiv::make(P.ncolseg);
  P.div_nch = FastDiv::make(P.nchunks_n);
  P.div_cols = FastDiv::make(P.ncols_in);
  P.w_tile = (uint32_t)P.Nn * 128;
  // weight tap images: resident (loaded once per CTA) when all of them fit next to >= 2 stages, else streamed per K step
  const size_t fixed = 1024 + 256 + (mode == cv::MODE_WGRAD ? 2 * 2 * 2 * 32 * 128 : 0);
  const size_t img_bytes = (size_t)P.nph * 2 * cv::kImg;
  const size_t all_w = (size_t)(mode == cv::MODE_DGRAD ? P.nchunks_n : P.nslab) * P.kh * P.kw * 2 * P.w_tile;
  P.w_res = 0;
  P.w_res_bytes = 0;
  if (mode != cv::MODE_WGRAD && fixed + all_w + 2 * img_bytes <= kSmemBudget) {
    P.w_res = 1;
    P.w_res_bytes = (uint32_t)all_w;
  }
  const bool wstream = mode != cv::MODE_WGRAD && !P.w_res;
  P.stage_bytes = (uint32_t)align_up(img_bytes + (wstream ? (size_t)P.kw * 2 * P.w_tile : 0), 1024);
  int stages = (int)((kSmemBudget - fixed - P.w_res_bytes) / P.stage_bytes);
  if (stages > cv::kMaxStages) stages = cv::kMaxStages;
  if (stages < 2) return false;
  P.stages = stages;
  // conversion items per thread
  if (mode != cv::MODE_DGRAD && (P.rpt * P.ncols_in * (cv::kSlab / 4) + cv::kConvThreads - 1) / cv::kConvThreads > cv::kMaxItems)
    return false;
  if (mode == cv::MODE_DGRAD && (P.rpt * P.ncols_in * P.nk4 * 2 + cv::kConvThreads - 1) / cv::kConvThreads > 2) return false;
  if (P.ncols_in > 255 || P.rpt > 8) return false;   // packed item fields
  // FWD / DGRAD accumulators are 2 * Nn columns wide (hi*hi + lo*hi | hi*lo), double-buffered
  const int nacc = (mode == cv::MODE_DGRAD && P.s == 2) ? 4 : 1;
  if (mode == cv::MODE_WGRAD) P.tmem_cols = conv_pow2_cols(P.kh * P.kw * P.Nn);
  else P.tmem_cols = conv_pow2_cols(2 * nacc * 2 * P.Nn);
  if (P.tmem_cols > 512) return false;
  return true;
}

static size_t conv_smem(const cv::Params& P, int mode) {
  return (size_t)P.stages * P.stage_bytes + (mode == cv::MODE_WGRAD ? 2 * 2 * 2 * 32 * 128 : 0) + P.w_res_bytes + 256 + 1024;
}

// warp-MMA kernels (dcn_conv_small.cu): narrow layers and whatever else the shifted-view kernels refuse
bool conv_small_supported(const Geo& g, int O);
size_t conv_small_wfrag_bytes(const Geo& g, int O);
int conv_small_forward(const Geo& g, int O, const float* xt, const float* woff, const float* boff, float* offset_out,
                       uint8_t* wfrag, cudaStream_t st, float* mask_out);
int conv_small_backward(const Geo& g, int O, const float* xt, float* gxt, const float* goff, const float* woff,
                        float* gwoff, uint8_t* wfrag, cudaStream_t st);

static bool conv_fwd_shifted(const Geo& g, int O) {
  cv::Params P;
  return conv_params(g, cv::MODE_FWD, &P, O);
}
static bool conv_bwd_shifted(const Geo& g, int O) {
  cv::Params P;
  return conv_params(g, cv::MODE_DGRAD, &P, O) && conv_params(g, cv::MODE_WGRAD, &P, O);
}

// O = the conv's output channels: 2N (offsets) or 3N (offsets and mask logits of the modulated layer)
bool conv_offset_fwd_supported(const Geo& g, int O) {
  return conv_fwd_shifted(g, O) || conv_small_supported(g, O);
}
bool conv_offset_bwd_supported(const Geo& g, int O) {
  // measured on the detector's layers (batch 1024): the warp-MMA backward wins below 64 channels (conv2 1.4 vs 1.8 ms,
  // conv3 0.7 vs 0.7 ms); at 64 / 128 channels the plain mode of the fused DCN backward kernel is faster (0.23 vs 0.35 ms)
  return conv_bwd_shifted(g, O) || (g.C < 64 && conv_small_supported(g, O));
}

// bytes of weight tap images one pass needs (the backward passes run one after the other and share the region)
size_t conv_offset_wtile_bytes(const Geo& g, int O) {
  cv::Params P;
  size_t need = 0;
  if (conv_params(g, cv::MODE_FWD, &P, O)) need = (size_t)P.nslab * P.kh * P.kw * 2 * P.w_tile;
  if (conv_params(g, cv::MODE_DGRAD, &P, O)) {
    const size_t d = (size_t)P.nchunks_n * P.kh * P.kw * 2 * P.w_tile;
    need = d > need ? d : need;
  }
  const size_t sm = conv_small_wfrag_bytes(g, O);
  need = sm > need ? sm : need;
  return align_up(need, 1024);
}

template <int MODE, bool MASK = false>
static int conv_launch(const cv::Params& P, int grid, cudaStream_t st, const char* name, float* mask = nullptr) {
  const size_t smem = conv_smem(P, MODE);
  DCN_CUDA_TRY(cudaFuncSetAttribute(cv::conv_kernel<MODE, MASK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  KernelScope scope(name, st);
  cv::conv_kernel<MODE, MASK><<<grid, cv::kThreads, smem, st>>>(P, mask);
  DCN_KERNEL_CHECK(name);
  return DCN_OK;
}

static int conv_weight_tiles(const cv::Params& P, int dgrad, const float* w, uint8_t* tiles, cudaStream_t st) {
  const int total = (dgrad ? P.nchunks_n : P.nslab) * P.kh * P.kw * P.Nn * 64;
  KernelScope scope("conv_weight_tiles_kernel", st);
  cv::conv_weight_tiles_kernel<<<(total + 255) / 256 < 1024 ? (total + 255) / 256 : 1024, 256, 0, st>>>(P, dgrad, w, tiles);
  DCN_KERNEL_CHECK("conv_weight_tiles_kernel");
  return DCN_OK;
}

// offset[B, 2N, Ho, Wo] = conv(x) + bias; xt = the layer's framed channels-last copy of x; wtiles = scratch of
// conv_offset_wtile_bytes().  mask_out != nullptr: the modulated layer's conv, woff / boff have 3N output channels and
// channels [2N, 3N) are written to mask_out [B, N, Ho, Wo] through the sigmoid (same pass, same kernels).
int conv_offset_forward(const Geo& g, const float* xt, const float* woff, const float* boff, float* offset_out,
                        uint8_t* wtiles, cudaStream_t st, float* mask_out) {
  cv::Params P;
  const int O = (mask_out ? 3 : 2) * g.N;
  if (!conv_fwd_shifted(g, O) && conv_small_supported(g, O))
    return conv_small_forward(g, O, xt, woff, boff, offset_out, wtiles, st, mask_out);
  if (!conv_params(g, cv::MODE_FWD, &P, O)) {
    set_error("offset conv (shifted-view kernel): shape not supported");
    return DCN_ERR_UNSUPPORTED;
  }
  int rc;
  if ((rc = conv_weight_tiles(P, 0, woff, wtiles, st))) return rc;
  P.xt = xt;
  P.bias = boff;
  P.out = offset_out;
  P.wtiles = wtiles;
  const int sms = num_sms();
  if (mask_out)
    return conv_launch<cv::MODE_FWD, true>(P, P.num_tiles < sms ? P.num_tiles : sms, st, "conv_offset_mask_fwd_kernel",
                                           mask_out);
  return conv_launch<cv::MODE_FWD>(P, P.num_tiles < sms ? P.num_tiles : sms, st, "conv_offset_fwd_kernel");
}

// backward of the offset conv: gxt += dgrad (may be null), gwoff = wgrad (zeroed here).  goff = the gradient of the
// conv's O output channels [B, O, Ho, Wo] (grad_offset, or the modulated layer's 3N-channel gradient).
int conv_offset_backward(const Geo& g, int O, const float* xt, float* gxt, const float* goff, const float* woff,
                         float* gwoff, uint8_t* wtiles, cudaStream_t st) {
  cv::Params P;
  int rc;
  if (!conv_bwd_shifted(g, O) && g.C < 64 && conv_small_supported(g, O))
    return conv_small_backward(g, O, xt, gxt, goff, woff, gwoff, wtiles, st);
  const int sms = num_sms();
  if (gxt) {
    if (!conv_params(g, cv::MODE_DGRAD, &P, O)) {
      set_error("offset conv backward (shifted-view kernel): shape not supported");
      return DCN_ERR_UNSUPPORTED;
    }
    if ((rc = conv_weight_tiles(P, 1, woff, wtiles, st))) return rc;
    P.gxt = gxt;
    P.goff = goff;
    P.wtiles = wtiles;
    if ((rc = conv_launch<cv::MODE_DGRAD>(P, P.num_tiles < sms ? P.num_tiles : sms, st, "conv_offset_dgrad_kernel")))
      return rc;
  }
  if (!conv_params(g, cv::MODE_WGRAD, &P, O)) {
    set_error("offset conv weight gradient (shifted-view kernel): shape not supported");
    return DCN_ERR_UNSUPPORTED;
  }
  DCN_CUDA_TRY(cudaMemsetAsync(gwoff, 0, sizeof(float) * (size_t)P.O * P.C * P.kh * P.kw, st));
  P.xt = xt;
  P.goff = goff;
  P.gw = gwoff;
  P.w_nchunks = sms / P.nslab;
  if (P.w_nchunks < 1) P.w_nchunks = 1;
  if (P.w_nchunks > P.num_tiles) P.w_nchunks = P.num_tiles;
  return conv_launch<cv::MODE_WGRAD>(P, P.nslab * P.w_nchunks, st, "conv_offset_wgrad_kernel");
}

}  // namespace dcn
