// dcn_umma_bwd_data.cu — grad_x and grad_offset on the tensor path (both column layouts).
//
// The autograd of train.py:102-134 (SURVEY.md A.4) as ONE kernel per 128-row tile:
//   GEMM-1    gA[rows, j] = gout[rows, :] * Wm[:, j]              (tcgen05.mma, TMEM accumulator)
//   scatter   grad_x[corner] += w_corner * gA                     (red.global.add.f32, coalesced:
//                                                                   32 lanes = 32 contiguous channels
//                                                                   of the channels-last grad copy)
//   coord     g_ix, g_iy = sum_c gA * d(sample)/d(ix, iy)         (butterfly warp-shuffle
//                                                                   reduce-scatter, then one
//                                                                   red.global per column)
// gA never leaves TMEM/registers, and a TMEM lane IS a channel:
//   Torch layout  (train.py:129-131): D[rows, j] = g[rows, :] * Wm^T; tile rows are ordered
//                 (class instance, channel), so lane l holds, for every column j, the gradient of
//                 sample (channel base(j) + l, sampling point q(r0, j)) — dcn_umma_common.cuh:Tiling.
//                 Resident operand A = converted grad_out rows, streamed operand B = Wm^T.
//   Jittor layout (deform_conv.py:72-73): the transposed product D[j, pixels] = Wm^T * g^T; lane l
//                 of column block jb is column j = 128*jb + l = (tap j / C, channel j % C), the
//                 TMEM columns are 128 consecutive output pixels.  Streamed operand A = Wm^T,
//                 resident operand B = converted grad_out pixels.
//
// Warp roles (640 or 704 threads, 1 CTA / SM, persistent over row tiles):
//   warps  0-15  scatter / coord-grad epilogue (quarter = w % 4 of the TMEM lanes, w / 4 = column part)
//   warp   16    MMA issuer          warp 17  loader: lane 0 streams the Wm^T tiles, lane 1 the staged
//                grad_out tiles (cp.async.bulk)
//   warps 18-19 / 18-21  plan: offsets -> bit-exact coordinate chain -> scatter entries (2-deep ring)
// The grad_out operand is never converted here: staging kernels (gout_tiles_torch_kernel — Torch-layout
// rows are R floats apart — and gout_tiles_pix_kernel for the pixel-row layouts) pre-build every tile's
// UMMA images once per backward pass.
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "dcn_umma.h"
#include "dcn_umma_common.cuh"

namespace dcn {

using namespace ptx;

namespace bd {

constexpr int kScatWarps = 16;
constexpr int kMmaWarp = kScatWarps, kLoadWarp = kScatWarps + 1;
constexpr int kFirstPlanWarp = kScatWarps + 2;
// Role layout by the number of plan warps PW:
//   <= 128 plan entries per block (Torch layout with Gt = 64, Jittor layout with C >= 64): PW = 2 = 20 warps,
//                 i.e. 5 per SM sub-partition and 96 registers per thread for the scatter loop;
//   more sampling points per block: PW = 4, 22 warps, 80 registers.
__host__ __device__ constexpr int threads_of(int pw) { return (kFirstPlanWarp + pw) * 32; }
constexpr int kPlanPerThread = 8;
__host__ __device__ constexpr int plan_max_of(int pw) { return pw * 32 * kPlanPerThread; }
constexpr uint32_t kGImg = 128 * 64 * 2;                 // one bf16 image of a grad_out K block

// what the scatter warps need for one (class instance, column): 16 bytes = ONE shared-memory load.
// The framed staging layout (dcn_umma_common.cuh) makes the four corners base + {0, C, pitch,
// pitch + C} for the value loads AND the scatter alike, with no validity mask; the corner weights
// are re-formed from (fx, fy) in registers exactly as the forward pass forms them.
struct __align__(16) ScatEntry {
  uint32_t base;  // BYTE offset (float image) of the top-left corner inside the framed image
  float fx, fy;
  uint32_t gidx;  // index of the grad_offset element that receives g_iy (the channel moving the row);
                  // g_ix goes ix_delta further (Params).  kDeadEntry: dead entry (padding column / row of
                  // no instance / no corner inside the image): nothing to scatter, sample 0.
                  // Unsigned: grad_offset has B * 2N * HW elements, up to 2^32 - 2 under make_geo's bound
                  // B * N * HW < 2^31, so a live index is at most 2^32 - 3 and never meets the sentinel
};
constexpr uint32_t kDeadEntry = 0xffffffffu;

struct Params {
  Geo g;
  Tiling t;
  const void* xt;        // channels-last x, float or bfloat16 (coordinate gradient needs the corner values)
  float* gxt;            // channels-last grad_x accumulator (zeroed), may be null
  const float* off;
  const void* gout;      // float or bfloat16
  const uint8_t* wtiles; // [cblocks][OB][hi|lo][ncols x 64] K-major SW128 images of Wm^T
  const uint8_t* gtiles; // Torch layout: [tile][OB][hi|lo][128 rows x 64 o] K-major SW128 images of grad_out
  float* gb_fused;       // staging kernel only (Torch layout): grad_bias [O] accumulated from the tiles it stages
                         // (zeroed by the caller), or null
  int row_v;             // staging kernel only: 0 = rows ordered (instance, channel) as this kernel wants them;
                         // V = 4 / 8: the forward-kernel order (channel / V, instance, channel % V) for MODE_WGRAD
  float* goff;           // grad_offset accumulators (zeroed)
  float scale_iy, scale_ix;  // chain-rule factors of the coordinate normalisation (1 for DCNv1)
  // Torch layout: t's row tiling, copied here by copy_row_tiling.  The kernels read it from these fields: their parameter
  // offsets keep the scatter loop's schedule (read from t, ptxas pairs the constant loads differently and the fused
  // Torch kernels spill more).
  int Gt, Rt, chunks, num_inst;
  int num_tiles;         // row tiles: t.num_tiles (Torch), or B * pix_blocks
  FastDiv divR, divChunks;
  int pix_blocks;        // pixel-row layouts: ceil(HW / ncols) pixel blocks per image
  int ix_delta;          // distance, in floats, from a tap's g_iy slot in grad_offset to its g_ix slot
  int ncols;             // TMEM columns per accumulator block: 128 or 64 (Torch: j's; Jittor: pixels)
  int cblocks;           // blocks per tile: Torch ceil(K / ncols) column blocks, Jittor ceil(K / 128) lane blocks
  int OB;                // ceil(O / 64) K blocks of the GEMM
  int plan_cap;          // entries per plan buffer = Rt * ncols
  // fused weight gradient (Torch layout, O <= 256 while the grad_out tile fits): the scatter warps also form the blended
  // sample S = sum_k w_k v_k they already hold the corners of, store it as a bf16 hi/lo B
  // operand, and a second accumulator set collects gW[o, j] += g^T S over all tiles of the CTA
  int fuse_w;            // 0 / 1
  int o_halves;          // Torch layout, fused: 128-channel halves of the o axis (1, or 2 when 128 < O <= 256), one gW
                         // accumulator set per half
  int o_cols;            // Jittor layout, fused: TMEM columns of one gW accumulator block = O rounded up to 16
  float* gw;             // [O, K], zeroed
  int nslices, nchunks, cb_per_slice;  // CTA = (slice of column blocks, chunk of tiles)
  int g_imgs;            // grad_out images the MMAs address per tile: OB, or 2 when fused (M = 128 of the o axis)
  int g_nbuf;            // 1 or 2 buffers of the converted grad_out tile (2 hides the conversion of the next tile)
  uint32_t g_img;        // bytes of one bf16 image of the resident grad_out operand (rows x 128 B)
  uint32_t w_stage;      // bytes of one Wm^T stage (hi | lo)
  uint32_t tmem_cols;
  // fused kernels give every CTA a FIXED slice of column blocks for all its tiles: when the slice's Wm^T
  // images (cb_per_slice * OB stages) fit in shared memory they are loaded ONCE and stay resident instead of
  // being re-streamed from L2 for every tile through the 2-stage ring
  int w_resident;        // 0 = ring of w_ring stages, else the number of resident stages
  int w_ring;            // 2, or 1 when only that leaves room for the second grad_out buffer (the loads of the
                         // next block then serialise with its MMAs, but both hide behind the previous scatter pass)
};

struct PlanWork {
  float ox, oy;
  int h, w, n, chan_base, valid;
  uint32_t gidx;  // ScatEntry::gidx
  float mk;  // MOD: the mask value, loaded on the same prefetch as the offsets
};

template <int VARIANT, bool PLAIN = false, bool MOD = false>
__device__ __forceinline__ void plan_prepare(const Params& P, int tile, int cb, int e, PlanWork& pw,
                                             const float* __restrict__ mask = nullptr) {
  const Geo& g = P.g;
  pw.valid = 0;
  pw.ox = pw.oy = 0.f;
  pw.h = pw.w = pw.n = pw.chan_base = 0;
  pw.gidx = kDeadEntry;
  uint32_t p, n, h, w;
  int b;
  if (VARIANT == DCN_VARIANT_TORCH) {
    const int il = e >> (P.ncols == 128 ? 7 : 6), cc = e & (P.ncols - 1), j = cb * P.ncols + cc;  // ncols = 64 | 128
    const TileRowInfo ri = decode_inst(P, tile * P.Rt + il);
    if (!ri.valid || j >= g.K) return;
    uint32_t cbase, q;
    P.t.divP.divmod((uint32_t)(ri.r0 * g.K + j), cbase, q);
    P.t.divN.divmod(q, p, n);
    pw.chan_base = (int)cbase * P.t.G + ri.chunk * P.Gt;
    b = ri.b;
  } else {
    // entry (tap slot tl of lane block cb, pixel column cc)
    const int tl = e >> (P.ncols == 128 ? 7 : 6), cc = e & (P.ncols - 1);
    b = tile / P.pix_blocks;
    p = (uint32_t)((tile - b * P.pix_blocks) * P.ncols + cc);
    n = P.t.divC.div((uint32_t)(cb * 128)) + (uint32_t)tl;
    if ((int)p >= g.HW || (int)n >= g.N) return;
  }
  P.t.divWo.divmod(p, h, w);
  pw.h = (int)h;
  pw.w = (int)w;
  pw.n = (int)n;
  if (PLAIN) {
    pw.gidx = 0;  // live entry; a plain problem has no offsets and no coordinate gradient
  } else {
    // target of g_iy, formed in 64 bits: it passes 2^31 in the tail of a large batch
    const size_t gi = ((size_t)b * 2 * g.N + off_row_ch(g, (int)n)) * g.HW + p;
    DCN_DEV_ASSERT(gi < (size_t)g.B * 2 * g.N * g.HW);
    pw.gidx = (uint32_t)gi;
    const float* ob = P.off + (size_t)b * 2 * g.N * g.HW;
    pw.ox = __ldg(ob + (size_t)off_row_ch(g, (int)n) * g.HW + p);
    pw.oy = __ldg(ob + (size_t)off_col_ch(g, (int)n) * g.HW + p);
  }
  if constexpr (MOD) {
    static_assert(VARIANT != DCN_VARIANT_TORCH && !PLAIN, "modulation exists for the pixel-row DCNv1 layout only");
    DCN_DEV_ASSERT(((size_t)b * g.N + n) * g.HW + p < (size_t)g.B * g.N * g.HW);
    pw.mk = __ldg(mask + ((size_t)b * g.N + n) * g.HW + p);
  }
  pw.valid = 1;
}

// PLAIN: the one pixel a (pixel, tap) pair reads / its gradient goes to (dcn_umma_common.cuh:plain_base)
__device__ __forceinline__ ScatEntry plan_finish_plain(const Geo& g, const PlanWork& pw) {
  ScatEntry e;
  int base = xt_null_base(g);
  e.fx = e.fy = 0.f;
  e.gidx = kDeadEntry;
  if (pw.valid) {
    bool inside;
    base = plain_base(g, pw.h, pw.w, pw.n, inside);
    if (inside) e.gidx = 0;
  }
  e.base = 4u * (uint32_t)(base + pw.chan_base);
  return e;
}

__device__ __forceinline__ ScatEntry plan_finish(const Geo& g, const PlanWork& pw) {
  ScatEntry e;
  int base = xt_null_base(g);
  e.fx = e.fy = 0.f;
  e.gidx = kDeadEntry;
  if (pw.valid) {
    const Tap tp = tap_of(g, pw.h, pw.w, pw.n, pw.ox, pw.oy);
    bool inside;
    base = xt_corner_base(g, tp.y0, tp.x0, inside);
    if (inside) {
      e.fx = tp.fx;
      e.fy = tp.fy;
      e.gidx = pw.gidx;
    }
  }
  e.base = 4u * (uint32_t)(base + pw.chan_base);
  return e;
}

// Butterfly reduce-scatter of NV values over the lanes that differ in lane bits S, S/2, ... (log2 NV bits): at the
// step over bit s a lane keeps the half of its values that bit selects and adds the partner's copy of that half.
// Afterwards v[0] is the sum over those lanes of value index (lane bit S, ..., lane bit 2S/NV) read as a binary number.
template <int S, int NV>
__device__ __forceinline__ void reduce_scatter(float (&v)[NV], unsigned mask, int lane) {
#pragma unroll
  for (int s = S, n = NV / 2; n >= 1; s >>= 1, n >>= 1) {
    const bool up = (lane & s) != 0;
#pragma unroll
    for (int k = 0; k < n; ++k) {
      const float send = up ? v[k] : v[k + n];
      const float keep = up ? v[k + n] : v[k];
      v[k] = keep + __shfl_xor_sync(mask, send, s);
    }
  }
}

// RW = lanes that share one sampling point (32, or 16 when only 16 channels do)
// BF  = bf16 operand mode: x / weight / grad_out are bfloat16, one image per operand, one MMA per K step
// PLAIN = backward of a regular convolution (the companion offset conv, Geo::plain): one exact pixel per column
//         instead of four weighted corners — one red.global per column, the "sample" of the fused weight gradient
//         is the pixel itself, no coordinate gradient
// MOD = modulated DCNv1 (DCNv2; pixel-row layout): the plan ring carries one mask value per entry beside the scatter
//       entries; per column the accumulator value gs is scaled by it once (grad_x and grad_offset then follow unchanged
//       in form), a third per-column partial gs * bilinear sample is reduced over the lanes of the sampling point into
//       ONE red.global per column of grad_mask, and the fused weight gradient's sample operand is m * sample.
//       mask / gmask [B, N, Ho, Wo] (gmask zeroed) are trailing kernel arguments rather than Params fields: Params is
//       also passed by value to gout_tiles_torch_kernel, whose following argument would move if Params grew.
template <int VARIANT, int RW, bool FUSE, bool BF, int PW, bool PLAIN = false, bool MOD = false>
__global__ void __launch_bounds__(threads_of(PW), 1) bwd_data_kernel(const __grid_constant__ Params P,
                                                                     const float* __restrict__ mask,
                                                                     float* __restrict__ gmask) {
  constexpr int NIMG = BF ? 1 : 2;
  typedef typename std::conditional<BF, __nv_bfloat16, float>::type XT;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const Geo& g = P.g;
  // carve-up: [grad_out tile: OB x (hi | lo)] [2 Wm^T stages] [plan x2] [barriers]
  // [g_nbuf buffers x OB real images][zero images completing the M = 128 o-axis when fused]
  uint8_t* gtile = smem;
  const uint32_t g_buf = (uint32_t)P.OB * NIMG * P.g_img;
  const uint32_t g_zero_off = (uint32_t)P.g_nbuf * g_buf;
  uint8_t* wstage = gtile + g_zero_off + (size_t)(P.g_imgs - P.OB) * NIMG * P.g_img;
  // fused: 2 buffers of the sample operand S, each [hi | lo][128 tile rows x 64 columns], MN-major
  // (the 64 columns of a block are contiguous in a row, so a lane stores 8 columns with one STS.128)
  uint8_t* sbuf = wstage + (size_t)(P.w_resident ? P.w_resident : P.w_ring) * P.w_stage;
  const uint32_t s_img = 128u * 128u, s_buf = FUSE ? NIMG * s_img : 0u;
  ScatEntry* plan = reinterpret_cast<ScatEntry*>(sbuf + 2 * (size_t)s_buf);
  // MOD: [2 x plan_cap] mask values, parallel to the plan ring
  float* mplan = reinterpret_cast<float*>(plan + 2 * P.plan_cap);
  uint64_t* bars = MOD ? reinterpret_cast<uint64_t*>(mplan + 2 * P.plan_cap)
                       : reinterpret_cast<uint64_t*>(plan + 2 * P.plan_cap);
  uint64_t* wfull = bars;        // [2]
  uint64_t* wempty = bars + 2;   // [2]
  uint64_t* tfull = bars + 4;    // [2]
  uint64_t* tempty = bars + 6;   // [2]
  uint64_t* pfull = bars + 8;    // [2]
  uint64_t* pempty = bars + 10;  // [2]
  uint64_t* gfull = bars + 12;   // [2] converted grad_out tile
  uint64_t* gempty = bars + 14;  // [2]
  uint64_t* sfull = bars + 16;   // [2] sample operand written (fused)
  uint64_t* sempty = bars + 18;  // [2]
  uint64_t* dfull = bars + 20;   // [1] weight-gradient accumulators final
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 21);
  {
    // the host sizes the allocation with little alignment slack when shared memory is tight: fail loudly
    // rather than run past the end
    uint32_t dyn;
    asm volatile("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn));
    if (smem_u32(tmem_slot + 1) - smem_u32(smem_raw) > dyn) __trap();
  }

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ncols = P.ncols;

  if (tid == 0) {
    for (int a = 0; a < 2; ++a) {
      mbar_init(&wfull[a], 1);
      mbar_init(&wempty[a], 1);
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], kScatWarps);
      mbar_init(&pfull[a], PW);
      mbar_init(&pempty[a], kScatWarps);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&gfull[a], 1);
      mbar_init(&gempty[a], 1);
      mbar_init(&sfull[a], kScatWarps);
      mbar_init(&sempty[a], 1);
    }
    mbar_init(dfull, 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(tmem_slot)),
                 "r"(P.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (FUSE) {
    // images beyond OB (the o >= 64*OB half of the M = 128 weight-gradient MMA) stay zero
    const uint32_t zero_end = g_zero_off + (uint32_t)(P.g_imgs - P.OB) * NIMG * P.g_img;
    for (uint32_t i = g_zero_off + tid * 16; i < zero_end; i += threads_of(PW) * 16)
      *reinterpret_cast<uint4*>(gtile + i) = make_uint4(0, 0, 0, 0);
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const size_t img_stride = xt_image_stride(g);
  // (tile, block) pairs of this CTA: all blocks of every gridDim-th tile, or — fused — one slice
  // of the column blocks for one chunk of the tiles (the gW accumulators live in TMEM throughout)
  int tile0, tile_step, cb0, cb1;
  if (!FUSE) {
    tile0 = blockIdx.x;
    tile_step = gridDim.x;
    cb0 = 0;
    cb1 = P.cblocks;
  } else {
    const int slice = blockIdx.x % P.nslices;
    tile0 = blockIdx.x / P.nslices;
    tile_step = P.nchunks;
    cb0 = slice * P.cb_per_slice;
    cb1 = min(P.cblocks, cb0 + P.cb_per_slice);
  }
  const uint32_t d2_base = tmem_base + 2u * (uint32_t)P.ncols;  // gW accumulators after the 2 gA buffers

  if (warp < kScatWarps) {
    // ================================================================ scatter + coordinate gradient
    const int quarter = warp & 3, part = warp >> 2;
    const int m = quarter * 32 + lane;          // TMEM lane
    const int cols_per_part = ncols >> 2;       // 32 or 16
    const unsigned grp_mask = RW == 32 ? 0xffffffffu : (0xffffu << (lane & 16));
    const int gl = lane & (RW - 1);             // lane inside its reduction group
    int acc = 0, pb = 0, sb = 0;
    uint32_t acc_phase = 0, pphase = 0, sphase = 0;
    // byte distances to the east / south corner in the framed images (x: float or bfloat16; grad: float)
    const int dg1 = 4 * g.C, dg2 = 4 * xt_row_pitch(g);
    const int dx1 = (int)sizeof(XT) * g.C, dx2 = (int)sizeof(XT) * xt_row_pitch(g);
    for (int tile = tile0; tile < P.num_tiles; tile += tile_step) {
      // Torch: lane = (class instance il, channel i_lo) for the whole tile
      int slot = 0, chan = 0, bimg = 0;
      if (VARIANT == DCN_VARIANT_TORCH) {
        slot = m / P.Gt;
        chan = m - slot * P.Gt;
        bimg = decode_inst(P, tile * P.Rt + slot).b;
      } else {
        bimg = tile / P.pix_blocks;
      }
      for (int cb = cb0; cb < cb1; ++cb) {
        int mrow = 0;  // MOD: grad_mask index of this block's pixel column 0 for the lane's tap
        if (VARIANT != DCN_VARIANT_TORCH) {
          // Jittor: lane = column j = 128*cb + m = (tap j / C, channel j % C); slot = tap inside the block
          const int j = cb * 128 + m, n = j / g.C;
          chan = j - n * g.C;
          slot = n - (cb * 128) / g.C;
          if (MOD) mrow = (bimg * g.N + n) * g.HW + (tile - bimg * P.pix_blocks) * ncols;
        }
        // byte-addressed image bases: address = base + zero-extended 32-bit offset (2 instructions)
        const char* ximg =
            reinterpret_cast<const char*>(reinterpret_cast<const XT*>(P.xt) + (size_t)bimg * img_stride + chan);
        char* gimg = P.gxt ? reinterpret_cast<char*>(P.gxt + (size_t)bimg * img_stride + chan) : nullptr;
        mbar_wait_relaxed(&tfull[acc], acc_phase, 32);
        mbar_wait_relaxed(&pfull[pb], pphase, 32);
        if (FUSE) mbar_wait_relaxed(&sempty[sb], sphase ^ 1, 32);
        tc_fence_after();
        // fused: this lane's row m of the sample operand (8-row groups of 1024 B, 128 B per row)
        uint8_t* s_row = sbuf + (size_t)sb * s_buf + (size_t)(m >> 3) * 1024 + (m & 7) * 128;
        const ScatEntry* pl = plan + pb * P.plan_cap + slot * ncols;
        const float* mkp = mplan + pb * P.plan_cap + slot * ncols;  // MOD only
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * ncols);
        // (reducing the coordinate gradient in batches of 16 columns was measured slower: DESIGN.md §5)
        // MOD: one grad_mask RED per column, after an 8-value reduce-scatter over the RW lanes of the sampling points
        auto mask_red = [&](const int cc, float (&part_m)[8]) {
          if (RW == 32) {
#pragma unroll
            for (int k = 0; k < 8; ++k) part_m[k] += __shfl_xor_sync(0xffffffffu, part_m[k], 16);
          }
          reduce_scatter<8>(part_m, grp_mask, lane);
          part_m[0] += __shfl_xor_sync(grp_mask, part_m[0], 1);
          if ((gl & 1) == 0 && (RW == 16 || lane < 16)) {
            const int col = cc + ((gl >> 1) & 7);
            DCN_DEV_ASSERT(pl[col].gidx == kDeadEntry || (size_t)(mrow + col) < (size_t)g.B * g.N * g.HW);
            if (pl[col].gidx != kDeadEntry && part_m[0] != 0.f) atomicAdd(gmask + mrow + col, part_m[0]);
          }
        };
        // one pass = 8 columns whose accumulator values are already in registers
        auto pass = [&](const int cc, const uint32_t* raw) {
          float part_g[16];  // [0 .. 8) g_ix of the batch's columns, [8 .. 16) g_iy
          float part_m[8];   // MOD: gA * sample of the batch's columns
          float smp8[8];     // fused: the 8 samples of this row
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const float ga = __uint_as_float(raw[u]);
            const float mkv = MOD ? mkp[cc + u] : 1.f;
            const float gs = MOD ? ga * mkv : ga;
            const uint4 e4 = *reinterpret_cast<const uint4*>(pl + cc + u);  // {base, fx, fy, gidx}
            const float fx = __uint_as_float(e4.y), fy = __uint_as_float(e4.z);
            // entry offsets are bytes of the float grad image; the bf16 x image is half as wide
            constexpr int XS = BF ? 1 : 0;
            const char* xp = ximg + (e4.x >> XS);
            const float v0 = (float)__ldg(reinterpret_cast<const XT*>(xp));
            if (PLAIN) {
              if (gimg && e4.w != kDeadEntry) atomicAdd(reinterpret_cast<float*>(gimg + e4.x), gs);
              part_g[u] = part_g[8 + u] = 0.f;
              if (FUSE) smp8[u] = v0;   // dead entries read the all-zero frame-only block
              continue;
            }
            const float v1 = (float)__ldg(reinterpret_cast<const XT*>(xp + dx1));
            const float v2 = (float)__ldg(reinterpret_cast<const XT*>(xp + dx2));
            const float v3 = (float)__ldg(reinterpret_cast<const XT*>(xp + dx2 + dx1));
            // corner weights as the forward pass forms them (dcn_common.cuh:corner_weights)
            const float ex = __fsub_rn(1.0f, fx), sy = __fsub_rn(1.0f, fy);
            const float w0 = __fmul_rn(sy, ex), w1 = __fmul_rn(sy, fx), w2 = __fmul_rn(fy, ex),
                        w3 = __fmul_rn(fy, fx);
            if (gimg && e4.w != kDeadEntry) {
              // coalesced red.global.add.f32 x4; a corner outside the image lands on the frame
              char* gp = gimg + e4.x;
              atomicAdd(reinterpret_cast<float*>(gp), gs * w0);
              atomicAdd(reinterpret_cast<float*>(gp + dg1), gs * w1);
              atomicAdd(reinterpret_cast<float*>(gp + dg2), gs * w2);
              atomicAdd(reinterpret_cast<float*>(gp + dg2 + dg1), gs * w3);
            }
            part_g[u] = gs * ((v1 - v0) * sy + (v3 - v2) * fy);
            part_g[8 + u] = gs * ((v2 - v0) * ex + (v3 - v1) * fx);
            // the sample itself (same blend order as the forward pass)
            if (MOD) {
              const float bil = fmaf(v3, w3, fmaf(v2, w2, fmaf(v1, w1, v0 * w0)));
              part_m[u] = ga * bil;
              if (FUSE) smp8[u] = mkv * bil;
            } else if (FUSE) {
              smp8[u] = fmaf(v3, w3, fmaf(v2, w2, fmaf(v1, w1, v0 * w0)));
            }
          }
          if (FUSE) {
            // columns cc..cc+7 of row m: one 16-byte chunk of the MN-major operand, swizzled by m % 8
            uint4 hi, lo;
            split_pair(smp8[0], smp8[1], hi.x, lo.x);
            split_pair(smp8[2], smp8[3], hi.y, lo.y);
            split_pair(smp8[4], smp8[5], hi.z, lo.z);
            split_pair(smp8[6], smp8[7], hi.w, lo.w);
            const uint32_t so = (uint32_t)((((cc >> 3) ^ m) & 7) << 4);
            *reinterpret_cast<uint4*>(s_row + so) = hi;
            if (!BF) *reinterpret_cast<uint4*>(s_row + s_img + so) = lo;
          }
          if (PLAIN) return;
          if (MOD) mask_red(cc, part_m);
          // butterfly reduce-scatter over the RW lanes that share the sampling points:
          // afterwards lane gl (< 16) holds the total of value index gl
          if (RW == 32) {
#pragma unroll
            for (int k = 0; k < 16; ++k) part_g[k] += __shfl_xor_sync(0xffffffffu, part_g[k], 16);
          }
          reduce_scatter<8>(part_g, grp_mask, lane);
          if (gl < 16 && (RW == 16 || lane < 16)) {
            const int vi = gl & 15, col = vi & 7;
            const uint32_t gidx = pl[cc + col].gidx;
            DCN_DEV_ASSERT(gidx == kDeadEntry || (size_t)gidx + (size_t)P.ix_delta < (size_t)g.B * 2 * g.N * g.HW);
            // lower half of the values: g_ix -> the column-moving offset channel; upper half: g_iy -> the row-moving one
            if (gidx != kDeadEntry && part_g[0] != 0.f)
              atomicAdd(P.goff + (size_t)gidx + (vi < 8 ? (size_t)P.ix_delta : 0),
                        part_g[0] * (vi < 8 ? P.scale_ix : P.scale_iy));
          }
        };
        // PAIR mode (all 32 lanes of the warp share the sampling points): lane pairs (2k, 2k+1) swap half of their
        // accumulator values, so that a thread owns TWO adjacent channels for FOUR of the 8 columns.  Every corner
        // is then one 8-byte load and one red.global.add.v2.f32, entries and weights are needed for 4 columns
        // instead of 8, and the coordinate gradient (summed over the thread's two channels first) is an 8-value
        // reduce-scatter over the 16 lanes of equal parity: 15 shuffles instead of 31.  Per 8 columns the warp
        // issues 16 + 16 + 4 + 19 load/store-unit instructions instead of 32 + 33 + 8 + 31.
        auto pass2 = [&](const int cc, const uint32_t* raw) {
          const int odd = lane & 1;
          float ga[4], gb[4];  // accumulator values of the lower / upper channel of the pair, columns cu0 .. cu0+3
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const float own = __uint_as_float(odd ? raw[u + 4] : raw[u]);
            const float send = __uint_as_float(odd ? raw[u] : raw[u + 4]);
            const float got = __shfl_xor_sync(0xffffffffu, send, 1);
            ga[u] = odd ? got : own;
            gb[u] = odd ? own : got;
          }
          const int cu0 = cc + 4 * odd;
          // image pointers of the channel PAIR
          const char* xpair = ximg - odd * (int)sizeof(XT);
          char* gpair = gimg ? gimg - odd * 4 : nullptr;
          float part_g[8];  // [0..3] g_ix of this thread's 4 columns (both channels), [4..7] g_iy
          float sa[4], sb2[4];
          float part_m[4];  // MOD: gA * sample of this thread's 4 columns (both channels)
          float4 mk4 = make_float4(1.f, 1.f, 1.f, 1.f);
          if (MOD) mk4 = *reinterpret_cast<const float4*>(mkp + cu0);
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const uint4 e4 = *reinterpret_cast<const uint4*>(pl + cu0 + u);  // {base, fx, fy, gidx}
            const float fx = __uint_as_float(e4.y), fy = __uint_as_float(e4.z);
            constexpr int XS = BF ? 1 : 0;
            const char* xp = xpair + (e4.x >> XS);
            // the south-east corner's channel pair still lies inside this image of the framed copies
            DCN_DEV_ASSERT((size_t)(e4.x >> 2) + (size_t)(PLAIN ? 0 : xt_row_pitch(g) + g.C) + (size_t)(chan - odd) + 2 <= img_stride);
            float2 v0, v1, v2, v3;
            if (PLAIN) {
              if (BF) {
                const uint32_t r0 = __ldg(reinterpret_cast<const uint32_t*>(xp));
                v0 = make_float2(__uint_as_float(r0 << 16), __uint_as_float(r0 & 0xffff0000u));
              } else {
                v0 = __ldg(reinterpret_cast<const float2*>(xp));
              }
              if (gpair && e4.w != kDeadEntry) atomicAdd(reinterpret_cast<float2*>(gpair + e4.x), make_float2(ga[u], gb[u]));
              part_g[u] = part_g[4 + u] = 0.f;
              if (FUSE) {
                sa[u] = v0.x;   // dead entries read the all-zero frame-only block
                sb2[u] = v0.y;
              }
              continue;
            }
            if (BF) {
              const uint32_t r0 = __ldg(reinterpret_cast<const uint32_t*>(xp));
              const uint32_t r1 = __ldg(reinterpret_cast<const uint32_t*>(xp + dx1));
              const uint32_t r2 = __ldg(reinterpret_cast<const uint32_t*>(xp + dx2));
              const uint32_t r3 = __ldg(reinterpret_cast<const uint32_t*>(xp + dx2 + dx1));
              v0 = make_float2(__uint_as_float(r0 << 16), __uint_as_float(r0 & 0xffff0000u));
              v1 = make_float2(__uint_as_float(r1 << 16), __uint_as_float(r1 & 0xffff0000u));
              v2 = make_float2(__uint_as_float(r2 << 16), __uint_as_float(r2 & 0xffff0000u));
              v3 = make_float2(__uint_as_float(r3 << 16), __uint_as_float(r3 & 0xffff0000u));
            } else {
              v0 = __ldg(reinterpret_cast<const float2*>(xp));
              v1 = __ldg(reinterpret_cast<const float2*>(xp + dx1));
              v2 = __ldg(reinterpret_cast<const float2*>(xp + dx2));
              v3 = __ldg(reinterpret_cast<const float2*>(xp + dx2 + dx1));
            }
            const float ex = __fsub_rn(1.0f, fx), sy = __fsub_rn(1.0f, fy);
            const float w0 = __fmul_rn(sy, ex), w1 = __fmul_rn(sy, fx), w2 = __fmul_rn(fy, ex),
                        w3 = __fmul_rn(fy, fx);
            if (MOD) {
              const float mkv = u == 0 ? mk4.x : (u == 1 ? mk4.y : (u == 2 ? mk4.z : mk4.w));
              const float bila = fmaf(v3.x, w3, fmaf(v2.x, w2, fmaf(v1.x, w1, v0.x * w0)));
              const float bilb = fmaf(v3.y, w3, fmaf(v2.y, w2, fmaf(v1.y, w1, v0.y * w0)));
              part_m[u] = ga[u] * bila + gb[u] * bilb;
              ga[u] *= mkv;
              gb[u] *= mkv;
              if (FUSE) {
                sa[u] = mkv * bila;
                sb2[u] = mkv * bilb;
              }
            }
            if (gpair && e4.w != kDeadEntry) {
              char* gp = gpair + e4.x;
              atomicAdd(reinterpret_cast<float2*>(gp), make_float2(ga[u] * w0, gb[u] * w0));
              atomicAdd(reinterpret_cast<float2*>(gp + dg1), make_float2(ga[u] * w1, gb[u] * w1));
              atomicAdd(reinterpret_cast<float2*>(gp + dg2), make_float2(ga[u] * w2, gb[u] * w2));
              atomicAdd(reinterpret_cast<float2*>(gp + dg2 + dg1), make_float2(ga[u] * w3, gb[u] * w3));
            }
            part_g[u] = ga[u] * ((v1.x - v0.x) * sy + (v3.x - v2.x) * fy) +
                        gb[u] * ((v1.y - v0.y) * sy + (v3.y - v2.y) * fy);
            part_g[4 + u] = ga[u] * ((v2.x - v0.x) * ex + (v3.x - v1.x) * fx) +
                            gb[u] * ((v2.y - v0.y) * ex + (v3.y - v1.y) * fx);
            if (FUSE && !MOD) {
              sa[u] = fmaf(v3.x, w3, fmaf(v2.x, w2, fmaf(v1.x, w1, v0.x * w0)));
              sb2[u] = fmaf(v3.y, w3, fmaf(v2.y, w2, fmaf(v1.y, w1, v0.y * w0)));
            }
          }
          if (FUSE) {
            // 4 columns of the two rows m & ~1, m | 1: the lower / upper 8 bytes of the rows' 16-byte chunk
            const int ma = m & ~1;
            uint8_t* ra = sbuf + (size_t)sb * s_buf + (size_t)(ma >> 3) * 1024 + (ma & 7) * 128;
            const uint32_t soa = (uint32_t)((((cc >> 3) ^ ma) & 7) << 4) + 8u * odd;
            const uint32_t sob = (uint32_t)((((cc >> 3) ^ (ma + 1)) & 7) << 4) + 8u * odd;
            uint2 hi, lo;
            split_pair(sa[0], sa[1], hi.x, lo.x);
            split_pair(sa[2], sa[3], hi.y, lo.y);
            *reinterpret_cast<uint2*>(ra + soa) = hi;
            if (!BF) *reinterpret_cast<uint2*>(ra + s_img + soa) = lo;
            split_pair(sb2[0], sb2[1], hi.x, lo.x);
            split_pair(sb2[2], sb2[3], hi.y, lo.y);
            *reinterpret_cast<uint2*>(ra + 128 + sob) = hi;
            if (!BF) *reinterpret_cast<uint2*>(ra + 128 + s_img + sob) = lo;
          }
          if (PLAIN) return;
          // reduce-scatter of the 8 values over the 16 lanes of equal parity (lane bits 4..1)
#pragma unroll
          for (int k = 0; k < 8; ++k) part_g[k] += __shfl_xor_sync(0xffffffffu, part_g[k], 16);
          reduce_scatter<8>(part_g, 0xffffffffu, lane);
          if (lane < 16) {
            // value index: lane bit 3 -> component (0 g_ix, 1 g_iy), bits 2..1 -> column inside the thread's four
            const int vi = (lane >> 1) & 7, col = cu0 + (vi & 3);
            const uint32_t gidx = pl[col].gidx;
            DCN_DEV_ASSERT(gidx == kDeadEntry || (size_t)gidx + (size_t)P.ix_delta < (size_t)g.B * 2 * g.N * g.HW);
            if (gidx != kDeadEntry && part_g[0] != 0.f)
              atomicAdd(P.goff + (size_t)gidx + (vi < 4 ? (size_t)P.ix_delta : 0),
                        part_g[0] * (vi < 4 ? P.scale_ix : P.scale_iy));
          }
          if (MOD) {
            // grad_mask: the 4 values over the 16 lanes of equal parity, then one RED per column
#pragma unroll
            for (int k = 0; k < 4; ++k) part_m[k] += __shfl_xor_sync(0xffffffffu, part_m[k], 16);
            reduce_scatter<8>(part_m, 0xffffffffu, lane);
            part_m[0] += __shfl_xor_sync(0xffffffffu, part_m[0], 2);
            if (lane < 16 && (lane & 2) == 0) {
              // lane bits 3..2 -> column inside the thread's four
              const int col = cu0 + ((lane >> 2) & 3);
              DCN_DEV_ASSERT(pl[col].gidx == kDeadEntry || (size_t)(mrow + col) < (size_t)g.B * g.N * g.HW);
              if (pl[col].gidx != kDeadEntry && part_m[0] != 0.f) atomicAdd(gmask + mrow + col, part_m[0]);
            }
          }
        };
        constexpr bool PAIR = RW == 32;
        // (fetching both passes' accumulator values up front with one x16 load lets the compiler overlap the
        // second pass's loads with the first pass's shuffles, but measured slower: 11.85 vs 11.36 ms)
        for (int cc = part * cols_per_part; cc < (part + 1) * cols_per_part; cc += 8) {
          uint32_t raw[8];
          asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                       : "=r"(raw[0]), "=r"(raw[1]), "=r"(raw[2]), "=r"(raw[3]), "=r"(raw[4]), "=r"(raw[5]),
                         "=r"(raw[6]), "=r"(raw[7])
                       : "r"(taddr + cc)
                       : "memory");
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if constexpr (PAIR) pass2(cc, raw);
          else pass(cc, raw);
        }
        tc_fence_before();
        if (FUSE) fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(&tempty[acc]);
          mbar_arrive(&pempty[pb]);
          if (FUSE) mbar_arrive(&sfull[sb]);
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
        pb ^= 1;
        if (pb == 0) pphase ^= 1;
        if (FUSE) {
          sb ^= 1;
          if (sb == 0) sphase ^= 1;
        }
      }
    }
    if (FUSE) {
      // ---- one-shot epilogue of the weight gradient: accumulators -> gW (red.global.add)
      mbar_wait_relaxed(dfull, 0);
      tc_fence_after();
      if (VARIANT == DCN_VARIANT_TORCH) {
        const int wcols = (cb1 - cb0) * ncols, per_part = (wcols + 3) >> 2;
        for (int hf = 0; hf < P.o_halves; ++hf) {
          const int o = hf * 128 + quarter * 32 + lane;
          const uint32_t taddr = d2_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(hf * P.cb_per_slice * ncols);
          for (int c0 = part * per_part; c0 < min(wcols, (part + 1) * per_part); c0 += 8) {
            uint32_t raw[8];
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                         : "=r"(raw[0]), "=r"(raw[1]), "=r"(raw[2]), "=r"(raw[3]), "=r"(raw[4]), "=r"(raw[5]),
                           "=r"(raw[6]), "=r"(raw[7])
                         : "r"(taddr + c0)
                         : "memory");
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            if (o < g.O) {
#pragma unroll
              for (int u = 0; u < 8; ++u) {
                const int j = cb0 * ncols + c0 + u;
                if (j < g.K) atomicAdd(P.gw + (size_t)o * g.K + j, __uint_as_float(raw[u]));
              }
            }
          }
        }
      } else {
        // Jittor layout: lane = column j of a lane block, TMEM columns = output channels
        for (int cb = cb0; cb < cb1; ++cb) {
          const int j = cb * 128 + m;
          const uint32_t taddr = d2_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)((cb - cb0) * P.o_cols);
          for (int c0 = part * 8; c0 < P.o_cols; c0 += 32) {
            uint32_t raw[8];
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                         : "=r"(raw[0]), "=r"(raw[1]), "=r"(raw[2]), "=r"(raw[3]), "=r"(raw[4]), "=r"(raw[5]),
                           "=r"(raw[6]), "=r"(raw[7])
                         : "r"(taddr + c0)
                         : "memory");
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            if (j < g.K) {
#pragma unroll
              for (int u = 0; u < 8; ++u)
                if (c0 + u < g.O) atomicAdd(P.gw + wt_index(g, c0 + u, j), __uint_as_float(raw[u]));
            }
          }
        }
      }
      tc_fence_before();
    }
  } else if (warp == kMmaWarp) {
    // ================================================================ MMA issuer
    // The whole warp runs this (uniform) loop; elect.sync picks the issuing lane per group of instructions and every
    // descriptor is one 64-bit add onto a loop-invariant base (dcn_umma.cuh:elect_one, tools/mma_rate_probe.cu): inside
    // `if (lane == 0)` each tcgen05.mma sat in a waterfall loop behind ~10 dependent integer instructions per descriptor,
    // and this warp shares its scheduler with four scatter warps.
    {
      const uint32_t idesc = make_idesc_bf16(128, ncols, false, false);
      const uint32_t idesc_w = make_idesc_bf16(128, ncols, true, true);  // A = g^T and B = S, both MN-major
      int s = 0, acc = 0, sb = 0, gb = 0;
      uint32_t phase = 0, acc_phase = 0, gphase = 0, sphase = 0;
      bool first_tile = true;
      // gW[o, cols of block] += g^T[o, 128 rows] * S[128 rows, cols]; A = the resident grad_out
      // images read MN-major (o contiguous, 64-o atoms = consecutive images), B = sample operand
      const uint32_t idesc_wj = make_idesc_bf16(128, P.o_cols > 0 ? P.o_cols : 16, false, true);
      auto wgrad_mmas = [&](int cb, bool first, int gb) {
        mbar_wait_relaxed(&sfull[sb], sphase, 32);
        tc_fence_after();
        const uint32_t g_hi = smem_u32(gtile) + (uint32_t)gb * g_buf, g_lo = g_hi + P.g_img;
        const uint32_t sbase = smem_u32(sbuf + (size_t)sb * s_buf);
        if (VARIANT == DCN_VARIANT_TORCH) {
          // gW[o, cols of block] += g^T[o, 128 rows] * S[128 rows, cols]: A = the resident grad_out images read
          // MN-major (o contiguous; 64-o atoms = this buffer's image, then its second image or — O <= 64 — the
          // shared zero image), B = sample operand read MN-major
          // (128 < O <= 256: a second pass over images 2, 3 into the second accumulator set)
          const uint64_t ds0 = make_sdesc_sw128(sbase, 1024, 1024);
          const uint32_t gimg16 = P.g_img >> 4;
          for (int hf = 0; hf < P.o_halves; ++hf) {
            const uint32_t g_h = g_hi + (uint32_t)(2 * hf) * NIMG * P.g_img;
            const uint32_t g_lbo = 2 * hf + 1 < P.OB ? NIMG * P.g_img
                                                     : g_zero_off - (uint32_t)gb * g_buf - (uint32_t)(2 * hf) * NIMG * P.g_img;
            const uint32_t d_tmem = d2_base + (uint32_t)((hf * P.cb_per_slice + cb - cb0) * ncols);
            const uint64_t dg0 = make_sdesc_sw128(g_h, g_lbo, 1024);
            if (elect_one()) {
#pragma unroll
              for (int ks = 0; ks < 8; ++ks) {  // 8 steps of 16 tile rows
                const uint64_t dgh = dg0 + (uint64_t)(ks * 128), dsh = ds0 + (uint64_t)(ks * 128);
                umma_bf16(d_tmem, dgh, dsh, idesc_w, (first && ks == 0) ? 0u : 1u);
                if (!BF) {
                  umma_bf16(d_tmem, dgh, dsh + (s_img >> 4), idesc_w, 1u);
                  umma_bf16(d_tmem, dgh + gimg16, dsh, idesc_w, 1u);
                }
              }
            }
            __syncwarp();
          }
        } else {
          // Jittor layout: gW^T[j of this lane block, o] += S^T[j, pixels] * g[pixels, o]: A = the sample operand,
          // the same image read K-major (K = the tile's 64 pixels), B = the resident grad_out pixels read MN-major
          // (o contiguous; 64-o atoms = consecutive images): no padded operand rows at all
          const uint32_t g_lbo = NIMG * P.g_img;
          const uint32_t d_tmem = d2_base + (uint32_t)((cb - cb0) * P.o_cols);
          const uint64_t ds0 = make_sdesc_sw128(sbase, 16, 1024), dg0 = make_sdesc_sw128(g_hi, g_lbo, 1024);
          const uint32_t gimg16 = P.g_img >> 4;
          if (elect_one()) {
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4) {  // 4 steps of 16 pixels
              const uint64_t dsh = ds0 + (uint64_t)(k4 * 2), dgh = dg0 + (uint64_t)(k4 * 128);
              umma_bf16(d_tmem, dsh, dgh, idesc_wj, (first && k4 == 0) ? 0u : 1u);
              if (!BF) {
                umma_bf16(d_tmem, dsh, dgh + gimg16, idesc_wj, 1u);
                umma_bf16(d_tmem, dsh + (s_img >> 4), dgh, idesc_wj, 1u);
              }
            }
          }
        }
        if (elect_one()) umma_commit(&sempty[sb]);
        __syncwarp();
        sb ^= 1;
        if (sb == 0) sphase ^= 1;
      };
      if (P.w_resident && tile0 < P.num_tiles) {
        mbar_wait_relaxed(&wfull[0], 0, 32);  // the slice's Wm^T images, loaded once
        tc_fence_after();
      }
      // The weight-gradient MMAs of a block need its scatter pass finished (sfull), so they trail GEMM-1 by one
      // block: GEMM-1 of block i + 1 is in flight while the scatter warps work on block i.  With two grad_out
      // buffers the trailing continues across the tile boundary (a slice of ONE block per tile would otherwise
      // serialise GEMM-1 and scatter completely); with one buffer the tile is drained before the next begins.
      bool pend = false, pend_first = false, pend_last = false;
      int pend_cb = 0, pend_gb = 0;
      auto drain = [&]() {
        if (!pend) return;
        wgrad_mmas(pend_cb, pend_first, pend_gb);
        if (pend_last && elect_one()) umma_commit(&gempty[pend_gb]);  // grad_out tile buffer may be overwritten
        __syncwarp();
        pend = false;
      };
      for (int tile = tile0; tile < P.num_tiles; tile += tile_step) {
        mbar_wait_relaxed(&gfull[gb], gphase, 32);
        for (int cb = cb0; cb < cb1; ++cb) {
          mbar_wait_relaxed(&tempty[acc], acc_phase ^ 1, 32);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)(acc * ncols);
          for (int ob = 0; ob < P.OB; ++ob) {
            if (P.w_resident) {
              s = (cb - cb0) * P.OB + ob;
            } else {
              mbar_wait_relaxed(&wfull[s], phase, 32);
              tc_fence_after();
            }
            // resident converted grad_out image and streamed Wm^T image; Torch: A = grad_out rows,
            // B = Wm^T columns; Jittor: A = Wm^T lanes, B = grad_out pixels
            const uint32_t r_hi = smem_u32(gtile) + (uint32_t)gb * g_buf + (uint32_t)ob * NIMG * P.g_img;
            const uint32_t r_lo = r_hi + P.g_img;
            const uint32_t w_hi = smem_u32(wstage + (size_t)s * P.w_stage);
            const uint32_t w_lo = w_hi + (P.w_stage >> 1);
            const uint32_t a_hi = VARIANT == DCN_VARIANT_TORCH ? r_hi : w_hi;
            const uint32_t a_lo = VARIANT == DCN_VARIANT_TORCH ? r_lo : w_lo;
            const uint32_t b_hi = VARIANT == DCN_VARIANT_TORCH ? w_hi : r_hi;
            const uint32_t b_lo = VARIANT == DCN_VARIANT_TORCH ? w_lo : r_lo;
            const uint64_t da0 = make_sdesc_sw128(a_hi, 16, 1024), db0 = make_sdesc_sw128(b_hi, 16, 1024);
            const uint32_t alo16 = (a_lo - a_hi) >> 4, blo16 = (b_lo - b_hi) >> 4;
            if (elect_one()) {
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4) {
                const uint64_t dah = da0 + (uint64_t)(k4 * 2), dbh = db0 + (uint64_t)(k4 * 2);
                umma_bf16(d_tmem, dah, dbh, idesc, (ob | k4) ? 1u : 0u);
                if (!BF) {
                  umma_bf16(d_tmem, dah, dbh + blo16, idesc, 1u);
                  umma_bf16(d_tmem, dah + alo16, dbh, idesc, 1u);
                }
              }
              if (!P.w_resident) umma_commit(&wempty[s]);
            }
            __syncwarp();
            if (!P.w_resident) {
              if (++s == P.w_ring) {
                s = 0;
                phase ^= 1;
              }
            }
          }
          if (elect_one()) umma_commit(&tfull[acc]);
          __syncwarp();
          acc ^= 1;
          if (acc == 0) acc_phase ^= 1;
          if (FUSE) {
            drain();
            pend = true;
            pend_cb = cb;
            pend_gb = gb;
            pend_first = first_tile;
            pend_last = cb == cb1 - 1;
          }
        }
        if (!FUSE) {
          if (elect_one()) umma_commit(&gempty[gb]);
          __syncwarp();
        } else if (P.g_nbuf == 1) drain();
        if (++gb == P.g_nbuf) {
          gb = 0;
          gphase ^= 1;
        }
        first_tile = false;
      }
      if (FUSE) drain();
      if (FUSE && elect_one()) umma_commit(dfull);
      __syncwarp();
    }
  } else if (warp == kLoadWarp) {
    // ================================================================ Wm^T tile loader
    if (lane == 0) {
      int s = 0;
      uint32_t phase = 0;
      if (P.w_resident) {
        if (tile0 < P.num_tiles) {
          // the slice's images are contiguous in wtiles ([cb][ob] order): stage i = (cb - cb0) * OB + ob
          const int n = (cb1 - cb0) * P.OB;
          mbar_arrive_expect_tx(&wfull[0], (uint32_t)n * P.w_stage);
          for (int i = 0; i < n; ++i)
            bulk_g2s(wstage + (size_t)i * P.w_stage, P.wtiles + ((size_t)cb0 * P.OB + i) * P.w_stage, P.w_stage,
                     &wfull[0]);
        }
      } else
      for (int tile = tile0; tile < P.num_tiles; tile += tile_step) {
        for (int cb = cb0; cb < cb1; ++cb)
          for (int ob = 0; ob < P.OB; ++ob) {
            mbar_wait_relaxed(&wempty[s], phase ^ 1, 32);
            mbar_arrive_expect_tx(&wfull[s], P.w_stage);
            bulk_g2s(wstage + (size_t)s * P.w_stage, P.wtiles + (size_t)(cb * P.OB + ob) * P.w_stage,
                     P.w_stage, &wfull[s]);
            if (++s == P.w_ring) {
              s = 0;
              phase ^= 1;
            }
          }
      }
    } else if (lane == 1) {
      // the tile's grad_out operand images were staged by gout_tiles_*_kernel: bulk copies, no conversion here
      uint32_t gphase = 0;
      int gb = 0;
      for (int tile = tile0; tile < P.num_tiles; tile += tile_step) {
        mbar_wait_relaxed(&gempty[gb], gphase ^ 1, 64);
        mbar_arrive_expect_tx(&gfull[gb], g_buf);
        if (VARIANT == DCN_VARIANT_TORCH || ncols == 128) {
          // the tile's images are contiguous: one copy
          bulk_g2s(gtile + (size_t)gb * g_buf, P.gtiles + (size_t)tile * g_buf, g_buf, &gfull[gb]);
        } else {
          // Jittor layout, 64-pixel tiles: one half (64 rows = 8 KB) of every 128-pixel image
          const int b = tile / P.pix_blocks, pblk = tile - b * P.pix_blocks;
          const int pb128 = (g.HW + 127) / 128;
          const uint8_t* src = P.gtiles + ((size_t)(b * pb128 + (pblk >> 1)) * P.OB * NIMG) * kGImg + (pblk & 1) * (kGImg / 2);
          for (int i = 0; i < P.OB * NIMG; ++i)
            bulk_g2s(gtile + (size_t)gb * g_buf + (size_t)i * P.g_img, src + (size_t)i * kGImg, P.g_img, &gfull[gb]);
        }
        if (++gb == P.g_nbuf) {
          gb = 0;
          gphase ^= 1;
        }
      }
    }
  } else {
    // ================================================================ plan warps
    const int pt = tid - kFirstPlanWarp * 32;  // 0..63 / 0..127
    constexpr int kPlanThreads = PW * 32;
    const int n_ent = P.plan_cap;
    int pb = 0;
    uint32_t pphase = 0;
    PlanWork pw[kPlanPerThread];
    if (tile0 < P.num_tiles) {
#pragma unroll
      for (int u = 0; u < kPlanPerThread; ++u)
        if (pt + u * kPlanThreads < n_ent) plan_prepare<VARIANT, PLAIN, MOD>(P, tile0, cb0, pt + u * kPlanThreads, pw[u], mask);
    }
    for (int tile = tile0; tile < P.num_tiles; tile += tile_step) {
      for (int cb = cb0; cb < cb1; ++cb) {
        ScatEntry* pl = plan + pb * P.plan_cap;
        mbar_wait_relaxed(&pempty[pb], pphase ^ 1, 64);
#pragma unroll
        for (int u = 0; u < kPlanPerThread; ++u)
          if (pt + u * kPlanThreads < n_ent)
            pl[pt + u * kPlanThreads] = PLAIN ? plan_finish_plain(g, pw[u]) : plan_finish(g, pw[u]);
        if (MOD) {
          // dead entries get 0: their sample is 0, and m * 0 must stay finite for the fused weight gradient
          float* mpl = mplan + pb * P.plan_cap;
#pragma unroll
          for (int u = 0; u < kPlanPerThread; ++u)
            if (pt + u * kPlanThreads < n_ent) mpl[pt + u * kPlanThreads] = pw[u].valid ? pw[u].mk : 0.f;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&pfull[pb]);
        int ntile = tile, ncb = cb + 1;
        if (ncb == cb1) {
          ncb = cb0;
          ntile = tile + tile_step;
        }
        if (ntile < P.num_tiles) {
#pragma unroll
          for (int u = 0; u < kPlanPerThread; ++u)
            if (pt + u * kPlanThreads < n_ent) plan_prepare<VARIANT, PLAIN, MOD>(P, ntile, ncb, pt + u * kPlanThreads, pw[u], mask);
        }
        pb ^= 1;
        if (pb == 0) pphase ^= 1;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(P.tmem_cols)
                 : "memory");
  }
}

// grad_out rows of a Torch-layout tile are R floats apart (row (instance, i) = pixel r0 + i*R of
// channel plane o), so gathering them inside the main kernel costs one L1 wavefront per float.
// This staging pass reads 16 consecutive instances at a time (64-byte runs), transposes through
// shared memory and writes every tile's operand exactly as the MMAs read it:
//   gtiles[tile][ob][hi | lo][row m = il*Gt + i][64 o]  bf16, K-major, 128-byte swizzle.
// Block = (16 instances) x (16 of the Gt channels) x (32 output channels) = 32 KB of floats.
constexpr int kGtInst = 16, kGtCh = 16, kGtOsub = 32;
constexpr int kGtRow = kGtOsub + 1;        // floats per (instance, channel) row, odd
constexpr int kGtIS = kGtCh * kGtRow + 2;  // floats per instance: == 2 mod 32 -> (16 inst x 2 ch) lanes hit 32 banks

template <typename T>
__global__ void __launch_bounds__(256) gout_tiles_torch_kernel(const __grid_constant__ Params P,
                                                               uint8_t* __restrict__ gtiles) {
  constexpr int NIMG = sizeof(T) == 2 ? 1 : 2;
  __shared__ float gt_buf[kGtInst * kGtIS];
  const Geo& g = P.g;
  const int Gt = P.Gt, tid = threadIdx.x;
  const int ch_blocks = Gt / kGtCh;
  const int o0 = (blockIdx.y / ch_blocks) * kGtOsub, i0 = (blockIdx.y % ch_blocks) * kGtCh;
  {
    // lanes: 16 instances (one 64-byte run) x 2 channels; the instance of a thread is fixed
    const int r = tid & 15;
    const TileRowInfo ri = decode_inst(P, blockIdx.x * kGtInst + r);
    const T* src = reinterpret_cast<const T*>(P.gout) + ((size_t)ri.b * g.Oimg + o0) * g.HW + ri.r0 +
                   ((size_t)ri.chunk * Gt + i0) * P.t.R;
    float* dst = gt_buf + r * kGtIS;
    const int p0 = tid >> 4;  // 0..15: (ol, i2) pairs, i2 fastest
    float v[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) {
      const int it = p0 + 16 * k, ol = it / kGtCh, i2 = it % kGtCh;
      v[k] = 0.f;
      if (ri.valid && o0 + ol < g.O) v[k] = (float)__ldg(src + (size_t)ol * g.HW + (size_t)i2 * P.t.R);
    }
#pragma unroll
    for (int k = 0; k < 32; ++k) {
      const int it = p0 + 16 * k, ol = it / kGtCh, i2 = it % kGtCh;
      dst[i2 * kGtRow + ol] = v[k];
    }
  }
  __syncthreads();
  if (P.gb_fused) {
    // grad_bias rides along: the block holds 256 (instance, channel) rows x 32 output channels of grad_out; every
    // element of grad_out is staged exactly once, rows of no instance are zero.  Lanes = output channels (odd row
    // stride: no bank conflicts), 8 warps = 8 groups of 32 rows.
    __shared__ float gb_part[8][32];
    const int ol = tid & 31, part = tid >> 5;
    float sum = 0.f;
#pragma unroll 8
    for (int q = 0; q < 32; ++q) {
      const int row = part * 32 + q;  // (instance r, channel i2)
      sum += gt_buf[(row >> 4) * kGtIS + (row & 15) * kGtRow + ol];
    }
    gb_part[part][ol] = sum;
    __syncthreads();
    if (tid < 32 && o0 + tid < g.O) {
      float tot = 0.f;
#pragma unroll
      for (int q = 0; q < 8; ++q) tot += gb_part[q][tid];
      atomicAdd(P.gb_fused + o0 + tid, tot);
    }
  }
  // 16-byte chunks (8 o) of the images: lanes = 4 chunks x 8 consecutive rows of one instance
  const uint32_t img_bytes = 128u * 128u;
  const int ob = o0 >> 6, c_base = (o0 & 63) >> 3;
#pragma unroll
  for (int k = 0; k < kGtInst * kGtCh * (kGtOsub / 8) / 256; ++k) {
    const int it = tid + 256 * k;
    const int ck = it & 3, row = it >> 2, r = row / kGtCh, i2 = row % kGtCh;
    const int inst = blockIdx.x * kGtInst + r, tile = inst / P.Rt, il = inst - tile * P.Rt;
    if (tile >= P.num_tiles) continue;
    const float* srow = gt_buf + r * kGtIS + i2 * kGtRow + ck * 8;
    float v[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) v[q] = srow[q];
    uint4 hi, lo;
    split_pair(v[0], v[1], hi.x, lo.x);
    split_pair(v[2], v[3], hi.y, lo.y);
    split_pair(v[4], v[5], hi.z, lo.z);
    split_pair(v[6], v[7], hi.w, lo.w);
    const int ic = i0 + i2;
    const int m = P.row_v ? (ic / P.row_v) * (P.row_v * P.Rt) + il * P.row_v + ic % P.row_v : il * Gt + ic;
    uint8_t* img = gtiles + ((size_t)tile * P.OB + ob) * NIMG * img_bytes + kmajor_sw128_off(m, (c_base + ck) * 8);
    *reinterpret_cast<uint4*>(img) = hi;
    if (NIMG == 2) *reinterpret_cast<uint4*>(img + img_bytes) = lo;
  }
}

// Pixel-row layouts (Jittor / DCNv1): operand row = output pixel.  gout[b][o][p] -> images
//   gtiles[b][pixel block of 128][ob][hi | lo][128 pixels x 64 o]  bf16, K-major, 128-byte swizzle,
// i.e. a transposition (pixels are contiguous in gout, output channels in the image).  A 64-pixel tile of
// the data-gradient kernel is one half (64 rows = 8 KB) of an image.  Block = 128 pixels x 64 output channels.
template <typename T>
__global__ void __launch_bounds__(256) gout_tiles_pix_kernel(Geo g, int OB, const T* __restrict__ gout,
                                                             uint8_t* __restrict__ gtiles) {
  constexpr int NIMG = sizeof(T) == 2 ? 1 : 2;
  __shared__ float tile[64][129];
  const int pb = blockIdx.x, ob = blockIdx.y, b = blockIdx.z;
  const int tid = threadIdx.x, px = tid & 127, p = pb * 128 + px;
  const T* src = gout + ((size_t)b * g.Oimg + ob * 64) * g.HW + p;
#pragma unroll 8
  for (int it = 0; it < 32; ++it) {
    const int ol = (tid >> 7) + 2 * it;
    float v = 0.f;
    if (p < g.HW && ob * 64 + ol < g.O) v = (float)__ldg(src + (size_t)ol * g.HW);
    tile[ol][px] = v;
  }
  __syncthreads();
  const uint32_t img_bytes = 128u * 128u;
  uint8_t* img = gtiles + (((size_t)b * gridDim.x + pb) * OB + ob) * NIMG * img_bytes;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int it = tid + 256 * k, ck = it & 7, row = it >> 3;  // lanes: 8 chunks x 4 pixel rows
    float v[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) v[q] = tile[ck * 8 + q][row];
    uint4 hi, lo;
    split_pair(v[0], v[1], hi.x, lo.x);
    split_pair(v[2], v[3], hi.y, lo.y);
    split_pair(v[4], v[5], hi.z, lo.z);
    split_pair(v[6], v[7], hi.w, lo.w);
    const uint32_t so = kmajor_sw128_off(row, ck * 8);
    *reinterpret_cast<uint4*>(img + so) = hi;
    if (NIMG == 2) *reinterpret_cast<uint4*>(img + img_bytes + so) = lo;
  }
}

// Wm^T images: tiles[cb][ob][hl][K-major SW128 image of ncols rows (j) x 64 (o)]
template <typename T>
__global__ void __launch_bounds__(256) weight_tiles_bwd_kernel(Geo g, int ncols, int cblocks, int OB,
                                                               const T* __restrict__ wt,
                                                               uint8_t* __restrict__ tiles) {
  constexpr int NIMG = sizeof(T) == 2 ? 1 : 2;
  const int total = cblocks * ncols * OB * 64;
  const uint32_t img = (uint32_t)ncols * 128;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int o = i % (OB * 64), jj = i / (OB * 64);  // lanes along o: Wm[o, j] strided reads, small
    const int cb = jj / ncols, jl = jj - cb * ncols, ob = o >> 6, ol = o & 63;
    const float v = (o < g.O && jj < g.K) ? (float)wt[wt_index(g, o, jj)] : 0.f;
    __nv_bfloat16 hi, lo;
    ptx::split_bf16(v, hi, lo);
    uint8_t* base = tiles + (size_t)(cb * OB + ob) * NIMG * img + ptx::kmajor_sw128_off(jl, ol);
    *reinterpret_cast<__nv_bfloat16*>(base) = hi;
    if (NIMG == 2) *reinterpret_cast<__nv_bfloat16*>(base + img) = lo;
  }
}

}  // namespace bd

// Fused kernels: CTA = (slice of the column / lane blocks, chunk of the tiles).  Slices of equal size finish
// together: among the smallest slice counts pick the one that wastes the least (padding blocks of the last
// slice x SMs left without a CTA; cfg2: 9 blocks -> 3 x 3, not 5 + 4).  Then the shared-memory plan: two
// grad_out tile buffers first (the MMA issuer then runs GEMM-1 of the next tile while the weight-gradient MMAs
// of the previous one are still waiting for its scatter pass), and the slice's Wm^T images resident when they
// fit (loaded once instead of re-streamed from L2 for every tile).
//   real = bytes of one grad_out tile buffer, zero = shared zero images, other = everything but the grad_out
//   buffers and the Wm^T stages
static void choose_slices(bd::Params* P, int max_cb, size_t real, size_t zero, size_t other) {
  const int ns_min = (P->cblocks + max_cb - 1) / max_cb;
  double best = 1e30;
  for (int ns = ns_min; ns <= ns_min + 2 && ns <= P->cblocks; ++ns) {
    const int cbp = (P->cblocks + ns - 1) / ns;
    const int ns_eff = (P->cblocks + cbp - 1) / cbp;
    const double waste = (double)ns_eff * cbp / P->cblocks * 148.0 / (ns_eff * (148 / ns_eff));
    if (waste < best - 1e-9) {
      best = waste;
      P->nslices = ns_eff;
      P->cb_per_slice = cbp;
    }
  }
  const size_t n_res = (size_t)P->cb_per_slice * P->OB;
  // plans in order of preference: {grad_out buffers, resident?, ring stages}.  The 1-stage ring is taken only
  // to make room for the second grad_out buffer; its budget counts 256 instead of 1024 bytes of alignment slack
  // (the dynamic shared-memory window starts 1 KB-aligned in practice; the kernel traps if it would overrun).
  const int plans[5][3] = {{2, 1, 2}, {2, 0, 2}, {2, 0, 1}, {1, 1, 2}, {1, 0, 2}};
  for (const auto& pl : plans) {
    const size_t n_w = pl[1] ? n_res : (size_t)pl[2];
    const size_t need = pl[0] * real + zero + n_w * P->w_stage + other;
    if (need <= kSmemBudget || (pl[2] == 1 && need - 768 <= kSmemBudget)) {
      P->g_nbuf = pl[0];
      P->w_resident = pl[1] ? (int)n_res : 0;
      P->w_ring = pl[2];
      return;
    }
  }
}

// ---------------------------------------------------------------------------- host side
static bool copy_row_tiling(const Geo& g, bd::Params* P) {
  if (!make_tiling(g, &P->t)) return false;
  P->Gt = P->t.Gt;
  P->Rt = P->t.Rt;
  P->chunks = P->t.chunks;
  P->num_inst = P->t.num_inst;
  P->num_tiles = P->t.num_tiles;
  P->divR = P->t.divR;
  P->divChunks = P->t.divChunks;
  return true;
}

static bool bwd_data_tiling(const Geo& g, int operand, bd::Params* P) {
  const size_t nimg = operand == DCN_OPERAND_BF16 ? 1 : 2;
  if (!copy_row_tiling(g, P)) return false;
  P->fuse_w = 0;
  P->o_halves = 1;
  P->o_cols = 0;
  P->w_resident = 0;
  P->w_ring = 2;
  P->g_nbuf = 1;
  P->gw = nullptr;
  P->nslices = P->nchunks = 1;
  P->cb_per_slice = 0;
  // ScatEntry::gidx is an unsigned 32-bit grad_offset index with 0xffffffff reserved (make_geo's B*N*HW < 2^31 keeps
  // every shape inside this bound; the check states the limit where the index is formed)
  if ((long long)g.B * 2 * g.N * g.HW > 0xffffffffLL) return false;
  if ((long long)xt_image_stride(g) >= (1LL << 30)) return false;  // 32-bit byte offsets inside an image
  P->OB = (g.O + 63) / 64;
  if (P->OB > 4) return false;  // so O <= 256, and the fused weight gradient is always a candidate
  const bool torch = g.variant == DCN_VARIANT_TORCH;
  // pixel-row layouts: a lane block of 128 columns must hold whole taps
  if (!torch && !(g.C % 128 == 0 || g.C == 64 || g.C == 32 || g.C == 16)) return false;
  // What the layouts differ in.  Plan entries per block column: Torch the Rt class instances of a tile, pixel-row
  // the taps of a lane block.  Fused weight gradient: Torch one gW accumulator set per 128-channel half of the o axis
  // (the gW MMAs take two 64-o images at a time, zero images complete the second one), <= 6 blocks next to the
  // 2 gA buffers; pixel-row gW^T accumulator blocks of O columns rounded up to 16, <= 8 of them.
  const int ent = torch ? P->t.Rt : (g.C >= 128 ? 1 : 128 / g.C);
  const int halves = g.O > 128 ? 2 : 1;
  const int o_cols = (g.O + 15) / 16 * 16;
  const int max_cb = torch ? 6 / halves : min((512 - 2 * 64) / o_cols, 8);
  const size_t zero = torch ? (size_t)(2 * halves - P->OB) * nimg * bd::kGImg : 0;
  // candidates in order of preference: fused (64 columns), then unfused with 128 or 64 columns per accumulator block
  // (Torch: columns j; pixel-row: pixels)
  const struct { bool fuse; int ncols; } cands[3] = {{true, 64}, {false, 128}, {false, 64}};
  for (const auto& c : cands) {
    const int ncols = c.ncols;
    const int w_rows = torch ? ncols : 128;  // Wm^T rows of a block: its columns j, or a lane block
    const uint32_t g_img = torch ? bd::kGImg : (uint32_t)ncols * 128;  // grad_out image: 128 tile rows or ncols pixels
    const uint32_t w_stage = (uint32_t)nimg * w_rows * 128;
    const size_t real = (size_t)P->OB * nimg * g_img, z = c.fuse ? zero : 0;
    // Wm^T ring, sample operand (fused), plan ring, barriers, alignment slack
    const size_t rest = 2 * (size_t)w_stage + (c.fuse ? 2 * nimg * (size_t)(128 * 128) : 0) +
                        2 * (size_t)ent * ncols * sizeof(bd::ScatEntry) + 256 + 1024;
    if (ent * ncols > bd::plan_max_of(4) || real + z + rest > kSmemBudget) continue;
    P->ncols = ncols;
    P->cblocks = (g.K + w_rows - 1) / w_rows;
    P->plan_cap = ent * ncols;
    P->g_img = g_img;
    P->w_stage = w_stage;
    P->pix_blocks = torch ? 1 : (g.HW + ncols - 1) / ncols;
    P->num_tiles = torch ? P->t.num_tiles : g.B * P->pix_blocks;
    P->g_imgs = c.fuse && torch ? 2 * halves : P->OB;
    P->tmem_cols = c.fuse ? 512 : 2 * ncols;
    if (!c.fuse) {
      P->g_nbuf = (2 * real + rest <= kSmemBudget) ? 2 : 1;
      return true;
    }
    P->fuse_w = 1;
    if (torch) P->o_halves = halves;
    else P->o_cols = o_cols;
    choose_slices(P, max_cb, real, z, rest - 2 * (size_t)w_stage);
    return true;
  }
  return false;
}

bool umma_bwd_data_supported(const Geo& g, int operand) {
  if (operand != DCN_OPERAND_FP32 && operand != DCN_OPERAND_BF16) return false;
  bd::Params P;
  P.g = g;
  return bwd_data_tiling(g, operand, &P);
}

// does umma_bwd_data_any also produce grad_weight for this shape?
bool umma_bwd_data_fuses_wgrad(const Geo& g, int operand) {
  bd::Params P;
  P.g = g;
  return bwd_data_tiling(g, operand, &P) && P.fuse_w;
}

size_t umma_bwd_data_wtile_bytes(const Geo& g, int operand) {
  bd::Params P;
  P.g = g;
  if (!bwd_data_tiling(g, operand, &P)) return 0;
  return align_up((size_t)P.cblocks * P.OB * P.w_stage, 1024);
}

// the staging pass of the grad_out operand (Torch layout); P needs g, copy_row_tiling, OB, gout, row_v
static int launch_gout_tiles(const bd::Params& P, bool bf, uint8_t* gtiles, cudaStream_t st) {
  const dim3 grid((unsigned)(((size_t)P.num_tiles * P.t.Rt + bd::kGtInst - 1) / bd::kGtInst),
                  (unsigned)((P.OB * 64 / bd::kGtOsub) * (P.t.Gt / bd::kGtCh)));
  KernelScope scope("gout_tiles_kernel", st);
  if (bf)
    bd::gout_tiles_torch_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(P, gtiles);
  else
    bd::gout_tiles_torch_kernel<float><<<grid, 256, 0, st>>>(P, gtiles);
  DCN_KERNEL_CHECK("gout_tiles_kernel");
  return DCN_OK;
}

// pixel-row layouts: [b][ceil(HW / 128)][OB][hi | lo][128 x 64] images (see gout_tiles_pix_kernel)
static size_t gtile_pix_bytes(const Geo& g, int operand) {
  return align_up((size_t)g.B * ((g.HW + 127) / 128) * ((g.O + 63) / 64) * (operand == DCN_OPERAND_BF16 ? 1 : 2) *
                      bd::kGImg, 1024);
}
int launch_gout_tiles_pix(const Geo& g, int operand, const void* gout, uint8_t* gtiles, cudaStream_t st) {
  const int OB = (g.O + 63) / 64;
  const dim3 grid((unsigned)((g.HW + 127) / 128), (unsigned)OB, (unsigned)g.B);
  KernelScope scope("gout_tiles_kernel", st);
  if (operand == DCN_OPERAND_BF16)
    bd::gout_tiles_pix_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(g, OB, (const __nv_bfloat16*)gout, gtiles);
  else
    bd::gout_tiles_pix_kernel<float><<<grid, 256, 0, st>>>(g, OB, (const float*)gout, gtiles);
  DCN_KERNEL_CHECK("gout_tiles_kernel");
  return DCN_OK;
}

// grad_out tile images in the FORWARD kernel's row order, for its weight-gradient mode (MODE_WGRAD):
// [tile][OB = ceil(O / 64)][hi | lo][128 rows x 64 o].  V = channels per gather item (4 fp32 / 8 bf16).
size_t umma_wgrad_gtile_bytes(const Geo& g, int operand) {
  Tiling t;
  if (!make_tiling(g, &t)) return 0;
  if (g.variant != DCN_VARIANT_TORCH) return gtile_pix_bytes(g, operand);
  return align_up((size_t)t.num_tiles * ((g.O + 63) / 64) * (operand == DCN_OPERAND_BF16 ? 1 : 2) * bd::kGImg, 1024);
}
int launch_gout_tiles_fwd_order(const Geo& g, int operand, const void* gout, uint8_t* gtiles, cudaStream_t st) {
  if (g.variant != DCN_VARIANT_TORCH) return launch_gout_tiles_pix(g, operand, gout, gtiles, st);
  bd::Params P;
  memset(&P, 0, sizeof(P));
  P.g = g;
  if (!copy_row_tiling(g, &P)) return DCN_ERR_UNSUPPORTED;
  P.OB = (g.O + 63) / 64;
  P.gout = gout;
  P.row_v = operand == DCN_OPERAND_BF16 ? 8 : 4;
  return launch_gout_tiles(P, operand == DCN_OPERAND_BF16, gtiles, st);
}

// staged grad_out operand images
size_t umma_bwd_data_gtile_bytes(const Geo& g, int operand) {
  bd::Params P;
  P.g = g;
  if (!bwd_data_tiling(g, operand, &P)) return 0;
  if (g.variant != DCN_VARIANT_TORCH) return gtile_pix_bytes(g, operand);
  return align_up((size_t)P.num_tiles * P.OB * (operand == DCN_OPERAND_BF16 ? 1 : 2) * bd::kGImg, 1024);
}

// what every launch of the data-gradient kernel takes besides its template arguments
struct BdLaunch {
  const bd::Params& P;
  int grid;
  size_t smem;
  cudaStream_t st;
  const float* mask;
  float* gmask;
};

// one instantiation: opt in to its shared memory, launch it with its role layout, check the launch
template <int VARIANT, int RW, bool FUSE, bool BF, int PW, bool PLAIN, bool MOD>
static int launch_bd(const BdLaunch& L) {
  DCN_CUDA_TRY(cudaFuncSetAttribute(bd::bwd_data_kernel<VARIANT, RW, FUSE, BF, PW, PLAIN, MOD>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.smem));
  bd::bwd_data_kernel<VARIANT, RW, FUSE, BF, PW, PLAIN, MOD>
      <<<L.grid, bd::threads_of(PW), L.smem, L.st>>>(L.P, L.mask, L.gmask);
  DCN_KERNEL_CHECK("umma_bwd_data_kernel");
  return DCN_OK;
}

// lanes per sampling point and plan warps.  16 channels per point put 8 class instances / taps in a block column, so
// such a plan has >= 512 entries; <= 128 entries (2 per plan thread) leave the plan to 2 warps: 20 warps, 96 registers
// for the scatter loop.  Otherwise 4 plan warps keep up with the scatter.
template <int VARIANT, bool FUSE, bool BF, bool PLAIN, bool MOD>
static int launch_bd_split(const BdLaunch& L, bool narrow) {
  if (narrow) return launch_bd<VARIANT, 16, FUSE, BF, 4, PLAIN, MOD>(L);
  if (L.P.plan_cap <= 128) return launch_bd<VARIANT, 32, FUSE, BF, 2, PLAIN, MOD>(L);
  return launch_bd<VARIANT, 32, FUSE, BF, 4, PLAIN, MOD>(L);
}

template <int VARIANT, bool MOD>
static int launch_bd_operand(const BdLaunch& L, bool bf, bool narrow) {
  if (bf)
    return L.P.fuse_w ? launch_bd_split<VARIANT, true, true, false, MOD>(L, narrow)
                      : launch_bd_split<VARIANT, false, true, false, MOD>(L, narrow);
  return L.P.fuse_w ? launch_bd_split<VARIANT, true, false, false, MOD>(L, narrow)
                    : launch_bd_split<VARIANT, false, false, false, MOD>(L, narrow);
}

// gxt (channels-last grad_x, may be null), goff and — when the shape fuses the weight gradient
// (umma_bwd_data_fuses_wgrad) — gw must be zero on entry.
// gb_fused (Torch layout only, may be null): grad_bias [g.O], zeroed by the caller, summed by the grad_out staging pass
// mask / gmask (DCNv1 only, both or neither): modulated; gmask must be zero on entry like goff.
int umma_bwd_data_any(const Geo& g, int operand, const void* xt, float* gxt, const float* off, const void* wt,
                      const void* gout, float* goff, float* gw, uint8_t* wtiles, uint8_t* gtiles,
                      cudaStream_t st, float* gb_fused, const float* mask, float* gmask) {
  bd::Params P;
  P.g = g;
  const bool bf = operand == DCN_OPERAND_BF16;
  const size_t nimg = bf ? 1 : 2;
  if (!bwd_data_tiling(g, operand, &P)) {
    set_error("umma bwd_data: shape not tileable");
    return DCN_ERR_UNSUPPORTED;
  }
  {
    // Wm^T images: rows = the block's columns j (Torch: ncols per block, Jittor: 128 per block)
    const int rows = g.variant == DCN_VARIANT_TORCH ? P.ncols : 128;
    const int total = P.cblocks * rows * P.OB * 64;
    KernelScope scope("weight_tiles_bwd_kernel", st);
    if (bf)
      bd::weight_tiles_bwd_kernel<__nv_bfloat16><<<min((total + 255) / 256, 2048), 256, 0, st>>>(
          g, rows, P.cblocks, P.OB, (const __nv_bfloat16*)wt, wtiles);
    else
      bd::weight_tiles_bwd_kernel<float><<<min((total + 255) / 256, 2048), 256, 0, st>>>(g, rows, P.cblocks, P.OB,
                                                                                       (const float*)wt, wtiles);
    DCN_KERNEL_CHECK("weight_tiles_bwd_kernel");
  }
  P.xt = xt;
  P.gxt = gxt;
  P.off = off;
  P.gout = gout;
  P.wtiles = wtiles;
  P.gtiles = gtiles;
  P.row_v = 0;
  P.gb_fused = g.variant == DCN_VARIANT_TORCH ? gb_fused : nullptr;
  {
    int rc = g.variant == DCN_VARIANT_TORCH ? launch_gout_tiles(P, bf, gtiles, st)
                                            : launch_gout_tiles_pix(g, operand, gout, gtiles, st);
    if (rc) return rc;
  }
  P.goff = goff;
  P.gw = gw;
  P.ix_delta = (off_col_ch(g, 0) - off_row_ch(g, 0)) * g.HW;
  // grad_offset[row-moving channel] = g_iy * sy * 2 / Dx ; [column-moving channel] = g_ix * sx * 2 / Dy
  // (autograd of train.py:111-113 -> GridSampler.h:27-36; dcn_simt.cu:offset_scale_kernel)
  P.scale_iy = g.variant == DCN_VARIANT_DCNV1 ? 1.f : g.sy * 2.0f / g.Dx;
  P.scale_ix = g.variant == DCN_VARIANT_DCNV1 ? 1.f : g.sx * 2.0f / g.Dy;
  size_t smem = ((size_t)P.g_nbuf * P.OB + (P.g_imgs - P.OB)) * nimg * P.g_img +
                (size_t)(P.w_resident ? P.w_resident : P.w_ring) * P.w_stage +
                (P.fuse_w ? 2 * nimg * (size_t)(128 * 128) : 0) +
                2 * (size_t)P.plan_cap * sizeof(bd::ScatEntry) + 256 + 1024;
  // modulated: the mask values beside the plan ring (float per entry; the kernel traps if the window is too small)
  if (mask) smem += 2 * (size_t)P.plan_cap * sizeof(float);
  if (smem > kSmemBudget) smem = kSmemBudget;  // tight plan (choose_slices): less alignment slack, checked in the kernel
  const int sms = num_sms();
  int grid = P.num_tiles < sms ? P.num_tiles : sms;
  if (P.fuse_w) {
    P.nchunks = sms / P.nslices;
    if (P.nchunks < 1) P.nchunks = 1;
    if (P.nchunks > P.num_tiles) P.nchunks = P.num_tiles;
    grid = P.nslices * P.nchunks;
  }
  const BdLaunch L{P, grid, smem, st, mask, gmask};
  // 16 channels per sampling point: RW = 16 lanes share one
  const bool narrow = g.variant == DCN_VARIANT_TORCH ? P.t.Gt == 16 : g.C == 16;
  KernelScope scope(g.plain ? "umma_offset_conv_bwd_kernel" : "umma_bwd_data_kernel", st);
  if (g.plain) {
    // regular convolution (the companion offset conv): pixel-row layout, fp32, weight gradient fused
    if (g.variant == DCN_VARIANT_TORCH || bf || !P.fuse_w) {
      set_error("plain (offset-conv) backward: pixel-row layout, fp32 operands, fused weight gradient only");
      return DCN_ERR_UNSUPPORTED;
    }
    return launch_bd_split<DCN_VARIANT_JITTOR, true, false, true, false>(L, narrow);
  }
  if (mask) {
    // modulated DCNv1: the pixel-row instantiations with MOD
    if (g.variant != DCN_VARIANT_DCNV1 || !gmask) {
      set_error("umma bwd_data: a mask exists for the DCNv1 variant only, and needs grad_mask");
      return DCN_ERR_UNSUPPORTED;
    }
    return launch_bd_operand<DCN_VARIANT_JITTOR, true>(L, bf, narrow);
  }
  if (g.variant == DCN_VARIANT_TORCH) return launch_bd_operand<DCN_VARIANT_TORCH, false>(L, bf, narrow);
  return launch_bd_operand<DCN_VARIANT_JITTOR, false>(L, bf, narrow);
}

}  // namespace dcn
