// dcn_umma_fwd.cu — forward pass as ONE warp-specialised implicit GEMM on the 5th-gen tensor
// cores (tcgen05.mma, accumulators in TMEM).
//
// Replaces, per 128-row tile and without ever writing columns to HBM:
//   coordinates + bilinear sampling   deform_conv.py:62-68,30-54 / train.py:102-127
//   column layout                     deform_conv.py:72-73       / train.py:129-131
//   GEMM + bias + NCHW store          deform_conv.py:74-81       / train.py:133-140
//
// Warp roles (832 threads, 1 CTA per SM, persistent over tiles; the gather is issue/latency
// bound, so it gets most of the warps):
//   warps 0-3   epilogue : tcgen05.ld accumulator -> + bias -> out[B,O,Ho,Wo]
//   warp  4     MMA      : one lane issues tcgen05.mma (bf16 hi/lo split, 3 MMAs per K step)
//   warp  5     B loader : one lane streams the pre-tiled weight images with cp.async.bulk
//   warps 6-9   plan     : offsets -> bit-exact coordinate chain -> branch-free gather entries
//                          (corner offsets + masked weights) in a 2-deep smem ring, one K block
//                          ahead of the gather warps
//   warps 10-25 gather   : 4x LDG.128 per entry from the channels-last input -> blend ->
//                          bf16 hi/lo -> swizzled smem A images
// Pipelines (all mbarrier based): plan ring (plan -> gather -> back), smem stages
// (gather + loader -> MMA -> back), TMEM accumulators (MMA -> epilogue -> back; 2 buffers).
//
// fp32 parity: every fp32 operand v is split as hi = bf16(v), lo = bf16(v - hi) and the product
// is formed as hi*hi + hi*lo + lo*hi with fp32 accumulation (relative error ~5e-6, measured).
#include <cuda.h>

#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "dcn_umma.h"
#include "dcn_umma_common.cuh"

namespace dcn {

using namespace ptx;

// the plan and gather roles follow the epilogue, MMA and loader warps; their sizes are template arguments
constexpr int kEpiWarps = 4, kFirstPlanWarp = kEpiWarps + 2;
constexpr int kPlanMax = 512;                                    // plan entries per K block (32 B each)
constexpr uint32_t kATile = 128 * 64 * 2;                        // one bf16 A image (16 KB)
constexpr uint32_t kAMnLbo = 1024, kAMnSbo = 2048;               // MN-major A: atom strides
constexpr int kMaxStages = 4;
// forward pipeline depth (fewer when shared memory runs out): a few stages are enough to overlap the (fast) MMAs with
// the (slow) gather; every KB of shared memory not taken stays L1 for the gather's footprint (L1 + smem share 256 KB)
constexpr int kFwdStages = 3;

enum { MODE_FWD = 0, MODE_WGRAD = 1 };

struct FwdParams {
  Geo g;
  Tiling t;
  const void* xt;      // channels-last staging copy: float (fp32 mode) or bfloat16 (bf16 mode)
  const float* off;
  const uint8_t* wtiles;
  const float* bias;
  float* out;
  // weight-gradient mode (MODE_WGRAD): gW[o, j] += sum_rows gout[row, o] * S[row, j]
  const void* gout;    // float or bfloat16
  const uint8_t* gtiles;  // Torch layout: staged grad_out tile images [tile][OB][hi|lo][128 rows x 64 o] (rows in this kernel's order)
  int g_OB;               // ceil(O / 64) images per tile
  float* gw;
  int nslices, nchunks, kb_per_slice;  // CTA = (K slice, chunk of row tiles)
  int o_blocks;                        // ceil(O / 128) accumulators
  int n_gbuf;                          // 1 or 2 buffers for the converted grad_out tile
  uint32_t g_img;                      // bytes of one bf16 image of the grad_out tile: o_blocks*128 rows x 128 B
  int stages;
  int plan_cap;        // plan entries per buffer (n_ent rounded up to 256)
  uint32_t b_tile;     // bytes of one bf16 B image = O*128
  uint32_t stage_bytes;
  uint32_t tmem_cols;  // 2*O rounded to a power of two >= 32
  // Torch layout, forward: out[b, o, r0 + i*R] of a tile is Gt x O runs of only Rt floats, R floats
  // apart.  With tma_out the epilogue stages `tpg` consecutive tiles (box_r = tpg*Rt >= 4 adjacent
  // instances) in shared memory as [o][i][r] and ONE tensor-map store writes the 16-byte runs.
  int tma_out, tpg, box_r, n_ost;  // n_ost = 1 or 2 staging buffers
  uint32_t stage_out_bytes;         // of ONE staging buffer
  // Pixel-row layouts, forward: the K blocks of a tile are (tap, 64-channel slab) pairs, stored tap-major.
  // With kperm_slabs = C / 64 > 1 they are WALKED slab-major (step i -> tap i % N of slab i / N): consecutive
  // steps then gather the same 64 channels around the same pixels (only the tap's offset differs), so the
  // corner lines of one step are L1 hits of the next.  The accumulation order over K is irrelevant.
  int kperm_slabs;
  // modulated instantiations (MOD, DCNv1 only): mask [B, N, Ho, Wo] float32; every sample is scaled by
  // mask[b, n, p], folded into the four corner weights of its plan entry (appended last: the fields above keep
  // their parameter offsets)
  const float* mask;
};

// One plan entry in the making: the index math is done and the two offset loads are in
// flight (issued one K block ahead so that their latency hides behind the gather phase).
// mk: the modulation scalar (MOD instantiations only; loaded on the same prefetch as the offsets).
struct PlanWork {
  float ox, oy;
  int h, w, n, chan_base, valid;
  float mk;
};

template <int VARIANT, bool PLAIN = false, bool MOD = false>
__device__ __forceinline__ void plan_prepare(const Geo& g, const Tiling& t, const float* __restrict__ off,
                                             int tile, int kb, int e, PlanWork& pw,
                                             const float* __restrict__ mask = nullptr) {
  pw.valid = 0;
  pw.ox = pw.oy = 0.f;
  pw.h = pw.w = pw.n = pw.chan_base = 0;
  int b, p, n;
  if (VARIANT == DCN_VARIANT_TORCH) {
    // Rt <= 4: entries are instance-interleaved (e = kk * Rt + il) so that the entries a warp reads
    // together sit next to each other in shared memory, i.e. in different banks; Rt = 8 keeps the
    // instance-major order (e = il * 64 + kk), which measured faster there
    // (Rt is a power of two)
    const int sh = t.Rt == 4 ? 2 : 1;
    const int kk = t.Rt <= 4 ? (e >> sh) : (e & 63), il = t.Rt <= 4 ? (e & (t.Rt - 1)) : (e >> 6), j = kb * 64 + kk;
    const TileRowInfo ri = decode_inst(t, tile * t.Rt + il);
    if (!ri.valid || j >= g.K) return;
    uint32_t cb, q, pp, nn;
    t.divP.divmod((uint32_t)(ri.r0 * g.K + j), cb, q);
    t.divN.divmod(q, pp, nn);
    b = ri.b;
    p = (int)pp;
    n = (int)nn;
    pw.chan_base = (int)cb * t.G + ri.chunk * t.Gt;
  } else {
    const int tl = e >> 7, m = e & 127;
    b = tile / t.pix_blocks;
    p = (tile - b * t.pix_blocks) * 128 + m;
    n = (int)t.divC.div((uint32_t)(kb * 64)) + tl;
    if (p >= g.HW || n >= g.N) return;
  }
  uint32_t h, w;
  t.divWo.divmod((uint32_t)p, h, w);
  pw.h = (int)h;
  pw.w = (int)w;
  pw.n = n;
  if (!PLAIN) {
    const float* ob = off + (size_t)b * 2 * g.N * g.HW;
    pw.ox = __ldg(ob + (size_t)off_row_ch(g, n) * g.HW + p);
    pw.oy = __ldg(ob + (size_t)off_col_ch(g, n) * g.HW + p);
  }
  if constexpr (MOD) {
    static_assert(VARIANT != DCN_VARIANT_TORCH && !PLAIN, "modulation exists for the pixel-row DCNv1 layout only");
    DCN_DEV_ASSERT(((size_t)b * g.N + n) * g.HW + p < (size_t)g.B * g.N * g.HW);
    pw.mk = __ldg(mask + ((size_t)b * g.N + n) * g.HW + p);
  }
  pw.valid = 1;
}

__device__ __forceinline__ PlanEntry plan_finish_plain(const Geo& g, const PlanWork& pw) {
  PlanEntry e;
  int base = xt_null_base(g);
#pragma unroll
  for (int k = 0; k < 4; ++k) e.w[k] = 0.f;
  if (pw.valid) {
    bool inside;
    base = plain_base(g, pw.h, pw.w, pw.n, inside);
    e.w[0] = inside ? 1.f : 0.f;
  }
  base += pw.chan_base;
  e.off[0] = e.off[1] = e.off[2] = e.off[3] = base;
  return e;
}

// coordinate chain (bit-exact, dcn_common.cuh:tap_of) -> branch-free gather entry: corners
// outside the image fall on the zero frame of the staging copy, samples with no corner inside
// (and padding rows / columns) on the frame-only block with zero weights.
// MOD: the corner weights carry the sample's mask (m * w_k; m == 1 leaves them bit-identical)
template <bool MOD = false>
__device__ __forceinline__ PlanEntry plan_finish(const Geo& g, const PlanWork& pw) {
  PlanEntry e;
  int base = xt_null_base(g);
#pragma unroll
  for (int k = 0; k < 4; ++k) e.w[k] = 0.f;
  if (pw.valid) {
    const Tap tp = tap_of(g, pw.h, pw.w, pw.n, pw.ox, pw.oy);
    bool inside;
    base = xt_corner_base(g, tp.y0, tp.x0, inside);
    if (inside) corner_weights(tp, e.w);
    if constexpr (MOD) {
#pragma unroll
      for (int k = 0; k < 4; ++k) e.w[k] = __fmul_rn(e.w[k], pw.mk);
    }
  }
  base += pw.chan_base;
  const int pitch = xt_row_pitch(g);
  e.off[0] = base;
  e.off[1] = base + g.C;
  e.off[2] = base + pitch;
  e.off[3] = base + pitch + g.C;
  return e;
}

__device__ __forceinline__ float4 blend4(const float4 v[4], const PlanEntry& e) {
  float4 r;
  r.x = fmaf(v[3].x, e.w[3], fmaf(v[2].x, e.w[2], fmaf(v[1].x, e.w[1], v[0].x * e.w[0])));
  r.y = fmaf(v[3].y, e.w[3], fmaf(v[2].y, e.w[2], fmaf(v[1].y, e.w[1], v[0].y * e.w[0])));
  r.z = fmaf(v[3].z, e.w[3], fmaf(v[2].z, e.w[2], fmaf(v[1].z, e.w[1], v[0].z * e.w[0])));
  r.w = fmaf(v[3].w, e.w[3], fmaf(v[2].w, e.w[2], fmaf(v[1].w, e.w[1], v[0].w * e.w[0])));
  return r;
}

// float4 -> 4 bf16 hi + 4 bf16 lo, each packed in 8 bytes
__device__ __forceinline__ void split4(const float4& v, uint2& hi, uint2& lo) {
  split_pair(v.x, v.y, hi.x, lo.x);
  split_pair(v.z, v.w, hi.y, lo.y);
}

// BF = bf16 operand mode (DCN_OPERAND_BF16): x / weight / grad_out are bfloat16 in HBM, every
// operand is ONE bf16 image and every K step ONE MMA; otherwise fp32 with the hi/lo split (two
// images, three MMAs).  A gather item is one 16-byte load per corner: V = 4 fp32 or 8 bf16 channels.
// PLAIN = regular convolution on the same machinery (the companion offset conv): one exact pixel per entry.
// PW / GW = plan / gather warps.  4 + 16 everywhere except the Torch layout with 16 channels per sampling point
// (Rt = 8: 512 coordinate chains per K block for 2048 gather items — the 4 plan warps, one per scheduler, were the
// critical path and the gather warps waited 40 % of the time, profiles/r1_ncu_det2.txt): 8 + 8 there.
// MOD = modulated deformable convolution (DCNv2, pixel-row layout): the plan warps scale each entry's corner weights
// by its mask value, so the gather, MMA and epilogue roles are the unmodulated ones.
template <int VARIANT, int MODE, bool BF, bool PLAIN = false, int PW = 4, int GW = 16, bool MOD = false>
__global__ void __launch_bounds__((kFirstPlanWarp + PW + GW) * 32, 1)
    umma_gemm_kernel(const __grid_constant__ FwdParams P, const __grid_constant__ CUtensorMap tmap_out) {
  // role layout of this instantiation
  constexpr int kPlanWarps = PW, kProdWarps = GW;
  constexpr int kPlanThreads = PW * 32, kProdThreads = GW * 32;
  constexpr int kFirstProdWarp = kFirstPlanWarp + PW;
  constexpr int kFwdThreads = (kFirstProdWarp + GW) * 32;
  static_assert(kPlanMax % kPlanThreads == 0, "every plan thread owns the same number of plan slots");
  constexpr int kPlanPerThread = kPlanMax / kPlanThreads;
  constexpr int V = BF ? 8 : 4;
  constexpr int NIMG = BF ? 1 : 2;
  constexpr int kIt = 128 * 64 / V / kProdThreads;  // gather items per thread and K block: 4 or 2
  typedef typename std::conditional<BF, __nv_bfloat16, float>::type XT;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 1024-byte alignment by pointer arithmetic (a uintptr_t round trip would lose the shared
  // address space and turn every LDS/STS below into a slow generic LD/ST)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const Geo& g = P.g;
  const Tiling& t = P.t;
  // carve-up: [stages x (A_hi | A_lo | B_hi | B_lo)] [grad_out tile buffers (WGRAD)] [plan x2] [barriers]
  uint8_t* stage_base = smem;
  uint8_t* gbuf_base = smem + (size_t)P.stages * P.stage_bytes;
  const uint32_t gbuf_bytes = MODE == MODE_WGRAD ? 2u * NIMG * P.g_img : 0u;  // 2 row halves x (hi | lo)
  float* ostage = reinterpret_cast<float*>(gbuf_base);  // forward + tma_out: [O][Gt][box_r] floats
  PlanEntry* plan = reinterpret_cast<PlanEntry*>(gbuf_base + (size_t)(MODE == MODE_WGRAD ? P.n_gbuf : 0) * gbuf_bytes +
                                                 (MODE == MODE_FWD ? P.n_ost * P.stage_out_bytes : 0u));
  uint64_t* bars = reinterpret_cast<uint64_t*>(plan + 2 * P.plan_cap);
  uint64_t* full = bars;                   // [stages]
  uint64_t* empty = bars + kMaxStages;     // [stages]
  uint64_t* tfull = bars + 2 * kMaxStages; // [2]
  uint64_t* tempty = tfull + 2;            // [2]
  uint64_t* pfull = tempty + 2;            // [2] plan ring
  uint64_t* pempty = pfull + 2;            // [2]
  uint64_t* afull = pempty + 2;            // [2] converted grad_out tile (WGRAD)
  uint64_t* aempty = afull + 2;            // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(aempty + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  DCN_DBG_ONLY(__shared__ int dbg_steps[5]; if (tid < 5) dbg_steps[tid] = -1; int dbg_n = 0;)
  const int O = g.O;
  // which (tile, K block) pairs this CTA walks: forward = all K blocks of every gridDim-th tile;
  // weight gradient = one slice of K blocks for one chunk of the row tiles
  int tile0, tile_step, kb0, kb1;
  if (MODE == MODE_FWD) {
    tile0 = blockIdx.x;
    tile_step = gridDim.x;
    kb0 = 0;
    kb1 = t.KB;
    if (P.tpg == 2) tile0 = 2 * blockIdx.x;  // CTAs walk PAIRS of tiles: 2c, 2c+1, 2(c+grid), ...
  } else {
    const int slice = blockIdx.x % P.nslices;
    tile0 = blockIdx.x / P.nslices;
    tile_step = P.nchunks;
    kb0 = slice * P.kb_per_slice;
    kb1 = min(t.KB, kb0 + P.kb_per_slice);
  }
  const bool pairs = MODE == MODE_FWD && P.tpg == 2;
  auto next_tile = [&](int tile) {
    return pairs ? ((tile & 1) ? tile + 2 * (int)gridDim.x - 1 : tile + 1) : tile + tile_step;
  };
  // step of the K loop -> K block (see FwdParams::kperm_slabs)
  auto kb_of = [&](int i) {
    if (MODE != MODE_FWD || P.kperm_slabs <= 1) return i;
    uint32_t slab, tap;
    t.divN.divmod((uint32_t)i, slab, tap);
    return (int)(tap * (uint32_t)P.kperm_slabs + slab);
  };

  if (tid == 0) {
    for (int s = 0; s < P.stages; ++s) {
      mbar_init(&full[s], MODE == MODE_FWD ? kProdWarps + 1 : kProdWarps);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], kEpiWarps);
      mbar_init(&pfull[a], kPlanWarps);
      mbar_init(&pempty[a], kProdWarps);
      mbar_init(&afull[a], 1);
      mbar_init(&aempty[a], 1);
    }
    fence_barrier_init();
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(tmem_slot)),
                 "r"(P.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (MODE == MODE_WGRAD && (P.g_OB & 1)) {
    // O is not a multiple of 128: the upper 64-o half of the last M = 128 operand stays zero
    for (int ab = 0; ab < P.n_gbuf; ++ab) {
      uint8_t* z = gbuf_base + (size_t)ab * gbuf_bytes + (size_t)P.g_OB * NIMG * kATile;
      for (uint32_t i = tid * 16; i < NIMG * kATile; i += kFwdThreads * 16)
        *reinterpret_cast<uint4*>(z + i) = make_uint4(0, 0, 0, 0);
    }
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < kEpiWarps) {
    if constexpr (MODE == MODE_FWD) {
    // ================================================================ epilogue (forward)
    uint32_t acc_phase = 0;
    int acc = 0, ost = 0;
    const int m = warp * 32 + lane;  // TMEM lane == tile row
    for (int tile = tile0; tile < t.num_tiles; tile = next_tile(tile)) {
      size_t out_off = 0;
      bool valid;
      int il = 0, ich = 0;           // Torch: class instance inside the tile, channel inside the Gt chunk
      TileRowInfo ri0 = {0, 0, 0, 0};
      if (VARIANT == DCN_VARIANT_TORCH) {
        // tile row m = grp*(V*Rt) + il*V + ch: V channels of class instance il are V consecutive rows
        const int grp = m / (V * t.Rt), ch = m % V;
        il = (m / V) % t.Rt;
        ich = V * grp + ch;
        const TileRowInfo ri = decode_inst(t, tile * t.Rt + il);
        valid = ri.valid;
        const int i = ri.chunk * t.Gt + ich;
        out_off = (size_t)ri.b * g.Oimg * g.HW + (size_t)(ri.r0 + i * t.R);
        if (P.tma_out) ri0 = decode_inst(t, (tile - (tile % P.tpg)) * t.Rt);  // first instance of the group
      } else {
        const int b = tile / t.pix_blocks, p = (tile - b * t.pix_blocks) * 128 + m;
        valid = p < g.HW;
        out_off = (size_t)b * g.Oimg * g.HW + p;
      }
      mbar_wait_relaxed(&tfull[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(acc * O);
      if (VARIANT == DCN_VARIANT_TORCH && P.tma_out) {
        const int sub = tile % P.tpg;  // position of this tile inside its staging group
        if (sub == 0) {
          // the store that last used this staging buffer must have finished reading it
          if (tid == 0) {
            if (P.n_ost == 2) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            else asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          }
          asm volatile("bar.sync 1, 128;" ::: "memory");
        }
        float* obuf = ostage + (size_t)ost * (P.stage_out_bytes >> 2);
        float* dst = obuf + (size_t)ich * P.box_r + sub * t.Rt + il;
        const int o_stride = t.Gt * P.box_r;
        for (int c0 = 0; c0 < O; c0 += 16) {
          float v[16];
          tmem_ld16(taddr + c0, v);
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float bv = P.bias ? __ldg(P.bias + c0 + i) : 0.f;
            const float r = v[i] + bv;
            dst[(size_t)(c0 + i) * o_stride] = g.relu_out ? fmaxf(r, 0.f) : r;
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[acc]);
        if (sub == P.tpg - 1) {
          fence_proxy_async_smem();  // generic-proxy writes -> visible to the bulk-copy engine
          asm volatile("bar.sync 1, 128;" ::: "memory");
          if (tid == 0) {
            // box {box_r, Gt, O, 1} at (r0, chunk*Gt, 0, b) of out viewed as [B][O][G][R]
            asm volatile(
                "cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                    reinterpret_cast<uint64_t>(&tmap_out)),
                "r"(smem_u32(obuf)), "r"(ri0.r0), "r"(ri0.chunk * t.Gt), "r"(0), "r"(ri0.b)
                : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
          if (P.n_ost == 2) ost ^= 1;
        }
      } else if (!PLAIN && g.out_framed) {
        // chained inference: this row's pixel of the CONSUMER's framed channels-last copy (Geo::out_framed)
        const int bimg = (int)(out_off / ((size_t)g.Oimg * g.HW)), pix = (int)(out_off - (size_t)bimg * g.Oimg * g.HW);
        uint32_t oh, ow;
        t.divWo.divmod((uint32_t)(valid ? pix : 0), oh, ow);
        float* dst = P.out + (((size_t)bimg * (g.Ho + 3) + oh + 1) * (g.Wo + 2) + ow + 1) * g.O;
        for (int c0 = 0; c0 < O; c0 += 16) {
          float v[16];
          tmem_ld16(taddr + c0, v);
          if (valid) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int o = c0 + i;
              const float bv = P.bias ? __ldg(P.bias + o) : 0.f;
              const float r = v[i] + bv;
              const int od = g.out_G ? (o % g.out_Cs) * g.out_G + o / g.out_Cs : o;
              dst[od] = g.relu_out ? fmaxf(r, 0.f) : r;
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[acc]);
      } else {
        for (int c0 = 0; c0 < O; c0 += 16) {
          float v[16];
          tmem_ld16(taddr + c0, v);
          if (valid) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              if (PLAIN && c0 + i >= g.o_valid) break;   // padded accumulator columns of a plain problem
              const float bv = P.bias ? __ldg(P.bias + c0 + i) : 0.f;
              const float r = v[i] + bv;
              DCN_DEV_ASSERT(out_off + (size_t)(c0 + i) * g.HW < (size_t)g.B * g.Oimg * g.HW);
              P.out[out_off + (size_t)(c0 + i) * g.HW] = g.relu_out ? fmaxf(r, 0.f) : r;
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[acc]);
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    // the last tensor store must have left shared memory before the CTA exits
    if (VARIANT == DCN_VARIANT_TORCH && P.tma_out && tid == 0)
      asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    } else {
    // ================================================================ grad_out tile loader, then the
    // one-shot epilogue (weight gradient).  The tile's operand images [ob][hi | lo][128 rows x 64 o] were staged
    // once per backward pass (gout_tiles_*_kernel, rows in this kernel's order): one bulk copy per tile.
    if (tid == 0) {
      int ab = 0;
      uint32_t aphase = 0;
      const uint32_t bytes = (uint32_t)P.g_OB * NIMG * kATile;
      for (int tile = tile0; tile < t.num_tiles; tile = next_tile(tile)) {
        mbar_wait_relaxed(&aempty[ab], aphase ^ 1);
        mbar_arrive_expect_tx(&afull[ab], bytes);
        bulk_g2s(gbuf_base + (size_t)ab * gbuf_bytes, P.gtiles + (size_t)tile * bytes, bytes, &afull[ab]);
        if (P.n_gbuf == 2) {
          ab ^= 1;
          if (ab == 0) aphase ^= 1;
        } else {
          aphase ^= 1;
        }
      }
    }
    // ---- epilogue: accumulators -> gW (one red.global.add per element; each CTA owns a K slice
    // for a chunk of the rows, so O*K*nchunks adds in total)
    mbar_wait_relaxed(&tfull[0], 0);
    tc_fence_after();
    const int ncols = (kb1 - kb0) * 64;
    for (int ob = 0; ob < P.o_blocks; ++ob) {
      const int o = ob * 128 + warp * 32 + lane;
      const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(ob * ncols);
      for (int c0 = 0; c0 < ncols; c0 += 16) {
        float v[16];
        tmem_ld16(taddr + c0, v);
        if (o < O) {
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const int j = kb0 * 64 + c0 + i;
            if (j < g.K) atomicAdd(P.gw + wt_index(g, o, j), v[i]);
          }
        }
      }
    }
    tc_fence_before();
    }
  } else if (warp == kEpiWarps) {
    if constexpr (MODE == MODE_FWD) {
    // ================================================================ MMA issuer (forward)
    // The whole warp runs this (uniform) loop and elect.sync picks the issuing lane per instruction; every descriptor
    // is one 64-bit add onto a per-stage base (the address field is the low 14 bits, 18-bit shared addresses never
    // carry out of it).  Inside `if (lane == 0)` the compiler wraps every tcgen05.mma in a waterfall loop and the
    // four descriptors of a K = 16 step cost ~40 dependent integer instructions: ~130 issue cycles per MMA, which is
    // what an N = 256 MMA takes to EXECUTE (tools/mma_rate_probe.cu) — the issuer, not the tensor pipe, set the pace of
    // the O = 256 layers.
    {
      const uint32_t idesc = make_idesc_bf16(128, O, VARIANT == DCN_VARIANT_TORCH, false);
      const uint64_t adesc0 = VARIANT == DCN_VARIANT_TORCH ? make_sdesc_sw128(smem_u32(stage_base), kAMnLbo, kAMnSbo)
                                                           : make_sdesc_sw128(smem_u32(stage_base), 16, 1024);
      const uint64_t bdesc0 = make_sdesc_sw128(smem_u32(stage_base) + NIMG * kATile, 16, 1024);
      const uint32_t stage16 = P.stage_bytes >> 4, btile16 = P.b_tile >> 4;
      constexpr uint32_t kATile16 = kATile >> 4;
      constexpr uint32_t kAStep16 = VARIANT == DCN_VARIANT_TORCH ? (2 * kAMnSbo) >> 4 : 2;   // K = 16 step of the A image
      int s = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      for (int tile = tile0; tile < t.num_tiles; tile = next_tile(tile)) {
        mbar_wait_relaxed(&tempty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * O);
        for (int kb = 0; kb < t.KB; ++kb) {
          mbar_wait_relaxed(&full[s], phase, 64);
          tc_fence_after();
          const uint64_t a_hi = adesc0 + (uint64_t)((uint32_t)s * stage16), b_hi = bdesc0 + (uint64_t)((uint32_t)s * stage16);
          if (elect_one()) {
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4) {
              const uint64_t dah = a_hi + (uint64_t)(k4 * kAStep16), dbh = b_hi + (uint64_t)(k4 * 2);
              umma_bf16(d_tmem, dah, dbh, idesc, (kb | k4) ? 1u : 0u);
              if (!BF) {
                umma_bf16(d_tmem, dah, dbh + btile16, idesc, 1u);
                umma_bf16(d_tmem, dah + kATile16, dbh, idesc, 1u);
              }
            }
            umma_commit(&empty[s]);  // stage reusable once these MMAs have read it
            if (kb == t.KB - 1) umma_commit(&tfull[acc]);
          }
          __syncwarp();
          DCN_DBG_ONLY(++dbg_n;)
          if (++s == P.stages) {
            s = 0;
            phase ^= 1;
          }
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
      DCN_DBG_ONLY(if (lane == 0) dbg_steps[0] = dbg_n;)
    }
    } else {
    // ================================================================ MMA issuer (weight gradient)
    // D[o, j] += g^T[o, rows] * S[rows, j]: A = converted grad_out tile (K-major, K = tile rows),
    // B = the sample image the gather warps wrote — the forward's A image read as a B operand:
    //   Torch  image (rows contiguous per column) = K-major B, 8-column groups 2048 B apart,
    //          row half h at +1024;
    //   Jittor image (columns contiguous per row) = MN-major B, 8-row groups 1024 B apart.
    if (lane == 0) {
      // A = staged grad_out images [row][64 o] read MN-major (o contiguous, 64-o atoms = consecutive images);
      // B = the sample image: K-major for the Torch layout, MN-major for the pixel-row layouts
      const uint32_t idesc = make_idesc_bf16(128, 64, true, VARIANT != DCN_VARIANT_TORCH);
      const int ncols = (kb1 - kb0) * 64;
      int s = 0, ab = 0;
      uint32_t phase = 0, aphase = 0;
      bool first_tile = true;
      for (int tile = tile0; tile < t.num_tiles; tile = next_tile(tile)) {
        mbar_wait_relaxed(&afull[ab], aphase, 64);
        const uint32_t gb = smem_u32(gbuf_base + (size_t)ab * gbuf_bytes);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait_relaxed(&full[s], phase, 64);
          tc_fence_after();
          const uint32_t s_hi = smem_u32(stage_base + (size_t)s * P.stage_bytes);
          const uint32_t s_lo = s_hi + kATile;
#pragma unroll
          for (int ks = 0; ks < 8; ++ks) {  // 8 steps of 16 tile rows
            const int h = ks >> 2, k4 = ks & 3;
            uint64_t dsh, dsl;
            if (VARIANT == DCN_VARIANT_TORCH) {
              dsh = make_sdesc_sw128(s_hi + h * 1024 + k4 * 32, 16, 2048);
              dsl = make_sdesc_sw128(s_lo + h * 1024 + k4 * 32, 16, 2048);
            } else {
              dsh = make_sdesc_sw128(s_hi + ks * 2048, 1024, 1024);
              dsl = make_sdesc_sw128(s_lo + ks * 2048, 1024, 1024);
            }
            for (int ob = 0; ob < P.o_blocks; ++ob) {
              const uint32_t g_hi = gb + (uint32_t)(2 * ob) * NIMG * kATile + ks * 2048;
              const uint64_t dgh = make_sdesc_sw128(g_hi, NIMG * kATile, 1024);
              const uint64_t dgl = make_sdesc_sw128(g_hi + kATile, NIMG * kATile, 1024);
              const uint32_t d_tmem = tmem_base + (uint32_t)(ob * ncols + (kb - kb0) * 64);
              umma_bf16(d_tmem, dgh, dsh, idesc, (first_tile && ks == 0) ? 0u : 1u);
              if (!BF) {
                umma_bf16(d_tmem, dgh, dsl, idesc, 1u);
                umma_bf16(d_tmem, dgl, dsh, idesc, 1u);
              }
            }
          }
          umma_commit(&empty[s]);
          if (++s == P.stages) {
            s = 0;
            phase ^= 1;
          }
        }
        umma_commit(&aempty[ab]);  // grad_out tile buffer reusable
        first_tile = false;
        if (P.n_gbuf == 2) {
          ab ^= 1;
          if (ab == 0) aphase ^= 1;
        } else {
          aphase ^= 1;
        }
      }
      umma_commit(&tfull[0]);
    }
    }
  } else if (warp == kEpiWarps + 1) {
    // ================================================================ weight (B) loader (forward only)
    if (MODE == MODE_FWD && lane == 0) {
      int s = 0;
      uint32_t phase = 0;
      for (int tile = tile0; tile < t.num_tiles; tile = next_tile(tile)) {
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait_relaxed(&empty[s], phase ^ 1);
          uint8_t* dst = stage_base + (size_t)s * P.stage_bytes + NIMG * kATile;
          mbar_arrive_expect_tx(&full[s], NIMG * P.b_tile);
          bulk_g2s(dst, P.wtiles + (size_t)kb_of(kb) * NIMG * P.b_tile, NIMG * P.b_tile, &full[s]);
          DCN_DBG_ONLY(++dbg_n;)
          if (++s == P.stages) {
            s = 0;
            phase ^= 1;
          }
        }
      }
      DCN_DBG_ONLY(dbg_steps[1] = dbg_n;)
    }
  } else if (warp < kFirstProdWarp) {
    // ================================================================ plan warps
    const int pt = tid - kFirstPlanWarp * 32;  // 0..63
    const int n_ent = VARIANT == DCN_VARIANT_TORCH ? t.Rt * 64 : 128 * t.taps_per_kb;
    int pbuf = 0;
    uint32_t pphase = 0;
    PlanWork pw[kPlanPerThread];
    if (tile0 < t.num_tiles) {
#pragma unroll
      for (int u = 0; u < kPlanPerThread; ++u)
        if (pt + u * kPlanThreads < n_ent)
          plan_prepare<VARIANT, PLAIN, MOD>(g, t, P.off, tile0, kb_of(kb0), pt + u * kPlanThreads, pw[u], P.mask);
    }
    for (int tile = tile0; tile < t.num_tiles; tile = next_tile(tile)) {
      for (int kb = kb0; kb < kb1; ++kb) {
        PlanEntry* pl = plan + pbuf * P.plan_cap;
        mbar_wait_relaxed(&pempty[pbuf], pphase ^ 1, 64);
        // finish this K block's entries (their offset loads were issued one block ago) ...
#pragma unroll
        for (int u = 0; u < kPlanPerThread; ++u)
          if (pt + u * kPlanThreads < n_ent)
            pl[pt + u * kPlanThreads] = PLAIN ? plan_finish_plain(g, pw[u]) : plan_finish<MOD>(g, pw[u]);
        __syncwarp();
        if (lane == 0) mbar_arrive(&pfull[pbuf]);
        // ... and start the next block's
        int ntile = tile, nkb = kb + 1;
        if (nkb == kb1) {
          nkb = kb0;
          ntile = next_tile(tile);
        }
        if (ntile < t.num_tiles) {
#pragma unroll
          for (int u = 0; u < kPlanPerThread; ++u)
            if (pt + u * kPlanThreads < n_ent)
              plan_prepare<VARIANT, PLAIN, MOD>(g, t, P.off, ntile, kb_of(nkb), pt + u * kPlanThreads, pw[u], P.mask);
        }
        pbuf ^= 1;
        if (pbuf == 0) pphase ^= 1;
        DCN_DBG_ONLY(++dbg_n;)
      }
    }
    DCN_DBG_ONLY(if (pt == 0) dbg_steps[2] = dbg_n;)
  } else {
    // ================================================================ gather warps
    // kIt items (one 16-byte load per corner: 4 fp32 or 8 bf16 channels) per thread and K block,
    // software pipelined one item deep: the 4 LDG.128 of item i+1 (possibly the first item of the
    // NEXT K block) are issued before item i is blended, so every warp always has gathers in flight.
    const int pt = tid - kFirstProdWarp * 32;  // 0..511
    const size_t img_stride = xt_image_stride(g);
    const XT* xt = reinterpret_cast<const XT*>(P.xt);
    // `groups` lanes share one sampling point; a "pair" is one (class instance, column) of the
    // Torch tile or one row of the Jittor tile
    const int groups = VARIANT == DCN_VARIANT_TORCH ? (t.Gt / V) : (64 / V);
    int grp = pt % groups, slot = pt / groups;
    const int pairs_per_pass = kProdThreads / groups;
    // fp32, Gt = 64 (two class instances of 16 groups): a 64-bit shared store is served per half-warp,
    // and the 8-byte pieces of a half-warp must fall into 32 different banks.  Lanes are therefore
    // laid out (group low 3 bits, instance, group high bit): each quarter-warp still gathers one
    // contiguous 128-byte run of ONE entry, while a half-warp stores both 8-byte halves (instance 0 / 1)
    // of 8 different 16-byte chunks — conflict-free, where the plain order was a 2-way conflict.
    const bool paired = VARIANT == DCN_VARIANT_TORCH && !BF && t.Rt == 2;
    if (paired) grp = (lane & 7) | ((lane >> 4) << 3);
    int ent_idx[kIt], item_il[kIt];
    uint32_t st_off[kIt];
#pragma unroll
    for (int it = 0; it < kIt; ++it) {
      const int pair = slot + it * pairs_per_pass;
      if (VARIANT == DCN_VARIANT_TORCH) {
        // consecutive slots read consecutive plan entries (see plan_prepare)
        int il = t.Rt <= 4 ? pair % t.Rt : (pair >> 6), kk = t.Rt <= 4 ? pair / t.Rt : (pair & 63);
        if (paired) {
          il = (lane >> 3) & 1;
          kk = (warp - kFirstProdWarp) + kProdWarps * it;
        }
        item_il[it] = il;
        ent_idx[it] = t.Rt <= 4 ? kk * t.Rt + il : il * 64 + kk;
        st_off[it] = mnmajor_sw128_off(grp * (V * t.Rt) + il * V, kk, kAMnLbo, kAMnSbo);
      } else {
        item_il[it] = 0;
        ent_idx[it] = pair;  // row m
        st_off[it] = kmajor_sw128_off(pair, grp * V);
      }
    }
    // position of one K block in the three rings it touches
    struct Pos {
      int tile, kb, s, pbuf;
      uint32_t phase, pphase;
      int kbm;  // the K block this step works on: kb_of(kb)
    };
    auto advance = [&](Pos& q) {
      if (++q.kb == kb1) {
        q.kb = kb0;
        q.tile = next_tile(q.tile);
      }
      if (++q.s == P.stages) {
        q.s = 0;
        q.phase ^= 1;
      }
      q.pbuf ^= 1;
      if (q.pbuf == 0) q.pphase ^= 1;
      q.kbm = kb_of(q.kb);
    };
    const XT* img[kIt];  // load side: image base (+ channel group) of each item's rows
    auto set_images = [&](int tile) {
#pragma unroll
      for (int it = 0; it < kIt; ++it) {
        if (VARIANT == DCN_VARIANT_TORCH)
          img[it] = xt + (size_t)decode_inst(t, tile * t.Rt + item_il[it]).b * img_stride + grp * V;
        else
          img[it] = xt + (size_t)(tile / t.pix_blocks) * img_stride;
      }
    };
    // Jittor layout: channel offset / tap slot of this thread's V columns inside K block kb
    auto jit_cols = [&](int kb, int& c, int& tl, bool& ok) {
      // (multiply-high division: this runs twice per gather item, a hardware-less `/` cost 12 % of the
      // bf16 forward kernel's issue slots)
      const int j = kb * 64 + grp * V;
      const int n = (int)t.divC.div((uint32_t)j);
      c = j - n * g.C;
      tl = n - (int)t.divC.div((uint32_t)(kb * 64));
      ok = j < g.K;
    };
    uint4 v[2][4];  // [buffer][corner], 16 raw bytes each
    auto issue = [&](const Pos& q, int it, int buf) {
      const PlanEntry* pl = plan + q.pbuf * P.plan_cap;
      int jc = 0, tl = 0;
      bool ok = true;
      if (VARIANT != DCN_VARIANT_TORCH) {
        jit_cols(q.kbm, jc, tl, ok);
        pl += tl * 128;
      }
      const XT* base = img[it] + jc;
      DCN_DEV_ASSERT(base >= xt && pl[ent_idx[it]].off[0] >= 0 &&
                     (size_t)(base - xt) + (size_t)pl[ent_idx[it]].off[3] + V <= (size_t)g.B * img_stride);
      if (PLAIN) {
        v[buf][0] = __ldg(reinterpret_cast<const uint4*>(base + pl[ent_idx[it]].off[0]));
      } else {
        const int4 off = *reinterpret_cast<const int4*>(pl[ent_idx[it]].off);
        v[buf][0] = __ldg(reinterpret_cast<const uint4*>(base + off.x));
        v[buf][1] = __ldg(reinterpret_cast<const uint4*>(base + off.y));
        v[buf][2] = __ldg(reinterpret_cast<const uint4*>(base + off.z));
        v[buf][3] = __ldg(reinterpret_cast<const uint4*>(base + off.w));
      }
    };
    // blend one pair of channels held as the two bf16 halves of a word (bf16 mode)
    auto blend_bf = [](uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, const float4& w) {
      const float lo = fmaf(__uint_as_float(a3 << 16), w.w,
                            fmaf(__uint_as_float(a2 << 16), w.z,
                                 fmaf(__uint_as_float(a1 << 16), w.y, __uint_as_float(a0 << 16) * w.x)));
      const float hi = fmaf(__uint_as_float(a3 & 0xffff0000u), w.w,
                            fmaf(__uint_as_float(a2 & 0xffff0000u), w.z,
                                 fmaf(__uint_as_float(a1 & 0xffff0000u), w.y,
                                      __uint_as_float(a0 & 0xffff0000u) * w.x)));
      return pack_bf16x2(lo, hi);
    };
    auto blend_f = [](uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, const float4& w) {
      return fmaf(__uint_as_float(a3), w.w,
                  fmaf(__uint_as_float(a2), w.z, fmaf(__uint_as_float(a1), w.y, __uint_as_float(a0) * w.x)));
    };
    Pos cur{tile0, kb0, 0, 0, 0u, 0u, kb_of(kb0)};
    if constexpr (PLAIN) {
      // One exact pixel per item = ONE 16-byte load: with the one-item-deep pipeline below a thread had a single load
      // in flight and the kernel ran at the L2 latency (2.45 ms for the cfg2 offset conv, 4x the L1 time of its
      // gathers).  Here every thread issues ALL kIt loads of the NEXT K block before it converts the current one:
      // kIt .. 2*kIt loads in flight per thread, two register sets used alternately (static indexing).
      uint4 va[kIt], vb[kIt];
      auto issue_all = [&](const Pos& q, uint4 (&dst)[kIt]) {
        const PlanEntry* pl = plan + q.pbuf * P.plan_cap;
        int jc, tl;
        bool ok;
        jit_cols(q.kbm, jc, tl, ok);
        pl += tl * 128;
#pragma unroll
        for (int it = 0; it < kIt; ++it)
          dst[it] = __ldg(reinterpret_cast<const uint4*>(img[it] + jc + pl[ent_idx[it]].off[0]));
      };
      auto convert = [&](const Pos& q, const uint4 (&src)[kIt]) {
        const PlanEntry* pl = plan + q.pbuf * P.plan_cap;
        int jc, tl;
        bool col_ok;
        jit_cols(q.kbm, jc, tl, col_ok);
        pl += tl * 128;
        uint8_t* a_hi = stage_base + (size_t)q.s * P.stage_bytes;
        uint8_t* a_lo = a_hi + kATile;
#pragma unroll
        for (int it = 0; it < kIt; ++it) {
          const float w = col_ok ? pl[ent_idx[it]].w[0] : 0.f;  // 1, or 0 for padding columns / positions off the frame
          float4 r;
          r.x = __uint_as_float(src[it].x) * w;
          r.y = __uint_as_float(src[it].y) * w;
          r.z = __uint_as_float(src[it].z) * w;
          r.w = __uint_as_float(src[it].w) * w;
          uint2 hi, lo;
          split4(r, hi, lo);
          *reinterpret_cast<uint2*>(a_hi + st_off[it]) = hi;
          *reinterpret_cast<uint2*>(a_lo + st_off[it]) = lo;
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(&full[q.s]);
          mbar_arrive(&pempty[q.pbuf]);
        }
        DCN_DBG_ONLY(++dbg_n;)
      };
      auto start = [&](const Pos& q, const Pos& prev, uint4 (&dst)[kIt]) {
        if (q.tile != prev.tile) set_images(q.tile);
        mbar_wait(&pfull[q.pbuf], q.pphase);
        mbar_wait(&empty[q.s], q.phase ^ 1);
        issue_all(q, dst);
      };
      if (cur.tile < t.num_tiles) {
        set_images(cur.tile);
        start(cur, cur, va);
      }
      while (cur.tile < t.num_tiles) {
        Pos nxt = cur;
        advance(nxt);
        const bool nv = nxt.tile < t.num_tiles;
        if (nv) start(nxt, cur, vb);
        convert(cur, va);
        if (!nv) break;
        Pos nn = nxt;
        advance(nn);
        if (nn.tile < t.num_tiles) start(nn, nxt, va);
        convert(nxt, vb);
        cur = nn;
      }
    } else {
    if (cur.tile < t.num_tiles) {
      set_images(cur.tile);
      mbar_wait(&pfull[cur.pbuf], cur.pphase);
      mbar_wait(&empty[cur.s], cur.phase ^ 1);
      issue(cur, 0, 0);
    }
    while (cur.tile < t.num_tiles) {
      Pos nxt = cur;
      advance(nxt);
      const PlanEntry* pl = plan + cur.pbuf * P.plan_cap;
      bool col_ok = true;
      if (VARIANT != DCN_VARIANT_TORCH) {
        int jc, tl;
        jit_cols(cur.kbm, jc, tl, col_ok);
        pl += tl * 128;
      }
      uint8_t* a_hi = stage_base + (size_t)cur.s * P.stage_bytes;
      uint8_t* a_lo = a_hi + kATile;
#pragma unroll
      for (int it = 0; it < kIt; ++it) {
        // keep the L1 fed: next item first
        if (it < kIt - 1) {
          issue(cur, it + 1, (it + 1) & 1);
        } else if (nxt.tile < t.num_tiles) {
          if (nxt.tile != cur.tile) set_images(nxt.tile);
          mbar_wait(&pfull[nxt.pbuf], nxt.pphase);
          mbar_wait(&empty[nxt.s], nxt.phase ^ 1);
          issue(nxt, 0, 0);
        }
        float4 w = *reinterpret_cast<const float4*>(pl[ent_idx[it]].w);
        if (VARIANT != DCN_VARIANT_TORCH && !col_ok) w = make_float4(0.f, 0.f, 0.f, 0.f);
        const uint4* c4 = v[it & 1];
        if (PLAIN) {
          // one exact pixel: the "blend" is a product with 1 (or with 0 for padding columns / positions off the frame)
          float4 r;
          r.x = __uint_as_float(c4[0].x) * w.x;
          r.y = __uint_as_float(c4[0].y) * w.x;
          r.z = __uint_as_float(c4[0].z) * w.x;
          r.w = __uint_as_float(c4[0].w) * w.x;
          uint2 hi, lo;
          split4(r, hi, lo);
          *reinterpret_cast<uint2*>(a_hi + st_off[it]) = hi;
          *reinterpret_cast<uint2*>(a_lo + st_off[it]) = lo;
        } else if (BF) {
          // 8 channels: blend in fp32, ONE bf16 rounding of the sample, one 16-byte store
          uint4 r;
          r.x = blend_bf(c4[0].x, c4[1].x, c4[2].x, c4[3].x, w);
          r.y = blend_bf(c4[0].y, c4[1].y, c4[2].y, c4[3].y, w);
          r.z = blend_bf(c4[0].z, c4[1].z, c4[2].z, c4[3].z, w);
          r.w = blend_bf(c4[0].w, c4[1].w, c4[2].w, c4[3].w, w);
          *reinterpret_cast<uint4*>(a_hi + st_off[it]) = r;
        } else {
          float4 r;
          r.x = blend_f(c4[0].x, c4[1].x, c4[2].x, c4[3].x, w);
          r.y = blend_f(c4[0].y, c4[1].y, c4[2].y, c4[3].y, w);
          r.z = blend_f(c4[0].z, c4[1].z, c4[2].z, c4[3].z, w);
          r.w = blend_f(c4[0].w, c4[1].w, c4[2].w, c4[3].w, w);
          uint2 hi, lo;
          split4(r, hi, lo);
          *reinterpret_cast<uint2*>(a_hi + st_off[it]) = hi;
          *reinterpret_cast<uint2*>(a_lo + st_off[it]) = lo;
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&full[cur.s]);
        mbar_arrive(&pempty[cur.pbuf]);
      }
      DCN_DBG_ONLY(++dbg_n;)
      cur = nxt;
    }
    }
    DCN_DBG_ONLY(if (pt == 0) dbg_steps[3] = dbg_n;)
  }

  tc_fence_before();
  __syncthreads();
#ifdef DCN_DEBUG_CHECKS
  // every role that exchanges stages through the mbarrier rings walked the same number of K steps
  if (tid == 0) {
    const int ref = dbg_steps[3];   // gather warps
    DCN_DEV_ASSERT(dbg_steps[2] == ref);                                   // plan warps
    if (MODE == MODE_FWD) DCN_DEV_ASSERT(dbg_steps[0] == ref && dbg_steps[1] == ref);   // MMA issuer, weight loader
  }
#endif
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(P.tmem_cols)
                 : "memory");
  }
}

// ---------------------------------------------------------------------------- host side
static uint32_t pow2_cols(int cols) {
  uint32_t c = 32;
  while ((int)c < cols) c <<= 1;
  return c;
}

static bool tiling_ok(const Geo& g, Tiling* t) {
  if (!make_tiling(g, t)) return false;
  if (g.variant == DCN_VARIANT_TORCH && t->Rt * 64 > kPlanMax) return false;
  if (g.variant != DCN_VARIANT_TORCH && 128 * t->taps_per_kb > kPlanMax) return false;
  return true;
}

bool umma_fwd_supported(const Geo& g, int operand) {
  if (operand != DCN_OPERAND_FP32 && operand != DCN_OPERAND_BF16) return false;
  if (g.O % 16 || g.O < 16 || g.O > 256) return false;
  if (operand == DCN_OPERAND_BF16 && g.C % 8) return false;
  Tiling t;
  return tiling_ok(g, &t);
}

bool umma_wgrad_supported(const Geo& g, int operand) {
  if (operand != DCN_OPERAND_FP32 && operand != DCN_OPERAND_BF16) return false;
  if (g.O > 256) return false;
  if (operand == DCN_OPERAND_BF16 && g.C % 8) return false;
  Tiling t;
  return tiling_ok(g, &t);
}

static size_t elem_bytes(int operand) { return operand == DCN_OPERAND_BF16 ? 2 : 4; }

size_t umma_xt_bytes(const Geo& g, int operand) {
  return align_up(elem_bytes(operand) * (size_t)g.B * xt_image_stride(g), 1024);
}

size_t umma_fwd_workspace(const Geo& g, int operand) {
  Tiling t;
  make_tiling(g, &t);
  const int nimg = operand == DCN_OPERAND_BF16 ? 1 : 2;
  return umma_xt_bytes(g, operand) + align_up((size_t)t.KB * nimg * g.O * 128, 1024);
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}

// out[B, O, Ho*Wo] of the Torch layout viewed as a 4-D tensor [B][O][G][R] (pixel = i*R + r), box
// {box_r, Gt, O, 1}: what one staged tile group covers.  false if the driver call is unavailable.
static bool make_out_tensor_map(const Geo& g, const Tiling& t, int box_r, float* out, CUtensorMap* map) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return false;
  const cuuint64_t dims[4] = {(cuuint64_t)t.R, (cuuint64_t)t.G, (cuuint64_t)g.O, (cuuint64_t)g.B};
  const cuuint64_t strides[3] = {(cuuint64_t)t.R * 4, (cuuint64_t)g.HW * 4, (cuuint64_t)g.Oimg * g.HW * 4};
  const cuuint32_t box[4] = {(cuuint32_t)box_r, (cuuint32_t)t.Gt, (cuuint32_t)g.O, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, out, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static void common_params(const Geo& g, FwdParams& P) {
  const int n_ent = g.variant == DCN_VARIANT_TORCH ? P.t.Rt * 64 : 128 * P.t.taps_per_kb;
  P.plan_cap = (n_ent + 255) / 256 * 256;
  P.gout = nullptr;
  P.gw = nullptr;
  P.gtiles = nullptr;
  P.g_OB = 0;
  P.nslices = P.nchunks = P.kb_per_slice = 1;
  P.o_blocks = 1;
  P.n_gbuf = 0;
  P.g_img = 0;
  P.tma_out = 0;
  P.tpg = 1;
  P.n_ost = 1;
  P.box_r = 0;
  P.stage_out_bytes = 0;
  P.kperm_slabs = 0;
  P.mask = nullptr;
}

// one instantiation: opt in to its shared memory, launch it with its role layout, check the launch
template <int VARIANT, int MODE, bool BF, bool PLAIN, int PW, int GW, bool MOD>
static int launch_umma_gemm(const FwdParams& P, const CUtensorMap& tmap, int grid, size_t smem, cudaStream_t st) {
  DCN_CUDA_TRY(cudaFuncSetAttribute(umma_gemm_kernel<VARIANT, MODE, BF, PLAIN, PW, GW, MOD>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  umma_gemm_kernel<VARIANT, MODE, BF, PLAIN, PW, GW, MOD>
      <<<grid, (kFirstPlanWarp + PW + GW) * 32, smem, st>>>(P, tmap);
  DCN_KERNEL_CHECK(MODE == MODE_FWD ? "umma_fwd_kernel" : "umma_bwd_weight_kernel");
  return DCN_OK;
}

// the plan / gather split: 8 + 8 warps when more than 256 coordinate chains per K block (16 channels per sampling
// point), else 4 + 16
template <int VARIANT, int MODE, bool MOD>
static int launch_umma_gemm_split(bool bf, bool many_chains, const FwdParams& P, const CUtensorMap& tmap, int grid,
                                  size_t smem, cudaStream_t st) {
  if (many_chains)
    return bf ? launch_umma_gemm<VARIANT, MODE, true, false, 8, 8, MOD>(P, tmap, grid, smem, st)
              : launch_umma_gemm<VARIANT, MODE, false, false, 8, 8, MOD>(P, tmap, grid, smem, st);
  return bf ? launch_umma_gemm<VARIANT, MODE, true, false, 4, 16, MOD>(P, tmap, grid, smem, st)
            : launch_umma_gemm<VARIANT, MODE, false, false, 4, 16, MOD>(P, tmap, grid, smem, st);
}

template <int MODE>
static int launch_gemm(const Geo& g, int operand, const FwdParams& P, const CUtensorMap& tmap, int grid,
                       size_t smem, cudaStream_t st) {
  if (g.plain) {
    // regular convolution: pixel-row tiling, fp32 operands, 4 + 16 warps; forward only (the weight gradient of the
    // companion offset conv is fused into the data-gradient kernel)
    if constexpr (MODE == MODE_FWD) {
      if (g.variant != DCN_VARIANT_TORCH && operand == DCN_OPERAND_FP32)
        return launch_umma_gemm<DCN_VARIANT_JITTOR, MODE, false, true, 4, 16, false>(P, tmap, grid, smem, st);
    }
    set_error("plain (offset-conv) problems run forward only, in the pixel-row layout with fp32 operands");
    return DCN_ERR_UNSUPPORTED;
  }
  const bool bf = operand == DCN_OPERAND_BF16;
  // more than 256 coordinate chains per K block: Torch layout with Rt = 8, pixel-row layouts with 4 taps per K block
  // (measured at 256 and 128 chains per block — det3, c3, cfg2 — the 8 + 8 split is 18 - 43 % SLOWER: those are gather-bound)
  const int n_ent = g.variant == DCN_VARIANT_TORCH ? P.t.Rt * 64 : 128 * P.t.taps_per_kb;
  const bool many_chains = n_ent > 256;
  if (P.mask) {
    // modulated (DCNv1 only): the pixel-row instantiations with the mask folded into the plan entries
    if (g.variant != DCN_VARIANT_DCNV1) {
      set_error("umma: a mask exists for the DCNv1 variant only");
      return DCN_ERR_UNSUPPORTED;
    }
    return launch_umma_gemm_split<DCN_VARIANT_JITTOR, MODE, true>(bf, many_chains, P, tmap, grid, smem, st);
  }
  if (g.variant == DCN_VARIANT_TORCH)
    return launch_umma_gemm_split<DCN_VARIANT_TORCH, MODE, false>(bf, many_chains, P, tmap, grid, smem, st);
  return launch_umma_gemm_split<DCN_VARIANT_JITTOR, MODE, false>(bf, many_chains, P, tmap, grid, smem, st);
}

// stage_x = false: the head of the workspace already holds the staged copy of x (an earlier
// output-channel group of the same call wrote it)
int umma_forward_any(const Geo& g, int operand, const void* x, const float* off, const void* wt,
                     const float* bias, float* out, void* workspace, cudaStream_t st, bool stage_x,
                     const float* mask) {
  FwdParams P;
  P.g = g;
  if (!make_tiling(g, &P.t)) {
    set_error("umma forward: shape not tileable");
    return DCN_ERR_UNSUPPORTED;
  }
  common_params(g, P);
  const int nimg = operand == DCN_OPERAND_BF16 ? 1 : 2;
  void* xt = workspace;
  uint8_t* wtiles = (uint8_t*)workspace + umma_xt_bytes(g, operand);
  int rc;
  if (stage_x && (rc = launch_nchw_to_nhwc(g, P.t, x, xt, operand, st))) return rc;
  if ((rc = launch_weight_tiles_fwd(g, P.t, wt, wtiles, operand, st))) return rc;
  P.xt = xt;
  P.off = off;
  P.wtiles = wtiles;
  P.bias = bias;
  P.out = out;
  P.mask = mask;
  P.b_tile = (uint32_t)g.O * 128;
  P.stage_bytes = nimg * (kATile + P.b_tile);
  size_t fixed = 2 * (size_t)P.plan_cap * sizeof(PlanEntry) + 256 + 1024;  // plan ring, barriers, align slack
  // Torch layout: stage the output of box_r >= 4 adjacent class instances and write it with one
  // tensor-map store (16-byte runs) instead of 4-byte stores R floats apart
  alignas(64) CUtensorMap tmap;
  memset(&tmap, 0, sizeof(tmap));
  // (Rt = 2 only: with Rt >= 4 the direct stores already write 16-byte runs, and the staged path
  // measured slower there)
  if (g.variant == DCN_VARIANT_TORCH && P.t.Rt == 2 && !g.out_framed) {
    const int box_r = P.t.Rt < 4 ? 4 : P.t.Rt;
    const size_t bytes = sizeof(float) * (size_t)g.O * P.t.Gt * box_r;
    if (P.t.R % box_r == 0 && bytes <= 64 * 1024 && g.O <= 256 &&
        (size_t)2 * P.stage_bytes + bytes + fixed <= kSmemBudget && make_out_tensor_map(g, P.t, box_r, out, &tmap)) {
      P.tma_out = 1;
      P.box_r = box_r;
      P.tpg = box_r / P.t.Rt;
      P.stage_out_bytes = (uint32_t)align_up(bytes, 1024);
      // two staging buffers when three pipeline stages still fit next to them
      P.n_ost = (size_t)3 * P.stage_bytes + 2 * P.stage_out_bytes + fixed <= kSmemBudget ? 2 : 1;
      fixed += (size_t)P.n_ost * P.stage_out_bytes;
    }
  }
  const int stages = (int)((kSmemBudget - fixed) / P.stage_bytes);
  P.stages = stages > kFwdStages ? kFwdStages : stages;
  if (P.stages < 2) {
    set_error("umma forward: not enough shared memory for 2 stages");
    return DCN_ERR_UNSUPPORTED;
  }
  P.tmem_cols = pow2_cols(2 * g.O);
  if (g.variant != DCN_VARIANT_TORCH && g.C % 64 == 0 && g.C > 64 && P.t.KB == g.N * (g.C / 64))
    P.kperm_slabs = g.C / 64;
  const size_t smem = (size_t)P.stages * P.stage_bytes + fixed;
  const int sms = num_sms();
  const int groups = (P.t.num_tiles + P.tpg - 1) / P.tpg;  // CTAs walk groups of tpg tiles
  const int grid = groups < sms ? groups : sms;
  KernelScope scope(g.plain ? "umma_offset_conv_fwd_kernel" : "umma_fwd_kernel", st);
  return launch_gemm<MODE_FWD>(g, operand, P, tmap, grid, smem, st);
}

// ---- the companion offset convolution (deform_conv.py:16-21,58 / train.py:80-85,98) as a PLAIN problem -----------
// g is the DCN layer; the staged copy of x at the head of the workspace is the layer's (channel-permuted for the
// Torch layout), so offset conv, dcn_forward and dcn_backward share ONE staging pass.
// shifted-view convolution kernels (dcn_conv.cu): preferred when they cover the shape
bool conv_offset_fwd_supported(const Geo& g, int O);
size_t conv_offset_wtile_bytes(const Geo& g, int O);
int conv_offset_forward(const Geo& g, const float* xt, const float* woff, const float* boff, float* offset_out,
                        uint8_t* wtiles, cudaStream_t st, float* mask_out);

// n_out = 3N (the modulated layer's offset-and-mask conv): shifted-view or warp-MMA kernels only (the plain mode's
// epilogue has no mask output)
bool umma_offset_conv_fwd_supported(const Geo& g, int n_out) {
  Tiling t;
  if (!make_tiling(g, &t)) return false;          // the layer's own staging layout
  if (conv_offset_fwd_supported(g, n_out)) return true;
  return n_out == 2 * g.N && umma_fwd_supported(plain_geo(g, t, true), DCN_OPERAND_FP32);
}

size_t umma_offset_conv_fwd_workspace(const Geo& g, int n_out) {
  const size_t b = umma_xt_bytes(g, DCN_OPERAND_FP32) + conv_offset_wtile_bytes(g, n_out);
  if (n_out != 2 * g.N) return b;
  Tiling t;
  if (!make_tiling(g, &t)) return 0;
  const size_t a = umma_fwd_workspace(plain_geo(g, t, true), DCN_OPERAND_FP32);
  return a > b ? a : b;
}

int umma_offset_conv_forward(const Geo& g, const void* x, const float* woff, const float* boff, float* offset_out,
                             void* workspace, cudaStream_t st, bool stage_x, float* mask_out) {
  Tiling t;
  if (!make_tiling(g, &t)) {
    set_error("offset conv: layer shape not tileable");
    return DCN_ERR_UNSUPPORTED;
  }
  if (mask_out && !conv_offset_fwd_supported(g, 3 * g.N)) {
    set_error("offset-and-mask conv: shape not supported by the shifted-view or warp-MMA kernels");
    return DCN_ERR_UNSUPPORTED;
  }
  int rc;
  if (stage_x && (rc = launch_nchw_to_nhwc(g, t, x, workspace, DCN_OPERAND_FP32, st))) return rc;
  if (mask_out || conv_offset_fwd_supported(g, 2 * g.N))
    return conv_offset_forward(g, (const float*)workspace, woff, boff, offset_out,
                               (uint8_t*)workspace + umma_xt_bytes(g, DCN_OPERAND_FP32), st, mask_out);
  const Geo gp = plain_geo(g, t, true);
  return umma_forward_any(gp, DCN_OPERAND_FP32, x, nullptr, woff, boff, offset_out, workspace, st, false, nullptr);
}

// grad_weight[O, K] (zeroed here) = sum over all rows of gout^T * S, S re-sampled by the same
// plan / gather warps as the forward pass (mask != null: S = m * bilinear sample, as in the modulated forward).
// xt = channels-last staging copy (already built).
size_t umma_wgrad_gtile_bytes(const Geo& g, int operand);
int launch_gout_tiles_fwd_order(const Geo& g, int operand, const void* gout, uint8_t* gtiles, cudaStream_t st);

// gtiles: scratch of umma_wgrad_gtile_bytes() for the staged grad_out tile images (Torch layout; unused otherwise)
int umma_wgrad_any(const Geo& g, int operand, const void* xt, const float* off, const void* gout, float* gw,
                   uint8_t* gtiles, cudaStream_t st, const float* mask) {
  FwdParams P;
  P.g = g;
  if (!make_tiling(g, &P.t)) {
    set_error("umma wgrad: shape not tileable");
    return DCN_ERR_UNSUPPORTED;
  }
  common_params(g, P);
  const int nimg = operand == DCN_OPERAND_BF16 ? 1 : 2;
  DCN_CUDA_TRY(cudaMemsetAsync(gw, 0, sizeof(float) * (size_t)g.O * g.K, st));
  P.xt = xt;
  P.off = off;
  P.wtiles = nullptr;
  P.bias = nullptr;
  P.out = nullptr;
  P.gout = gout;
  P.gw = gw;
  P.gtiles = gtiles;
  P.mask = mask;
  P.g_OB = (g.O + 63) / 64;
  {
    int rc = launch_gout_tiles_fwd_order(g, operand, gout, gtiles, st);
    if (rc) return rc;
  }
  P.o_blocks = (g.O + 127) / 128;
  P.g_img = (uint32_t)P.o_blocks * 128 * 128;
  const int kb_max = 8 / P.o_blocks;  // 512 TMEM columns
  P.nslices = (P.t.KB + kb_max - 1) / kb_max;
  P.kb_per_slice = (P.t.KB + P.nslices - 1) / P.nslices;
  P.nslices = (P.t.KB + P.kb_per_slice - 1) / P.kb_per_slice;
  const int sms = num_sms();
  P.nchunks = sms / P.nslices;
  if (P.nchunks < 1) P.nchunks = 1;
  if (P.nchunks > P.t.num_tiles) P.nchunks = P.t.num_tiles;
  P.b_tile = 0;
  P.stage_bytes = nimg * kATile;
  P.stages = 2;
  P.tmem_cols = pow2_cols(P.o_blocks * P.kb_per_slice * 64);
  const size_t fixed = 2 * (size_t)P.plan_cap * sizeof(PlanEntry) + 256 + 1024;
  const size_t gbuf = 2 * (size_t)nimg * P.g_img;
  P.n_gbuf = ((size_t)P.stages * P.stage_bytes + 2 * gbuf + fixed <= kSmemBudget) ? 2 : 1;
  const size_t smem = (size_t)P.stages * P.stage_bytes + (size_t)P.n_gbuf * gbuf + fixed;
  if (smem > kSmemBudget) {
    set_error("umma wgrad: %zu bytes of shared memory needed", smem);
    return DCN_ERR_UNSUPPORTED;
  }
  const int grid = P.nslices * P.nchunks;
  KernelScope scope("umma_bwd_weight_kernel", st);
  alignas(64) CUtensorMap tmap;
  memset(&tmap, 0, sizeof(tmap));
  return launch_gemm<MODE_WGRAD>(g, operand, P, tmap, grid, smem, st);
}

}  // namespace dcn
