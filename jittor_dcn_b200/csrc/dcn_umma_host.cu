// dcn_umma_host.cu — dispatch of the tcgen05 kernel family behind dcn_umma.h.
//
// Output-channel groups: the tensor kernels keep a whole output row (forward: O accumulator columns,
// double-buffered in the 512 TMEM columns; backward: ceil(O / 64) <= 4 resident grad_out images) on
// chip, i.e. O <= 256 per launch.  A wider layer (ResNet-50 C5: 512 -> 512, BASELINE configs[3]) is run
// as ceil(O / 256) balanced groups of output channels: the same kernels on a Geo whose O is the group
// size and whose Oimg (image stride of out / grad_out) stays the layer's O, with weight / bias / out /
// grad_out / grad_weight pointers advanced to the group.  x is staged once, grad_x and grad_offset
// accumulate over the groups (both are sums over o).
#include "dcn_umma.h"
#include "dcn_umma_common.cuh"

namespace dcn {

bool umma_fwd_supported(const Geo& g, int operand);
size_t umma_fwd_workspace(const Geo& g, int operand);
int umma_forward_any(const Geo& g, int operand, const void* x, const float* off, const void* wt,
                     const float* bias, float* out, void* workspace, cudaStream_t st, bool stage_x,
                     const float* mask);
bool umma_bwd_supported(const Geo& g, int operand);
size_t umma_bwd_workspace(const Geo& g, int operand);
int umma_backward_any(const Geo& g, int operand, int flags, const void* x, const float* off, const void* wt,
                      const void* gout, float* gx, float* goff, float* gw, float* gb, void* workspace,
                      cudaStream_t st, const float* woff, float* gwoff, float* gboff, const float* mask,
                      float* gmask, float* g3);

bool o_groups(const Geo& g, int* size) {
  if (g.O <= 256) {
    *size = g.O;
    return true;
  }
  if (g.O % 16) return false;
  const int n = (g.O + 255) / 256;
  *size = ((g.O + n - 1) / n + 15) / 16 * 16;
  return true;
}

Geo o_group_geo(const Geo& g, int o0, int size) {
  Geo c = g;
  c.O = g.O - o0 < size ? g.O - o0 : size;
  c.o_valid = c.O;
  return c;
}

bool umma_supported(const Geo& g, int operand, int phase) {
  int size;
  if (!o_groups(g, &size)) return false;
  // the first and the last group cover every group size of this layer
  const Geo first = o_group_geo(g, 0, size), last = o_group_geo(g, (g.O - 1) / size * size, size);
  if (phase == DCN_PHASE_FORWARD) return umma_fwd_supported(first, operand) && umma_fwd_supported(last, operand);
  if (phase == DCN_PHASE_BACKWARD) return umma_bwd_supported(first, operand) && umma_bwd_supported(last, operand);
  return false;
}

size_t umma_workspace_bytes(const Geo& g, int operand, int phase) {
  int size;
  if (!o_groups(g, &size)) return 0;
  const Geo first = o_group_geo(g, 0, size);  // the largest group
  return phase == DCN_PHASE_FORWARD ? umma_fwd_workspace(first, operand) : umma_bwd_workspace(first, operand);
}

int umma_forward(const Geo& g, int operand, int flags, const void* x, const float* off, const void* wt,
                 const float* bias, void* out, void* workspace, cudaStream_t st, const float* mask) {
  int size;
  if (!o_groups(g, &size)) {
    set_error("umma forward: O = %d cannot be split into groups", g.O);
    return DCN_ERR_UNSUPPORTED;
  }
  const size_t esz = operand == DCN_OPERAND_BF16 ? 2 : 4;
  for (int o0 = 0; o0 < g.O; o0 += size) {
    const Geo gc = o_group_geo(g, o0, size);
    const int rc = umma_forward_any(gc, operand, x, off, (const uint8_t*)wt + (size_t)o0 * g.K * esz,
                                    bias ? bias + o0 : nullptr, (float*)out + (size_t)o0 * g.HW, workspace, st,
                                    o0 == 0 && !(flags & DCN_FLAG_XT_STAGED), mask);
    if (rc) return rc;
  }
  return DCN_OK;
}

int umma_backward(const Geo& g, int operand, int flags, const void* x, const float* off, const void* wt,
                  const void* gout, float* gx, float* goff, float* gw, float* gb, void* workspace,
                  cudaStream_t st, const float* mask, float* gmask) {
  return umma_backward_any(g, operand, flags, x, off, wt, gout, gx, goff, gw, gb, workspace, st, nullptr, nullptr,
                           nullptr, mask, gmask, nullptr);
}

}  // namespace dcn
