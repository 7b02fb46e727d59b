// dcn_api.cu — the C ABI declared in include/dcn_b200.h: validation, workspace carving and
// dispatch to a kernel family.  No torch types, no allocation, no device synchronisation.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <atomic>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "dcn_common.cuh"
#include "dcn_umma.h"
#include "dcn_umma_common.cuh"

namespace dcn {

static thread_local char g_err[512] = "";
// process-wide: autograd runs the backward on its own thread, bench.py reads from the main one
static std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
  return DCN_ERR_CUDA;
}

void count_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

// ---- per-kernel event profiler ------------------------------------------------------
struct ProfRec {
  const char* name;
  cudaEvent_t a, b;
};
static std::atomic<bool> g_prof_on{false};
static std::vector<ProfRec>* g_prof = nullptr;
static std::mutex g_prof_mu;
static thread_local int g_prof_slot = -1;  // record opened by this thread's KernelScope

void profile_mark(const char* name, cudaStream_t st, bool begin) {
  if (!g_prof_on.load(std::memory_order_relaxed)) return;
  std::lock_guard<std::mutex> lock(g_prof_mu);
  if (!g_prof) return;
  if (begin) {
    ProfRec r{name, nullptr, nullptr};
    if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
    cudaEventRecord(r.a, st);
    g_prof->push_back(r);
    g_prof_slot = (int)g_prof->size() - 1;
  } else if (g_prof_slot >= 0 && g_prof_slot < (int)g_prof->size()) {
    cudaEventRecord((*g_prof)[g_prof_slot].b, st);
    g_prof_slot = -1;
  }
}

static int check_ptr(const void* p, const char* name, bool required = true) {
  if (!p) {
    if (!required) return DCN_OK;
    set_error("%s is NULL", name);
    return DCN_ERR_NULL_POINTER;
  }
  if ((uintptr_t)p & 15u) {
    set_error("%s (%p) is not 16-byte aligned", name, p);
    return DCN_ERR_MISALIGNED;
  }
  return DCN_OK;
}

static int geo_or_error(const DcnShape* s, Geo* g) {
  int rc = make_geo(s, g);
  if (rc == DCN_ERR_NULL_POINTER) set_error("DcnShape is NULL");
  if (rc == DCN_ERR_BAD_SHAPE)
    set_error("bad shape B=%d C=%d O=%d H=%d W=%d k=(%d,%d) s=(%d,%d) p=(%d,%d) variant=%d", s->B,
              s->C, s->O, s->H, s->W, s->kh, s->kw, s->sh, s->sw, s->ph, s->pw, s->variant);
  if (rc == DCN_OK && s->operand != DCN_OPERAND_FP32 && s->operand != DCN_OPERAND_BF16) {
    set_error("unknown operand mode %d", s->operand);
    rc = DCN_ERR_UNSUPPORTED;
  }
  return rc;
}

static size_t plan_bytes(const Geo& g) { return align_up(sizeof(Tap) * (size_t)g.B * g.P, 256); }

// Generic kernels in bf16 storage mode: fp32 scratch copies of the bfloat16 operands, behind the plan.
static size_t f32_copy_bytes(size_t n) { return align_up(sizeof(float) * n, 256); }
static size_t n_x(const Geo& g) { return (size_t)g.B * g.C * g.H * g.W; }
static size_t n_w(const Geo& g) { return (size_t)g.O * g.K; }
static size_t n_out(const Geo& g) { return (size_t)g.B * g.O * g.HW; }
static size_t simt_workspace(const Geo& g, int operand, int phase) {
  size_t b = plan_bytes(g);
  if (operand == DCN_OPERAND_BF16) {
    b += f32_copy_bytes(n_x(g)) + f32_copy_bytes(n_w(g));
    if (phase == DCN_PHASE_BACKWARD) b += f32_copy_bytes(n_out(g));
  }
  return b;
}

size_t bn_workspace_bytes(int C);
int bn_relu_forward_staged(const Geo& g, const Tiling& t, int training, const float* x, const float* gamma,
                           const float* beta, float* running_mean, float* running_var, float momentum, float eps,
                           float* xt, float* saved, void* workspace, cudaStream_t st);
int bn_relu_backward_staged(const Geo& g, const Tiling& t, int training, const float* x, const float* gxt,
                            const float* saved, float* grad_x, float* grad_gamma, float* grad_beta, void* workspace,
                            cudaStream_t st);

int bn_relu_forward(int B, int C, int HW, int training, const float* x, const float* gamma, const float* beta,
                    float* running_mean, float* running_var, float momentum, float eps, float* y, float* saved,
                    void* workspace, cudaStream_t st);
int bn_relu_backward(int B, int C, int HW, int training, const float* x, const float* grad_y, const float* saved,
                     float* grad_x, float* grad_gamma, float* grad_beta, void* workspace, cudaStream_t st);

static int bn_shape_ok(int B, int C, int HW) {
  if (B <= 0 || C <= 0 || HW <= 0 || (long long)B * C * HW > (1LL << 40) || (long long)B * HW > 0x7fffffffLL) {
    set_error("bad batch-norm shape B=%d C=%d HW=%d", B, C, HW);
    return DCN_ERR_BAD_SHAPE;
  }
  return DCN_OK;
}

static bool use_umma(const DcnShape* s, const Geo& g, int phase) {
  if (s->flags & DCN_FLAG_FORCE_SIMT) return false;
  return umma_supported(g, s->operand, phase);
}

// Torch column layout with too few channels per sampling point for the fused kernels (dcn_gemm_path.cu):
// materialised samples + plain GEMMs
bool gemm_path_supported(const Geo& g, int operand);
size_t gemm_path_workspace(const Geo& g, int operand, int phase);
int gemm_path_forward(const Geo& g, int operand, const void* x, const float* off, const void* wt, const float* bias,
                      float* out, void* workspace, cudaStream_t st);
int gemm_path_backward(const Geo& g, int operand, int flags, const void* x, const float* off, const void* wt,
                       const void* gout, float* gx, float* goff, float* gw, float* gb, void* workspace, cudaStream_t st);
static bool use_gemm(const DcnShape* s, const Geo& g, int phase) {
  if ((s->flags & DCN_FLAG_FORCE_SIMT) || (phase != DCN_PHASE_FORWARD && phase != DCN_PHASE_BACKWARD)) return false;
  return !umma_supported(g, s->operand, phase) && gemm_path_supported(g, s->operand);
}

// mask: the modulated calls (dcn_forward_modulated / dcn_backward_modulated): DCNv1 only, float32 [B, N, Ho, Wo]
static int check_modulated(const DcnShape* s, const void* mask, const char* mname, const void* gmask = nullptr,
                           bool backward = false) {
  int rc;
  if ((rc = check_ptr(mask, mname)) || (backward && (rc = check_ptr(gmask, "grad_mask")))) return rc;
  if (s->variant != DCN_VARIANT_DCNV1) {
    set_error("a mask (modulated deformable convolution, DCNv2) exists for DCN_VARIANT_DCNV1 only, not variant %d: "
              "the reference's two variants have no modulated form", s->variant);
    return DCN_ERR_UNSUPPORTED;
  }
  return DCN_OK;
}

// ---- whole-layer calls (offset conv + DCN span), phases DCN_PHASE_LAYER_*: fp32 operands on the tensor path only.
// The modulated layer (phases *_MODULATED; mmcv's ModulatedDeformConv2dPack) is DCNv1 only and its conv has 3N
// outputs (offsets, then one mask logit per tap) instead of 2N.
static bool is_layer_phase(int phase) {
  return phase >= DCN_PHASE_LAYER_FORWARD && phase <= DCN_PHASE_LAYER_BACKWARD_MODULATED;
}
static bool modulated_phase(int phase) {
  return phase == DCN_PHASE_LAYER_FORWARD_MODULATED || phase == DCN_PHASE_LAYER_BACKWARD_MODULATED;
}
static bool backward_phase(int phase) {
  return phase == DCN_PHASE_LAYER_BACKWARD || phase == DCN_PHASE_LAYER_BACKWARD_MODULATED;
}
static int conv_outputs(const Geo& g, int phase) { return (modulated_phase(phase) ? 3 : 2) * g.N; }

static bool layer_ok(const DcnShape* s, const Geo& g, int phase) {
  if ((s->flags & DCN_FLAG_FORCE_SIMT) || s->operand != DCN_OPERAND_FP32) return false;
  if (modulated_phase(phase) && s->variant != DCN_VARIANT_DCNV1) return false;
  const int n_out = conv_outputs(g, phase);
  if (!umma_supported(g, DCN_OPERAND_FP32, DCN_PHASE_FORWARD) || !umma_offset_conv_fwd_supported(g, n_out)) return false;
  return !backward_phase(phase) || umma_layer_bwd_supported(g, n_out);
}

static size_t layer_workspace(const Geo& g, int phase) {
  const int n_out = conv_outputs(g, phase);
  if (backward_phase(phase)) return umma_layer_bwd_workspace(g, n_out);
  const size_t f1 = umma_offset_conv_fwd_workspace(g, n_out), f2 = umma_workspace_bytes(g, DCN_OPERAND_FP32, DCN_PHASE_FORWARD);
  return f1 > f2 ? f1 : f2;
}

// the refusal of a whole-layer call `what` that layer_ok turns down, with its reason: variant, operand, shape / flags
static int layer_refusal(const DcnShape* s, const Geo& g, int phase, const char* what) {
  if (layer_ok(s, g, phase)) return DCN_OK;
  static const char* const names[] = {"DCN_PHASE_LAYER_FORWARD", "DCN_PHASE_LAYER_BACKWARD",
                                      "DCN_PHASE_LAYER_FORWARD_MODULATED", "DCN_PHASE_LAYER_BACKWARD_MODULATED"};
  if (modulated_phase(phase) && s->variant != DCN_VARIANT_DCNV1)
    set_error("%s: a mask (modulated deformable convolution, DCNv2) exists for DCN_VARIANT_DCNV1 only, not variant %d",
              what, s->variant);
  else if (s->operand != DCN_OPERAND_FP32)
    set_error("%s: fp32 operands only (operand %d)", what, s->operand);
  else
    set_error("%s: shape / flags not supported (dcn_path_name(s, %s))", what, names[phase - DCN_PHASE_LAYER_FORWARD]);
  return DCN_ERR_UNSUPPORTED;
}

// DCN_FLAG_GRAD_X_FRAMED: grad_x is the consumer's framed channels-last accumulator.  Only the tensor-path data
// gradient writes that layout, and it overwrites; any other data gradient, or an accumulating one, would leave NCHW
// values (or a sum) in a buffer the caller reads as framed.  data_on_umma: the data gradient of this call runs there.
static int grad_x_framed_refusal(const DcnShape* s, bool data_on_umma, const char* what) {
  if (!(s->flags & DCN_FLAG_GRAD_X_FRAMED)) return DCN_OK;
  if (s->flags & DCN_FLAG_ACCUM_GRAD_X)
    set_error("%s: DCN_FLAG_GRAD_X_FRAMED excludes DCN_FLAG_ACCUM_GRAD_X (the framed grad_x is overwritten)", what);
  else if (!data_on_umma)
    set_error("%s: DCN_FLAG_GRAD_X_FRAMED needs the data gradient on the tensor path, which this shape / operand / "
              "flags does not take", what);
  else
    return DCN_OK;
  return DCN_ERR_UNSUPPORTED;
}

static int check_workspace(size_t have, size_t need, const char* what) {
  if (have >= need) return DCN_OK;
  set_error("%s workspace: have %zu bytes, need %zu", what, have, need);
  return DCN_ERR_WORKSPACE;
}

// multi-scale deformable attention (dcn_msda.cu)
int msda_forward(const DcnMsdaShape& s, const float* value, const int64_t* shapes, const int64_t* starts,
                 const float* loc, const float* attn, float* out, cudaStream_t st);
int msda_backward(const DcnMsdaShape& s, const float* value, const int64_t* shapes, const int64_t* starts,
                  const float* loc, const float* attn, const float* gout, float* gvalue, float* gloc, float* gattn,
                  cudaStream_t st);

static int msda_shape_ok(const DcnMsdaShape* s, const char* what) {
  if (!s) {
    set_error("%s: DcnMsdaShape is NULL", what);
    return DCN_ERR_NULL_POINTER;
  }
  if (s->B <= 0 || s->S <= 0 || s->Q <= 0 || s->M <= 0 || s->D <= 0 || s->L <= 0 || s->P <= 0) {
    set_error("%s: bad shape B=%d S=%d Q=%d M=%d D=%d L=%d P=%d", what, s->B, s->S, s->Q, s->M, s->D, s->L, s->P);
    return DCN_ERR_BAD_SHAPE;
  }
  if ((long long)s->B * s->Q * s->M > 0x7fffffffLL) {
    set_error("%s: B*Q*M = %lld exceeds the limit 2^31 - 1", what, (long long)s->B * s->Q * s->M);
    return DCN_ERR_BAD_SHAPE;
  }
  if (s->flags != 0) {
    set_error("%s: flags must be 0 (reserved), got %d", what, s->flags);
    return DCN_ERR_UNSUPPORTED;
  }
  if (s->D != 16 && s->D != 32 && s->D != 64 && s->D != 128 && s->D != 256) {
    set_error("%s: D = %d channels per head is not supported (D in {16, 32, 64, 128, 256})", what, s->D);
    return DCN_ERR_UNSUPPORTED;
  }
  if (s->L > 16) {
    set_error("%s: L = %d levels exceeds the limit L <= 16", what, s->L);
    return DCN_ERR_UNSUPPORTED;
  }
  if (s->P > 32) {
    set_error("%s: P = %d points exceeds the limit P <= 32", what, s->P);
    return DCN_ERR_UNSUPPORTED;
  }
  return DCN_OK;
}

// DCNv3 (dcn_dcnv3.cu)
int dcnv3_forward(const DcnV3Shape& s, int Ho, int Wo, float offset_scale, const float* input, const float* offset,
                  const float* mask, float* out, cudaStream_t st);
int dcnv3_backward(const DcnV3Shape& s, int Ho, int Wo, float offset_scale, const float* input, const float* offset,
                   const float* mask, const float* gout, float* ginput, float* goffset, float* gmask, cudaStream_t st);

// floor((in + 2*pad - (dil*(k-1) + 1)) / stride) + 1, or 0 when the dilated kernel does not fit the padded input
static long long dcnv3_out_extent(long long in, long long k, long long stride, long long pad, long long dil) {
  const long long room = in + 2 * pad - (dil * (k - 1) + 1);
  return room < 0 ? 0 : room / stride + 1;
}

// The shape checks of dcn_v3_forward / _backward: bad shapes (DCN_ERR_BAD_SHAPE) -> Ho, Wo.
static int dcnv3_shape_ok(const DcnV3Shape* s, const char* what, int* Ho, int* Wo) {
  if (!s) {
    set_error("%s: DcnV3Shape is NULL", what);
    return DCN_ERR_NULL_POINTER;
  }
  if (s->N <= 0 || s->H <= 0 || s->W <= 0 || s->G <= 0 || s->Gc <= 0 || s->kh <= 0 || s->kw <= 0 || s->sh <= 0 ||
      s->sw <= 0 || s->dh <= 0 || s->dw <= 0 || s->ph < 0 || s->pw < 0) {
    set_error("%s: bad shape N=%d H=%d W=%d G=%d Gc=%d k=(%d,%d) s=(%d,%d) p=(%d,%d) d=(%d,%d)", what, s->N, s->H, s->W,
              s->G, s->Gc, s->kh, s->kw, s->sh, s->sw, s->ph, s->pw, s->dh, s->dw);
    return DCN_ERR_BAD_SHAPE;
  }
  const long long ho = dcnv3_out_extent(s->H, s->kh, s->sh, s->ph, s->dh);
  const long long wo = dcnv3_out_extent(s->W, s->kw, s->sw, s->pw, s->dw);
  if (ho < 1 || wo < 1) {
    set_error("%s: empty output Ho=%lld Wo=%lld (the dilated kernel does not fit the padded input)", what, ho, wo);
    return DCN_ERR_BAD_SHAPE;
  }
  const long long items = (long long)s->N * ho * wo * s->G, pixels = (long long)s->N * s->H * s->W;
  if (items > 0x7fffffffLL) {
    set_error("%s: N*Ho*Wo*G = %lld exceeds the limit 2^31 - 1", what, items);
    return DCN_ERR_BAD_SHAPE;
  }
  if (pixels > 0x7fffffffLL) {
    set_error("%s: N*H*W = %lld exceeds the limit 2^31 - 1", what, pixels);
    return DCN_ERR_BAD_SHAPE;
  }
  *Ho = (int)ho;
  *Wo = (int)wo;
  return DCN_OK;
}

// What the kernels cover (DCN_ERR_UNSUPPORTED), checked after the pointers.
static int dcnv3_supported(const DcnV3Shape* s, const char* what) {
  if (s->Gc != 16 && s->Gc != 32 && s->Gc != 64 && s->Gc != 128 && s->Gc != 256) {
    set_error("%s: Gc = %d channels per group is not supported (Gc in {16, 32, 64, 128, 256})", what, s->Gc);
    return DCN_ERR_UNSUPPORTED;
  }
  if ((long long)s->kh * s->kw > 32) {
    set_error("%s: P = kh*kw = %lld points exceeds the limit P <= 32", what, (long long)s->kh * s->kw);
    return DCN_ERR_UNSUPPORTED;
  }
  if (s->flags & ~DCN_V3_FLAG_SOFTMAX_MASK) {
    set_error("%s: unknown flags 0x%x (only DCN_V3_FLAG_SOFTMAX_MASK = 1 is defined)", what,
              (unsigned)s->flags & ~(unsigned)DCN_V3_FLAG_SOFTMAX_MASK);
    return DCN_ERR_UNSUPPORTED;
  }
  return DCN_OK;
}

// DCNv4 (dcn_dcnv3.cu)
long long dcnv4_row_floats(const DcnV3Shape& s);
int dcnv4_forward(const DcnV3Shape& s, int Ho, int Wo, float offset_scale, const float* input, const float* offset_mask,
                  float* out, cudaStream_t st);
int dcnv4_backward(const DcnV3Shape& s, int Ho, int Wo, float offset_scale, const float* input, const float* offset_mask,
                   const float* gout, float* ginput, float* goffset_mask, cudaStream_t st);

// The shape checks of dcn_v4_forward / _backward: DCNv3's, then K >= 1 and the row width Cm.
static int dcnv4_shape_ok(const DcnV3Shape* s, const char* what, int* Ho, int* Wo) {
  int rc;
  if ((rc = dcnv3_shape_ok(s, what, Ho, Wo))) return rc;
  if ((long long)s->kh * s->kw == 1 && (s->flags & DCN_V4_FLAG_REMOVE_CENTER)) {
    set_error("%s: K = 0 points: a 1 x 1 kernel with remove_center has none", what);
    return DCN_ERR_BAD_SHAPE;
  }
  const long long cm = dcnv4_row_floats(*s);
  if (cm > 0x7fffffffLL) {
    set_error("%s: Cm = ceil(3*G*K / 8)*8 = %lld exceeds the limit 2^31 - 1", what, cm);
    return DCN_ERR_BAD_SHAPE;
  }
  return DCN_OK;
}

// What the DCNv4 kernels cover (DCN_ERR_UNSUPPORTED), checked after the pointers.
static int dcnv4_supported(const DcnV3Shape* s, const char* what) {
  if (s->Gc != 16 && s->Gc != 32 && s->Gc != 64 && s->Gc != 128 && s->Gc != 256) {
    set_error("%s: Gc = %d channels per group is not supported (Gc in {16, 32, 64, 128, 256})", what, s->Gc);
    return DCN_ERR_UNSUPPORTED;
  }
  if (s->flags & ~DCN_V4_FLAG_REMOVE_CENTER) {
    set_error("%s: unknown flags 0x%x (only DCN_V4_FLAG_REMOVE_CENTER = 2 is defined; DCNv4 has no softmax)", what,
              (unsigned)s->flags & ~(unsigned)DCN_V4_FLAG_REMOVE_CENTER);
    return DCN_ERR_UNSUPPORTED;
  }
  if ((s->flags & DCN_V4_FLAG_REMOVE_CENTER) && (s->kh % 2 == 0 || s->kw % 2 == 0)) {
    set_error("%s: remove_center needs an odd kernel, got %d x %d (no centre point)", what, s->kh, s->kw);
    return DCN_ERR_UNSUPPORTED;
  }
  return DCN_OK;
}

}  // namespace dcn

using namespace dcn;

extern "C" {

int dcn_version(void) { return DCN_B200_VERSION; }

const char* dcn_last_error(void) { return g_err; }

const char* dcn_status_string(int status) {
  switch (status) {
    case DCN_OK: return "ok";
    case DCN_ERR_BAD_SHAPE: return "bad shape";
    case DCN_ERR_NULL_POINTER: return "null pointer";
    case DCN_ERR_MISALIGNED: return "misaligned pointer";
    case DCN_ERR_WORKSPACE: return "workspace too small";
    case DCN_ERR_CUDA: return "CUDA error";
    case DCN_ERR_UNSUPPORTED: return "unsupported configuration";
    case DCN_ERR_NCCL: return "NCCL error";
    default: return "unknown status";
  }
}

int dcn_output_hw(const DcnShape* s, int32_t* h_out, int32_t* w_out) {
  Geo g;
  int rc = geo_or_error(s, &g);
  if (rc) return rc;
  if (h_out) *h_out = g.Ho;
  if (w_out) *w_out = g.Wo;
  return DCN_OK;
}

size_t dcn_workspace_bytes(const DcnShape* s, int phase) {
  Geo g;
  if (geo_or_error(s, &g)) return 0;
  if (phase == DCN_PHASE_CORNERS) return 0;
  if (is_layer_phase(phase)) return layer_ok(s, g, phase) ? layer_workspace(g, phase) : 0;
  if (use_umma(s, g, phase)) return umma_workspace_bytes(g, s->operand, phase);
  if (use_gemm(s, g, phase)) return gemm_path_workspace(g, s->operand, phase);
  return simt_workspace(g, s->operand, phase);
}

const char* dcn_path_name(const DcnShape* s, int phase) {
  Geo g;
  if (geo_or_error(s, &g)) return "invalid";
  if (is_layer_phase(phase)) return layer_ok(s, g, phase) ? "umma" : "unsupported";
  return use_umma(s, g, phase) ? "umma" : (use_gemm(s, g, phase) ? "gemm" : "simt");
}

int dcn_profile_begin(void) {
  std::lock_guard<std::mutex> lock(g_prof_mu);
  if (!g_prof) g_prof = new std::vector<ProfRec>();
  for (auto& r : *g_prof) {
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  g_prof->clear();
  g_prof_on = true;
  return DCN_OK;
}

int dcn_profile_end(char* out, size_t cap) {
  g_prof_on = false;
  std::lock_guard<std::mutex> lock(g_prof_mu);
  if (!g_prof) return DCN_OK;
  std::map<std::string, std::pair<int, double>> agg;
  std::vector<std::string> order;
  for (auto& r : *g_prof) {
    float ms = 0.f;
    if (r.b && cudaEventSynchronize(r.b) == cudaSuccess && cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
      auto it = agg.find(r.name);
      if (it == agg.end()) {
        order.push_back(r.name);
        agg[r.name] = {1, (double)ms};
      } else {
        it->second.first += 1;
        it->second.second += ms;
      }
    }
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  g_prof->clear();
  size_t used = 0;
  if (out && cap) out[0] = 0;
  for (auto& n : order) {
    char line[256];
    int len = snprintf(line, sizeof line, "%s %d %.6f\n", n.c_str(), agg[n].first, agg[n].second);
    if (out && used + (size_t)len + 1 < cap) {
      memcpy(out + used, line, (size_t)len + 1);
      used += (size_t)len;
    }
  }
  return DCN_OK;
}

uint64_t dcn_launch_count(void) { return g_launches.load(); }
void dcn_launch_count_reset(void) { g_launches.store(0); }

}  // extern "C"

namespace dcn {

// dcn_forward and dcn_forward_modulated: mask == nullptr = unmodulated
static int forward_impl(const DcnShape* s, const void* x, const void* offset, const float* mask, const void* weight,
                        const void* bias, void* out, void* workspace, size_t workspace_bytes, void* stream) {
  Geo g;
  int rc = geo_or_error(s, &g);
  if (rc) return rc;
  if ((rc = check_ptr(x, "x")) || (rc = check_ptr(offset, "offset")) ||
      (rc = check_ptr(weight, "weight")) || (rc = check_ptr(bias, "bias", false)) ||
      (rc = check_ptr(out, "out")))
    return rc;
  const size_t need = dcn_workspace_bytes(s, DCN_PHASE_FORWARD);
  if (need && (rc = check_ptr(workspace, "workspace"))) return rc;
  if ((rc = check_workspace(workspace_bytes, need, "forward"))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (use_umma(s, g, DCN_PHASE_FORWARD))
    return umma_forward(g, s->operand, s->flags, x, (const float*)offset, weight, (const float*)bias,
                        out, workspace, st, mask);
  if (use_gemm(s, g, DCN_PHASE_FORWARD))
    return gemm_path_forward(g, s->operand, x, (const float*)offset, weight, (const float*)bias, (float*)out, workspace,
                             st);
  Tap* plan = (Tap*)workspace;
  if (s->operand == DCN_OPERAND_BF16) {
    // shapes the tensor path does not tile: widen the bf16 operands once, run the fp32 kernels
    float* xf = (float*)((uint8_t*)workspace + plan_bytes(g));
    float* wf = (float*)((uint8_t*)xf + f32_copy_bytes(n_x(g)));
    if ((rc = launch_widen_bf16(x, xf, n_x(g), st)) || (rc = launch_widen_bf16(weight, wf, n_w(g), st))) return rc;
    x = xf;
    weight = wf;
  }
  // (the plan of the DCNv1 layout is [b][n][p], the order of the mask: the sampling kernels index both alike)
  if ((rc = launch_plan(g, (const float*)offset, plan, st))) return rc;
  return simt_forward(g, (const float*)x, plan, (const float*)weight, (const float*)bias, (float*)out,
                      st, mask);
}

// dcn_backward and dcn_backward_modulated: mask == nullptr = unmodulated (grad_mask unused)
static int backward_impl(const DcnShape* s, const void* x, const void* offset, const float* mask, const void* weight,
                         const void* grad_out, void* grad_x, void* grad_offset, float* grad_mask, void* grad_weight,
                         void* grad_bias, void* workspace, size_t workspace_bytes, void* stream) {
  Geo g;
  int rc = geo_or_error(s, &g);
  if (rc) return rc;
  const bool want_gx = !(s->flags & DCN_FLAG_NO_GRAD_X);
  if ((rc = check_ptr(x, "x")) || (rc = check_ptr(offset, "offset")) ||
      (rc = check_ptr(weight, "weight")) || (rc = check_ptr(grad_out, "grad_out")) ||
      (rc = check_ptr(grad_x, "grad_x", want_gx)) || (rc = check_ptr(grad_offset, "grad_offset")) ||
      (rc = check_ptr(grad_weight, "grad_weight")) || (rc = check_ptr(grad_bias, "grad_bias", false)))
    return rc;
  const bool data_on_umma = use_umma(s, g, DCN_PHASE_BACKWARD) && umma_bwd_data_on_tensor_path(g, s->operand);
  if ((rc = grad_x_framed_refusal(s, data_on_umma, mask ? "modulated backward" : "backward"))) return rc;
  const size_t need = dcn_workspace_bytes(s, DCN_PHASE_BACKWARD);
  if (need && (rc = check_ptr(workspace, "workspace"))) return rc;
  if ((rc = check_workspace(workspace_bytes, need, "backward"))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (use_umma(s, g, DCN_PHASE_BACKWARD))
    return umma_backward(g, s->operand, s->flags, x, (const float*)offset, weight, grad_out,
                         (float*)grad_x, (float*)grad_offset, (float*)grad_weight,
                         (float*)grad_bias, workspace, st, mask, grad_mask);
  if (use_gemm(s, g, DCN_PHASE_BACKWARD))
    return gemm_path_backward(g, s->operand, s->flags, x, (const float*)offset, weight, grad_out, (float*)grad_x,
                              (float*)grad_offset, (float*)grad_weight, (float*)grad_bias, workspace, st);
  Tap* plan = (Tap*)workspace;
  if (s->operand == DCN_OPERAND_BF16) {
    float* xf = (float*)((uint8_t*)workspace + plan_bytes(g));
    float* wf = (float*)((uint8_t*)xf + f32_copy_bytes(n_x(g)));
    float* gf = (float*)((uint8_t*)wf + f32_copy_bytes(n_w(g)));
    if ((rc = launch_widen_bf16(x, xf, n_x(g), st)) || (rc = launch_widen_bf16(weight, wf, n_w(g), st)) ||
        (rc = launch_widen_bf16(grad_out, gf, n_out(g), st)))
      return rc;
    x = xf;
    weight = wf;
    grad_out = gf;
  }
  if ((rc = launch_plan(g, (const float*)offset, plan, st))) return rc;
  return simt_backward(g, s->flags, (const float*)x, plan, (const float*)weight,
                       (const float*)grad_out, (float*)grad_x, (float*)grad_offset,
                       (float*)grad_weight, (float*)grad_bias, st, SIMT_BWD_ALL, mask, grad_mask);
}

// ---- whole-layer calls: phase DCN_PHASE_LAYER_FORWARD / _BACKWARD, or the *_MODULATED one with a mask; every call
// checks shape, pointers, support, workspace, in that order, then launches

// dcn_offset_conv_forward and dcn_offset_conv_forward_modulated
static int offset_conv_impl(const DcnShape* s, int phase, const char* what, const void* x, const void* offset_weight,
                            const void* offset_bias, void* offset, void* mask, void* workspace, size_t workspace_bytes,
                            void* stream) {
  Geo g;
  int rc;
  if ((rc = geo_or_error(s, &g)) || (rc = check_ptr(x, "x")) || (rc = check_ptr(offset_weight, "offset_weight")) ||
      (rc = check_ptr(offset_bias, "offset_bias", false)) || (rc = check_ptr(offset, "offset")) ||
      (rc = check_ptr(mask, "mask", modulated_phase(phase))) || (rc = check_ptr(workspace, "workspace")) ||
      (rc = layer_refusal(s, g, phase, what)) ||
      (rc = check_workspace(workspace_bytes, umma_offset_conv_fwd_workspace(g, conv_outputs(g, phase)), what)))
    return rc;
  return umma_offset_conv_forward(g, x, (const float*)offset_weight, (const float*)offset_bias, (float*)offset,
                                  workspace, (cudaStream_t)stream, !(s->flags & DCN_FLAG_XT_STAGED), (float*)mask);
}

// chained inference (SURVEY 8f.2): the producer's epilogue writes the consumer's staged input.
// Geo of the producer with out_framed set from the consumer's staging layout, or an error.
static int chained_geo(const DcnShape* s, const DcnShape* consumer, Geo* g) {
  int rc = geo_or_error(s, g);
  if (rc) return rc;
  Geo gc;
  if ((rc = geo_or_error(consumer, &gc))) return rc;
  if (s->operand != DCN_OPERAND_FP32 || consumer->operand != DCN_OPERAND_FP32 || g->O > 256 ||
      gc.B != g->B || gc.C != g->O || gc.H != g->Ho || gc.W != g->Wo) {
    set_error("chained forward: consumer must take this layer's output (B=%d C=%d H=%d W=%d, fp32, O <= 256); got "
              "B=%d C=%d H=%d W=%d", g->B, g->O, g->Ho, g->Wo, gc.B, gc.C, gc.H, gc.W);
    return DCN_ERR_BAD_SHAPE;
  }
  if (!use_umma(s, *g, DCN_PHASE_FORWARD) || !use_umma(consumer, gc, DCN_PHASE_FORWARD)) {
    set_error("chained forward: both layers must run on the tensor path (dcn_path_name == \"umma\")");
    return DCN_ERR_UNSUPPORTED;
  }
  Tiling tc;
  if (!make_tiling(gc, &tc)) return DCN_ERR_UNSUPPORTED;
  g->out_framed = 1;
  g->out_G = gc.variant == DCN_VARIANT_TORCH ? tc.G : 0;
  g->out_Cs = gc.variant == DCN_VARIANT_TORCH ? tc.Cs : 0;
  return DCN_OK;
}

// dcn_layer_forward, dcn_layer_forward_chained (consumer != nullptr: out is the consumer's workspace) and
// dcn_layer_forward_modulated.  The offset conv and the span share one staging pass of x.
static int layer_forward_impl(const DcnShape* s, const DcnShape* consumer, int phase, const char* what, const void* x,
                              const void* offset_weight, const void* offset_bias, const void* weight, const void* bias,
                              void* offset, void* mask, void* out, void* workspace, size_t workspace_bytes,
                              void* stream) {
  Geo g;
  int rc;
  if ((rc = consumer ? chained_geo(s, consumer, &g) : geo_or_error(s, &g)) || (rc = check_ptr(x, "x")) ||
      (rc = check_ptr(offset_weight, "offset_weight")) || (rc = check_ptr(offset_bias, "offset_bias", false)) ||
      (rc = check_ptr(weight, "weight")) || (rc = check_ptr(bias, "bias", false)) ||
      (rc = check_ptr(offset, "offset")) || (rc = check_ptr(mask, "mask", modulated_phase(phase))) ||
      (rc = check_ptr(out, consumer ? "consumer_workspace" : "out")) || (rc = check_ptr(workspace, "workspace")) ||
      (rc = layer_refusal(s, g, phase, what)) ||
      (rc = check_workspace(workspace_bytes, layer_workspace(g, phase), what)))
    return rc;
  // (out_framed of a chained Geo only concerns the span's epilogue: the offset conv ignores it)
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = umma_offset_conv_forward(g, x, (const float*)offset_weight, (const float*)offset_bias, (float*)offset,
                                     workspace, st, !(s->flags & DCN_FLAG_XT_STAGED), (float*)mask)))
    return rc;
  return umma_forward(g, DCN_OPERAND_FP32, s->flags | DCN_FLAG_XT_STAGED, x, (const float*)offset, weight,
                      (const float*)bias, out, workspace, st, (const float*)mask);
}

// dcn_layer_backward and dcn_layer_backward_modulated
static int layer_backward_impl(const DcnShape* s, int phase, const char* what, const void* x, const void* offset,
                               const void* mask, const void* offset_weight, const void* weight, const void* grad_out,
                               void* grad_x, void* grad_offset_weight, void* grad_offset_bias, void* grad_weight,
                               void* grad_bias, void* workspace, size_t workspace_bytes, void* stream) {
  Geo g;
  int rc = geo_or_error(s, &g);
  if (rc) return rc;
  const bool want_gx = !(s->flags & DCN_FLAG_NO_GRAD_X);
  if ((rc = check_ptr(x, "x")) || (rc = check_ptr(offset, "offset")) ||
      (rc = check_ptr(mask, "mask", modulated_phase(phase))) || (rc = check_ptr(offset_weight, "offset_weight")) ||
      (rc = check_ptr(weight, "weight")) || (rc = check_ptr(grad_out, "grad_out")) ||
      (rc = check_ptr(grad_x, "grad_x", want_gx)) || (rc = check_ptr(grad_offset_weight, "grad_offset_weight")) ||
      (rc = check_ptr(grad_offset_bias, "grad_offset_bias", false)) || (rc = check_ptr(grad_weight, "grad_weight")) ||
      (rc = check_ptr(grad_bias, "grad_bias", false)) || (rc = check_ptr(workspace, "workspace")) ||
      (rc = layer_refusal(s, g, phase, what)) ||
      (rc = grad_x_framed_refusal(s, umma_bwd_data_on_tensor_path(g, DCN_OPERAND_FP32), what)))
    return rc;
  const size_t need = layer_workspace(g, phase);
  if ((rc = check_workspace(workspace_bytes, need, what))) return rc;
  return umma_layer_backward(g, s->flags, x, (const float*)offset, (const float*)mask, (const float*)offset_weight,
                             weight, grad_out, (float*)grad_x, (float*)grad_offset_weight, (float*)grad_offset_bias,
                             (float*)grad_weight, (float*)grad_bias, workspace, need, (cudaStream_t)stream);
}

}  // namespace dcn

extern "C" {

int dcn_forward(const DcnShape* s, const void* x, const void* offset, const void* weight,
                const void* bias, void* out, void* workspace, size_t workspace_bytes,
                void* stream) {
  return forward_impl(s, x, offset, nullptr, weight, bias, out, workspace, workspace_bytes, stream);
}

int dcn_backward(const DcnShape* s, const void* x, const void* offset, const void* weight,
                 const void* grad_out, void* grad_x, void* grad_offset, void* grad_weight,
                 void* grad_bias, void* workspace, size_t workspace_bytes, void* stream) {
  return backward_impl(s, x, offset, nullptr, weight, grad_out, grad_x, grad_offset, nullptr, grad_weight, grad_bias,
                       workspace, workspace_bytes, stream);
}

int dcn_forward_modulated(const DcnShape* s, const void* x, const void* offset, const void* mask,
                          const void* weight, const void* bias, void* out,
                          void* workspace, size_t workspace_bytes, void* stream) {
  Geo g;
  int rc = geo_or_error(s, &g);
  if (rc || (rc = check_modulated(s, mask, "mask"))) return rc;
  return forward_impl(s, x, offset, (const float*)mask, weight, bias, out, workspace, workspace_bytes, stream);
}

int dcn_backward_modulated(const DcnShape* s, const void* x, const void* offset, const void* mask,
                           const void* weight, const void* grad_out, void* grad_x, void* grad_offset,
                           void* grad_mask, void* grad_weight, void* grad_bias,
                           void* workspace, size_t workspace_bytes, void* stream) {
  Geo g;
  int rc = geo_or_error(s, &g);
  if (rc || (rc = check_modulated(s, mask, "mask", grad_mask, true))) return rc;
  return backward_impl(s, x, offset, (const float*)mask, weight, grad_out, grad_x, grad_offset, (float*)grad_mask,
                       grad_weight, grad_bias, workspace, workspace_bytes, stream);
}

int dcn_offset_conv_forward(const DcnShape* s, const void* x, const void* offset_weight, const void* offset_bias,
                            void* offset, void* workspace, size_t workspace_bytes, void* stream) {
  return offset_conv_impl(s, DCN_PHASE_LAYER_FORWARD, "offset conv", x, offset_weight, offset_bias, offset, nullptr,
                          workspace, workspace_bytes, stream);
}

int dcn_layer_forward(const DcnShape* s, const void* x, const void* offset_weight, const void* offset_bias,
                      const void* weight, const void* bias, void* offset, void* out, void* workspace,
                      size_t workspace_bytes, void* stream) {
  return layer_forward_impl(s, nullptr, DCN_PHASE_LAYER_FORWARD, "layer forward", x, offset_weight, offset_bias, weight,
                            bias, offset, nullptr, out, workspace, workspace_bytes, stream);
}

size_t dcn_staged_input_bytes(const DcnShape* s) {
  Geo g;
  if (geo_or_error(s, &g)) return 0;
  return align_up(sizeof(float) * (size_t)g.B * xt_image_stride(g), 1024);
}

int dcn_staged_input_clear(const DcnShape* s, void* workspace, void* stream) {
  Geo g;
  int rc = geo_or_error(s, &g);
  if (rc) return rc;
  if ((rc = check_ptr(workspace, "workspace"))) return rc;
  DCN_CUDA_TRY(cudaMemsetAsync(workspace, 0, dcn_staged_input_bytes(s), (cudaStream_t)stream));
  return DCN_OK;
}

int dcn_layer_forward_chained(const DcnShape* s, const DcnShape* consumer, const void* x, const void* offset_weight,
                              const void* offset_bias, const void* weight, const void* bias, void* offset,
                              void* consumer_workspace, void* workspace, size_t workspace_bytes, void* stream) {
  return layer_forward_impl(s, consumer, DCN_PHASE_LAYER_FORWARD, "chained layer forward", x, offset_weight,
                            offset_bias, weight, bias, offset, nullptr, consumer_workspace, workspace, workspace_bytes,
                            stream);
}

static int staged_consumer(const DcnShape* consumer, Geo* g, Tiling* t) {
  int rc = geo_or_error(consumer, g);
  if (rc) return rc;
  if (consumer->operand != DCN_OPERAND_FP32 || !use_umma(consumer, *g, DCN_PHASE_FORWARD) || !make_tiling(*g, t)) {
    set_error("staged post-op: the consumer layer must run on the tensor path with fp32 operands");
    return DCN_ERR_UNSUPPORTED;
  }
  return DCN_OK;
}

int dcn_bn_relu_forward_staged(const DcnShape* consumer, int training, const void* x, const void* gamma, const void* beta,
                               void* running_mean, void* running_var, float momentum, float eps,
                               void* consumer_workspace, void* saved, void* workspace, size_t workspace_bytes,
                               void* stream) {
  Geo g;
  Tiling t;
  int rc = staged_consumer(consumer, &g, &t);
  if (rc) return rc;
  if ((rc = check_ptr(x, "x")) || (rc = check_ptr(consumer_workspace, "consumer_workspace")) ||
      (rc = check_ptr(saved, "saved")) || (rc = check_ptr(workspace, "workspace")))
    return rc;
  if (!training && (!running_mean || !running_var)) {
    set_error("staged post-op: eval mode needs running_mean / running_var");
    return DCN_ERR_NULL_POINTER;
  }
  if (workspace_bytes < bn_workspace_bytes(g.C)) {
    set_error("staged post-op workspace: have %zu bytes, need %zu", workspace_bytes, bn_workspace_bytes(g.C));
    return DCN_ERR_WORKSPACE;
  }
  return bn_relu_forward_staged(g, t, training, (const float*)x, (const float*)gamma, (const float*)beta,
                                (float*)running_mean, (float*)running_var, momentum, eps, (float*)consumer_workspace,
                                (float*)saved, workspace, (cudaStream_t)stream);
}

int dcn_bn_relu_backward_staged(const DcnShape* consumer, int training, const void* x, const void* grad_staged,
                                const void* saved, void* grad_x, void* grad_gamma, void* grad_beta, void* workspace,
                                size_t workspace_bytes, void* stream) {
  Geo g;
  Tiling t;
  int rc = staged_consumer(consumer, &g, &t);
  if (rc) return rc;
  if ((rc = check_ptr(x, "x")) || (rc = check_ptr(grad_staged, "grad_staged")) || (rc = check_ptr(saved, "saved")) ||
      (rc = check_ptr(grad_x, "grad_x", false)) || (rc = check_ptr(workspace, "workspace")))
    return rc;
  if (workspace_bytes < bn_workspace_bytes(g.C)) {
    set_error("staged post-op workspace: have %zu bytes, need %zu", workspace_bytes, bn_workspace_bytes(g.C));
    return DCN_ERR_WORKSPACE;
  }
  return bn_relu_backward_staged(g, t, training, (const float*)x, (const float*)grad_staged, (const float*)saved,
                                 (float*)grad_x, (float*)grad_gamma, (float*)grad_beta, workspace, (cudaStream_t)stream);
}

int dcn_layer_backward(const DcnShape* s, const void* x, const void* offset, const void* offset_weight,
                       const void* weight, const void* grad_out, void* grad_x, void* grad_offset_weight,
                       void* grad_offset_bias, void* grad_weight, void* grad_bias, void* workspace,
                       size_t workspace_bytes, void* stream) {
  return layer_backward_impl(s, DCN_PHASE_LAYER_BACKWARD, "layer backward", x, offset, nullptr, offset_weight, weight,
                             grad_out, grad_x, grad_offset_weight, grad_offset_bias, grad_weight, grad_bias, workspace,
                             workspace_bytes, stream);
}

// ---- whole modulated layer (mmcv's ModulatedDeformConv2dPack) -----------------------------------------------------
int dcn_offset_conv_forward_modulated(const DcnShape* s, const void* x, const void* offset_weight,
                                      const void* offset_bias, void* offset, void* mask, void* workspace,
                                      size_t workspace_bytes, void* stream) {
  return offset_conv_impl(s, DCN_PHASE_LAYER_FORWARD_MODULATED, "offset-and-mask conv", x, offset_weight, offset_bias,
                          offset, mask, workspace, workspace_bytes, stream);
}

int dcn_layer_forward_modulated(const DcnShape* s, const void* x, const void* offset_weight, const void* offset_bias,
                                const void* weight, const void* bias, void* offset, void* mask, void* out,
                                void* workspace, size_t workspace_bytes, void* stream) {
  return layer_forward_impl(s, nullptr, DCN_PHASE_LAYER_FORWARD_MODULATED, "modulated layer forward", x, offset_weight,
                            offset_bias, weight, bias, offset, mask, out, workspace, workspace_bytes, stream);
}

int dcn_layer_backward_modulated(const DcnShape* s, const void* x, const void* offset, const void* mask,
                                 const void* offset_weight, const void* weight, const void* grad_out, void* grad_x,
                                 void* grad_offset_weight, void* grad_offset_bias, void* grad_weight, void* grad_bias,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  return layer_backward_impl(s, DCN_PHASE_LAYER_BACKWARD_MODULATED, "modulated layer backward", x, offset, mask,
                             offset_weight, weight, grad_out, grad_x, grad_offset_weight, grad_offset_bias,
                             grad_weight, grad_bias, workspace, workspace_bytes, stream);
}

int dcn_debug_corners(const DcnShape* s, const void* offset, int32_t* y0, int32_t* x0, float* w4,
                      void* stream) {
  Geo g;
  int rc = geo_or_error(s, &g);
  if (rc) return rc;
  if ((rc = check_ptr(offset, "offset")) || (rc = check_ptr(y0, "y0")) ||
      (rc = check_ptr(x0, "x0")) || (rc = check_ptr(w4, "w4")))
    return rc;
  return launch_corners(g, (const float*)offset, y0, x0, w4, (cudaStream_t)stream);
}

int dcn_msda_forward(const DcnMsdaShape* s, const void* value, const int64_t* spatial_shapes,
                     const int64_t* level_start_index, const void* sampling_locations, const void* attention_weights,
                     void* out, void* stream) {
  int rc;
  if ((rc = msda_shape_ok(s, "dcn_msda_forward")) || (rc = check_ptr(value, "value")) ||
      (rc = check_ptr(spatial_shapes, "spatial_shapes")) || (rc = check_ptr(level_start_index, "level_start_index")) ||
      (rc = check_ptr(sampling_locations, "sampling_locations")) ||
      (rc = check_ptr(attention_weights, "attention_weights")) || (rc = check_ptr(out, "out")))
    return rc;
  return msda_forward(*s, (const float*)value, spatial_shapes, level_start_index, (const float*)sampling_locations,
                      (const float*)attention_weights, (float*)out, (cudaStream_t)stream);
}

int dcn_msda_backward(const DcnMsdaShape* s, const void* value, const int64_t* spatial_shapes,
                      const int64_t* level_start_index, const void* sampling_locations, const void* attention_weights,
                      const void* grad_out, void* grad_value, void* grad_sampling_locations,
                      void* grad_attention_weights, void* stream) {
  int rc;
  if ((rc = msda_shape_ok(s, "dcn_msda_backward")) || (rc = check_ptr(value, "value")) ||
      (rc = check_ptr(spatial_shapes, "spatial_shapes")) || (rc = check_ptr(level_start_index, "level_start_index")) ||
      (rc = check_ptr(sampling_locations, "sampling_locations")) ||
      (rc = check_ptr(attention_weights, "attention_weights")) || (rc = check_ptr(grad_out, "grad_out")) ||
      (rc = check_ptr(grad_value, "grad_value", false)) ||
      (rc = check_ptr(grad_sampling_locations, "grad_sampling_locations", false)) ||
      (rc = check_ptr(grad_attention_weights, "grad_attention_weights", false)))
    return rc;
  return msda_backward(*s, (const float*)value, spatial_shapes, level_start_index, (const float*)sampling_locations,
                       (const float*)attention_weights, (const float*)grad_out, (float*)grad_value,
                       (float*)grad_sampling_locations, (float*)grad_attention_weights, (cudaStream_t)stream);
}

int dcn_v3_forward(const DcnV3Shape* s, float offset_scale, const void* input, const void* offset, const void* mask,
                   void* out, void* stream) {
  int rc, Ho, Wo;
  if ((rc = dcnv3_shape_ok(s, "dcn_v3_forward", &Ho, &Wo)) || (rc = check_ptr(input, "input")) ||
      (rc = check_ptr(offset, "offset")) || (rc = check_ptr(mask, "mask")) || (rc = check_ptr(out, "out")) ||
      (rc = dcnv3_supported(s, "dcn_v3_forward")))
    return rc;
  return dcnv3_forward(*s, Ho, Wo, offset_scale, (const float*)input, (const float*)offset, (const float*)mask,
                       (float*)out, (cudaStream_t)stream);
}

int dcn_v3_backward(const DcnV3Shape* s, float offset_scale, const void* input, const void* offset, const void* mask,
                    const void* grad_out, void* grad_input, void* grad_offset, void* grad_mask, void* stream) {
  int rc, Ho, Wo;
  if ((rc = dcnv3_shape_ok(s, "dcn_v3_backward", &Ho, &Wo)) || (rc = check_ptr(input, "input")) ||
      (rc = check_ptr(offset, "offset")) || (rc = check_ptr(mask, "mask")) || (rc = check_ptr(grad_out, "grad_out")) ||
      (rc = check_ptr(grad_input, "grad_input", false)) || (rc = check_ptr(grad_offset, "grad_offset", false)) ||
      (rc = check_ptr(grad_mask, "grad_mask", false)) || (rc = dcnv3_supported(s, "dcn_v3_backward")))
    return rc;
  return dcnv3_backward(*s, Ho, Wo, offset_scale, (const float*)input, (const float*)offset, (const float*)mask,
                        (const float*)grad_out, (float*)grad_input, (float*)grad_offset, (float*)grad_mask,
                        (cudaStream_t)stream);
}

int dcn_v4_forward(const DcnV3Shape* s, float offset_scale, const void* input, const void* offset_mask, void* out,
                   void* stream) {
  int rc, Ho, Wo;
  if ((rc = dcnv4_shape_ok(s, "dcn_v4_forward", &Ho, &Wo)) || (rc = check_ptr(input, "input")) ||
      (rc = check_ptr(offset_mask, "offset_mask")) || (rc = check_ptr(out, "out")) ||
      (rc = dcnv4_supported(s, "dcn_v4_forward")))
    return rc;
  return dcnv4_forward(*s, Ho, Wo, offset_scale, (const float*)input, (const float*)offset_mask, (float*)out,
                       (cudaStream_t)stream);
}

int dcn_v4_backward(const DcnV3Shape* s, float offset_scale, const void* input, const void* offset_mask,
                    const void* grad_out, void* grad_input, void* grad_offset_mask, void* stream) {
  int rc, Ho, Wo;
  if ((rc = dcnv4_shape_ok(s, "dcn_v4_backward", &Ho, &Wo)) || (rc = check_ptr(input, "input")) ||
      (rc = check_ptr(offset_mask, "offset_mask")) || (rc = check_ptr(grad_out, "grad_out")) ||
      (rc = check_ptr(grad_input, "grad_input", false)) ||
      (rc = check_ptr(grad_offset_mask, "grad_offset_mask", false)) || (rc = dcnv4_supported(s, "dcn_v4_backward")))
    return rc;
  return dcnv4_backward(*s, Ho, Wo, offset_scale, (const float*)input, (const float*)offset_mask,
                        (const float*)grad_out, (float*)grad_input, (float*)grad_offset_mask, (cudaStream_t)stream);
}

size_t dcn_bn_workspace_bytes(int32_t C) { return C > 0 ? bn_workspace_bytes(C) : 0; }

int dcn_bn_relu_forward(int32_t B, int32_t C, int32_t HW, int32_t training, const void* x, const void* gamma,
                        const void* beta, void* running_mean, void* running_var, float momentum, float eps,
                        void* y, void* saved, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = bn_shape_ok(B, C, HW);
  if (rc) return rc;
  if ((rc = check_ptr(x, "x")) || (rc = check_ptr(y, "y")) || (rc = check_ptr(saved, "saved")) ||
      (rc = check_ptr(workspace, "workspace")))
    return rc;
  if (!training && (!running_mean || !running_var)) {
    set_error("eval-mode batch norm needs running_mean and running_var");
    return DCN_ERR_NULL_POINTER;
  }
  if (workspace_bytes < bn_workspace_bytes(C)) {
    set_error("batch-norm workspace: have %zu bytes, need %zu", workspace_bytes, bn_workspace_bytes(C));
    return DCN_ERR_WORKSPACE;
  }
  return bn_relu_forward(B, C, HW, training, (const float*)x, (const float*)gamma, (const float*)beta,
                         (float*)running_mean, (float*)running_var, momentum, eps, (float*)y, (float*)saved,
                         workspace, (cudaStream_t)stream);
}

int dcn_bn_relu_backward(int32_t B, int32_t C, int32_t HW, int32_t training, const void* x, const void* grad_y,
                         const void* saved, void* grad_x, void* grad_gamma, void* grad_beta, void* workspace,
                         size_t workspace_bytes, void* stream) {
  int rc = bn_shape_ok(B, C, HW);
  if (rc) return rc;
  if ((rc = check_ptr(x, "x")) || (rc = check_ptr(grad_y, "grad_y")) || (rc = check_ptr(saved, "saved")) ||
      (rc = check_ptr(workspace, "workspace")))
    return rc;
  if (workspace_bytes < bn_workspace_bytes(C)) {
    set_error("batch-norm workspace: have %zu bytes, need %zu", workspace_bytes, bn_workspace_bytes(C));
    return DCN_ERR_WORKSPACE;
  }
  return bn_relu_backward(B, C, HW, training, (const float*)x, (const float*)grad_y, (const float*)saved,
                          (float*)grad_x, (float*)grad_gamma, (float*)grad_beta, workspace, (cudaStream_t)stream);
}

}  // extern "C"
