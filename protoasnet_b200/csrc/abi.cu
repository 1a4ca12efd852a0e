// extern "C" entry points of libpasn_b200.so (declared in include/pasn.h) and path dispatch.
#include "common.cuh"
#include "tc_gemm.cuh"

using namespace pasn;

static bool dims_ok(const pasn_dims* d) {
  if (!d) return false;
  if (d->N < 0 || d->C <= 0 || d->D <= 0 || d->P <= 0 || d->K <= 0 || d->S <= 0) return false;
  if (d->D % 2 != 0) return false;  // occurrence_module hidden width is D // 2
  if (d->dtype != PASN_F32 && d->dtype != PASN_BF16 && d->dtype != PASN_F16) return false;
  if (d->layout != PASN_LAYOUT_NCS && d->layout != PASN_LAYOUT_NSC) return false;
  if (d->occ_act != PASN_OCC_ABS) return false;
  if (d->path < PASN_PATH_AUTO || d->path > PASN_PATH_TILED) return false;
  return true;
}

// which kernel family serves these dims: 0 generic, 1 fused token kernel, 2 tiled GEMM chain; *err when an explicitly
// requested family cannot run them.  fp16 feature maps are served by the tensor-core families only (the CUDA-core path is
// the fp32 correctness path): without one of them *err is PASN_ERR_UNSUPPORTED.
enum { FAM_GENERIC = 0, FAM_FUSED = 1, FAM_TILED = 2 };
static int resolve_family_any(const pasn_dims& d, int* err);
static int resolve_family(const pasn_dims& d, int* err) {
  const int fam = resolve_family_any(d, err);
  if (d.dtype == PASN_F16 && fam == FAM_GENERIC) *err = PASN_ERR_UNSUPPORTED;
  return fam;
}
static int resolve_family_any(const pasn_dims& d, int* err) {
  *err = PASN_OK;
  switch (d.path) {
    case PASN_PATH_GENERIC: return FAM_GENERIC;
    case PASN_PATH_TCGEN05:
      if (sm100_supported(d)) return FAM_FUSED;
      *err = PASN_ERR_UNSUPPORTED;
      return FAM_GENERIC;
    case PASN_PATH_TILED:
      if (tiled_supported(d)) return FAM_TILED;
      *err = PASN_ERR_UNSUPPORTED;
      return FAM_GENERIC;
    default:
      if (sm100_supported(d)) return FAM_FUSED;
      if (tiled_supported(d)) return FAM_TILED;
      return FAM_GENERIC;
  }
}

// ---- sticky fault word: pinned host memory mapped into the device address space -------------------
static volatile int* g_fault_host = nullptr;
static int* g_fault_dev = nullptr;
namespace pasn {
int* fault_word() {
  static bool tried = false;
  if (!tried) {
    tried = true;
    int* h = nullptr;
    if (cudaHostAlloc(reinterpret_cast<void**>(&h), 64, cudaHostAllocMapped | cudaHostAllocPortable) == cudaSuccess) {
      *h = 0;
      void* d = nullptr;
      if (cudaHostGetDevicePointer(&d, h, 0) == cudaSuccess) { g_fault_host = h; g_fault_dev = reinterpret_cast<int*>(d); }
    }
    (void)cudaGetLastError();
  }
  return g_fault_dev;
}
}  // namespace pasn
static inline bool faulted() { return g_fault_host != nullptr && *g_fault_host != 0; }
extern "C" int pasn_debug_fault(void) { return g_fault_host ? *g_fault_host : 0; }
extern "C" int pasn_debug_set_fault(int code) {
  if (fault_word() == nullptr) return PASN_ERR_CUDA;
  *g_fault_host = code;
  return PASN_OK;
}

// ---- measurement hooks ------------------------------------------------------------------------
static unsigned long long g_launches = 0;
static int g_time_main = 0;
static cudaEvent_t g_ev0 = nullptr, g_ev1 = nullptr;
namespace pasn {
void count_launch(int n) { g_launches += (unsigned long long)n; }
void main_kernel_begin(cudaStream_t st) {
  if (!g_time_main) return;
  if (!g_ev0) { cudaEventCreate(&g_ev0); cudaEventCreate(&g_ev1); }
  cudaEventRecord(g_ev0, st);
}
void main_kernel_end(cudaStream_t st) {
  if (g_time_main && g_ev1) cudaEventRecord(g_ev1, st);
}
}  // namespace pasn
extern "C" unsigned long long pasn_debug_launch_count(void) { return g_launches; }
extern "C" int pasn_debug_time_main_kernel(int enable) { g_time_main = enable; return PASN_OK; }
extern "C" float pasn_debug_last_main_kernel_ms(void) {
  if (!g_ev0 || !g_ev1) return -1.f;
  if (cudaEventSynchronize(g_ev1) != cudaSuccess) return -1.f;
  float ms = -1.f;
  if (cudaEventElapsedTime(&ms, g_ev0, g_ev1) != cudaSuccess) return -1.f;
  return ms;
}

extern "C" int pasn_similarity_stats(const float* similarity, const int64_t* labels, int32_t N, int32_t P, int32_t K,
                                     int32_t abstain, int32_t n_specific, int32_t top_specific, int32_t top_rest,
                                     float* class_max, int32_t* class_arg, double* sums, uint64_t* counts,
                                     double* sim_cumsum, void* stream) {
  if (N < 0 || P <= 0 || K <= 0 || (sums && !labels)) return PASN_ERR_INVALID;
  if (N > 0 && !similarity) return PASN_ERR_INVALID;
  return launch_sim_stats(similarity, labels, N, P, K, abstain, n_specific, top_specific, top_rest, class_max, class_arg,
                          sums, reinterpret_cast<unsigned long long*>(counts), sim_cumsum,
                          reinterpret_cast<cudaStream_t>(stream));
}
extern "C" int pasn_occurrence_lnorm(const void* occ, int32_t dtype, int64_t rows, int32_t S, int32_t p, double* sum,
                                     float* row_norm, void* stream) {
  if (rows < 0 || S <= 0 || !sum || (rows > 0 && !occ)) return PASN_ERR_INVALID;
  if (dtype != PASN_F32 && dtype != PASN_BF16 && dtype != PASN_F16) return PASN_ERR_INVALID;
  return launch_occ_lnorm(occ, dtype, rows, S, p, sum, row_norm, reinterpret_cast<cudaStream_t>(stream));
}

// fp16 feature maps: tensor-core backward only
static bool backward_ok(const pasn_dims* d) { return dims_ok(d) && (d->dtype != PASN_F16 || tiled_backward_supported(*d)); }
extern "C" size_t pasn_head_backward_workspace_bytes(const pasn_dims* dims) {
  return backward_ok(dims) ? backward_workspace_bytes(*dims) : 0;
}
extern "C" int pasn_head_backward(const void* feat, const pasn_weights* w, const pasn_dims* dims, const float* grad_logits,
                                  const float* grad_similarity, const float* grad_occurrence, const pasn_grads* grads,
                                  float* grad_feat, void* workspace, size_t workspace_bytes, void* stream) {
  if (!dims_ok(dims) || !w || !grads) return PASN_ERR_INVALID;
  if (!backward_ok(dims)) return PASN_ERR_UNSUPPORTED;
  if (faulted()) return PASN_ERR_FAULT;
  if (dims->N == 0) return PASN_OK;
  if (!feat || !workspace) return PASN_ERR_INVALID;
  const float* const* gp = reinterpret_cast<const float* const*>(grads);
  for (int i = 0; i < 11; ++i)
    if (!gp[i]) return PASN_ERR_INVALID;
  return head_backward(feat, *w, *dims, grad_logits, grad_similarity, grad_occurrence, *grads, grad_feat, workspace,
                       workspace_bytes, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int pasn_debug_sm100_error(const void* workspace, const pasn_dims* dims, void* stream) {
  if (!workspace || !dims_ok(dims) || !sm100_supported(*dims)) return 0;
  return sm100_last_error(workspace, *dims, (cudaStream_t)stream);
}

extern "C" int pasn_debug_set_trace(void* device_buffer) { sm100_set_trace(device_buffer); return PASN_OK; }

// test hook: one launch of the internal tiled tcgen05 GEMM (descriptor = pasn::tcg::Gemm, see csrc/tc_gemm.cuh)
extern "C" size_t pasn_debug_tc_gemm_desc_bytes(void) { return sizeof(tcg::Gemm); }
extern "C" int pasn_debug_tc_gemm(const void* desc_host, size_t desc_bytes, void* stream) {
  if (!desc_host || desc_bytes != sizeof(tcg::Gemm)) return PASN_ERR_INVALID;
  if (faulted()) return PASN_ERR_FAULT;
  if (!tcg::available()) return PASN_ERR_UNSUPPORTED;
  return tcg::launch(*reinterpret_cast<const tcg::Gemm*>(desc_host), reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int pasn_debug_set_gemm_trace(void* device_buffer) { tcg::set_trace(device_buffer); return PASN_OK; }

extern "C" int pasn_abi_version(void) { return PASN_ABI_VERSION; }

extern "C" const char* pasn_strerror(int status) {
  switch (status) {
    case PASN_OK: return "ok";
    case PASN_ERR_INVALID: return "invalid argument or unsupported shape";
    case PASN_ERR_WORKSPACE: return "workspace too small (see pasn_head_workspace_bytes)";
    case PASN_ERR_CUDA: return "CUDA runtime call or kernel launch failed";
    case PASN_ERR_UNSUPPORTED: return "requested kernel path is not available for these dims";
    case PASN_ERR_ALIGN: return "pointer alignment requirement violated";
    case PASN_ERR_FAULT: return "an earlier kernel reported an internal pipeline fault (bounded wait expired); results are invalid";
    default: return "unknown pasn status";
  }
}

extern "C" int pasn_tcgen05_supported(const pasn_dims* dims) {
  if (!dims_ok(dims)) return 0;
  int err;
  const int fam = resolve_family(*dims, &err);
  return fam != FAM_GENERIC && err == PASN_OK ? 1 : 0;
}

extern "C" size_t pasn_head_workspace_bytes(const pasn_dims* dims) {
  if (!dims_ok(dims)) return 0;
  int err;
  const int fam = resolve_family(*dims, &err);
  if (dims->dtype == PASN_F16 && err) return 0;   // no family can run them
  size_t need = generic_workspace_bytes(*dims);   // the generic path stays available as the NULL-`packed` fallback
  if (dims->path == PASN_PATH_TCGEN05 || dims->path == PASN_PATH_TILED || dims->dtype == PASN_F16) need = 0;
  if (fam == FAM_FUSED) { const size_t t = sm100_workspace_bytes(*dims); need = t > need ? t : need; }
  if (fam == FAM_TILED) {   // (pasn_occurrence_only runs in the same family as the forward)
    const size_t t = tiled_workspace_bytes(*dims);
    need = t > need ? t : need;
  }
  return need;
}

extern "C" size_t pasn_packed_weights_bytes(const pasn_dims* dims) {
  if (!dims_ok(dims)) return 0;
  int err;
  const int fam = resolve_family(*dims, &err);
  return fam == FAM_FUSED ? sm100_packed_bytes(*dims) : (fam == FAM_TILED ? tiled_packed_bytes(*dims) : 0);
}

extern "C" int pasn_pack_weights(const pasn_weights* w, const pasn_dims* dims, void* packed, void* stream) {
  if (!w || !dims_ok(dims) || !packed) return PASN_ERR_INVALID;
  int err;
  const int fam = resolve_family(*dims, &err);
  if (fam == FAM_FUSED) return sm100_pack_weights(*w, *dims, packed, (cudaStream_t)stream);
  if (fam == FAM_TILED) return tiled_pack_weights(*w, *dims, packed, (cudaStream_t)stream);
  return PASN_ERR_UNSUPPORTED;
}

extern "C" int pasn_head_forward(const void* feat, const pasn_weights* w, const void* packed, const pasn_dims* dims,
                                 float* logits, float* similarity, void* occurrence_map, float* features_extracted,
                                 float* distance, const pasn_push_args* push, void* workspace, size_t workspace_bytes,
                                 void* stream) {
  if (!dims_ok(dims) || !w || !logits || !similarity) return PASN_ERR_INVALID;
  if (faulted()) return PASN_ERR_FAULT;
  if (dims->N == 0) return PASN_OK;
  if (!feat || !workspace) return PASN_ERR_INVALID;
  if (push && (!push->labels || !push->proto_class || !push->best_key)) return PASN_ERR_INVALID;   // best_vec is optional
  if (push && (push->global_offset < 0 || push->global_offset + dims->N > 0xFFFFFFFFll)) return PASN_ERR_INVALID;
  int err;
  int fam = resolve_family(*dims, &err);
  if (err) return err;
  if (fam != FAM_GENERIC && packed == nullptr) {
    if (dims->path != PASN_PATH_AUTO || dims->dtype == PASN_F16) return PASN_ERR_UNSUPPORTED;
    fam = FAM_GENERIC;
  }
  if (fam == FAM_FUSED)
    return sm100_head_forward(feat, *w, packed, *dims, logits, similarity, occurrence_map, features_extracted,
                              distance, push, workspace, workspace_bytes, (cudaStream_t)stream);
  if (fam == FAM_TILED)
    return tiled_head_forward(feat, *w, packed, *dims, logits, similarity, occurrence_map, features_extracted, distance,
                              push, workspace, workspace_bytes, (cudaStream_t)stream);
  return generic_head_forward(feat, *w, *dims, logits, similarity, occurrence_map, features_extracted, distance, push,
                              workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int pasn_occurrence_only(const void* feat, const pasn_weights* w, const void* packed, const pasn_dims* dims,
                                    void* occurrence_map, void* workspace, size_t workspace_bytes, void* stream) {
  if (!dims_ok(dims) || !w || !occurrence_map) return PASN_ERR_INVALID;
  if (faulted()) return PASN_ERR_FAULT;
  if (dims->N == 0) return PASN_OK;
  if (!feat || !workspace) return PASN_ERR_INVALID;
  int err;
  int fam = resolve_family(*dims, &err);   // same family (and therefore the same packed weights) as pasn_head_forward
  if (err) return err;
  if (fam != FAM_GENERIC && packed == nullptr) {
    if (dims->path != PASN_PATH_AUTO || dims->dtype == PASN_F16) return PASN_ERR_UNSUPPORTED;
    fam = FAM_GENERIC;
  }
  if (fam == FAM_FUSED)
    return sm100_occurrence_only(feat, *w, packed, *dims, occurrence_map, workspace, workspace_bytes, (cudaStream_t)stream);
  if (fam == FAM_TILED)
    return tiled_occurrence_only(feat, *w, packed, *dims, occurrence_map, workspace, workspace_bytes, (cudaStream_t)stream);
  return generic_occurrence_only(feat, *w, *dims, occurrence_map, workspace, workspace_bytes, (cudaStream_t)stream);
}
