// Shared device/host helpers for libpasn_b200 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pasn.h"

namespace pasn {

#define PASN_LAUNCH_CHECK()                           \
  do {                                                \
    if (cudaGetLastError() != cudaSuccess) return PASN_ERR_CUDA; \
  } while (0)

__host__ __device__ inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
// most clips one chunk of the generic or tiled path takes: kernels of both put the clip index in gridDim.y / z
constexpr int kMaxChunkClips = 65535;

// bytes per element of a feature / occurrence map of this pasn_dtype (the one place that knows the element sizes)
__host__ __device__ inline size_t dtype_bytes(int dtype) { return dtype == PASN_F32 ? 4 : 2; }

template <typename T>
__device__ __forceinline__ float to_f32(T v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <>
__device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }

__device__ __forceinline__ float round_bf16(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

// Monotone map fp32 -> u32 (total order incl. negatives), used for packed argmin keys.
__host__ __device__ __forceinline__ uint32_t f32_orderable(float f) {
#ifdef __CUDA_ARCH__
  uint32_t u = __float_as_uint(f);
#else
  union { float f; uint32_t u; } c; c.f = f; uint32_t u = c.u;
#endif
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float f32_from_orderable(uint32_t o) {
  uint32_t u = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  union { float f; uint32_t u; } c; c.u = u; return c.f;
#endif
}
__host__ __device__ __forceinline__ unsigned long long pack_key(float dist, uint32_t gidx) {
  return ((unsigned long long)f32_orderable(dist) << 32) | (unsigned long long)gidx;
}
#define PASN_KEY_NONE 0xFFFFFFFFFFFFFFFFull
// Keys are kept as unsigned (orderable(dist) << 32 | index) inside a kernel; in global memory (pasn_push_args.best_key)
// the top bit is flipped so that SIGNED 64-bit order equals the unsigned key order -- an NCCL all-reduce(MIN) over
// int64 then merges ranks directly.  "No candidate" is INT64_MAX.
#define PASN_KEY_SIGN 0x8000000000000000ull
__device__ __forceinline__ void key_atomic_min_global(unsigned long long* best_key_signed, unsigned long long key_u) {
  atomicMin(reinterpret_cast<long long*>(best_key_signed), (long long)(key_u ^ PASN_KEY_SIGN));
}

// programmatic dependent launch (see launch_pdl): let the next kernel of the stream start setting itself up / wait until the
// kernel in front has completed and flushed its writes.  Both are no-ops for a kernel that was launched the ordinary way.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// kernel<<<grid, block, smem, st>>>(args...) with programmatic stream serialization allowed: the kernel may be scheduled while
// the previous kernel of the stream drains; it must call pdl_wait() before its first global-memory access.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- generic path (generic.cu) -------------------------------------------------------------
size_t generic_workspace_bytes(const pasn_dims& d);
int launch_sim_stats(const float* sim, const int64_t* labels, int N, int P, int K, int abstain, int n_specific, int top_a,
                     int top_b, float* class_max, int32_t* class_arg, double* sums, unsigned long long* counts, double* simsum,
                     cudaStream_t st);
int launch_occ_lnorm(const void* occ, int dtype, long long rows, int S, int p, double* sums, float* row_norm, cudaStream_t st);
int generic_head_forward(const void* feat, const pasn_weights& w, const pasn_dims& d, float* logits, float* sim,
                         void* occ, float* feats, float* dist, const pasn_push_args* push, void* ws, size_t ws_bytes,
                         cudaStream_t st);
int generic_occurrence_only(const void* feat, const pasn_weights& w, const pasn_dims& d, void* occ, void* ws,
                            size_t ws_bytes, cudaStream_t st);
// backward on the CUDA cores: fp32 / bf16 feature maps, any shape; the shapes tiled_backward_supported() rejects
size_t generic_backward_workspace_bytes(const pasn_dims& d);
int generic_head_backward(const void* feat, const pasn_weights& w, const pasn_dims& d, const pasn_upstream& up,
                          const pasn_grads& g, float* gX, void* ws, size_t ws_bytes, cudaStream_t st);
// gWl[k][p] += sum_n gL[n][k] sim[n][p] (one FFMA GEMM, each output tile summed by one block: deterministic)
int generic_last_layer_backward(const float* gL, const float* sim, int N, int P, int K, float* gWl, cudaStream_t st);

// Which intermediate gradients of the head's backward some wanted output depends on.  A NULL member of pasn_grads (or a
// NULL grad_feat) is not wanted, and work that serves only unwanted outputs is skipped; both backward families prune by
// this table.  Every wanted output depends on the prototype stage, so `proto` is false exactly when nothing is wanted.
struct BwdNeeds {
  bool gH1, gF, gG1, gG2, gOpre, proto;
};
inline BwdNeeds bwd_needs(const pasn_grads& g, const float* gX) {
  BwdNeeds n;
  n.gH1 = g.addon_w1 || g.addon_b1 || gX;
  n.gF = g.addon_w2 || g.addon_b2 || n.gH1;
  n.gG1 = g.occ_w1 || g.occ_b1 || gX;
  n.gG2 = g.occ_w2 || g.occ_b2 || n.gG1;
  n.gOpre = g.occ_w3 || n.gG2;
  n.proto = g.prototypes || g.last_layer || n.gF || n.gOpre;
  return n;
}

// ---- prototype stage (proto_stage.cu): cosine -> (.+1)/2 -> logits -> 1-s -> running argmin keys ----
int launch_proto_stage(const float* feats /*[N,P,D]*/, const float* protos, const float* last_layer, int N, int P,
                       int D, int K, float* logits, float* sim, float* dist, const pasn_push_args* push,
                       cudaStream_t st);

// prototype stage from per-row statistics left by the GEMM that made the pooled features (tiled path, plain forward):
// stat[(n*P + p) * nparts + t] = (||f||^2, <f, v_p>, ||v_p||^2, -) over the columns of part t
int launch_proto_from_stats(const float* stat, int nparts, const float* last_layer, int N, int P, int K, float* logits, float* sim,
                            float* dist, cudaStream_t st);

// ---- tiled tcgen05 path (tiled.cu, tc_gemm.cu): chain of TMA-fed GEMMs, bf16 or fp32 (hi/lo split) -----------------
bool tiled_supported(const pasn_dims& d);
size_t tiled_workspace_bytes(const pasn_dims& d);
size_t tiled_packed_bytes(const pasn_dims& d);
int tiled_pack_weights(const pasn_weights& w, const pasn_dims& d, void* packed, cudaStream_t st);
int tiled_head_forward(const void* feat, const pasn_weights& w, const void* packed, const pasn_dims& d, float* logits,
                       float* sim, void* occ, float* feats, float* dist, const pasn_push_args* push, void* ws,
                       size_t ws_bytes, cudaStream_t st);
int tiled_occurrence_only(const void* feat, const pasn_weights& w, const void* packed, const pasn_dims& d, void* occ, void* ws,
                          size_t ws_bytes, cudaStream_t st);

// backward on the tensor cores (tiled.cu): fp32-grade hi/lo GEMM chain; serves the shapes tiled_supported() takes unless
// dims.path asks for the generic CUDA-core kernels
bool tiled_backward_supported(const pasn_dims& d);
size_t tiled_backward_workspace_bytes(const pasn_dims& d);
int tiled_head_backward(const void* feat, const pasn_weights& w, const pasn_dims& d, const pasn_upstream& up,
                        const pasn_grads& g, float* gX, void* ws, size_t ws_bytes, cudaStream_t st);

// ---- fused tcgen05 path (head_sm100.cu) -----------------------------------------------------
bool sm100_supported(const pasn_dims& d);
size_t sm100_workspace_bytes(const pasn_dims& d);
size_t sm100_packed_bytes(const pasn_dims& d);
int sm100_pack_weights(const pasn_weights& w, const pasn_dims& d, void* packed, cudaStream_t st);
int sm100_head_forward(const void* feat, const pasn_weights& w, const void* packed, const pasn_dims& d, float* logits,
                       float* sim, void* occ, float* feats, float* dist, const pasn_push_args* push, void* ws,
                       size_t ws_bytes, cudaStream_t st);
int sm100_occurrence_only(const void* feat, const pasn_weights& w, const void* packed, const pasn_dims& d, void* occ, void* ws,
                          size_t ws_bytes, cudaStream_t st);
int sm100_last_error(const void* ws, const pasn_dims& d, cudaStream_t st);
void sm100_set_trace(void* dev_buf);

}  // namespace pasn

// ---- debug / measurement hooks (abi.cu) -----------------------------------------------------
namespace pasn {
int* fault_word();                                // device-visible alias of the host-mapped sticky fault word (or nullptr)
void count_launch(int n = 1);                     // every kernel launch of the library is counted
void main_kernel_begin(cudaStream_t st);          // bracket the dominant kernel with CUDA events when enabled
void main_kernel_end(cudaStream_t st);
}
