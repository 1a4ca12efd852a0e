// Definitions shared by the fused head's token kernel (head_sm100_k1.cu) and its host side and prototype kernel
// (head_sm100.cu): tile constants, packed-weight layout, kernel parameters, bounded waits, epilogue helpers.
#pragma once
#include "common.cuh"
#include "sm100_prims.cuh"

namespace pasn {
namespace k1 {
using namespace sm100;

constexpr int TILE_M = 128;
constexpr int DD = 256;            // prototype depth D handled by this kernel
constexpr int DH = DD / 2;         // occurrence hidden width
constexpr int PP_MAX = 48;         // padded prototype count limit (multiple of 8)
constexpr uint32_t FE_TILE_BYTES = 131072;  // K2 operand images of one 128-row tile: hi 64 KB | lo 64 KB

// packed weight buffer (bf16 stage images + fp32 biases), see pack_weights_kernel
struct PackedLayout {
  size_t off_l1, off_w4, off_w5, off_bias, off_w2, off_b2, total;
};
__host__ __device__ inline PackedLayout packed_layout(int C) {
  PackedLayout L;
  const int nkc = C / 64;
  L.off_l1 = 0;
  L.off_w4 = (size_t)2 * nkc * 32768;
  L.off_w5 = L.off_w4 + 65536;
  L.off_bias = L.off_w5 + 16384;
  L.off_w2 = (L.off_bias + (DD + DD + DH) * 4 + 1023) / 1024 * 1024;
  L.off_b2 = L.off_w2 + 4 * 32768;
  L.total = L.off_b2 + DD * 4;
  return L;
}

struct K1Params {
  const __nv_bfloat16* feat;   // [N][C][S] (bf16 input)
  const float* feat32;         // same buffer seen as fp32 when f32_in (bf16-compute mode for fp32 feature maps)
  float* occ32;                // occurrence map as fp32 when f32_in
  int f32_in;
  int nsc;                     // feature map is [N][S][C] (channels_last): bf16 or fp16
  const uint8_t* packed;
  __nv_bfloat16* occ;          // [N][P][S] or null
  uint8_t* feimg;              // K2 operand images, FE_TILE_BYTES per K2 tile
  float* osum;                 // [N][P]
  int N, C, P, S, nkc, clips_per_cta, cpt;  // cpt = clips per K2 tile = 128 / PP
  // small batches: every clip is cut into G voxel groups of S voxels that are processed as G independent "clips"
  // (pooling is linear in the voxels; the partial sums are added after K2).  N and S above are the virtual counts,
  // SR the real voxel count per clip (= row pitch of the feature map and of the occurrence map).  G = 1: no split.
  int G, SR;
  int* err;
  int* fault;                  // host-mapped sticky fault word (or null)
  long long* trace;            // optional [3][16][16] clock64 stamps of CTA 0 (MMA thread, epilogue warp 4)
  int f16_in;                  // fp16 feature map (read as it is; layer-1 MMAs fp16 x fp16 with fp16 weight images), map in fp16
};

struct Ctx {
  int* err;
  volatile int* abort_s;
  int* fault;   // host-mapped sticky fault word (may be null)
};

// bounded wait: returns false (and raises the CTA-wide abort flag) instead of hanging on a protocol bug.  The spin is
// out of line so that the fast path at every call site is a single try_wait.
static __device__ __noinline__ bool bwait_slow(uint64_t* bar, uint32_t parity, int* err, volatile int* abort_s, int* fault, int code) {
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (*abort_s) return false;
    if (clock64() - t0 > 4000000000ll) {
      *abort_s = 1;
      atomicCAS(err, 0, code);
      if (fault != nullptr) *reinterpret_cast<volatile int*>(fault) = code;
      return false;
    }
  }
  return true;
}
__device__ __forceinline__ bool bwait(uint64_t* bar, uint32_t parity, const Ctx& c, int code) {
  if (mbar_try_wait(bar, parity)) return true;
  return bwait_slow(bar, parity, c.err, c.abort_s, c.fault, code);
}

__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// 32 fp32 accumulator columns + bias -> ReLU -> 16 packed bf16x2 (bias: 32 floats in smem, 16-byte aligned)
__device__ __forceinline__ void bias_relu_pack(const uint32_t (&r)[32], const float* bias, uint32_t* pk) {
#pragma unroll
  for (int j4 = 0; j4 < 8; ++j4) {
    const float4 b = *reinterpret_cast<const float4*>(bias + 4 * j4);
    pk[2 * j4] = pack_bf16x2_relu(__uint_as_float(r[4 * j4 + 0]) + b.x, __uint_as_float(r[4 * j4 + 1]) + b.y);
    pk[2 * j4 + 1] = pack_bf16x2_relu(__uint_as_float(r[4 * j4 + 2]) + b.z, __uint_as_float(r[4 * j4 + 3]) + b.w);
  }
}

#define K1_TRACE(role, tile, slot)                                                            \
  do {                                                                                        \
    if (p.trace != nullptr && blockIdx.x == 0 && (tile) < 16)                                 \
      p.trace[((role) * 16 + (tile)) * 16 + (slot)] = clock64();                              \
  } while (0)


}  // namespace k1

// token kernel (head_sm100_k1.cu)
int launch_k1(const k1::K1Params& k1p, int ppad, int grid, cudaStream_t st);

}  // namespace pasn
