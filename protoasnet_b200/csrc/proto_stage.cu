// Prototype stage: pooled features -> cosine similarity vs prototype vectors -> (cos+1)/2 -> last-layer logits
// -> push distance 1-s -> class-restricted running argmin keys.
//
// Reference arithmetic being restated (fp32 throughout):
//   nn.CosineSimilarity(dim=2, eps=1e-8): each norm clamped separately, normalise, then dot
//                                                       src/models/Video_XProtoNet.py:65, :90-92
//   similarity = (similarity + 1) / 2.0                 :93
//   logits = last_layer(similarity)  (no bias)          :96
//   distance = 1 - similarity                           :130
//   running argmin with class mask                      src/utils/push_abs_revision.py:288-307
// Bit-exact push indices need this exact rounding chain: argmin is taken over d = 1-(cos+1)/2, never over
// raw cos (SURVEY.md section 0 row 4).  Ties resolve to the lowest global index through the packed key.
#include "common.cuh"

namespace pasn {

constexpr int PS_THREADS = 256;
constexpr int PS_WARPS = PS_THREADS / 32;

// One warp per (clip, prototype) row: cosine vs the prototype vector, (cos+1)/2, 1-s, push key.  Rows are spread over
// the whole grid (N*P rows / 8 per block), so P = 40 and P = 4096 both fill the machine.
// The warp stride over the rows is a multiple of P, so a warp keeps ONE prototype: its vector, already divided by its
// clamped norm, lives in registers (NV = D / 32 values per lane), and a feature row is read from memory exactly once
// (NV independent coalesced loads in flight).  Element -> lane mapping and the order of every sum are those of the
// generic loop below (d = lane + 32 i), so both forms give the same bits.
template <int NV>
__global__ void __launch_bounds__(256) proto_rows_reg_kernel(
    const float* __restrict__ feats, const float* __restrict__ protos, long long rows, int P,
    float* __restrict__ sim, float* __restrict__ dist, const int64_t* __restrict__ labels,
    const int32_t* __restrict__ proto_class, long long global_offset, unsigned long long* __restrict__ best_key) {
  constexpr int D = NV * 32;
  pdl_launch_dependents();
  pdl_wait();   // the features come from the kernel in front (pooling / W2 GEMM)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long w0 = (long long)blockIdx.x * 8 + warp, wstride = (long long)gridDim.x * 8;   // wstride % P == 0 (host)
  if (w0 >= rows) return;
  const int p = (int)(w0 % P);
  float vq[NV];
  {
    const float* v = protos + (size_t)p * D;
    float vv = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) { vq[i] = v[lane + 32 * i]; vv = fmaf(vq[i], vq[i], vv); }
    vv = warp_sum(vv);
    const float nv = fmaxf(sqrtf(vv), 1e-8f);
#pragma unroll
    for (int i = 0; i < NV; ++i) vq[i] = vq[i] / nv;
  }
  const int pc = best_key != nullptr ? proto_class[p] : 0;
  // the next row's loads are issued before this row's reductions: a warp walks its rows one after the other, and without
  // the prefetch each row would pay the full memory latency in front of its dependent shuffle / divide chain
  float nx[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) nx[i] = __ldcs(feats + (size_t)w0 * D + lane + 32 * i);
  for (long long r = w0; r < rows; r += wstride) {
    float a[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) a[i] = nx[i];
    if (r + wstride < rows) {
      const float* fn = feats + (size_t)(r + wstride) * D;
#pragma unroll
      for (int i = 0; i < NV; ++i) nx[i] = __ldcs(fn + lane + 32 * i);
    }
    float ff = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) ff = fmaf(a[i], a[i], ff);
    ff = warp_sum(ff);
    const float nf = fmaxf(sqrtf(ff), 1e-8f);
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) dot = fmaf(a[i] / nf, vq[i], dot);
    dot = warp_sum(dot);
    if (lane == 0) {
      const long long n = r / P;
      const float s = (dot + 1.0f) / 2.0f;
      const float dd = 1.0f - s;
      sim[r] = s;
      if (dist) dist[r] = dd;
      if (best_key != nullptr) {
        if (pc < 0 || (long long)pc == labels[n]) {
          const unsigned long long key = pack_key(dd, (uint32_t)(global_offset + n));
          // plain read as a filter (the value only ever decreases), atomic only for candidates
          if ((long long)(key ^ PASN_KEY_SIGN) < *reinterpret_cast<volatile long long*>(best_key + p))
            key_atomic_min_global(&best_key[p], key);
        }
      }
    }
  }
}

// any D: the same arithmetic with the row read twice
__global__ void __launch_bounds__(PS_THREADS) proto_rows_kernel(
    const float* __restrict__ feats, const float* __restrict__ protos, long long rows, int P, int D,
    float* __restrict__ sim, float* __restrict__ dist, const int64_t* __restrict__ labels,
    const int32_t* __restrict__ proto_class, long long global_offset, unsigned long long* __restrict__ best_key) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (long long r = (long long)blockIdx.x * PS_WARPS + warp; r < rows; r += (long long)gridDim.x * PS_WARPS) {
    const long long n = r / P;
    const int p = (int)(r - n * P);
    const float* f = feats + (size_t)r * D;
    const float* v = protos + (size_t)p * D;
    float ff = 0.f, vv = 0.f;
    for (int d = lane; d < D; d += 32) {
      float a = f[d], b = v[d];
      ff = fmaf(a, a, ff);
      vv = fmaf(b, b, vv);
    }
    ff = warp_sum(ff);
    vv = warp_sum(vv);
    const float nf = fmaxf(sqrtf(ff), 1e-8f), nv = fmaxf(sqrtf(vv), 1e-8f);
    float dot = 0.f;
    for (int d = lane; d < D; d += 32) dot = fmaf(f[d] / nf, v[d] / nv, dot);
    dot = warp_sum(dot);
    if (lane == 0) {
      const float s = (dot + 1.0f) / 2.0f;
      const float dd = 1.0f - s;
      sim[r] = s;
      if (dist) dist[r] = dd;
      if (best_key != nullptr) {
        const int pc = proto_class[p];
        if (pc < 0 || (long long)pc == labels[n]) {
          const unsigned long long key = pack_key(dd, (uint32_t)(global_offset + n));
          // plain read as a filter (the value only ever decreases), atomic only for candidates
          if ((long long)(key ^ PASN_KEY_SIGN) < *reinterpret_cast<volatile long long*>(best_key + p))
            key_atomic_min_global(&best_key[p], key);
        }
      }
    }
  }
}

// logits[n,k] = sum_p sim[n,p] * last_layer[k,p]: one block per clip, one warp per class
__global__ void __launch_bounds__(PS_THREADS) proto_logits_kernel(const float* __restrict__ sim,
                                                                  const float* __restrict__ last_layer, int N, int P, int K,
                                                                  float* __restrict__ logits) {
  pdl_launch_dependents();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int n = blockIdx.x; n < N; n += gridDim.x) {
    const float* s = sim + (size_t)n * P;
    for (int k = warp; k < K; k += PS_WARPS) {
      float acc = 0.f;
      for (int p = lane; p < P; p += 32) acc = fmaf(s[p], last_layer[(size_t)k * P + p], acc);
      acc = warp_sum(acc);
      if (lane == 0) logits[(size_t)n * K + k] = acc;
    }
  }
}
// thousands of prototypes, few clips: one block per (clip, class) pair
__global__ void __launch_bounds__(PS_THREADS) proto_logits_wide_kernel(const float* __restrict__ sim,
                                                                       const float* __restrict__ last_layer, int N, int P, int K,
                                                                       float* __restrict__ logits) {
  __shared__ float red[PS_WARPS];
  pdl_launch_dependents();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = blockIdx.x / K, k = blockIdx.x - n * K;
  const float* s = sim + (size_t)n * P;
  const float* wl = last_layer + (size_t)k * P;
  float acc = 0.f;
  for (int p = threadIdx.x; p < P; p += PS_THREADS) acc = fmaf(s[p], wl[p], acc);
  acc = warp_sum(acc);
  if (lane == 0) red[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < PS_WARPS; ++i) t += red[i];
    logits[(size_t)n * K + k] = t;
  }
}

// Prototype stage from per-row statistics: the GEMM that produced the pooled features left, per column half-tile,
// (||f||^2, <f, v_p>, ||v_p||^2) over its columns instead of the features themselves.
// cos = <f, v> / (max(||f||, eps) max(||v||, eps)), then the reference's fp32 chain (cos+1)/2 and 1 - s (the fused kernels form
// the cosine the same way).
__device__ __forceinline__ float sim_from_stats(const float4* sp, int nparts) {
  float ff = 0.f, dot = 0.f, vv = 0.f;
  for (int t = 0; t < nparts; ++t) { const float4 v = sp[t]; ff += v.x; dot += v.y; vv += v.z; }
  const float cosv = dot / (fmaxf(sqrtf(ff), 1e-8f) * fmaxf(sqrtf(vv), 1e-8f));
  return (cosv + 1.0f) / 2.0f;
}
// thousands of prototypes: one thread per (clip, prototype) row, the logits by proto_logits_wide_kernel
__global__ void __launch_bounds__(256) proto_from_stats_kernel(const float* __restrict__ stat, int nparts, long long rows,
                                                               float* __restrict__ sim, float* __restrict__ dist) {
  pdl_launch_dependents();
  pdl_wait();
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const float s = sim_from_stats(reinterpret_cast<const float4*>(stat) + (size_t)r * nparts, nparts);
  sim[r] = s;
  if (dist) dist[r] = 1.0f - s;
}
// up to 1024 prototypes: one block per clip -- similarities into shared memory, then one warp per class for the logits
__global__ void __launch_bounds__(PS_THREADS) proto_finish_stats_kernel(const float* __restrict__ stat, int nparts,
                                                                        const float* __restrict__ last_layer, int N, int P, int K,
                                                                        float* __restrict__ logits, float* __restrict__ sim,
                                                                        float* __restrict__ dist) {
  __shared__ float s_sim[1024];
  pdl_launch_dependents();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int n = blockIdx.x; n < N; n += gridDim.x) {
    for (int pp = threadIdx.x; pp < P; pp += PS_THREADS) {
      const size_t r = (size_t)n * P + pp;
      const float s = sim_from_stats(reinterpret_cast<const float4*>(stat) + r * nparts, nparts);
      s_sim[pp] = s;
      sim[r] = s;
      if (dist) dist[r] = 1.0f - s;
    }
    __syncthreads();
    for (int k = warp; k < K; k += PS_WARPS) {
      float acc = 0.f;
      for (int pp = lane; pp < P; pp += 32) acc = fmaf(s_sim[pp], last_layer[(size_t)k * P + pp], acc);
      acc = warp_sum(acc);
      if (lane == 0) logits[(size_t)n * K + k] = acc;
    }
    __syncthreads();
  }
}

// best_vec[p,:] = feats[n*,p,:] where n* = clip of this call that holds best_key[p] (keys carry the global clip index);
// prototypes whose best clip lies outside [offset, offset+N) keep their row.  One block per prototype.
__global__ void push_capture_dense_kernel(const unsigned long long* __restrict__ best_key, int P, int D, long long offset,
                                          int N, const float* __restrict__ feats, float* __restrict__ best_vec) {
  const int p = blockIdx.x;
  const unsigned long long key = best_key[p] ^ PASN_KEY_SIGN;
  if (key == PASN_KEY_NONE) return;
  const long long idx = (long long)(key & 0xFFFFFFFFull);
  if (idx < offset || idx >= offset + N) return;
  const float* src = feats + ((size_t)(idx - offset) * P + p) * D;
  for (int d = threadIdx.x; d < D; d += blockDim.x) best_vec[(size_t)p * D + d] = src[d];
}

int launch_proto_stage(const float* feats, const float* protos, const float* last_layer, int N, int P, int D, int K,
                       float* logits, float* sim, float* dist, const pasn_push_args* push, cudaStream_t st) {
  if (N <= 0) return PASN_OK;
  const long long rows = (long long)N * P;
  const int64_t* labels = push ? push->labels : nullptr;
  const int32_t* pcls = push ? push->proto_class : nullptr;
  const long long goff = push ? (long long)push->global_offset : 0;
  unsigned long long* bkey = push ? reinterpret_cast<unsigned long long*>(push->best_key) : nullptr;
  if (D == 128 || D == 256 || D == 512 || D == 1024) {
    // warps = P * m (so a warp keeps its prototype), 8 warps per block: blocks * 8 must be a multiple of P
    long long per = P;                                   // warps per "round" of all prototypes
    long long m = (148LL * 4 * 8 + per - 1) / per;       // rounds wanted: ~4 blocks per SM, several rows per warp so that
                                                         // the prototype set-up (load, norm, NV divisions) is amortised
    if (m > N) m = N;
    if (m < 1) m = 1;
    long long warps = per * m;
    while (warps % 8 != 0) warps += per;                 // at most 7 steps; stays a multiple of P
    const unsigned blocks = (unsigned)(warps / 8);
    cudaError_t e;
    if (D == 128) e = launch_pdl(proto_rows_reg_kernel<4>, dim3(blocks), dim3(256), 0, st, feats, protos, rows, P, sim, dist, labels, pcls, goff, bkey);
    else if (D == 256) e = launch_pdl(proto_rows_reg_kernel<8>, dim3(blocks), dim3(256), 0, st, feats, protos, rows, P, sim, dist, labels, pcls, goff, bkey);
    else if (D == 512) e = launch_pdl(proto_rows_reg_kernel<16>, dim3(blocks), dim3(256), 0, st, feats, protos, rows, P, sim, dist, labels, pcls, goff, bkey);
    else e = launch_pdl(proto_rows_reg_kernel<32>, dim3(blocks), dim3(256), 0, st, feats, protos, rows, P, sim, dist, labels, pcls, goff, bkey);
    if (e != cudaSuccess) return PASN_ERR_CUDA;
  } else {
    long long blocks = (rows + PS_WARPS - 1) / PS_WARPS;
    if (blocks > 148 * 32) blocks = 148 * 32;
    proto_rows_kernel<<<(unsigned)blocks, PS_THREADS, 0, st>>>(feats, protos, rows, P, D, sim, dist, labels, pcls, goff, bkey);
  }
  PASN_LAUNCH_CHECK();
  count_launch();
  if (P >= 1024 && (long long)N * K <= 148 * 64) {
    if (launch_pdl(proto_logits_wide_kernel, dim3(N * K), dim3(PS_THREADS), 0, st, sim, last_layer, N, P, K, logits) != cudaSuccess) return PASN_ERR_CUDA;
  } else {
    if (launch_pdl(proto_logits_kernel, dim3(N < 148 * 8 ? N : 148 * 8), dim3(PS_THREADS), 0, st, sim, last_layer, N, P, K, logits) != cudaSuccess)
      return PASN_ERR_CUDA;
  }
  PASN_LAUNCH_CHECK();
  count_launch();
  if (push && push->best_vec) {   // winner capture in the same pass (push_abs_revision.py:299-302)
    push_capture_dense_kernel<<<P, 128, 0, st>>>(reinterpret_cast<const unsigned long long*>(push->best_key), P, D,
                                                 (long long)push->global_offset, N, feats, push->best_vec);
    PASN_LAUNCH_CHECK();
    count_launch();
  }
  return PASN_OK;
}

int launch_proto_from_stats(const float* stat, int nparts, const float* last_layer, int N, int P, int K, float* logits, float* sim,
                            float* dist, cudaStream_t st) {
  if (N <= 0) return PASN_OK;
  if (P <= 1024) {
    if (launch_pdl(proto_finish_stats_kernel, dim3(N < 148 * 8 ? N : 148 * 8), dim3(PS_THREADS), 0, st, stat, nparts, last_layer, N, P, K,
                   logits, sim, dist) != cudaSuccess)
      return PASN_ERR_CUDA;
    count_launch();
    return PASN_OK;
  }
  const long long rows = (long long)N * P;
  if (launch_pdl(proto_from_stats_kernel, dim3((unsigned)((rows + 255) / 256)), dim3(256), 0, st, stat, nparts, rows, sim, dist) != cudaSuccess)
    return PASN_ERR_CUDA;
  count_launch();
  if ((long long)N * K <= 148 * 64) {
    if (launch_pdl(proto_logits_wide_kernel, dim3(N * K), dim3(PS_THREADS), 0, st, sim, last_layer, N, P, K, logits) != cudaSuccess) return PASN_ERR_CUDA;
  } else {
    if (launch_pdl(proto_logits_kernel, dim3(N < 148 * 8 ? N : 148 * 8), dim3(PS_THREADS), 0, st, sim, last_layer, N, P, K, logits) != cudaSuccess)
      return PASN_ERR_CUDA;
  }
  count_launch();
  return PASN_OK;
}

// ---------------------------------------------------------------------------------------------
// push bookkeeping
// ---------------------------------------------------------------------------------------------
__global__ void push_init_kernel(unsigned long long* k, int P) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < P) k[i] = PASN_KEY_NONE ^ PASN_KEY_SIGN;   // INT64_MAX in the signed-order global format
}
// decode: index / distance of the winner per prototype
__global__ void push_decode_kernel(const unsigned long long* k, int P, int64_t* index, float* distance) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  const unsigned long long key = k[i] ^ PASN_KEY_SIGN;
  long long idx = -1;
  float d = __int_as_float(0x7f800000);
  if (key != PASN_KEY_NONE) {
    idx = (long long)(key & 0xFFFFFFFFull);
    d = f32_from_orderable((uint32_t)(key >> 32));
  }
  index[i] = idx;
  if (distance) distance[i] = d;
}
// merge of R push records [keys P x u64 | vecs P x D x f32]: per prototype (one block) the smallest signed key wins
__global__ void push_reduce_kernel(const unsigned char* __restrict__ gathered, size_t rec_bytes, int R, int P, int D,
                                   int64_t* __restrict__ index, float* __restrict__ distance, int32_t* __restrict__ valid,
                                   float* __restrict__ vec) {
  const int p = blockIdx.x;
  long long best = 0x7FFFFFFFFFFFFFFFll;
  int rb = 0;
  for (int r = 0; r < R; ++r) {
    const long long k = reinterpret_cast<const long long*>(gathered + (size_t)r * rec_bytes)[p];
    if (k < best) { best = k; rb = r; }
  }
  const unsigned long long key = (unsigned long long)best ^ PASN_KEY_SIGN;
  const bool ok = key != PASN_KEY_NONE;
  if (threadIdx.x == 0) {
    index[p] = ok ? (long long)(key & 0xFFFFFFFFull) : -1;
    if (distance) distance[p] = ok ? f32_from_orderable((uint32_t)(key >> 32)) : __int_as_float(0x7f800000);
    if (valid) valid[p] = ok ? 1 : 0;
  }
  if (ok && vec) {
    const float* src = reinterpret_cast<const float*>(gathered + (size_t)rb * rec_bytes + (size_t)P * 8) + (size_t)p * D;
    for (int d = threadIdx.x; d < D; d += blockDim.x) vec[(size_t)p * D + d] = src[d];
  }
}
// Exchange + merge of the ranks' push records in ONE kernel over NVLink peer memory (no collective call): every rank's
// record [keys P x u64 | vectors P x D x f32] lives in memory that all ranks of the node have mapped (symmetric memory).
// Block p: (block 0 first publishes this rank's record by raising its epoch flag with system scope -- the record was
// written by earlier kernels of this stream), waits until every peer's flag has reached this push's epoch, reads the R
// keys of prototype p straight from the peers, keeps the smallest (lowest distance, ties -> lowest global index; equal
// keys cannot come from different ranks because they carry the global clip index) and copies the winner's vector.
// Records are double-buffered by epoch parity on the host side, so a rank that starts its next push cannot overwrite
// a record a slower peer is still reading.  The wait is bounded (fault word), like every wait in this library.
__device__ __forceinline__ unsigned ld_acquire_sys_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys_u32(unsigned* p, unsigned v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__global__ void __launch_bounds__(128) push_merge_peers_kernel(const unsigned long long* __restrict__ rec_ptrs,
                                                               const unsigned long long* __restrict__ flag_ptrs, int R, int my_rank,
                                                               unsigned epoch, int P, int D, int64_t* __restrict__ index,
                                                               float* __restrict__ distance, int32_t* __restrict__ valid,
                                                               float* __restrict__ vec, int* fault) {
  __shared__ long long s_key[64];
  __shared__ int s_who, s_fail;
  const int p = blockIdx.x, tid = threadIdx.x;
  if (tid == 0) s_fail = 0;
  if (blockIdx.x == 0 && tid == 0) {
    __threadfence_system();
    st_release_sys_u32(reinterpret_cast<unsigned*>(flag_ptrs[my_rank]), epoch);
  }
  __syncthreads();
  if (tid < R) {
    const unsigned* f = reinterpret_cast<const unsigned*>(flag_ptrs[tid]);
    const long long t0 = clock64();
    // flags only grow; the signed difference tolerates wrap-around of the 32-bit epoch
    while ((int)(ld_acquire_sys_u32(f) - epoch) < 0) {
      if (clock64() - t0 > 8000000000ll) {
        s_fail = 1;
        if (fault != nullptr) *reinterpret_cast<volatile int*>(fault) = 801;
        break;
      }
      __nanosleep(200);
    }
    s_key[tid] = reinterpret_cast<const long long*>(rec_ptrs[tid])[p];
  }
  __syncthreads();
  if (s_fail) return;
  if (tid == 0) {
    long long best = 0x7FFFFFFFFFFFFFFFll;
    int rb = 0;
    for (int r = 0; r < R; ++r)
      if (s_key[r] < best) { best = s_key[r]; rb = r; }
    const unsigned long long key = (unsigned long long)best ^ PASN_KEY_SIGN;
    const bool ok = key != PASN_KEY_NONE;
    index[p] = ok ? (long long)(key & 0xFFFFFFFFull) : -1;
    if (distance) distance[p] = ok ? f32_from_orderable((uint32_t)(key >> 32)) : __int_as_float(0x7f800000);
    if (valid) valid[p] = ok ? 1 : 0;
    s_who = ok ? rb : -1;
  }
  __syncthreads();
  if (vec != nullptr) {
    const int rb = s_who;
    if (rb >= 0) {
      const float* src = reinterpret_cast<const float*>(rec_ptrs[rb] + (size_t)P * 8) + (size_t)p * D;
      for (int d = tid; d < D; d += blockDim.x) vec[(size_t)p * D + d] = __ldcv(src + d);
    } else {
      for (int d = tid; d < D; d += blockDim.x) vec[(size_t)p * D + d] = 0.f;
    }
  }
}

__global__ void push_write_kernel(float* protos, const float* vec, const int32_t* valid, int P, int D) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)P * D) return;
  if (valid[i / D]) protos[i] = vec[i];
}

// Winner side data (pasn_push_capture): block (p, slot, part) copies part of row p of one slot when best_key[p] names a
// clip of this call.  The slots travel by value in the kernel parameters, so the call needs no host->device copy.
struct CaptureSlots {
  pasn_capture_slot s[PASN_CAPTURE_MAX_SLOTS];
};
__global__ void __launch_bounds__(256) push_capture_kernel(const unsigned long long* __restrict__ best_key, long long offset,
                                                           int N, const CaptureSlots slots) {
  const int p = blockIdx.x;
  const unsigned long long key = best_key[p] ^ PASN_KEY_SIGN;
  if (key == PASN_KEY_NONE) return;
  const long long idx = (long long)(key & 0xFFFFFFFFull);
  if (idx < offset || idx >= offset + N) return;
  const pasn_capture_slot& sl = slots.s[blockIdx.y];
  const char* src = reinterpret_cast<const char*>(sl.src) + (idx - offset) * sl.clip_stride_bytes + (long long)p * sl.proto_stride_bytes;
  char* dst = reinterpret_cast<char*>(sl.dst) + (long long)p * sl.row_bytes;
  const long long n = sl.row_bytes;
  const long long t0 = (long long)blockIdx.z * blockDim.x + threadIdx.x, step = (long long)gridDim.z * blockDim.x;
  if ((((uintptr_t)src | (uintptr_t)dst | (uintptr_t)n) & 15) == 0) {
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    uint4* d4 = reinterpret_cast<uint4*>(dst);
    for (long long i = t0; i < n / 16; i += step) d4[i] = s4[i];
  } else {
    for (long long i = t0; i < n; i += step) dst[i] = src[i];
  }
}

}  // namespace pasn

using namespace pasn;

extern "C" int pasn_push_init(uint64_t* best_key, int32_t P, void* stream) {
  if (!best_key || P <= 0) return PASN_ERR_INVALID;
  push_init_kernel<<<ceil_div(P, 256), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<unsigned long long*>(best_key), P);
  PASN_LAUNCH_CHECK();
  count_launch();
  return PASN_OK;
}
extern "C" size_t pasn_push_record_bytes(int32_t P, int32_t D) {
  return (P > 0 && D > 0) ? (size_t)P * 8 + (size_t)P * D * 4 : 0;
}
extern "C" int pasn_push_decode(const uint64_t* best_key, int32_t P, int64_t* index, float* distance, void* stream) {
  if (!best_key || !index || P <= 0) return PASN_ERR_INVALID;
  push_decode_kernel<<<ceil_div(P, 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const unsigned long long*>(best_key), P, index, distance);
  PASN_LAUNCH_CHECK();
  count_launch();
  return PASN_OK;
}
extern "C" int pasn_push_reduce(const void* gathered, int32_t R, int32_t P, int32_t D, int64_t* index, float* distance,
                                int32_t* valid, float* vec, void* stream) {
  if (!gathered || !index || R <= 0 || P <= 0 || D <= 0) return PASN_ERR_INVALID;
  if (((uintptr_t)gathered & 7) != 0) return PASN_ERR_ALIGN;
  push_reduce_kernel<<<P, 128, 0, (cudaStream_t)stream>>>(reinterpret_cast<const unsigned char*>(gathered),
                                                          pasn_push_record_bytes(P, D), R, P, D, index, distance, valid, vec);
  PASN_LAUNCH_CHECK();
  count_launch();
  return PASN_OK;
}
extern "C" int pasn_push_merge_peers(const uint64_t* peer_records, const uint64_t* peer_flags, int32_t R, int32_t my_rank,
                                     uint32_t epoch, int32_t P, int32_t D, int64_t* index, float* distance, int32_t* valid,
                                     float* vec, void* stream) {
  if (!peer_records || !peer_flags || !index || R <= 0 || R > 64 || my_rank < 0 || my_rank >= R || P <= 0 || D <= 0)
    return PASN_ERR_INVALID;
  push_merge_peers_kernel<<<P, 128, 0, (cudaStream_t)stream>>>(reinterpret_cast<const unsigned long long*>(peer_records),
                                                                reinterpret_cast<const unsigned long long*>(peer_flags), R, my_rank,
                                                                epoch, P, D, index, distance, valid, vec, fault_word());
  PASN_LAUNCH_CHECK();
  count_launch();
  return PASN_OK;
}
extern "C" int pasn_push_write_prototypes(float* prototypes, const float* vec, const int32_t* valid, int32_t P,
                                          int32_t D, void* stream) {
  if (!prototypes || !vec || !valid || P <= 0 || D <= 0) return PASN_ERR_INVALID;
  long long n = (long long)P * D;
  push_write_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(prototypes, vec, valid, P, D);
  PASN_LAUNCH_CHECK();
  count_launch();
  return PASN_OK;
}
extern "C" int pasn_push_capture(const uint64_t* best_key, int32_t P, int64_t global_offset, int32_t N,
                                 const pasn_capture_slot* slots_host, int32_t nslots, void* stream) {
  if (!best_key || P <= 0 || N < 0 || global_offset < 0 || global_offset + N > 0xFFFFFFFFll || !slots_host || nslots <= 0 ||
      nslots > PASN_CAPTURE_MAX_SLOTS)
    return PASN_ERR_INVALID;
  CaptureSlots cs{};
  long long max_row = 0;
  for (int i = 0; i < nslots; ++i) {
    const pasn_capture_slot& s = slots_host[i];
    if (s.row_bytes < 0 || s.clip_stride_bytes < 0 || s.proto_stride_bytes < 0) return PASN_ERR_INVALID;
    if (s.row_bytes > 0 && (!s.src || !s.dst)) return PASN_ERR_INVALID;
    cs.s[i] = s;
    if (s.row_bytes > max_row) max_row = s.row_bytes;
  }
  if (N == 0 || max_row == 0) return PASN_OK;
  // a whole input clip can be megabytes: split long rows over up to 32 blocks (16 KB each) so one SM does not copy it alone
  long long parts = (max_row + 16383) / 16384;
  if (parts > 32) parts = 32;
  push_capture_kernel<<<dim3(P, nslots, (unsigned)parts), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const unsigned long long*>(best_key), (long long)global_offset, N, cs);
  PASN_LAUNCH_CHECK();
  count_launch();
  return PASN_OK;
}
