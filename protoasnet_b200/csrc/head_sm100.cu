// Fused prototype-head kernels for sm_100a (tcgen05 tensor cores, TMEM accumulators, bulk-async weight streaming).
//
// Reference computation being replaced (per clip, S = T*H*W voxels; src/models/Video_XProtoNet.py:82-98):
//     H1 = relu(W1 x + b1)            add_on_layers[0..1]     :27-39
//     F  = W2 H1 + b2                 add_on_layers[2]
//     G1 = relu(W3 x + b3); G2 = relu(W4 G1 + b4); O = |W5 G2|   occurrence_module + abs   :42-62, :106-109
//     FE[p,:] = sum_s O[p,s] F[:,s]   occurrence-weighted pooling   :87
//     cos / (.+1)/2 / logits          :90-96
//
// Algorithmic restructuring (exact in real arithmetic): pooling commutes with the last add-on conv,
//     FE[p,:] = W2 (sum_s O[p,s] H1[:,s]) + b2 * (sum_s O[p,s]),
// so W2 is applied to P pooled vectors per clip instead of S voxels (D*D*S -> D*D*P MACs per clip).
//
// K1  head_tokens2_kernel  (head_sm100_k1.cu) one persistent CTA per SM walks a contiguous range of clips in tiles of 128 voxels
//                          ("tokens" = rows of the MMA M dimension).  Per tile, all on tensor cores:
//        acc_G = X W3^T, acc_A = X W1^T     (SS MMA, X tile MN-major from NCDHW, weights streamed by cp.async.bulk)
//        G1 -> TMEM (bf16) -> acc_G2 = G1 W4^T -> G2 -> TMEM -> acc_O = G2 W5^T        (A operand from TMEM)
//        O = |acc_O| -> Os in smem: B operand of the pooling MMA, source of the occurrence-map store and of Osum
//        FEpre^T[d, (slot,p)] += H1^T O      (MN-major SS MMA; "slot" separates the <=2 clips a tile touches)
//      Hidden activations never touch HBM.  Outputs: occurrence_map, Osum [N,P] fp32 and FEpre as bf16 hi/lo
//      operand images (already in the K-major SWIZZLE_128B byte order K2 feeds to its MMAs).
// K2  proto_w2_kernel      FE = FEpre W2^T + b2 Osum on tensor cores (hi/lo split keeps ~fp32 accuracy), then the fp32
//                          cosine -> (.+1)/2 -> logits -> 1-s -> packed argmin keys chain (cf. proto_stage.cu).
#include <cstdlib>

#include "head_sm100_shared.cuh"

namespace pasn {
using namespace sm100;

using namespace k1;

// =================================================================================================
// K2: FE = FEpre W2^T + b2 Osum (tensor cores), cosine / similarity / logits / distance / push keys (fp32)
//     warps 0..7 epilogue (row = TMEM lane, two column halves), warp 8 MMA issuer, warp 9 bulk-copy loader
// =================================================================================================
namespace {
constexpr int K2_THREADS = 320;
constexpr uint32_t K2_STAGE = 65536;                 // A_hi chunk 16 KB | A_lo chunk 16 KB | W2 chunk 32 KB
constexpr uint32_t K2_SM_V = 2 * K2_STAGE;           // prototypes fp32 [P][257]
constexpr uint32_t K2_V_BYTES = PP_MAX * 257 * 4;    // 49344
constexpr uint32_t K2_SM_MISC = K2_SM_V + 49408;     // 180480
constexpr uint32_t K2_SMEM = K2_SM_MISC + 8192;

struct K2Params {
  const uint8_t* feimg; const float* osum; const uint8_t* packed; size_t off_w2, off_b2;
  const float* protos; const float* last_layer;
  float* logits; float* sim; float* dist; float* feats;
  const int64_t* labels; const int32_t* proto_class; long long global_offset; unsigned long long* best_key;
  float* stash;   // push capture: [gridDim][P][256] fp32, FE row of this CTA's best clip per prototype (or null)
  int N, P, PP, K, cpt, ntiles;   // PP = padded P (row stride inside a tile), cpt = clips per tile = 128 / PP
  int* err;
  int* fault;         // host-mapped sticky fault word (or null)
  long long* trace;   // optional: K2 stamps of CTA 0 at trace[768 ...] (see tools/trace_k2.py)
};
__device__ __forceinline__ long long gtimer_ns() {
  long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
}  // namespace
#define K2_TRACE(slot) do { if (p.trace != nullptr && blockIdx.x == 0 && (slot) < 184) p.trace[768 + 16 + (slot)] = gtimer_ns(); } while (0)

__global__ void __launch_bounds__(K2_THREADS, 1) proto_w2_kernel(const K2Params p) {
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + K2_SM_MISC);   // full[0..1] empty[2..3] accfull[4..5] accempty[6..7]
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(smem + K2_SM_MISC + 64);
  volatile int* abort_s = reinterpret_cast<volatile int*>(smem + K2_SM_MISC + 72);
  float* s_vn = reinterpret_cast<float*>(smem + K2_SM_MISC + 128);             // [64] clamped prototype norms
  float* s_b2 = reinterpret_cast<float*>(smem + K2_SM_MISC + 512);             // [256]
  float* s_part = reinterpret_cast<float*>(smem + K2_SM_MISC + 1536);          // [2][128][2] (dot, ff) of column half 1
  float* s_sim = reinterpret_cast<float*>(smem + K2_SM_MISC + 3584);           // [2][128]
  unsigned long long* s_key = reinterpret_cast<unsigned long long*>(smem + K2_SM_MISC + 4608);  // [64]
  uint64_t* tbars = reinterpret_cast<uint64_t*>(smem + K2_SM_MISC + 5632);     // [4] tile-info slots published by the loader
  volatile int* s_tile = reinterpret_cast<volatile int*>(smem + K2_SM_MISC + 5696);   // [4] tile index or -1 (no more tiles)
  int* s_win = reinterpret_cast<int*>(smem + K2_SM_MISC + 5120);               // [128] push capture: row holds its prototype's best key
  float* s_v = reinterpret_cast<float*>(smem + K2_SM_V);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  Ctx ctx{p.err, abort_s, p.fault};
  if ((smem_u32(smem) & 1023u) != 0) {
    if (tid == 0) atomicCAS(p.err, 0, 901);
    return;
  }
  if (tid == 0) K2_TRACE(0);
  if (tid == 0) {
    *abort_s = 0;
    mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_init(&bars[2], 1); mbar_init(&bars[3], 1);
    mbar_init(&bars[4], 1); mbar_init(&bars[5], 1); mbar_init(&bars[6], 8); mbar_init(&bars[7], 8);
    for (int i = 0; i < 4; ++i) mbar_init(&tbars[i], 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(tmem_ptr_s, 512);
  for (int i = tid; i < DD; i += K2_THREADS) s_b2[i] = reinterpret_cast<const float*>(p.packed + p.off_b2)[i];
  // push capture: rows only matter if they beat the running global best, so the CTA-local minimum starts there (the
  // value read is never below the final minimum; a later read by another CTA would only be a tighter filter)
  if (tid < p.P) s_key[tid] = p.stash ? (p.best_key[tid] ^ PASN_KEY_SIGN) : PASN_KEY_NONE;
  {  // prototypes -> smem rows of 257 floats (conflict-free row-per-lane reads); 128-bit loads, several in flight
    const float4* src = reinterpret_cast<const float4*>(p.protos);
    const int n4 = p.P * (DD / 4);
#pragma unroll 4
    for (int i = tid; i < n4; i += K2_THREADS) {
      const float4 v = __ldg(src + i);
      float* dst = s_v + ((i * 4) >> 8) * 257 + ((i * 4) & 255);
      dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
    }
  }
  __syncthreads();
  for (int pp = warp; pp < p.P; pp += K2_THREADS / 32) {
    float vv = 0.f;
    for (int d = lane; d < DD; d += 32) { const float b = s_v[pp * 257 + d]; vv = fmaf(b, b, vv); }
    vv = warp_sum(vv);
    if (lane == 0) s_vn[pp] = fmaxf(sqrtf(vv), 1e-8f);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = *tmem_ptr_s;
  const uint32_t st_base = smem_u32(smem);
  // Tiles are dealt round-robin once the whole token kernel has completed.  The loader publishes each tile index (or -1)
  // in a 4-slot ring guarded by mbarriers; MMA issuer and epilogue follow.
  if (tid == 0) K2_TRACE(1);   // prologue done

  if (warp == 9) {
    // ---------------------------------------------------------------- loader
    if (lane == 0) {
      griddep_wait();   // the pooled-vector images are written by the token kernel
      K2_TRACE(2);
      const uint64_t pol_first = l2_policy_evict_first();
      uint32_t u = 0;
      bool ok = true;
      for (int it = 0; ok; ++it) {
        int tile = (int)blockIdx.x + it * (int)gridDim.x;
        if (tile >= p.ntiles) tile = -1;
        s_tile[it & 3] = tile;
        mbar_arrive(&tbars[it & 3]);
        if (tile < 0) break;
        const uint8_t* a_src = p.feimg + (size_t)tile * FE_TILE_BYTES;
        K2_TRACE(16 + it * 8 + 7);
        if (p.trace != nullptr && blockIdx.x == 0 && it < 32) p.trace[768 + 200 + it] = tile;
        for (int kc = 0; kc < 4; ++kc, ++u) {
          const uint32_t s = u & 1, ph = (u >> 1) & 1;
          if (!(ok = bwait(&bars[2 + s], ph ^ 1, ctx, 611))) break;
          const uint32_t dst = st_base + s * K2_STAGE;
          mbar_arrive_expect_tx(&bars[s], K2_STAGE);
          // the images were stored evict_last by the token kernel; read them once, then let them go
          bulk_g2s_hint(dst, a_src + (size_t)kc * 16384, 16384, &bars[s], pol_first);
          bulk_g2s_hint(dst + 16384, a_src + 65536 + (size_t)kc * 16384, 16384, &bars[s], pol_first);
          bulk_g2s(dst + 32768, p.packed + p.off_w2 + (size_t)kc * 32768, 16384, &bars[s]);
          bulk_g2s(dst + 49152, p.packed + p.off_w2 + (size_t)kc * 32768 + 16384, 16384, &bars[s]);
        }
      }
    }
  } else if (warp == 8) {
    // ---------------------------------------------------------------- MMA issuer (one elected thread, lean issue path:
    // see head_sm100_k1.cu -- descriptors as 32-bit halves in a single-thread region keep the UTCHMMAs back to back)
    if (elect_one()) {
      // A (pooled vectors): K-major rows (k = d contiguous), B (W2) K-major
      const uint32_t idesc = make_idesc_bf16(128, 256, 0, 0);
      constexpr uint32_t a_lbo = 16u, a_kstep = 2u;
      constexpr uint32_t HI = desc_hi(1024, SWZ_128B);
      const uint32_t bar0 = smem_u32(bars);
      uint32_t u = 0;
      bool ok = true;
      for (int it = 0; ok; ++it) {
        if (!(ok = bwait(&tbars[it & 3], (it >> 2) & 1, ctx, 623))) break;
        if (s_tile[it & 3] < 0) break;
        const uint32_t buf = it & 1;
        if (!(ok = bwait(&bars[6 + buf], ((it >> 1) & 1) ^ 1, ctx, 621))) break;
        tc_fence_after();
        for (int kc = 0; kc < 4 && ok; ++kc, ++u) {
          const uint32_t s = u & 1, ph = (u >> 1) & 1;
          if (!(ok = bwait(&bars[s], ph, ctx, 622))) break;
          K2_TRACE(16 + it * 8 + kc);
          const uint32_t sb = st_base + s * K2_STAGE;
          const uint32_t ah = desc_lo(sb, a_lbo), al = desc_lo(sb + 16384, a_lbo), bd = desc_lo(sb + 32768, 16);
          const uint32_t d = tbase + 256u * buf;
          mma_ss_x(d, ah, HI, bd, HI, idesc, kc ? 1u : 0u);
          mma_ss_x(d, al, HI, bd, HI, idesc, 1u);
#pragma unroll
          for (int k4 = 1; k4 < 4; ++k4) {
            mma_ss_x(d, ah + k4 * a_kstep, HI, bd + k4 * 2, HI, idesc, 1u);
            mma_ss_x(d, al + k4 * a_kstep, HI, bd + k4 * 2, HI, idesc, 1u);
          }
          mma_commit_a(bar0 + 8u * (2 + s));
        }
        if (ok) mma_commit(&bars[4 + buf]);
        K2_TRACE(16 + it * 8 + 4);
      }
    }
  } else {
    // ---------------------------------------------------------------- epilogue: row r = 32q + lane, columns [128ch, +128)
    const int q = warp & 3, ch = warp >> 2;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    const int r = q * 32 + lane;
    griddep_wait();   // Osum is written by the token kernel
    bool ok = true;
    for (int it = 0; ok; ++it) {
      if (!(ok = bwait(&tbars[it & 3], (it >> 2) & 1, ctx, 632))) break;
      const int tile = s_tile[it & 3];
      if (tile < 0) break;
      const uint32_t buf = it & 1;
      const int clip0 = tile * p.cpt;
      int nclip = p.N - clip0;
      if (nclip > p.cpt) nclip = p.cpt;
      const int cl_r = r / p.PP, pp_r = r - cl_r * p.PP;          // row = clip-in-tile * PP + prototype
      const bool rvalid = cl_r < nclip && pp_r < p.P;
      const int cl = rvalid ? cl_r : 0, pp = rvalid ? pp_r : 0;
      const int n = clip0 + cl;
      const float* vrow = s_v + pp * 257 + 128 * ch;
      const float* b2 = s_b2 + 128 * ch;
      float* frow = (p.feats && rvalid) ? p.feats + ((size_t)n * p.P + pp) * DD + 128 * ch : nullptr;
      if (!(ok = bwait(&bars[4 + buf], (it >> 1) & 1, ctx, 631))) break;
      tc_fence_after();
      if (tid == 0) K2_TRACE(16 + it * 8 + 5);
      const float os = rvalid ? p.osum[(size_t)n * p.P + pp] : 0.f;
      const uint32_t ta = tbase + lane_base + 256u * buf + 128u * ch;
      float ff = 0.f, dot = 0.f;
      uint32_t ra[32], rb[32];
      tmem_ld_x32(ta, ra);
      tmem_ld_wait();
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t* cur = (c & 1) ? rb : ra;
        uint32_t* nxt = (c & 1) ? ra : rb;
        if (c < 3) tmem_ld_x32(ta + 32 * (c + 1), *reinterpret_cast<uint32_t(*)[32]>(nxt));
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          float f[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            f[j] = fmaf(b2[32 * c + 4 * j4 + j], os, __uint_as_float(cur[4 * j4 + j]));
            ff = fmaf(f[j], f[j], ff);
            dot = fmaf(f[j], vrow[32 * c + 4 * j4 + j], dot);
          }
          if (frow) *reinterpret_cast<float4*>(frow + 32 * c + 4 * j4) = make_float4(f[0], f[1], f[2], f[3]);
        }
        if (c < 3) tmem_ld_wait();
      }
      const bool cap = p.stash != nullptr;
      if (!cap) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars[6 + buf]);   // accumulator buffer may be overwritten by tile it+2
      }
      unsigned long long mykey = PASN_KEY_NONE;
      float* part = s_part + buf * 256;
      float* ssim = s_sim + buf * 128;
      if (ch == 1) { part[2 * r] = dot; part[2 * r + 1] = ff; }
      named_bar_sync(1, 256);
      if (ch == 0) {
        dot += part[2 * r];
        ff += part[2 * r + 1];
        const float nf = fmaxf(sqrtf(ff), 1e-8f);
        const float cosv = dot / (nf * s_vn[pp]);
        const float s = (cosv + 1.0f) / 2.0f;
        const float dd = 1.0f - s;
        ssim[r] = rvalid ? s : 0.f;
        if (rvalid) {
          p.sim[(size_t)n * p.P + pp] = s;
          if (p.dist) p.dist[(size_t)n * p.P + pp] = dd;
          if (p.best_key) {
            const int pc = p.proto_class[pp];
            if (pc < 0 || (long long)pc == p.labels[n]) {
              mykey = pack_key(dd, (uint32_t)(p.global_offset + n));
              atomicMin(&s_key[pp], mykey);
            }
          }
        }
      }
      named_bar_sync(1, 256);
      if (tid < nclip * p.K) {
        const int c2 = tid / p.K, k = tid - c2 * p.K;
        float acc = 0.f;
        for (int qq = 0; qq < p.P; ++qq) acc = fmaf(ssim[c2 * p.PP + qq], p.last_layer[(size_t)k * p.P + qq], acc);
        p.logits[(size_t)(clip0 + c2) * p.K + k] = acc;
      }
      if (cap) {
        // Winner capture in the same pass (src/utils/push_abs_revision.py:299-302 stashes protoL_input[a, j] of the batch
        // that produced the minimum): a row that now holds its prototype's CTA-wide best key re-reads its accumulator
        // row and leaves features_extracted in this CTA's stash slot; push_capture_stash_kernel keeps the slot of the
        // CTA that owns the final key.  Keys are unique (they carry the clip index), rows of one tile are ordered by the
        // barriers, tiles by program order.
        if (ch == 0) s_win[r] = (mykey != PASN_KEY_NONE && s_key[pp] == mykey) ? 1 : 0;
        named_bar_sync(1, 256);
        const int win = s_win[r];
        if (__any_sync(0xffffffffu, win != 0)) {
          float* srow = p.stash + ((size_t)blockIdx.x * p.P + pp) * DD + 128 * ch;
#pragma unroll 1
          for (int c = 0; c < 4; ++c) {
            tmem_ld_x32(ta + 32 * c, ra);
            tmem_ld_wait();
            if (win) {
#pragma unroll
              for (int j4 = 0; j4 < 8; ++j4) {
                float f[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) f[j] = fmaf(b2[32 * c + 4 * j4 + j], os, __uint_as_float(ra[4 * j4 + j]));
                *reinterpret_cast<float4*>(srow + 32 * c + 4 * j4) = make_float4(f[0], f[1], f[2], f[3]);
              }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars[6 + buf]);
      }
      if (tid == 0) K2_TRACE(16 + it * 8 + 6);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (tid == 0) K2_TRACE(3);
  if (p.best_key && tid < p.P && s_key[tid] != PASN_KEY_NONE) key_atomic_min_global(&p.best_key[tid], s_key[tid]);
  if (warp == 0) tmem_dealloc(tbase, 512);
}

// =================================================================================================
// weight packing: fp32 state_dict tensors -> bf16 stage images in the exact smem byte order (f16: the layer-1 images W3 / W1
// in fp16, the operand type of an fp16 feature map)
// =================================================================================================
__global__ void pack_weights_kernel(pasn_weights w, int C, int P, int f16, uint8_t* out) {
  const PackedLayout PL = packed_layout(C);
  const int nkc = C / 64;
  const size_t n_l1 = (size_t)2 * nkc * 256 * 64, n_w4 = (size_t)4 * 128 * 64, n_w5 = (size_t)2 * 64 * 64;
  const size_t n_w2 = (size_t)4 * 256 * 64, n_bias = DD + DD + DH, n_b2 = DD;
  const size_t total = n_l1 + n_w4 + n_w5 + n_w2 + n_bias + n_b2;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    size_t j = i;
    if (j < n_l1) {  // stage = 2*kc + pass; pass 0: occ_w1 (W3), pass 1: addon_w1 (W1); image [256 rows][64 k]
      const int stage = (int)(j / (256 * 64)), e = (int)(j % (256 * 64));
      const int r = e / 64, k = e % 64, kc = stage >> 1, pass = stage & 1;
      const float v = (pass ? w.addon_w1 : w.occ_w1)[(size_t)r * C + kc * 64 + k];
      uint8_t* dst = out + PL.off_l1 + (size_t)stage * 32768 + off_kmajor_sw128(r, k);
      if (f16) *reinterpret_cast<__half*>(dst) = __float2half_rn(v);
      else *reinterpret_cast<__nv_bfloat16*>(dst) = __float2bfloat16_rn(v);
      continue;
    }
    j -= n_l1;
    if (j < n_w4) {  // occ_w2 [128][256]: 4 k-chunk images [128 rows][64 k]
      const int kc = (int)(j / (128 * 64)), e = (int)(j % (128 * 64)), r = e / 64, k = e % 64;
      *reinterpret_cast<__nv_bfloat16*>(out + PL.off_w4 + (size_t)kc * 16384 + off_kmajor_sw128(r, k)) =
          __float2bfloat16_rn(w.occ_w2[(size_t)r * DD + kc * 64 + k]);
      continue;
    }
    j -= n_w4;
    if (j < n_w5) {  // occ_w3 [P][128] zero-padded to 64 rows: 2 k-chunk images [64 rows][64 k]
      const int kc = (int)(j / (64 * 64)), e = (int)(j % (64 * 64)), r = e / 64, k = e % 64;
      const float v = r < P ? w.occ_w3[(size_t)r * DH + kc * 64 + k] : 0.f;
      *reinterpret_cast<__nv_bfloat16*>(out + PL.off_w5 + (size_t)kc * 8192 + off_kmajor_sw128(r, k)) = __float2bfloat16_rn(v);
      continue;
    }
    j -= n_w5;
    if (j < n_w2) {  // addon_w2 [256][256]: 4 k-chunk images [256 rows][64 k]
      const int kc = (int)(j / (256 * 64)), e = (int)(j % (256 * 64)), r = e / 64, k = e % 64;
      *reinterpret_cast<__nv_bfloat16*>(out + PL.off_w2 + (size_t)kc * 32768 + off_kmajor_sw128(r, k)) =
          __float2bfloat16_rn(w.addon_w2[(size_t)r * DD + kc * 64 + k]);
      continue;
    }
    j -= n_w2;
    if (j < n_bias) {  // b3 | b1 | b4, bf16-rounded values kept as fp32
      float v;
      if (j < DD) v = w.occ_b1[j];
      else if (j < 2 * DD) v = w.addon_b1[j - DD];
      else v = w.occ_b2[j - 2 * DD];
      reinterpret_cast<float*>(out + PL.off_bias)[j] = round_bf16(v);
      continue;
    }
    j -= n_bias;
    reinterpret_cast<float*>(out + PL.off_b2)[j] = round_bf16(w.addon_b2[j]);
  }
}

// =================================================================================================
// push capture: best_vec[p,:] = stash slot of the K2 CTA that processed the clip holding best_key[p], if that clip belongs
// to this call (keys carry the global clip index; K2 deals its tiles round-robin).  One block per prototype.
// =================================================================================================
__global__ void push_capture_stash_kernel(const unsigned long long* __restrict__ best_key, int P, long long offset, int N,
                                          int cpt, int grid2, const float* __restrict__ stash, float* __restrict__ best_vec) {
  const int pp = blockIdx.x;
  const unsigned long long key = best_key[pp] ^ PASN_KEY_SIGN;
  if (key == PASN_KEY_NONE) return;
  const long long idx = (long long)(key & 0xFFFFFFFFull);
  if (idx < offset || idx >= offset + N) return;
  const int tile = (int)((idx - offset) / cpt);
  const int cta = tile % grid2;
  const float* src = stash + ((size_t)cta * P + pp) * DD;
  for (int d = threadIdx.x; d < DD; d += blockDim.x) best_vec[(size_t)pp * DD + d] = src[d];
}

// =================================================================================================
// host side
// =================================================================================================
static long long* g_trace = nullptr;
void sm100_set_trace(void* dev_buf) { g_trace = reinterpret_cast<long long*>(dev_buf); }

bool sm100_supported(const pasn_dims& d) {
  // fp32 feature maps take the fused path only on explicit request (bf16 compute: inputs are rounded on the fly)
  // channels_last ([N,S,C]) feature maps: bf16 and fp16 only
  const bool half = d.dtype == PASN_BF16 || d.dtype == PASN_F16;
  if (d.layout != PASN_LAYOUT_NCS && !(d.layout == PASN_LAYOUT_NSC && half)) return false;
  if (!half && !(d.dtype == PASN_F32 && d.path == PASN_PATH_TCGEN05)) return false;
  if (d.D != DD) return false;
  if (d.C % 64 != 0 || d.C < 64 || d.C > 1024) return false;
  if (d.P < 1 || d.P > PP_MAX) return false;
  if (d.S % 4 != 0 || d.S < TILE_M) return false;   // a 128-voxel tile may touch at most two clips
  return true;
}

size_t sm100_packed_bytes(const pasn_dims& d) { return packed_layout(d.C).total; }

static inline int k2_ppad(const pasn_dims& d) {
  const int p8 = (d.P + 7) / 8 * 8;
  return p8 <= 16 ? 16 : p8 <= 32 ? 32 : p8 <= 40 ? 40 : 48;   // matches the head_tokens_kernel<PP> instantiations
}
// Small batches: one persistent CTA per clip range leaves most SMs idle when N < 148.  Pooling is linear in the voxels,
// so a clip of S voxels can be processed as G independent "virtual clips" of S/G voxels (each at least one 128-voxel
// tile, multiple of 4) whose pooled features are summed after K2.  G = 1 means no split.
static inline int split_groups(const pasn_dims& d) {
  if (d.N <= 0 || d.N > 74) return 1;
  int best = 1;
  for (int g = 2; g <= d.S / TILE_M; ++g) {
    if (d.S % g != 0) continue;
    const int sv = d.S / g;
    if (sv < TILE_M || sv % 4 != 0) continue;
    if ((long long)d.N * g > 148) break;         // one virtual clip range per SM is enough; beyond that the extra
                                                  // kernels of the split cost more than the parallelism gains
    best = g;
  }
  return best;
}
constexpr int K2_MAX_GRID = 160;   // upper bound of K2's grid (one CTA per SM)
struct WsLayout {
  int G, Nv, Sv, tiles2;
  size_t off_osum, off_err, off_stash, off_featsv, off_fe, off_simv, off_logv, total;
};
static inline WsLayout ws_layout(const pasn_dims& d) {
  WsLayout L;
  L.G = split_groups(d);
  L.Nv = d.N * L.G;
  L.Sv = d.S / L.G;
  L.tiles2 = ceil_div(L.Nv, TILE_M / k2_ppad(d));
  size_t o = (size_t)L.tiles2 * FE_TILE_BYTES;
  L.off_osum = o; o += align_up((size_t)L.Nv * d.P * 4, 256);
  L.off_err = o; o += 256;
  L.off_stash = o; o += align_up((size_t)K2_MAX_GRID * d.P * DD * 4, 256);   // push capture: FE row of each K2 CTA's best clip per prototype
  L.off_featsv = L.off_fe = L.off_simv = L.off_logv = o;
  if (L.G > 1) {
    L.off_featsv = o; o += align_up((size_t)L.Nv * d.P * DD * 4, 256);   // K2's features per virtual clip
    L.off_fe = o; o += align_up((size_t)d.N * d.P * DD * 4, 256);        // their sum per real clip
    L.off_simv = o; o += align_up((size_t)L.Nv * d.P * 4, 256);          // K2's per-virtual-clip similarity / logits: unused
    L.off_logv = o; o += align_up((size_t)L.Nv * d.K * 4, 256);
  }
  L.total = o;
  return L;
}

// workspace: K2 operand images [tiles2][128 KB] | Osum [Nv][P] fp32 | err int | capture stash | (split only) scratch, see ws_layout
size_t sm100_workspace_bytes(const pasn_dims& d) { return ws_layout(d).total; }

// FE[n][i] = sum_g FEv[n*G + g][i]   (i over P*D)
__global__ void sum_groups_kernel(const float* __restrict__ fev, float* __restrict__ fe, int N, int G, int PD) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)N * PD) return;
  const long long n = i / PD, r = i - n * PD;
  float a = 0.f;
  for (int g = 0; g < G; ++g) a += fev[((size_t)n * G + g) * PD + r];
  fe[i] = a;
}

int sm100_pack_weights(const pasn_weights& w, const pasn_dims& d, void* packed, cudaStream_t st) {
  if (((uintptr_t)packed & 15) != 0) return PASN_ERR_ALIGN;
  pack_weights_kernel<<<148 * 4, 256, 0, st>>>(w, d.C, d.P, d.dtype == PASN_F16 ? 1 : 0, reinterpret_cast<uint8_t*>(packed));
  PASN_LAUNCH_CHECK();
  count_launch();
  return PASN_OK;
}

int sm100_head_forward(const void* feat, const pasn_weights& w, const void* packed, const pasn_dims& d, float* logits,
                       float* sim, void* occ, float* feats, float* dist, const pasn_push_args* push, void* ws,
                       size_t ws_bytes, cudaStream_t st) {
  if (!sm100_supported(d)) return PASN_ERR_UNSUPPORTED;
  if (ws_bytes < sm100_workspace_bytes(d)) return PASN_ERR_WORKSPACE;
  if (((uintptr_t)feat & 15) != 0 || ((uintptr_t)packed & 15) != 0 || ((uintptr_t)ws & 15) != 0) return PASN_ERR_ALIGN;
  static bool attr_done = false;
  if (!attr_done) {
    if (cudaFuncSetAttribute(proto_w2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K2_SMEM) != cudaSuccess)
      return PASN_ERR_CUDA;
    attr_done = true;
  }
  const WsLayout L = ws_layout(d);
  char* wsp = reinterpret_cast<char*>(ws);
  uint8_t* feimg = reinterpret_cast<uint8_t*>(wsp);
  float* osum = reinterpret_cast<float*>(wsp + L.off_osum);
  int* err = reinterpret_cast<int*>(wsp + L.off_err);

  static const int num_sms = [] {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    return n > K2_MAX_GRID ? K2_MAX_GRID : n;
  }();
  K1Params k1{};
  k1.f32_in = d.dtype == PASN_F32;
  k1.f16_in = d.dtype == PASN_F16;
  k1.nsc = d.layout == PASN_LAYOUT_NSC;
  k1.feat = reinterpret_cast<const __nv_bfloat16*>(feat);
  k1.feat32 = reinterpret_cast<const float*>(feat);
  k1.packed = reinterpret_cast<const uint8_t*>(packed);
  k1.occ = k1.f32_in ? nullptr : reinterpret_cast<__nv_bfloat16*>(occ);
  k1.occ32 = k1.f32_in ? reinterpret_cast<float*>(occ) : nullptr;
  k1.feimg = feimg; k1.osum = osum;
  k1.N = L.Nv; k1.C = d.C; k1.P = d.P; k1.S = L.Sv; k1.nkc = d.C / 64;
  k1.G = L.G; k1.SR = d.S;
  k1.clips_per_cta = ceil_div(L.Nv, num_sms);
  k1.cpt = TILE_M / k2_ppad(d);
  k1.err = err;
  k1.fault = fault_word();
  k1.trace = g_trace;
  // The workspace's error word (what pasn_debug_sm100_error reads; faults themselves go to the sticky fault word) is only
  // cleared when somebody will look at it: a memset in front of every call is ~2 us of the step.
  static const int dbg_sync = [] { const char* e = getenv("PASN_DEBUG_SYNC"); return e ? atoi(e) : 0; }();
  if (dbg_sync && cudaMemsetAsync(err, 0, sizeof(int), st) != cudaSuccess) return PASN_ERR_CUDA;
  const int grid1 = ceil_div(L.Nv, k1.clips_per_cta);
  const int ppad = (d.P + 7) / 8 * 8;
  main_kernel_begin(st);
  const int rc = launch_k1(k1, ppad, grid1, st);
  if (rc) return rc;
  main_kernel_end(st);
  count_launch();
  if (logits == nullptr) return PASN_OK;   // occurrence map only (sm100_occurrence_only): the prototype kernel is not needed

  const PackedLayout PL = packed_layout(d.C);
  K2Params k2{};
  k2.feimg = feimg; k2.osum = osum; k2.packed = k1.packed; k2.off_w2 = PL.off_w2; k2.off_b2 = PL.off_b2;
  k2.protos = w.prototypes; k2.last_layer = w.last_layer;
  const bool split = L.G > 1;
  float* featsv = reinterpret_cast<float*>(wsp + L.off_featsv);
  k2.logits = split ? reinterpret_cast<float*>(wsp + L.off_logv) : logits;
  k2.sim = split ? reinterpret_cast<float*>(wsp + L.off_simv) : sim;
  k2.dist = split ? nullptr : dist;
  k2.feats = split ? featsv : feats;
  k2.labels = (push && !split) ? push->labels : nullptr;
  k2.proto_class = (push && !split) ? push->proto_class : nullptr;
  k2.global_offset = (push && !split) ? (long long)push->global_offset : 0;
  k2.best_key = (push && !split) ? reinterpret_cast<unsigned long long*>(push->best_key) : nullptr;
  k2.stash = (push && !split && push->best_vec) ? reinterpret_cast<float*>(wsp + L.off_stash) : nullptr;
  k2.N = L.Nv; k2.P = d.P; k2.K = d.K;
  k2.cpt = TILE_M / k2_ppad(d);
  k2.PP = k2_ppad(d);
  k2.ntiles = L.tiles2;
  k2.err = err;
  k2.fault = k1.fault;
  k2.trace = g_trace;
  const int grid2 = k2.ntiles < num_sms ? k2.ntiles : num_sms;   // <= K2_MAX_GRID
  {  // programmatic dependent launch: K2's prologue (TMEM, barriers, norms, the resident W2 images) overlaps K1's tail
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid2); cfg.blockDim = dim3(K2_THREADS); cfg.dynamicSmemBytes = K2_SMEM; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    if (cudaLaunchKernelEx(&cfg, proto_w2_kernel, k2) != cudaSuccess) return PASN_ERR_CUDA;
  }
  PASN_LAUNCH_CHECK();
  count_launch();
  if (k2.stash) {
    push_capture_stash_kernel<<<d.P, 128, 0, st>>>(k2.best_key, d.P, k2.global_offset, L.Nv, k2.cpt, grid2, k2.stash, push->best_vec);
    PASN_LAUNCH_CHECK();
    count_launch();
  }
  if (split) {   // sum the pooled features of the voxel groups, then the fp32 cosine / logits / push stage on real clips
    float* fe = feats ? feats : reinterpret_cast<float*>(wsp + L.off_fe);
    const long long tot = (long long)d.N * d.P * DD;
    sum_groups_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(featsv, fe, d.N, L.G, d.P * DD);
    PASN_LAUNCH_CHECK();
    count_launch();
    const int rc2 = launch_proto_stage(fe, w.prototypes, w.last_layer, d.N, d.P, DD, d.K, logits, sim, dist, push, st);
    if (rc2) return rc2;
  }
  return PASN_OK;
}

// compute_occurence_map (src/models/Video_XProtoNet.py:100-109) for the shapes the fused path takes: the token kernel alone
// (it writes the map on its way; the pooled vectors it also produces stay in the workspace).
int sm100_occurrence_only(const void* feat, const pasn_weights& w, const void* packed, const pasn_dims& d, void* occ, void* ws,
                          size_t ws_bytes, cudaStream_t st) {
  return sm100_head_forward(feat, w, packed, d, nullptr, nullptr, occ, nullptr, nullptr, nullptr, ws, ws_bytes, st);
}

// surfaced for tests / debugging: non-zero if a kernel hit its bounded-wait limit (protocol bug) on the last call
int sm100_last_error(const void* ws, const pasn_dims& d, cudaStream_t st) {
  const char* wsp = reinterpret_cast<const char*>(ws);
  const int* err = reinterpret_cast<const int*>(wsp + ws_layout(d).off_err);
  int h = 0;
  if (cudaMemcpyAsync(&h, err, 4, cudaMemcpyDeviceToHost, st) != cudaSuccess) return -1;
  if (cudaStreamSynchronize(st) != cudaSuccess) return -1;
  return h;
}

}  // namespace pasn
