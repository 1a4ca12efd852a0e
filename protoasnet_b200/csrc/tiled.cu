// "Tiled" tensor-core path of the prototype head: the head as a chain of tcgen05 GEMMs (tc_gemm.cu) over token-major
// activations, for the shapes the fused token kernel (head_sm100*.cu) does not take -- D != 256, feature maps with fewer
// than 128 voxels (image head, BASELINE config 2), thousands of prototypes (config 5: the O layer and the pooling
// contraction are then the dominant GEMMs) -- and for fp32 feature maps, where every product runs as a three-pass bf16
// hi/lo split (x*w ~ xh*wh + xh*wl + xl*wh, fp32 accumulation), i.e. fp32-grade results on the tensor cores.
//
// Reference computation (src/models/Video_XProtoNet.py:82-98, src/models/XProtoNet.py:51-67), per clip with S voxels:
//   [H1 | G1] = relu([W1; W3] x + [b1; b3])          one GEMM over all tokens        (add_on_layers[0], occurrence_module[0])
//   G2 = relu(W4 G1 + b4)                                                              (occurrence_module[2])
//   O  = |W5 G2|            per clip, written straight in the [N,P,S] layout of occurrence_map   (occurrence_module[4], abs)
//   pooled[p,:] = sum_s O[p,s] H1[:,s]     per clip, K = S; H1 (token-major) is the MN-major B operand
//   FE = pooled W2^T + (sum_s O[p,s]) b2     W2 applied after pooling (exact in real arithmetic, see DESIGN.md 2.1)
//   ... when that is the cheaper order (P rows per clip, times the hi/lo passes of the pooled vectors, against S voxels);
//   otherwise (image head: S = 49, config 5: P = 4096 > S) the reference's order is kept:
//   F = W2 H1 + b2 over all tokens, FE[p,:] = sum_s O[p,s] F[:,s] straight out of the pooling GEMM in fp32.
//   cosine / (.+1)/2 / logits / 1-s / push keys: proto_stage.cu (fp32)
// Hidden activations are bf16 in HBM between the GEMMs (hi|lo planes in fp32 mode).
#include <cstdlib>
#include <type_traits>

#include "tc_gemm.cuh"

namespace pasn {

namespace {

struct Plan {
  int ex;        // bf16 planes per activation / weight: 1 (bf16 mode), 2 (fp32 mode: hi | lo)
  int C, D, D2, P, K, S, Sp;   // Sp: column pitch of one plane of the pooling A operand (occurrence values)
  bool occ_direct;             // bf16 mode and 16-byte aligned rows: the pooling reads the occurrence_map buffer itself
                               // (fp16 mode: the map is fp16, the pooling reads a bf16 copy of it, see DESIGN.md 2.7)
  bool w2_first;               // F = W2 H1 + b2 before the pooling (cheaper when S is small against P)
  bool tok_c;                  // few prototypes: O over all tokens at once (token-major), the map leaves channel-major per clip
  int Pp;                      // column pitch of one plane of the token-major occurrence values
  int bn_c, tiles_n_c;         // tile width / count along S of the O GEMM (psum parts = 2 * tiles_n_c)
  int nb;                      // clips per chunk
  size_t off_xt, off_y, off_g2, off_occ, off_psum, off_pool, off_f, off_fe, off_stat, total;
  int stat_parts;              // column half-tiles of the GEMM that produces features_extracted (row statistics per part)
};

inline int pick_bn(int n) { return n <= 64 ? 64 : (n <= 128 ? 128 : 256); }

Plan make_plan(const pasn_dims& d) {
  Plan p{};
  p.ex = d.dtype == PASN_F32 ? 2 : 1;
  p.C = d.C; p.D = d.D; p.D2 = d.D / 2; p.P = d.P; p.K = d.K; p.S = d.S;
  p.occ_direct = d.dtype == PASN_BF16 && (d.S * 2) % 16 == 0;
  // MACs of the W2 stage per clip: S*D*D*passes before the pooling, P*D*D*passes after it (bf16 mode: the pooled vectors
  // go in as hi + lo planes, two passes; fp32 mode: three passes either way)
  p.w2_first = p.ex == 1 ? (d.S < 2 * d.P) : (d.S < d.P);
  p.tok_c = d.P <= 64;         // (the full chain uses it only together with w2_first: the other order needs row sums over s)
  p.Pp = (d.P + 7) / 8 * 8;
  p.Sp = p.ex == 2 ? (d.S + 63) / 64 * 64 : (d.S + 7) / 8 * 8;
  p.bn_c = pick_bn(p.ex == 2 ? p.Sp : d.S);
  p.tiles_n_c = ceil_div(p.ex == 2 ? p.Sp : d.S, p.bn_c);
  const size_t S = d.S, ex = p.ex;
  const size_t occ_elems = (size_t)d.P * p.Sp > S * p.Pp ? (size_t)d.P * p.Sp : S * p.Pp;   // either orientation
  const size_t per_clip = S * ex * d.C * 2 + S * ex * 2 * d.D * 2 + S * ex * p.D2 * 2 + occ_elems * ex * 2 +
                          (size_t)d.P * 2 * p.tiles_n_c * 4 + (size_t)d.P * 2 * d.D * 2 + S * ex * d.D * 2 +
                          (size_t)d.P * d.D * 4 + 2048;
  long long nb = (long long)(((size_t)2 << 30) / per_clip);
  static const int chunk_env = [] { const char* e = getenv("PASN_TILED_CHUNK"); return e ? atoi(e) : 0; }();   // tests: force chunking
  if (chunk_env > 0 && nb > chunk_env) nb = chunk_env;
  if (nb < 1) nb = 1;
  if (nb > d.N) nb = d.N > 0 ? d.N : 1;
  p.nb = (int)nb;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += align_up(bytes, 1024); return r; };
  p.off_xt = take((size_t)p.nb * S * ex * d.C * 2);
  p.off_y = take((size_t)p.nb * S * ex * 2 * d.D * 2);
  p.off_g2 = take((size_t)p.nb * S * ex * p.D2 * 2);
  p.off_occ = take((size_t)p.nb * occ_elems * ex * 2);
  p.off_psum = take((size_t)p.nb * d.P * 2 * p.tiles_n_c * 4);
  p.off_pool = take(p.w2_first ? 0 : (size_t)p.nb * d.P * 2 * d.D * 2);
  p.off_f = take(p.w2_first ? (size_t)p.nb * S * ex * d.D * 2 : 0);
  p.off_fe = take((size_t)p.nb * d.P * d.D * 4);
  p.stat_parts = 2 * ceil_div(d.D, 128);   // (upper bound: 128-wide tiles; the chunk passes the count its GEMM really wrote)
  p.off_stat = take((size_t)p.nb * d.P * p.stat_parts * 16);
  p.total = o + 256;
  return p;
}

struct PackLayout {
  size_t off_w13, off_w4, off_w5, off_w2, off_b13, off_b4, off_b2, total;
};
PackLayout pack_layout(const pasn_dims& d) {
  const size_t ex = d.dtype == PASN_F32 ? 2 : 1, D2 = d.D / 2;
  PackLayout L;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += align_up(bytes, 256); return r; };
  L.off_w13 = take((size_t)2 * d.D * ex * d.C * 2);
  L.off_w4 = take(D2 * ex * d.D * 2);
  L.off_w5 = take((size_t)d.P * ex * D2 * 2);
  L.off_w2 = take((size_t)d.D * ex * d.D * 2);
  L.off_b13 = take((size_t)2 * d.D * 4);
  L.off_b4 = take(D2 * 4);
  L.off_b2 = take((size_t)d.D * 4);
  L.total = o;
  return L;
}

// fp32 [rows][cols] -> bf16 planes [rows][ex*cols]: plane 0 = bf16(w), plane 1 = bf16(w - plane 0)
__global__ void pack_planes_kernel(const float* __restrict__ w, int rows, int cols, int ex, __nv_bfloat16* __restrict__ out) {
  const long long n = (long long)rows * cols;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i - (long long)r * cols);
    const float v = w[i];
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    out[(size_t)r * ex * cols + c] = hi;
    if (ex == 2) *(out + (size_t)r * ex * cols + cols + c) = __float2bfloat16_rn(v - __bfloat162float(hi));
  }
}
// fp16 mode's first-layer weights: fp32 [n] -> fp16 (the operand type of the fp16 feature map)
__global__ void pack_f16_kernel(const float* __restrict__ w, long long n, __half* __restrict__ out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = __float2half_rn(w[i]);
}
__global__ void pack_bias_kernel(const float* __restrict__ b, int n, int round, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = round ? round_bf16(b[i]) : b[i];
}

// feature map -> token-major bf16 planes XT[(n*S + s)][ex*C] (O = __half: one fp16 plane, the fp16 chain's first-layer operand)
//   NCS ([n][C][S]): 64-channel x 32-voxel tiles through shared memory: loads run along s (one channel row segment per warp
//   instruction), stores along c (one full 128-byte line of bf16 channel pairs per token and plane);
//   NSC fp32 / fp16 ([n][S][C]): plane split only
template <typename T, typename O = __nv_bfloat16>
__global__ void __launch_bounds__(256) to_tokens_ncs_kernel(const T* __restrict__ x, int C, int S, int ex, O* __restrict__ out) {
  __shared__ float tile[64][33];
  const int n = blockIdx.z, c0 = blockIdx.y * 64, s0 = blockIdx.x * 32;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const T* xn = x + (size_t)n * C * S;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int cl = warp * 8 + j, c = c0 + cl, s = s0 + lane;
    tile[cl][lane] = (c < C && s < S) ? to_f32<T>(xn[(size_t)c * S + s]) : 0.f;
  }
  __syncthreads();
  const int c = c0 + 2 * lane;           // C is a multiple of 64 on this path
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int sl = warp * 4 + j, s = s0 + sl;
    if constexpr (std::is_same<O, __half>::value) {
      if (s < S && c < C)
        *reinterpret_cast<__half2*>(out + ((size_t)n * S + s) * C + c) = __floats2half2_rn(tile[2 * lane][sl], tile[2 * lane + 1][sl]);
    } else if (s < S && c < C) {
      const float v0 = tile[2 * lane][sl], v1 = tile[2 * lane + 1][sl];
      const __nv_bfloat16 h0 = __float2bfloat16_rn(v0), h1 = __float2bfloat16_rn(v1);
      __nv_bfloat16* row = out + ((size_t)n * S + s) * ex * C;
      *reinterpret_cast<__nv_bfloat162*>(row + c) = __nv_bfloat162(h0, h1);
      if (ex == 2)
        *reinterpret_cast<__nv_bfloat162*>(row + C + c) =
            __nv_bfloat162(__float2bfloat16_rn(v0 - __bfloat162float(h0)), __float2bfloat16_rn(v1 - __bfloat162float(h1)));
    }
  }
}
// small bf16 (or fp16: the kernel only moves bytes) clips (C*S*2 bytes fit in shared memory, e.g. the 7 x 7 image head): a clip's [C][S] block is one contiguous
// run in memory, so it is copied in with 16-byte vectors and transposed out of shared memory (rows of S bf16 are not
// 4-byte aligned, which makes the tiled kernel above read half-empty sectors).  One block per clip.
__global__ void __launch_bounds__(256) to_tokens_small_bf16_kernel(const __nv_bfloat16* __restrict__ x, int C, int S,
                                                                   __nv_bfloat16* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char tsm[];
  __nv_bfloat16* t = reinterpret_cast<__nv_bfloat16*>(tsm);
  const int n = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total = C * S;                                     // multiple of 8 (host checks): whole 16-byte vectors
  const uint4* src = reinterpret_cast<const uint4*>(x + (size_t)n * total);
  for (int i = threadIdx.x; i < total / 8; i += 256) reinterpret_cast<uint4*>(tsm)[i] = __ldg(src + i);
  __syncthreads();
  for (int s = warp; s < S; s += 8) {
    __nv_bfloat16* row = out + ((size_t)n * S + s) * C;
    for (int c = 2 * lane; c < C; c += 64)
      *reinterpret_cast<__nv_bfloat162*>(row + c) = __nv_bfloat162(t[c * S + s], t[(c + 1) * S + s]);
  }
}

template <typename T>
__global__ void to_tokens_nsc_split_kernel(const T* __restrict__ x, long long rows, int C, __nv_bfloat16* __restrict__ out) {
  const long long n = rows * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / C;
    const int c = (int)(i - r * C);
    const float v = to_f32<T>(x[i]);
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    out[r * 2 * C + c] = hi;
    *(out + r * 2 * C + C + c) = __float2bfloat16_rn(v - __bfloat162float(hi));
  }
}

// Osum[n][p] = sum_s (hi + lo)[n*S + s][p] of the token-major occurrence values: grid (P / 32, clips), 8 row groups per block
__global__ void __launch_bounds__(256) clip_colsum_kernel(const __nv_bfloat16* __restrict__ O, int S, int P, int ld, int lo_off,
                                                          float* __restrict__ out) {
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, wy = threadIdx.x >> 5;
  const int p = blockIdx.x * 32 + lane, n = blockIdx.y;
  float a = 0.f;
  if (p < P) {
    const __nv_bfloat16* base = O + (size_t)n * S * ld + p;
    for (int s = wy; s < S; s += 8) {
      a += __bfloat162float(base[(size_t)s * ld]);
      if (lo_off) a += __bfloat162float(base[(size_t)s * ld + lo_off]);
    }
  }
  red[wy][lane] = a;
  __syncthreads();
  if (wy == 0 && p < P) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i][lane];
    out[(size_t)n * P + p] = t;
  }
}

// passes of a product of two operands that each come as planes (hi at column 0, lo at column *_lo)
void set_passes(tcg::Gemm& g, int ex, int a_lo, int b_lo) {
  g.pair = 1;   // CTA pairs wherever the shape allows (tc_gemm.cu decides)
  for (int q = 0; q < 4; ++q) g.a_off[q] = g.b_off[q] = 0;
  if (ex == 1) { g.npass = 1; return; }
  // hi*hi, hi*lo, lo*hi.  The lo*lo term is below the representation error of the split itself (each operand keeps 16
  // significant bits: |x - xh - xl| <= 2^-17 |x|, and |xl wl| <= 2^-18 |x w|), so it is not computed.
  g.npass = 3;
  g.b_off[1] = b_lo;
  g.a_off[2] = a_lo;
}

}  // namespace

bool tiled_supported(const pasn_dims& d) {
  if (d.C % 64 != 0 || d.D % 128 != 0) return false;   // every K (C, D, D/2) is a whole number of 64-wide k-blocks
  if (d.P < 1 || d.S < 1) return false;
  return tcg::available();
}
size_t tiled_workspace_bytes(const pasn_dims& d) { return make_plan(d).total; }
size_t tiled_packed_bytes(const pasn_dims& d) { return pack_layout(d).total; }

int tiled_pack_weights(const pasn_weights& w, const pasn_dims& d, void* packed, cudaStream_t st) {
  if (((uintptr_t)packed & 255) != 0) return PASN_ERR_ALIGN;
  const PackLayout L = pack_layout(d);
  const int ex = d.dtype == PASN_F32 ? 2 : 1, D2 = d.D / 2;
  char* pk = reinterpret_cast<char*>(packed);
  auto planes = [&](const float* src, int rows, int cols, size_t off) {
    pack_planes_kernel<<<148 * 2, 256, 0, st>>>(src, rows, cols, ex, reinterpret_cast<__nv_bfloat16*>(pk + off));
    count_launch();
  };
  if (d.dtype == PASN_F16) {   // first layer fp16 x fp16 (one plane, same bytes as bf16 mode's)
    pack_f16_kernel<<<148 * 2, 256, 0, st>>>(w.addon_w1, (long long)d.D * d.C, reinterpret_cast<__half*>(pk + L.off_w13));
    pack_f16_kernel<<<148 * 2, 256, 0, st>>>(w.occ_w1, (long long)d.D * d.C, reinterpret_cast<__half*>(pk + L.off_w13) + (size_t)d.D * d.C);
    count_launch(2);
  } else {
    planes(w.addon_w1, d.D, d.C, L.off_w13);
    planes(w.occ_w1, d.D, d.C, L.off_w13 + (size_t)d.D * ex * d.C * 2);
  }
  planes(w.occ_w2, D2, d.D, L.off_w4);
  planes(w.occ_w3, d.P, D2, L.off_w5);
  planes(w.addon_w2, d.D, d.D, L.off_w2);
  const int rnd = ex == 1;
  auto bias = [&](const float* src, int n, size_t off) {
    pack_bias_kernel<<<ceil_div(n, 256), 256, 0, st>>>(src, n, rnd, reinterpret_cast<float*>(pk + off));
    count_launch();
  };
  bias(w.addon_b1, d.D, L.off_b13);
  bias(w.occ_b1, d.D, L.off_b13 + (size_t)d.D * 4);
  bias(w.occ_b2, D2, L.off_b4);
  bias(w.addon_b2, d.D, L.off_b2);
  PASN_LAUNCH_CHECK();
  return PASN_OK;
}

// the chain for clips [n0, n0+nb); occ_only stops after the occurrence map
static int tiled_chunk(const void* feat, const pasn_weights& w, const void* packed, const pasn_dims& d, const Plan& p, int n0,
                       int nb, float* logits, float* sim, void* occ, float* feats, float* dist, const pasn_push_args* push,
                       char* ws, bool occ_only, cudaStream_t st) {
  const PackLayout L = pack_layout(d);
  const char* pk = reinterpret_cast<const char*>(packed);
  const int ex = p.ex, C = p.C, D = p.D, D2 = p.D2, P = p.P, S = p.S;
  const long long T = (long long)nb * S;
  const size_t elt = dtype_bytes(d.dtype);
  const bool f16 = d.dtype == PASN_F16;   // layer 1 fp16 x fp16, the map stored in fp16; everything else as bf16 mode
  int rc;

  // ---- tokens
  const __nv_bfloat16* xt;
  const char* x = reinterpret_cast<const char*>(feat) + (size_t)n0 * C * S * elt;
  // bf16 / fp16 NCDHW feature maps with 16-byte aligned channel rows need no transposition: [C][S] per clip IS the MN-major form
  // of the A operand (voxels contiguous), which the TMA unit tiles straight out of the caller's buffer
  const bool x_direct = d.layout == PASN_LAYOUT_NCS && ex == 1 && (S * 2) % 16 == 0 && ((uintptr_t)x & 15) == 0;
  if (d.layout == PASN_LAYOUT_NSC && ex == 1) {
    xt = reinterpret_cast<const __nv_bfloat16*>(x);   // channels_last bf16 / fp16 feature map: already token-major
    if (((uintptr_t)xt & 15) != 0) return PASN_ERR_ALIGN;
  } else if (x_direct) {
    xt = reinterpret_cast<const __nv_bfloat16*>(x);
  } else {
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(ws + p.off_xt);
    if (d.layout == PASN_LAYOUT_NSC) {
      to_tokens_nsc_split_kernel<float><<<148 * 8, 256, 0, st>>>(reinterpret_cast<const float*>(x), T, C, dst);
    } else {
      dim3 grid(ceil_div(S, 32), ceil_div(C, 64), nb);
      const size_t clip_bytes = (size_t)C * S * 2;
      if (ex == 1 && S < 128 && clip_bytes <= 96 * 1024 && clip_bytes % 16 == 0 && ((uintptr_t)x & 15) == 0) {
        static bool attr_done = false;
        if (!attr_done) {
          if (cudaFuncSetAttribute(to_tokens_small_bf16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024) != cudaSuccess)
            return PASN_ERR_CUDA;
          attr_done = true;
        }
        to_tokens_small_bf16_kernel<<<nb, 256, clip_bytes, st>>>(reinterpret_cast<const __nv_bfloat16*>(x), C, S, dst);
      } else if (f16) {
        to_tokens_ncs_kernel<__half, __half><<<grid, 256, 0, st>>>(reinterpret_cast<const __half*>(x), C, S, 1,
                                                                   reinterpret_cast<__half*>(dst));
      } else if (ex == 1) {
        to_tokens_ncs_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(x), C, S, ex, dst);
      } else {
        to_tokens_ncs_kernel<float><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(x), C, S, ex, dst);
      }
    }
    PASN_LAUNCH_CHECK();
    count_launch();
    xt = dst;
  }
  __nv_bfloat16* Y = reinterpret_cast<__nv_bfloat16*>(ws + p.off_y);
  __nv_bfloat16* G2 = reinterpret_cast<__nv_bfloat16*>(ws + p.off_g2);
  __nv_bfloat16* OCC = reinterpret_cast<__nv_bfloat16*>(ws + p.off_occ);
  float* PSUM = reinterpret_cast<float*>(ws + p.off_psum);
  __nv_bfloat16* POOL = reinterpret_cast<__nv_bfloat16*>(ws + p.off_pool);
  float* FE = feats ? feats + (size_t)n0 * P * D : reinterpret_cast<float*>(ws + p.off_fe);
  // Plain forward (nobody asked for features_extracted, no push): the GEMM that would write the pooled features leaves the
  // two reductions the prototype stage needs (||f||^2, <f, v_p>) instead -- the features are neither stored nor read back.
  // Used where it pays: many prototypes (config 5: 8 MB of features per clip), and the per-clip pooling GEMM of few
  // prototypes straight into features (image head: the GEMM keeps the prototype slices in shared memory).  Elsewhere the
  // statistics' vector reads (a row per lane) cost the epilogue more than the round trip.  (Both are W2-before-pooling
  // shapes: the statistics ride in the per-clip pooling GEMM.)
  const bool fuse_stats = p.w2_first && (P >= 1024 || P <= 64) && !occ_only && feats == nullptr && push == nullptr;
  float* STAT = reinterpret_cast<float*>(ws + p.off_stat);
  int stat_parts = 2 * ceil_div(D, D >= 256 ? 256 : 128);   // column half-tiles of the GEMM that leaves the statistics
  const __nv_bfloat16* W13 = reinterpret_cast<const __nv_bfloat16*>(pk + L.off_w13);
  const __nv_bfloat16* W4 = reinterpret_cast<const __nv_bfloat16*>(pk + L.off_w4);
  const __nv_bfloat16* W5 = reinterpret_cast<const __nv_bfloat16*>(pk + L.off_w5);
  const __nv_bfloat16* W2 = reinterpret_cast<const __nv_bfloat16*>(pk + L.off_w2);
  const float* b13 = reinterpret_cast<const float*>(pk + L.off_b13);
  const float* b4 = reinterpret_cast<const float*>(pk + L.off_b4);
  const float* b2 = reinterpret_cast<const float*>(pk + L.off_b2);

  // ---- (A) [H1 | G1] = relu(X [W1; W3]^T + [b1; b3])        (occurrence only: G1 alone)
  const int nA = occ_only ? D : 2 * D;          // output columns per plane
  {
    tcg::Gemm g{};
    g.A = xt; g.lda = (long long)ex * C; g.a_bs = 0; g.a_batched = 0; g.ka = ex * C;
    g.B = occ_only ? W13 + (size_t)D * ex * C : W13; g.ldb = (long long)ex * C; g.b_bs = 0; g.b_batched = 0; g.kb = ex * C;
    g.M = (int)T; g.N = nA; g.K = C; g.batch = 1; g.bn = 256;
    set_passes(g, ex, C, C);
    g.bias = occ_only ? b13 + D : b13; g.act = tcg::ACT_RELU;
    g.ab_f16 = f16 ? 1 : 0;   // X and [W1; W3] both fp16 (pack: tiled_pack_weights)
    g.out[0] = {Y, ex == 1 ? tcg::OUT_BF16 : tcg::OUT_BF16_HILO, (long long)ex * nA, 0, nA};
    if (x_direct) {   // one GEMM per clip: rows = its S voxels, operand [C rows][S] as it lies in the feature map
      g.a_mn_major = 1; g.lda = S; g.a_bs = (long long)C * S; g.a_batched = 1; g.ka = S; g.a_rows = C;
      g.M = S; g.batch = nb;
      g.out[0].bs = (long long)S * ex * nA;
    }
    if ((rc = tcg::launch(g, st))) return rc;
  }
  // ---- (B) G2 = relu(G1 W4^T + b4)
  const int g1_off = occ_only ? 0 : D;          // column of G1 inside a plane of Y
  {
    tcg::Gemm g{};
    g.A = Y + g1_off; g.lda = (long long)ex * nA; g.a_batched = 0; g.ka = ex * nA - g1_off;
    g.B = W4; g.ldb = (long long)ex * D; g.b_batched = 0; g.kb = ex * D;
    g.M = (int)T; g.N = D2; g.K = D; g.batch = 1; g.bn = pick_bn(D2);
    set_passes(g, ex, nA, D);
    g.bias = b4; g.act = tcg::ACT_RELU;
    g.out[0] = {G2, ex == 1 ? tcg::OUT_BF16 : tcg::OUT_BF16_HILO, (long long)ex * D2, 0, D2};
    if ((rc = tcg::launch(g, st))) return rc;
  }
  // ---- (C) O[n] = |W5 G2[n]^T|  -> occurrence_map [n][P][S] (+ the pooling operand copy when the map cannot serve as one)
  void* occ_user = occ ? reinterpret_cast<char*>(occ) + (size_t)n0 * P * S * elt : nullptr;
  const int occ_mode = ex == 2 ? tcg::OUT_F32 : (f16 ? tcg::OUT_F16 : tcg::OUT_BF16);   // the map in the feature map's type
  const __nv_bfloat16* pool_a = nullptr;     // pooling A operand
  long long pool_lda = 0;
  // W2-after-pooling order: the row sums over s then come from a small column-sum kernel below.  (fp32 maps keep the
  // per-clip form there: their map leaves as 4-byte plain stores, which measured slower than the TMA rows -- 0.72 vs 0.64 ms)
  const bool tok_c = p.tok_c && (occ_only || p.w2_first || ex == 1);
  if (tok_c) {
    // few prototypes: O^T = |G2 W5^T| over all tokens in one GEMM (rows = tokens, N = P).  The occurrence map leaves
    // channel-major per clip through plain stores that are coalesced along the voxels; the token-major copy
    // [T][ex*Pp] is the pooling's MN-major A operand.
    tcg::Gemm g{};
    g.A = G2; g.lda = (long long)ex * D2; g.a_batched = 0; g.ka = ex * D2;
    g.B = W5; g.ldb = (long long)ex * D2; g.b_batched = 0; g.kb = ex * D2;
    g.M = (int)T; g.N = P; g.K = D2; g.batch = 1; g.bn = 64;
    set_passes(g, ex, D2, D2);
    g.act = tcg::ACT_ABS;
    int no = 0;
    if (occ_user != nullptr) {
      g.out[no] = {occ_user, occ_mode, (long long)S, (long long)P * S, 0, P, 0, S};
      ++no;
    }
    if (!occ_only) {
      g.out[no] = {OCC, ex == 1 ? tcg::OUT_BF16 : tcg::OUT_BF16_HILO, (long long)ex * p.Pp, 0, p.Pp, P, 0, 0};
      ++no;
      pool_a = OCC; pool_lda = (long long)ex * p.Pp;
    }
    if ((rc = tcg::launch(g, st))) return rc;
    if (!occ_only && !p.w2_first) {   // Osum[n][p] = sum_s O[n,s,p] (of the stored values: what the pooling will read)
      dim3 grid(ceil_div(P, 32), nb);
      clip_colsum_kernel<<<grid, 256, 0, st>>>(OCC, S, P, ex * p.Pp, ex == 2 ? p.Pp : 0, PSUM);
      PASN_LAUNCH_CHECK();
      count_launch();
    }
  } else {
    tcg::Gemm g{};
    g.A = W5; g.lda = (long long)ex * D2; g.a_batched = 0; g.ka = ex * D2;
    g.B = G2; g.ldb = (long long)ex * D2; g.b_bs = (long long)S * ex * D2; g.b_batched = 1; g.kb = ex * D2;
    g.b_rows = S;   // tokens of this clip; the padded columns of the operand copy come out as exact zeros
    g.M = P; g.K = D2; g.batch = nb; g.bn = p.bn_c;
    g.N = ex == 2 ? p.Sp : S;
    set_passes(g, ex, D2, D2);
    g.act = tcg::ACT_ABS;
    int no = 0;
    const bool need_copy = !occ_only && !(p.occ_direct && occ_user != nullptr);
    if (occ_user != nullptr) {
      g.out[no] = {occ_user, occ_mode, (long long)S, (long long)P * S, 0};
      g.out[no].ncols = S;
      ++no;
    }
    if (need_copy) {
      g.out[no] = {OCC, ex == 1 ? tcg::OUT_BF16 : tcg::OUT_BF16_HILO, (long long)ex * p.Sp, (long long)P * ex * p.Sp, p.Sp};
      g.out[no].ncols = ex == 2 ? p.Sp : S;
      ++no;
      pool_a = OCC; pool_lda = (long long)ex * p.Sp;
    } else if (!occ_only) {
      pool_a = reinterpret_cast<const __nv_bfloat16*>(occ_user); pool_lda = S;
    }
    g.psum = (occ_only || p.w2_first) ? nullptr : PSUM;
    g.psum_rounded = ex == 1;
    if ((rc = tcg::launch(g, st))) return rc;
  }
  if (occ_only) return PASN_OK;
  if (p.w2_first) {
    // ---- (D') F = H1 W2^T + b2 over all tokens, then FE[n] = O[n] F[n] (K = S) straight into fp32
    __nv_bfloat16* F = reinterpret_cast<__nv_bfloat16*>(ws + p.off_f);
    {
      tcg::Gemm g{};
      g.A = Y; g.lda = (long long)ex * 2 * D; g.a_batched = 0; g.ka = ex * 2 * D;
      g.B = W2; g.ldb = (long long)ex * D; g.b_batched = 0; g.kb = ex * D;
      g.M = (int)T; g.N = D; g.K = D; g.batch = 1; g.bn = D >= 256 ? 256 : 128;
      set_passes(g, ex, 2 * D, D);
      g.bias = b2; g.act = tcg::ACT_NONE;
      g.out[0] = {F, ex == 1 ? tcg::OUT_BF16 : tcg::OUT_BF16_HILO, (long long)ex * D, 0, D};
      if ((rc = tcg::launch(g, st))) return rc;
    }
    {
      tcg::Gemm g{};
      g.A = pool_a; g.lda = pool_lda; g.a_bs = (long long)P * pool_lda; g.a_batched = 1;
      g.ka = ex == 2 ? 2 * p.Sp : S;
      g.B = F; g.ldb = (long long)ex * D; g.b_bs = (long long)S * ex * D; g.b_batched = 1; g.kb = ex * D;
      g.b_mn_major = 1; g.b_rows = S;
      g.M = P; g.N = D; g.K = ex == 2 ? p.Sp : S; g.batch = nb; g.bn = D >= 256 ? 256 : 128;
      set_passes(g, ex, p.Sp, D);
      if (tok_c) {   // occurrence values token-major: [S rows][P] per clip, prototypes contiguous (MN-major A)
        g.a_mn_major = 1; g.a_bs = (long long)S * pool_lda; g.ka = ex * p.Pp; g.a_rows = S; g.K = S;
        set_passes(g, ex, p.Pp, D);
      }
      g.act = tcg::ACT_NONE;
      g.out[0] = {FE, tcg::OUT_F32, (long long)D, (long long)P * D, 0};
      if (fuse_stats) {
        g.out[0].mode = tcg::OUT_NONE;
        g.rowstat = STAT; g.dotvec = w.prototypes; g.dot_ld = D; g.dot_mod = P; g.dot_early = 1;   // (parameters: the chain does not write them)
        // few prototypes, few voxels (image head: 40 x 49): three clips share a 128-row tile, block-diagonally -- a clip alone
        // uses 40 of the tile's rows and two of the four epilogue row groups
        const int G = 128 / P < 4 ? 128 / P : 4;
        if (tok_c && ex == 1 && S <= 64 && G >= 2 && nb >= 2 * G) {
          g.group = G; g.group_rows = P; g.group_items = nb;
          g.M = G * P; g.batch = ceil_div(nb, G); g.bn = 128;
          g.stat_rows = (long long)nb * P;
          stat_parts = 2 * ceil_div(D, 128);
        }
      }
      if ((rc = tcg::launch(g, st))) return rc;
    }
  } else {
  // ---- (D) pooled[n] = O[n] H1[n]   (K = S; H1 token-major = MN-major B operand) -> bf16 hi | lo planes
  {
    tcg::Gemm g{};
    g.A = pool_a; g.lda = pool_lda; g.a_bs = (long long)P * pool_lda; g.a_batched = 1;
    g.ka = ex == 2 ? 2 * p.Sp : S;
    g.B = Y; g.ldb = (long long)ex * 2 * D; g.b_bs = (long long)S * ex * 2 * D; g.b_batched = 1; g.kb = ex * 2 * D;
    g.b_mn_major = 1; g.b_rows = S;
    g.M = P; g.N = D; g.K = ex == 2 ? p.Sp : S; g.batch = nb; g.bn = D >= 256 ? 256 : 128;
    set_passes(g, ex, p.Sp, 2 * D);
    if (tok_c) {   // occurrence values token-major: [S rows][P] per clip (MN-major A)
      g.a_mn_major = 1; g.a_bs = (long long)S * pool_lda; g.ka = ex * p.Pp; g.a_rows = S; g.K = S;
      set_passes(g, ex, p.Pp, 2 * D);
    }
    g.act = tcg::ACT_NONE;
    g.out[0] = {POOL, tcg::OUT_BF16_HILO, (long long)2 * D, (long long)P * 2 * D, D};
    if ((rc = tcg::launch(g, st))) return rc;
  }
  // ---- (E) FE = pooled W2^T + (sum_s O) b2^T   (pooled = hi + lo; fp32 mode: W2 = hi + lo as well)
  {
    tcg::Gemm g{};
    g.A = POOL; g.lda = 2 * D; g.a_batched = 0; g.ka = 2 * D;
    g.B = W2; g.ldb = (long long)ex * D; g.b_batched = 0; g.kb = ex * D;
    g.M = nb * P; g.N = D; g.K = D; g.batch = 1; g.bn = D >= 256 ? 256 : 128;
    set_passes(g, ex, D, D);
    if (ex == 1) { g.npass = 2; g.a_off[1] = D; }   // pooled = hi + lo planes, W2 bf16
    g.rowparts = PSUM; g.nparts = tok_c ? 1 : 2 * p.tiles_n_c; g.colvec = b2;
    g.act = tcg::ACT_NONE;
    g.out[0] = {FE, tcg::OUT_F32, (long long)D, 0, 0};
    if ((rc = tcg::launch(g, st))) return rc;
  }
  }
  // ---- cosine / similarity / logits / distance / push keys (+ winner capture)
  if (fuse_stats)
    return launch_proto_from_stats(STAT, stat_parts, w.last_layer, nb, P, d.K, logits + (size_t)n0 * d.K, sim + (size_t)n0 * P,
                                   dist ? dist + (size_t)n0 * P : nullptr, st);
  pasn_push_args pa;
  const pasn_push_args* pp = nullptr;
  if (push) { pa = *push; pa.labels += n0; pa.global_offset += n0; pp = &pa; }
  return launch_proto_stage(FE, w.prototypes, w.last_layer, nb, P, D, d.K, logits + (size_t)n0 * d.K, sim + (size_t)n0 * P,
                            dist ? dist + (size_t)n0 * P : nullptr, pp, st);
}

int tiled_head_forward(const void* feat, const pasn_weights& w, const void* packed, const pasn_dims& d, float* logits,
                       float* sim, void* occ, float* feats, float* dist, const pasn_push_args* push, void* ws,
                       size_t ws_bytes, cudaStream_t st) {
  if (!tiled_supported(d) || packed == nullptr) return PASN_ERR_UNSUPPORTED;
  const Plan p = make_plan(d);
  if (ws_bytes < p.total) return PASN_ERR_WORKSPACE;
  if (((uintptr_t)ws & 255) != 0 || ((uintptr_t)feat & 15) != 0) return PASN_ERR_ALIGN;
  main_kernel_begin(st);   // tiled path: the "dominant kernel" is the GEMM chain
  for (int n0 = 0; n0 < d.N; n0 += p.nb) {
    const int nb = d.N - n0 < p.nb ? d.N - n0 : p.nb;
    const int rc = tiled_chunk(feat, w, packed, d, p, n0, nb, logits, sim, occ, feats, dist, push, reinterpret_cast<char*>(ws),
                               false, st);
    if (rc) return rc;
  }
  main_kernel_end(st);
  return PASN_OK;
}

int tiled_occurrence_only(const void* feat, const pasn_weights& w, const void* packed, const pasn_dims& d, void* occ, void* ws,
                          size_t ws_bytes, cudaStream_t st) {
  if (!tiled_supported(d) || packed == nullptr) return PASN_ERR_UNSUPPORTED;
  const Plan p = make_plan(d);
  if (ws_bytes < p.total) return PASN_ERR_WORKSPACE;
  if (((uintptr_t)ws & 255) != 0 || ((uintptr_t)feat & 15) != 0) return PASN_ERR_ALIGN;
  for (int n0 = 0; n0 < d.N; n0 += p.nb) {
    const int nb = d.N - n0 < p.nb ? d.N - n0 : p.nb;
    const int rc = tiled_chunk(feat, w, packed, d, p, n0, nb, nullptr, nullptr, occ, nullptr, nullptr, nullptr,
                               reinterpret_cast<char*>(ws), true, st);
    if (rc) return rc;
  }
  return PASN_OK;
}


// =================================================================================================================
// Backward of the head on the tensor cores (SURVEY.md section 8(f) row 2; reference: loss.backward() through
// Video_XProtoNet.forward, src/agents/XProtoNet_Base.py:397, src/models/Video_XProtoNet.py:82-98).
//
// Every contraction of the fp32 gradient (backward.cu documents the math and the sub-gradient conventions) runs as a
// three-pass bf16 hi/lo GEMM of tc_gemm.cu over token-major planes, i.e. fp32-grade products with fp32 accumulation:
//   recomputed forward   XT -> [H1|G1] -> G2 -> Opre (sign carrier + |.| planes) ; F = W2 H1 + b2 ; FE = O^T F
//   prototype stage      gFE, gV, gWl                                     (two small CUDA-core kernels)
//   gOpre = ((F gFE^T) + gOcc) * sign(Opre)          per clip, the upstream map gradient is read transposed
//   gF    = O gFE                                    per clip
//   gH1   = (gF W2) masked by H1 > 0 ; gG2 = (gOpre W5) masked ; gG1 = (gG2 W4) masked      (ReLU masks in the epilogue)
//   weight gradients     gW[m][n] = sum_tokens gY[t][m] X[t][n]: both operands token-major (MN-major), the token range
//                        split over the machine, fp32 partials reduced by one small kernel; biases: column sums
//   gX    = [gH1|gG1] [W1;W3]                        stored channel-major per clip (NCDHW) in fp32
// =================================================================================================================
namespace {

struct BPlan {
  int C, D, D2, P, Pp, K, S, xe;   // xe: planes of the token-major feature copy (1: bf16 input is exact, 2: fp32 input, or
                                   // fp16 input: its 11 significant bits are exact in a bf16 hi | lo pair)
  int nb;
  size_t off_pk, off_xt, off_y, off_g2, off_os, off_oa, off_f, off_fe, off_gfe, off_rs, off_go, off_gf, off_gy, off_gg2,
      off_part, part_bytes, total;
};

inline int split_parts(long long T, int tiles, int* kper) {
  int parts = (148 + tiles - 1) / tiles;
  if (parts < 1) parts = 1;
  long long k = (T + parts - 1) / parts;
  if (k < 256) k = 256;
  k = (k + 63) / 64 * 64;
  *kper = (int)k;
  return (int)((T + k - 1) / k);
}

BPlan make_bplan(const pasn_dims& d) {
  BPlan b{};
  b.C = d.C; b.D = d.D; b.D2 = d.D / 2; b.P = d.P; b.Pp = (d.P + 7) / 8 * 8; b.K = d.K; b.S = d.S;
  b.xe = d.dtype == PASN_BF16 ? 1 : 2;
  pasn_dims d2 = d;
  d2.dtype = PASN_F32;
  const size_t pk = align_up(pack_layout(d2).total, 1024);
  const size_t S = d.S;
  const size_t per_tok = (size_t)b.xe * d.C * 2 + 4 * d.D * 2 + 2 * b.D2 * 2 + 3 * b.Pp * 2 + 2 * d.D * 2 +   // XT Y G2 OS OA F
                         2 * b.Pp * 2 + 2 * d.D * 2 + 4 * d.D * 2 + 2 * b.D2 * 2;                             // GO GF GY GG2
  const size_t per_clip = per_tok * S + (size_t)d.P * d.D * 4 + (size_t)d.P * 2 * d.D * 2 + (size_t)d.P * 16 + 4096;
  // fp32 partials of the largest weight gradient at full machine width
  const size_t m13 = (size_t)2 * d.D * d.C, m2 = (size_t)d.D * d.D;
  b.part_bytes = align_up((m13 > m2 ? m13 : m2) * 4 * 80, 1024);
  long long nb = (long long)(((size_t)1500 << 20) / per_clip);
  static const int chunk_env = [] { const char* e = getenv("PASN_TILED_CHUNK"); return e ? atoi(e) : 0; }();
  if (chunk_env > 0 && nb > chunk_env) nb = chunk_env;
  if (nb < 1) nb = 1;
  if (nb > d.N) nb = d.N > 0 ? d.N : 1;
  b.nb = (int)nb;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += align_up(bytes, 1024); return r; };
  const size_t T = (size_t)b.nb * S;
  b.off_pk = take(pk);
  b.off_xt = take(T * b.xe * d.C * 2);
  b.off_y = take(T * 4 * d.D * 2);
  b.off_g2 = take(T * 2 * b.D2 * 2);
  b.off_os = take(T * b.Pp * 2);
  b.off_oa = take(T * 2 * b.Pp * 2);
  b.off_f = take(T * 2 * d.D * 2);
  b.off_fe = take((size_t)b.nb * d.P * d.D * 4);
  b.off_gfe = take((size_t)b.nb * d.P * 2 * d.D * 2);
  b.off_rs = take((size_t)b.nb * d.P * 16);
  b.off_go = take(T * 2 * b.Pp * 2);
  b.off_gf = take(T * 2 * d.D * 2);
  b.off_gy = take(T * 4 * d.D * 2);
  b.off_gg2 = take(T * 2 * b.D2 * 2);
  b.off_part = take(b.part_bytes);
  b.total = o + 256;
  return b;
}

// three-pass product of two plane pairs; an operand without a lo plane (bf16-exact feature map) drops its pass
void set_passes_b(tcg::Gemm& g, int a_lo, int b_lo, bool a_has_lo = true, bool b_has_lo = true) {
  g.pair = 1;
  for (int q = 0; q < 4; ++q) g.a_off[q] = g.b_off[q] = 0;
  int n = 1;
  if (b_has_lo) { g.b_off[n] = b_lo; ++n; }
  if (a_has_lo) { g.a_off[n] = a_lo; ++n; }
  g.npass = n;
}

// prototype stage backward, part 1: one warp per (clip, prototype) row.
//   gs = gSim + sum_k gLogits[n,k] Wl[k,p];  gcos = gs / 2;  cos = <f,v> / (nf nv) with each norm clamped at eps (a clamped
//   norm is a constant);  gFE = gcos (v / (nf nv) - cos f / nf^2)  -> bf16 hi|lo planes (operand of the next GEMMs);
//   row scalars for part 2: a = gcos / (nf nv), b = gcos cos / nv^2 (0 when nv is clamped), sim
__global__ void __launch_bounds__(256) proto_bwd_rows_kernel(const float* __restrict__ FE, const float* __restrict__ protos,
                                                             const float* __restrict__ last_layer, const float* __restrict__ gLogits,
                                                             const float* __restrict__ gSim, long long rows, int P, int D, int K,
                                                             __nv_bfloat16* __restrict__ gfe, float4* __restrict__ rs) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr float eps = 1e-8f;
  for (long long r = (long long)blockIdx.x * 8 + warp; r < rows; r += (long long)gridDim.x * 8) {
    const long long n = r / P;
    const int p = (int)(r - n * P);
    const float* f = FE + (size_t)r * D;
    const float* v = protos + (size_t)p * D;
    float ff = 0.f, vv = 0.f, dot = 0.f;
    for (int d = lane; d < D; d += 32) {
      const float a = f[d], b = v[d];
      ff = fmaf(a, a, ff); vv = fmaf(b, b, vv); dot = fmaf(a, b, dot);
    }
    ff = warp_sum(ff); vv = warp_sum(vv); dot = warp_sum(dot);
    const float fnorm = sqrtf(ff), vnorm = sqrtf(vv);
    const float nf = fmaxf(fnorm, eps), nv = fmaxf(vnorm, eps);
    const float inv = 1.0f / (nf * nv);
    const float cosv = dot * inv;
    float gs = gSim ? gSim[r] : 0.f;
    if (gLogits)
      for (int k = 0; k < K; ++k) gs = fmaf(gLogits[(size_t)n * K + k], last_layer[(size_t)k * P + p], gs);
    const float gcos = 0.5f * gs;
    const float cf = (fnorm > eps) ? cosv / (nf * nf) : 0.f;
    const float cv = (vnorm > eps) ? cosv / (nv * nv) : 0.f;
    __nv_bfloat16* grow = gfe + (size_t)r * 2 * D;
    for (int d = lane; d < D; d += 32) {
      const float gv = gcos * (v[d] * inv - cf * f[d]);
      const __nv_bfloat16 hi = __float2bfloat16_rn(gv);
      grow[d] = hi;
      grow[D + d] = __float2bfloat16_rn(gv - __bfloat162float(hi));
    }
    if (lane == 0) rs[r] = make_float4(gcos * inv, gcos * cv, (cosv + 1.0f) * 0.5f, 0.f);
  }
}
// part 2: gV[p,:] += sum_n a[n,p] FE[n,p,:] - (sum_n b[n,p]) v[p,:];  gWl[k,p] += sum_n gLogits[n,k] sim[n,p].
// grid (P, slices of the clip range); every slice adds its share with atomics
__global__ void __launch_bounds__(256) proto_bwd_reduce_kernel(const float* __restrict__ FE, const float* __restrict__ protos,
                                                               const float* __restrict__ gLogits, const float4* __restrict__ rs,
                                                               int nb, int P, int D, int K, float* __restrict__ gV,
                                                               float* __restrict__ gWl) {
  const int p = blockIdx.x, tid = threadIdx.x;
  const int per = (nb + gridDim.y - 1) / gridDim.y;
  const int n_begin = blockIdx.y * per, n_end = min(nb, n_begin + per);
  if (n_begin >= n_end) return;
  __shared__ float red[8];
  float bsum = 0.f;
  for (int n = n_begin + tid; n < n_end; n += 256) bsum += rs[(size_t)n * P + p].y;
  bsum = warp_sum(bsum);
  if ((tid & 31) == 0) red[tid >> 5] = bsum;
  __syncthreads();
  float sb = 0.f;
  for (int i = 0; i < 8; ++i) sb += red[i];
  for (int d = tid; d < D; d += 256) {
    float acc = 0.f;
#pragma unroll 4
    for (int n = n_begin; n < n_end; ++n) acc = fmaf(rs[(size_t)n * P + p].x, FE[((size_t)n * P + p) * D + d], acc);
    atomicAdd(gV + (size_t)p * D + d, acc - sb * protos[(size_t)p * D + d]);
  }
  if (gLogits && tid < K) {
    float acc = 0.f;
    for (int n = n_begin; n < n_end; ++n) acc = fmaf(gLogits[(size_t)n * K + tid], rs[(size_t)n * P + p].z, acc);
    atomicAdd(gWl + (size_t)tid * P + p, acc);
  }
}

// dst[m][n] += sum_parts part[q][m][n]; rows >= rows0 continue in dst1 (stacked [W1; W3] gradient)
__global__ void reduce_parts_kernel(const float* __restrict__ part, int nparts, int M, int N, float* __restrict__ dst0, int rows0,
                                    float* __restrict__ dst1) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)M * N) return;
  float a = 0.f;
  for (int q = 0; q < nparts; ++q) a += part[(size_t)q * M * N + i];
  const int m = (int)(i / N);
  if (m < rows0) dst0[i] += a;
  else dst1[i - (long long)rows0 * N] += a;
}

// gb[c] += sum over rows of (hi + lo) planes: X [rows][ld] with the lo plane at column lo_off.  A warp covers 64 columns
// (one bf16 pair per lane and plane: 128-byte row segments), a block 8 x 32 rows per step; grid (ncols / 64, row chunks)
__global__ void __launch_bounds__(256) colsum_planes_kernel(const __nv_bfloat16* __restrict__ X, long long rows, long long ld,
                                                            int lo_off, int ncols, float* __restrict__ gb0, int cols0,
                                                            float* __restrict__ gb1) {
  __shared__ float red[8][64];
  const int lane = threadIdx.x & 31, wy = threadIdx.x >> 5;
  const int c = blockIdx.x * 64 + 2 * lane;
  const long long r0 = (long long)blockIdx.y * 512, r1 = r0 + 512 < rows ? r0 + 512 : rows;
  float a0 = 0.f, a1 = 0.f;
  if (c < ncols) {
#pragma unroll 4
    for (long long r = r0 + wy; r < r1; r += 8) {
      const __nv_bfloat16* row = X + r * ld;
      const float2 h = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(row + c));
      const float2 l = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(row + lo_off + c));
      a0 += h.x + l.x; a1 += h.y + l.y;
    }
  }
  red[wy][2 * lane] = a0; red[wy][2 * lane + 1] = a1;
  __syncthreads();
  if (threadIdx.x < 64) {
    const int cc = blockIdx.x * 64 + threadIdx.x;
    if (cc < ncols) {
      float t = 0.f;
      for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x];
      atomicAdd(cc < cols0 ? gb0 + cc : gb1 + (cc - cols0), t);
    }
  }
}

// occurrence-only backward: gOpre[(n,s)][p] = gOcc[n][p][s] * sign(Opre[(n,s)][p]) as hi|lo planes (32 x 32 tiles through
// shared memory: reads run along s, writes along p); pad columns [P, Pp) are written as zeros
__global__ void __launch_bounds__(256) gopre_from_gocc_kernel(const float* __restrict__ gOcc, const __nv_bfloat16* __restrict__ OS,
                                                              int P, int Pp, int S, __nv_bfloat16* __restrict__ GO) {
  __shared__ float tile[32][33];
  const int n = blockIdx.z, p0 = blockIdx.y * 32, s0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int j = ty; j < 32; j += 8) {
    const int p = p0 + j, s = s0 + tx;
    tile[j][tx] = (p < P && s < S) ? gOcc[((size_t)n * P + p) * S + s] : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const int s = s0 + j, p = p0 + tx;
    if (s < S && p < Pp) {
      const size_t t = (size_t)n * S + s;
      float v = tile[tx][j];
      const float o = __bfloat162float(OS[t * Pp + p]);
      v = o > 0.f ? v : (o < 0.f ? -v : 0.f);
      const __nv_bfloat16 hi = __float2bfloat16_rn(v);
      GO[t * 2 * Pp + p] = hi;
      GO[t * 2 * Pp + Pp + p] = __float2bfloat16_rn(v - __bfloat162float(hi));
    }
  }
}

}  // namespace

bool tiled_backward_supported(const pasn_dims& d) { return tiled_supported(d) && d.path != PASN_PATH_GENERIC; }
size_t tiled_backward_workspace_bytes(const pasn_dims& d) { return make_bplan(d).total; }

int tiled_head_backward(const void* feat, const pasn_weights& w, const pasn_dims& d, const float* gLogits, const float* gSim,
                        const float* gOcc, const pasn_grads& gr, float* gX, void* ws_, size_t ws_bytes, cudaStream_t st) {
  const BPlan b = make_bplan(d);
  if (ws_bytes < b.total) return PASN_ERR_WORKSPACE;
  if (((uintptr_t)ws_ & 255) != 0) return PASN_ERR_ALIGN;
  char* ws = reinterpret_cast<char*>(ws_);
  const int C = b.C, D = b.D, D2 = b.D2, P = b.P, Pp = b.Pp, S = b.S, xe = b.xe;
  int rc;
  // weight planes (hi | lo), the forward's fp32-mode packing
  pasn_dims d2 = d;
  d2.dtype = PASN_F32;
  const PackLayout L = pack_layout(d2);
  if ((rc = tiled_pack_weights(w, d2, ws + b.off_pk, st))) return rc;
  const char* pk = ws + b.off_pk;
  const __nv_bfloat16* W13 = reinterpret_cast<const __nv_bfloat16*>(pk + L.off_w13);   // [2D][2C]
  const __nv_bfloat16* W4 = reinterpret_cast<const __nv_bfloat16*>(pk + L.off_w4);     // [D2][2D]
  const __nv_bfloat16* W5 = reinterpret_cast<const __nv_bfloat16*>(pk + L.off_w5);     // [P][2 D2]
  const __nv_bfloat16* W2 = reinterpret_cast<const __nv_bfloat16*>(pk + L.off_w2);     // [D][2D]
  const float* b13 = reinterpret_cast<const float*>(pk + L.off_b13);
  const float* b4 = reinterpret_cast<const float*>(pk + L.off_b4);
  const float* b2 = reinterpret_cast<const float*>(pk + L.off_b2);
  auto bf = [&](size_t off) { return reinterpret_cast<__nv_bfloat16*>(ws + off); };
  __nv_bfloat16 *XT = bf(b.off_xt), *Y = bf(b.off_y), *G2 = bf(b.off_g2), *OS = bf(b.off_os), *OA = bf(b.off_oa), *F = bf(b.off_f),
                *GFE = bf(b.off_gfe), *GO = bf(b.off_go), *GF = bf(b.off_gf), *GY = bf(b.off_gy), *GG2 = bf(b.off_gg2);
  float* FE = reinterpret_cast<float*>(ws + b.off_fe);
  float4* RS = reinterpret_cast<float4*>(ws + b.off_rs);
  float* PART = reinterpret_cast<float*>(ws + b.off_part);
  const size_t elt = dtype_bytes(d.dtype);
  const bool x_lo = xe == 2;
  // No gradient arrives through logits / similarity: backward of compute_occurence_map alone (TransformLoss re-entry,
  // src/loss/loss.py:302) -- only the occurrence branch is recomputed and differentiated.
  const bool occ_only = gLogits == nullptr && gSim == nullptr;
  if (occ_only && gOcc == nullptr) {
    if (gX) cudaMemsetAsync(gX, 0, (size_t)d.N * C * S * 4, st);
    return PASN_OK;
  }

  // gW[m][n] (+)= sum_t A[t][m] B[t][n] over the tokens of the chunk (hi|lo planes, lo at column a_lo / b_lo)
  auto wgrad = [&](const __nv_bfloat16* A, long long lda, int a_lo, int M, const __nv_bfloat16* B, long long ldb, int b_lo,
                   bool b_has_lo, int N, long long T, float* dst0, int rows0, float* dst1) -> int {
    const int bn = N >= 256 ? 256 : (N >= 128 ? 128 : 64);
    const int tiles = ceil_div(M, 256) * ceil_div(N, bn) * 2;
    int kper;
    int parts = split_parts(T, tiles > 148 ? 148 : tiles, &kper);
    while ((size_t)parts * M * N * 4 > b.part_bytes && parts > 1) { kper *= 2; parts = (int)((T + kper - 1) / kper); }
    tcg::Gemm g{};
    g.A = A; g.lda = lda; g.ka = (int)lda; g.a_mn_major = 1; g.a_rows = (int)T;
    g.B = B; g.ldb = ldb; g.kb = (int)ldb; g.b_mn_major = 1; g.b_rows = (int)T;
    g.M = M; g.N = N; g.K = kper; g.batch = parts; g.k_rows_per_batch = kper; g.bn = bn;
    set_passes_b(g, a_lo, b_lo, true, b_has_lo);
    g.out[0] = {PART, tcg::OUT_F32, (long long)N, (long long)M * N, 0, 0, 0, 0};
    int r = tcg::launch(g, st);
    if (r) return r;
    const long long tot = (long long)M * N;
    reduce_parts_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(PART, parts, M, N, dst0, rows0, dst1 ? dst1 : dst0);
    if (cudaGetLastError() != cudaSuccess) return PASN_ERR_CUDA;
    count_launch();
    return PASN_OK;
  };
  auto colsum = [&](const __nv_bfloat16* X, long long T, long long ld, int lo_off, int ncols, float* g0, int cols0, float* g1) -> int {
    dim3 grid(ceil_div(ncols, 64), (unsigned)((T + 511) / 512));   // ncols is even on every caller (channel counts)
    colsum_planes_kernel<<<grid, 256, 0, st>>>(X, T, ld, lo_off, ncols, g0, cols0, g1 ? g1 : g0);
    if (cudaGetLastError() != cudaSuccess) return PASN_ERR_CUDA;
    count_launch();
    return PASN_OK;
  };

  for (int n0 = 0; n0 < d.N; n0 += b.nb) {
    const int nb = d.N - n0 < b.nb ? d.N - n0 : b.nb;
    const long long T = (long long)nb * S;
    const char* x = reinterpret_cast<const char*>(feat) + (size_t)n0 * C * S * elt;
    // ---- token-major feature planes
    const __nv_bfloat16* xt = XT;
    if (d.layout == PASN_LAYOUT_NSC && xe == 1) {
      xt = reinterpret_cast<const __nv_bfloat16*>(x);
      if (((uintptr_t)xt & 15) != 0) return PASN_ERR_ALIGN;
    } else if (d.layout == PASN_LAYOUT_NSC) {
      if (d.dtype == PASN_F16) to_tokens_nsc_split_kernel<__half><<<148 * 8, 256, 0, st>>>(reinterpret_cast<const __half*>(x), T, C, XT);
      else to_tokens_nsc_split_kernel<float><<<148 * 8, 256, 0, st>>>(reinterpret_cast<const float*>(x), T, C, XT);
      count_launch();
    } else {
      dim3 grid(ceil_div(S, 32), ceil_div(C, 64), nb);
      if (xe == 1) to_tokens_ncs_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(x), C, S, 1, XT);
      else if (d.dtype == PASN_F16) to_tokens_ncs_kernel<__half><<<grid, 256, 0, st>>>(reinterpret_cast<const __half*>(x), C, S, 2, XT);
      else to_tokens_ncs_kernel<float><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(x), C, S, 2, XT);
      count_launch();
    }
    PASN_LAUNCH_CHECK();
    const long long ldx = (long long)xe * C;

    // ================= forward, recomputed
    {  // [H1 | G1] = relu(X [W1; W3]^T + b)
      tcg::Gemm g{};
      g.A = xt; g.lda = ldx; g.ka = (int)ldx;
      g.B = W13; g.ldb = 2 * C; g.kb = 2 * C;
      g.M = (int)T; g.N = 2 * D; g.K = C; g.batch = 1; g.bn = 256;
      set_passes_b(g, C, C, x_lo, true);
      g.bias = b13; g.act = tcg::ACT_RELU;
      g.out[0] = {Y, tcg::OUT_BF16_HILO, (long long)4 * D, 0, 2 * D, 0, 0, 0};
      if (occ_only) {   // G1 alone, into its usual columns [D, 2D) of the planes
        g.B = W13 + (size_t)D * 2 * C; g.N = D; g.bias = b13 + D; g.bn = D >= 256 ? 256 : 128;
        g.out[0] = {Y + D, tcg::OUT_BF16_HILO, (long long)4 * D, 0, 2 * D, D, 0, 0};
      }
      if ((rc = tcg::launch(g, st))) return rc;
    }
    {  // G2 = relu(G1 W4^T + b4)
      tcg::Gemm g{};
      g.A = Y + D; g.lda = 4 * D; g.ka = 4 * D - D;
      g.B = W4; g.ldb = 2 * D; g.kb = 2 * D;
      g.M = (int)T; g.N = D2; g.K = D; g.batch = 1; g.bn = pick_bn(D2);
      set_passes_b(g, 2 * D, D);
      g.bias = b4; g.act = tcg::ACT_RELU;
      g.out[0] = {G2, tcg::OUT_BF16_HILO, (long long)2 * D2, 0, D2, 0, 0, 0};
      if ((rc = tcg::launch(g, st))) return rc;
    }
    {  // Opre = G2 W5^T over all tokens: signed bf16 copy (sign carrier) and |.| as hi|lo planes; pad columns come out as zeros
      tcg::Gemm g{};
      g.A = G2; g.lda = 2 * D2; g.ka = 2 * D2;
      g.B = W5; g.ldb = 2 * D2; g.kb = 2 * D2;
      g.M = (int)T; g.N = P; g.K = D2; g.batch = 1; g.bn = pick_bn(P);
      set_passes_b(g, D2, D2);
      g.act = tcg::ACT_NONE;
      g.out[0] = {OS, tcg::OUT_BF16, (long long)Pp, 0, 0, Pp, 0, 0};
      if (!occ_only) g.out[1] = {OA, tcg::OUT_BF16_HILO, (long long)2 * Pp, 0, Pp, Pp, 1, 0};
      if ((rc = tcg::launch(g, st))) return rc;
    }
    if (occ_only) {
      dim3 grid(ceil_div(S, 32), ceil_div(Pp, 32), nb);
      gopre_from_gocc_kernel<<<grid, 256, 0, st>>>(gOcc + (size_t)n0 * P * S, OS, P, Pp, S, GO);
      PASN_LAUNCH_CHECK();
      count_launch();
    } else {
    {  // F = H1 W2^T + b2
      tcg::Gemm g{};
      g.A = Y; g.lda = 4 * D; g.ka = 4 * D;
      g.B = W2; g.ldb = 2 * D; g.kb = 2 * D;
      g.M = (int)T; g.N = D; g.K = D; g.batch = 1; g.bn = D >= 256 ? 256 : 128;
      set_passes_b(g, 2 * D, D);
      g.bias = b2;
      g.out[0] = {F, tcg::OUT_BF16_HILO, (long long)2 * D, 0, D, 0, 0, 0};
      if ((rc = tcg::launch(g, st))) return rc;
    }
    {  // FE[n] = O[n]^T F[n]   (K = S; both operands token-major)
      tcg::Gemm g{};
      g.A = OA; g.lda = 2 * Pp; g.a_bs = (long long)S * 2 * Pp; g.a_batched = 1; g.ka = 2 * Pp; g.a_mn_major = 1; g.a_rows = S;
      g.B = F; g.ldb = 2 * D; g.b_bs = (long long)S * 2 * D; g.b_batched = 1; g.kb = 2 * D; g.b_mn_major = 1; g.b_rows = S;
      g.M = P; g.N = D; g.K = S; g.batch = nb; g.bn = D >= 256 ? 256 : 128;
      set_passes_b(g, Pp, D);
      g.out[0] = {FE, tcg::OUT_F32, (long long)D, (long long)P * D, 0, 0, 0, 0};
      if ((rc = tcg::launch(g, st))) return rc;
    }
    // ================= prototype stage
    {
      const long long rows = (long long)nb * P;
      long long blocks = (rows + 7) / 8;
      if (blocks > 148 * 16) blocks = 148 * 16;
      proto_bwd_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>(FE, w.prototypes, w.last_layer, gLogits ? gLogits + (size_t)n0 * d.K : nullptr,
                                                              gSim ? gSim + (size_t)n0 * P : nullptr, rows, P, D, d.K, GFE, RS);
      PASN_LAUNCH_CHECK();
      count_launch();
      proto_bwd_reduce_kernel<<<dim3(P, nb >= 64 ? 16 : 1), 256, 0, st>>>(FE, w.prototypes, gLogits ? gLogits + (size_t)n0 * d.K : nullptr, RS, nb, P, D, d.K,
                                                 gr.prototypes, gr.last_layer);
      PASN_LAUNCH_CHECK();
      count_launch();
    }
    // ================= pooling backward
    {  // gOpre[n][s][p] = ((F[n] gFE[n]^T)[s][p] + gOcc[n][p][s]) * sign(Opre[n][s][p])
      tcg::Gemm g{};
      g.A = F; g.lda = 2 * D; g.a_bs = (long long)S * 2 * D; g.a_batched = 1; g.ka = 2 * D;
      g.B = GFE; g.ldb = 2 * D; g.b_bs = (long long)P * 2 * D; g.b_batched = 1; g.kb = 2 * D;
      g.M = S; g.N = P; g.K = D; g.batch = nb; g.bn = pick_bn(P);
      set_passes_b(g, D, D);
      if (gOcc) g.addin = {gOcc + (size_t)n0 * P * S, 1, (long long)P * S, (long long)S};
      g.signin = {OS, (long long)Pp, (long long)S * Pp, 0};
      g.out[0] = {GO, tcg::OUT_BF16_HILO, (long long)2 * Pp, (long long)S * 2 * Pp, Pp, Pp, 0, 0};
      if ((rc = tcg::launch(g, st))) return rc;
    }
    {  // gF[n][s][d] = sum_p O[n][s][p] gFE[n][p][d]
      tcg::Gemm g{};
      g.A = OA; g.lda = 2 * Pp; g.a_bs = (long long)S * 2 * Pp; g.a_batched = 1; g.ka = 2 * Pp;
      g.B = GFE; g.ldb = 2 * D; g.b_bs = (long long)P * 2 * D; g.b_batched = 1; g.kb = 2 * D; g.b_mn_major = 1; g.b_rows = P;
      g.M = S; g.N = D; g.K = P; g.batch = nb; g.bn = D >= 256 ? 256 : 128;
      set_passes_b(g, Pp, D);
      g.out[0] = {GF, tcg::OUT_BF16_HILO, (long long)2 * D, (long long)S * 2 * D, D, 0, 0, 0};
      if ((rc = tcg::launch(g, st))) return rc;
    }
    // ================= add-on branch
    if ((rc = wgrad(GF, 2 * D, D, D, Y, 4 * D, 2 * D, true, D, T, gr.addon_w2, D, nullptr))) return rc;     // gW2 += gF^T H1
    if ((rc = colsum(GF, T, 2 * D, D, D, gr.addon_b2, D, nullptr))) return rc;
    {  // gH1 = (gF W2) masked by H1 > 0   -> columns [0, D) of the [gH1 | gG1] planes
      tcg::Gemm g{};
      g.A = GF; g.lda = 2 * D; g.ka = 2 * D;
      g.B = W2; g.ldb = 2 * D; g.kb = 2 * D; g.b_mn_major = 1; g.b_rows = D;
      g.M = (int)T; g.N = D; g.K = D; g.batch = 1; g.bn = D >= 256 ? 256 : 128;
      set_passes_b(g, D, D);
      g.mask = {Y, (long long)4 * D, 0, 0};
      g.out[0] = {GY, tcg::OUT_BF16_HILO, (long long)4 * D, 0, 2 * D, 0, 0, 0};
      if ((rc = tcg::launch(g, st))) return rc;
    }
    }   // !occ_only
    // ================= occurrence branch
    if ((rc = wgrad(GO, 2 * Pp, Pp, P, G2, 2 * D2, D2, true, D2, T, gr.occ_w3, P, nullptr))) return rc;      // gW5 += gOpre^T G2
    {  // gG2 = (gOpre W5) masked by G2 > 0
      tcg::Gemm g{};
      g.A = GO; g.lda = 2 * Pp; g.ka = 2 * Pp;
      g.B = W5; g.ldb = 2 * D2; g.kb = 2 * D2; g.b_mn_major = 1; g.b_rows = P;
      g.M = (int)T; g.N = D2; g.K = P; g.batch = 1; g.bn = pick_bn(D2);
      set_passes_b(g, Pp, D2);
      g.mask = {G2, (long long)2 * D2, 0, 0};
      g.out[0] = {GG2, tcg::OUT_BF16_HILO, (long long)2 * D2, 0, D2, 0, 0, 0};
      if ((rc = tcg::launch(g, st))) return rc;
    }
    if ((rc = wgrad(GG2, 2 * D2, D2, D2, Y + D, 4 * D, 2 * D, true, D, T, gr.occ_w2, D2, nullptr))) return rc;   // gW4 += gG2^T G1
    if ((rc = colsum(GG2, T, 2 * D2, D2, D2, gr.occ_b2, D2, nullptr))) return rc;
    {  // gG1 = (gG2 W4) masked by G1 > 0   -> columns [D, 2D) of the [gH1 | gG1] planes
      tcg::Gemm g{};
      g.A = GG2; g.lda = 2 * D2; g.ka = 2 * D2;
      g.B = W4; g.ldb = 2 * D; g.kb = 2 * D; g.b_mn_major = 1; g.b_rows = D2;
      g.M = (int)T; g.N = D; g.K = D2; g.batch = 1; g.bn = D >= 256 ? 256 : 128;
      set_passes_b(g, D2, D);
      g.mask = {Y + D, (long long)4 * D, 0, 0};
      g.out[0] = {GY + D, tcg::OUT_BF16_HILO, (long long)4 * D, 0, 2 * D, D, 0, 0};
      if ((rc = tcg::launch(g, st))) return rc;
    }
    // ================= first layer: g[W1; W3] += [gH1 | gG1]^T X, biases, feature-map gradient
    if (occ_only) {
      if ((rc = wgrad(GY + D, 4 * D, 2 * D, D, xt, ldx, C, x_lo, C, T, gr.occ_w1, D, nullptr))) return rc;
      if ((rc = colsum(GY + D, T, 4 * D, 2 * D, D, gr.occ_b1, D, nullptr))) return rc;
    } else {
      if ((rc = wgrad(GY, 4 * D, 2 * D, 2 * D, xt, ldx, C, x_lo, C, T, gr.addon_w1, D, gr.occ_w1))) return rc;
      if ((rc = colsum(GY, T, 4 * D, 2 * D, 2 * D, gr.addon_b1, D, gr.occ_b1))) return rc;
    }
    if (gX) {   // gX[n][c][s] = sum_o [gH1|gG1][n,s][o] [W1;W3][o][c]
      tcg::Gemm g{};
      g.A = GY; g.lda = 4 * D; g.ka = 4 * D;
      g.B = W13; g.ldb = 2 * C; g.kb = 2 * C; g.b_mn_major = 1; g.b_rows = 2 * D;
      g.M = (int)T; g.N = C; g.K = 2 * D; g.batch = 1; g.bn = C >= 256 ? 256 : (C >= 128 ? 128 : 64);
      set_passes_b(g, 2 * D, C);
      if (occ_only) {   // the G1 half alone: gG1 [W3]
        g.A = GY + D; g.ka = 4 * D - D; g.B = W13 + (size_t)D * 2 * C; g.b_rows = D; g.K = D;
      }
      g.out[0] = {gX + (size_t)n0 * C * S, tcg::OUT_F32, (long long)S, (long long)C * S, 0, 0, 0, S};
      if ((rc = tcg::launch(g, st))) return rc;
    }
  }
  return PASN_OK;
}

}  // namespace pasn
