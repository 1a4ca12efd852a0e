// Generic prototype-head path: CUDA-core FFMA kernels, fp32 accumulate, any shape / dtype / layout.
// This is the fp32 correctness mode (1e-5 parity; TF32/bf16 tensor cores would not meet it) and the
// path for shapes the fused tcgen05 kernel does not cover.  Op order follows the reference exactly:
//   add-on  conv->ReLU->conv              src/models/Video_XProtoNet.py:27-39, :85
//   occ     conv->ReLU->conv->ReLU->conv->abs   :42-62, :106-109
//   pooling sum_s occ[p,s] * fmap[d,s]    :87
//   cosine / (.+1)/2 / logits             :90-96   (proto_stage.cu)
//
// Backward of the head (SURVEY.md section 8(f) row 2): gradients of
//     logits, similarity, occurrence_map  =  head(feature map; W1,b1,W2,b2,W3,b3,W4,b4,W5, prototypes, last_layer)
// with respect to the feature map and every parameter, so that training (reference: src/agents/XProtoNet_Base.py:397,
// src/agents/Video_XProtoNet_e2e.py:138 call loss.backward() through Video_XProtoNet.forward, src/models/Video_XProtoNet.py:82-98)
// can run through this library instead of a PyTorch composite.
//
// First correct path, like the forward above: CUDA-core FFMA GEMMs, fp32 throughout, forward intermediates
// recomputed per chunk of clips (nothing is saved by the forward).  Sub-gradients follow PyTorch: relu'(0) = 0,
// d|x|/dx at 0 = 0, CosineSimilarity clamps each norm at eps = 1e-8 (a clamped norm is a constant).
//   H1 = relu(W1 x + b1), F = W2 H1 + b2, G1 = relu(W3 x + b3), G2 = relu(W4 G1 + b4), Opre = W5 G2, O = |Opre|
//   FE[p,:] = sum_s O[p,s] F[:,s];  cos = <FE/nf, v/nv>;  sim = (cos+1)/2;  logits = sim Wl^T
// push_forward's extra outputs, features_extracted = FE and distance = 1 - sim, pass their gradients in at gFE and gsim.
// bf16 feature maps are read exactly (converted to fp32); weights are used unrounded: this is the gradient of the fp32
// formulation, which is also what the reference's autograd computes.
#include "common.cuh"

namespace pasn {

namespace {

enum { ACT_NONE = 0, ACT_RELU = 1, ACT_ABS = 2 };

struct GemmArgs {
  const void* A; const void* B; const float* bias;
  float* C;                // optional when C_bf16 is given (and nothing accumulates)
  __nv_bfloat16* C_bf16;   // optional bf16 copy of the result
  float* C_abs;            // optional |result| copy
  const float* mask;       // optional, same indexing as C: result zeroed where mask <= 0
  int M, N, K;
  long long a_sb, a_sm, a_sk;  // element strides: batch, row(m), k
  long long b_sb, b_sk, b_sn;
  long long c_sb, c_sm, c_sn;
  int nbatch;
  int act;
  int round_a_bf16;   // round A (weights) to bf16 on load
  int round_bias_bf16;
  int accumulate;     // C += result
  int reduce_batch;   // sum the products of all `nbatch` batches into one C (weight gradients)
};

constexpr int BM = 64, BN = 64, BK = 16;

// C[b][m][n] = epilogue(sum_k A[b][m][k] * B[b][k][n]); 256 threads, 4x4 outputs per thread.  Epilogue, in this order:
// + bias[m] (optionally bf16-rounded), act, mask, += C (accumulate), store C, C_bf16, C_abs.
// ROUND_A = g.round_a_bf16, as a template flag: read at run time it cost the loop its batching of the global loads (48
// registers instead of 64) and the backward GEMMs 1.8x their time (B200, 1000 W).  The per-batch output pointers are formed
// once, before the loop, so that ptxas emits global (LDG / STG) rather than generic accesses for them.
template <typename TA, typename TB, bool ROUND_A>
__global__ void __launch_bounds__(256) gemm_kernel(GemmArgs g) {
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Bs[BK][BN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int b_begin = g.reduce_batch ? 0 : blockIdx.z, b_end = g.reduce_batch ? g.nbatch : blockIdx.z + 1;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const bool a_k_contig = (g.a_sk == 1);
  const bool b_n_contig = (g.b_sn == 1);

  for (int b = b_begin; b < b_end; ++b) {
    const TA* A = reinterpret_cast<const TA*>(g.A) + (long long)b * g.a_sb;
    const TB* B = reinterpret_cast<const TB*>(g.B) + (long long)b * g.b_sb;
    for (int k0 = 0; k0 < g.K; k0 += BK) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int m, k;
        if (a_k_contig) { k = tid & 15; m = (tid >> 4) + 16 * i; }
        else            { m = tid & 63; k = (tid >> 6) + 4 * i; }
        float v = 0.f;
        if (m0 + m < g.M && k0 + k < g.K) {
          v = to_f32<TA>(A[(long long)(m0 + m) * g.a_sm + (long long)(k0 + k) * g.a_sk]);
          if (ROUND_A) v = round_bf16(v);
        }
        As[k][m] = v;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int n, k;
        if (b_n_contig) { n = tid & 63; k = (tid >> 6) + 4 * i; }
        else            { k = tid & 15; n = (tid >> 4) + 16 * i; }
        float v = 0.f;
        if (n0 + n < g.N && k0 + k < g.K)
          v = to_f32<TB>(B[(long long)(k0 + k) * g.b_sk + (long long)(n0 + n) * g.b_sn]);
        Bs[k][n] = v;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < BK; ++kk) {
        const float4 a4 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
        const float4 b4 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
        const float a[4] = {a4.x, a4.y, a4.z, a4.w};
        const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
      }
      __syncthreads();
    }
  }

  const long long cb = g.reduce_batch ? 0 : (long long)blockIdx.z * g.c_sb;
  float* const C = g.C ? g.C + cb : nullptr;
  __nv_bfloat16* const C_bf16 = g.C_bf16 ? g.C_bf16 + cb : nullptr;
  float* const C_abs = g.C_abs ? g.C_abs + cb : nullptr;
  const float* const mask = g.mask ? g.mask + cb : nullptr;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= g.M) continue;
    float bv = 0.f;
    if (g.bias) { bv = g.bias[m]; if (g.round_bias_bf16) bv = round_bf16(bv); }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= g.N) continue;
      const long long off = (long long)m * g.c_sm + (long long)n * g.c_sn;
      float v = acc[i][j] + bv;
      if (g.act == ACT_RELU) v = fmaxf(v, 0.f);
      else if (g.act == ACT_ABS) v = fabsf(v);
      if (mask && !(mask[off] > 0.f)) v = 0.f;
      if (g.accumulate) v += C[off];
      if (C) C[off] = v;
      if (C_bf16) C_bf16[off] = __float2bfloat16_rn(v);
      if (C_abs) C_abs[off] = fabsf(v);
    }
  }
}

// A is fp32 (weights, gradients, intermediates); B is fp32 or, when b_bf16, a bf16 feature map
int launch_gemm(const GemmArgs& g, bool b_bf16, cudaStream_t st) {
  if (g.nbatch <= 0 || g.M <= 0 || g.N <= 0) return PASN_OK;
  dim3 grid(ceil_div(g.N, BN), ceil_div(g.M, BM), g.reduce_batch ? 1 : g.nbatch);
  if (b_bf16) {
    if (g.round_a_bf16) gemm_kernel<float, __nv_bfloat16, true><<<grid, 256, 0, st>>>(g);
    else gemm_kernel<float, __nv_bfloat16, false><<<grid, 256, 0, st>>>(g);
  } else {
    if (g.round_a_bf16) gemm_kernel<float, float, true><<<grid, 256, 0, st>>>(g);
    else gemm_kernel<float, float, false><<<grid, 256, 0, st>>>(g);
  }
  PASN_LAUNCH_CHECK();
  count_launch();
  return PASN_OK;
}

// conv1x1: Y[n][o][s] = act(W[o][:] . X[n][:][s] + b[o]); X is either the user's feature map (dtype/layout from dims)
// or an fp32 NCS intermediate.  round_bf16: weights and bias rounded to bf16 (the forward's bf16 mode).
int conv1x1(const void* X, bool x_is_input, const pasn_dims& d, int nb, const float* W, const float* bias, int O, int Cin,
            float* Y, __nv_bfloat16* Y_bf16, float* Y_abs, int act, bool round_bf16, cudaStream_t st) {
  GemmArgs g{};
  g.A = W; g.B = X; g.bias = bias; g.C = Y; g.C_bf16 = Y_bf16; g.C_abs = Y_abs;
  g.M = O; g.N = d.S; g.K = Cin; g.nbatch = nb;
  g.a_sb = 0; g.a_sm = Cin; g.a_sk = 1;
  g.b_sb = (long long)Cin * d.S;
  if (x_is_input && d.layout == PASN_LAYOUT_NSC) { g.b_sk = 1; g.b_sn = Cin; }
  else { g.b_sk = d.S; g.b_sn = 1; }
  g.c_sb = (long long)O * d.S; g.c_sm = d.S; g.c_sn = 1;
  g.act = act;
  g.round_a_bf16 = g.round_bias_bf16 = round_bf16;
  return launch_gemm(g, x_is_input && d.dtype == PASN_BF16, st);
}

// FE[b][p][d] = sum_s O[b][p][s] F[b][d][s]
int pool(const float* O, const float* F, float* FE, const pasn_dims& d, int nb, cudaStream_t st) {
  GemmArgs g{};
  g.A = O; g.B = F; g.C = FE;
  g.M = d.P; g.N = d.D; g.K = d.S; g.nbatch = nb;
  g.a_sb = (long long)d.P * d.S; g.a_sm = d.S; g.a_sk = 1;
  g.b_sb = (long long)d.D * d.S; g.b_sk = 1; g.b_sn = d.S;
  g.c_sb = (long long)d.P * d.D; g.c_sm = d.D; g.c_sn = 1;
  return launch_gemm(g, false, st);
}

// clips per chunk when a clip needs per_clip bytes of scratch and the chunk may take cap bytes (at most kMaxChunkClips:
// launch_gemm puts the clip index in gridDim.z)
int chunk_clips(const pasn_dims& d, size_t per_clip, size_t cap) {
  long long c = (long long)(cap / (per_clip ? per_clip : 1));
  if (c > kMaxChunkClips) c = kMaxChunkClips;
  if (c < 1) c = 1;
  if (c > d.N) c = d.N > 0 ? d.N : 1;
  return (int)c;
}

// per-clip workspace of the forward (fp32): H [D,S] | F [D,S] | G2 [D/2,S] | O [P,S] | FE [P,D]; chunks bounded to ~256 MB
size_t fwd_per_clip(const pasn_dims& d) {
  return ((size_t)2 * d.D * d.S + (size_t)(d.D / 2) * d.S + (size_t)d.P * d.S + (size_t)d.P * d.D) * 4;
}
int fwd_chunk(const pasn_dims& d) { return chunk_clips(d, fwd_per_clip(d), (size_t)256 << 20); }

}  // namespace

size_t generic_workspace_bytes(const pasn_dims& d) { return align_up(fwd_per_clip(d) * fwd_chunk(d), 256) + 256; }

int generic_head_forward(const void* feat, const pasn_weights& w, const pasn_dims& d, float* logits, float* sim,
                         void* occ, float* feats, float* dist, const pasn_push_args* push, void* ws, size_t ws_bytes,
                         cudaStream_t st) {
  if (d.dtype == PASN_F16) return PASN_ERR_UNSUPPORTED;   // the CUDA-core path is the fp32 / bf16 correctness path
  if (ws_bytes < generic_workspace_bytes(d)) return PASN_ERR_WORKSPACE;
  const int nb_max = fwd_chunk(d);
  const int D2 = d.D / 2;
  const bool rnd = d.dtype == PASN_BF16;
  float* H = reinterpret_cast<float*>(ws);
  float* F = H + (size_t)nb_max * d.D * d.S;
  float* G2 = F + (size_t)nb_max * d.D * d.S;
  float* O = G2 + (size_t)nb_max * D2 * d.S;
  float* FE = O + (size_t)nb_max * d.P * d.S;
  const size_t elt = dtype_bytes(d.dtype);
  main_kernel_begin(st);  // generic path: the "dominant kernel" is the whole GEMM chain
  for (int n0 = 0; n0 < d.N; n0 += nb_max) {
    const int nb = (d.N - n0 < nb_max) ? d.N - n0 : nb_max;
    const char* x = reinterpret_cast<const char*>(feat) + (size_t)n0 * d.C * d.S * elt;
    int rc;
    // add-on branch
    if ((rc = conv1x1(x, true, d, nb, w.addon_w1, w.addon_b1, d.D, d.C, H, nullptr, nullptr, ACT_RELU, rnd, st))) return rc;
    if ((rc = conv1x1(H, false, d, nb, w.addon_w2, w.addon_b2, d.D, d.D, F, nullptr, nullptr, ACT_NONE, rnd, st))) return rc;
    // occurrence branch (H reused for the first hidden layer)
    if ((rc = conv1x1(x, true, d, nb, w.occ_w1, w.occ_b1, d.D, d.C, H, nullptr, nullptr, ACT_RELU, rnd, st))) return rc;
    if ((rc = conv1x1(H, false, d, nb, w.occ_w2, w.occ_b2, D2, d.D, G2, nullptr, nullptr, ACT_RELU, rnd, st))) return rc;
    float* o32 = O;
    __nv_bfloat16* o16 = nullptr;
    if (occ) {
      if (d.dtype == PASN_F32) o32 = reinterpret_cast<float*>(occ) + (size_t)n0 * d.P * d.S;
      else o16 = reinterpret_cast<__nv_bfloat16*>(occ) + (size_t)n0 * d.P * d.S;
    }
    if ((rc = conv1x1(G2, false, d, nb, w.occ_w3, nullptr, d.P, D2, o32, o16, nullptr, ACT_ABS, rnd, st))) return rc;
    float* fe = feats ? feats + (size_t)n0 * d.P * d.D : FE;
    if ((rc = pool(o32, F, fe, d, nb, st))) return rc;
    pasn_push_args pa;
    const pasn_push_args* pp = nullptr;
    if (push) { pa = *push; pa.labels += n0; pa.global_offset += n0; pp = &pa; }
    if ((rc = launch_proto_stage(fe, w.prototypes, w.last_layer, nb, d.P, d.D, d.K, logits + (size_t)n0 * d.K,
                                 sim + (size_t)n0 * d.P, dist ? dist + (size_t)n0 * d.P : nullptr, pp, st)))
      return rc;
  }
  main_kernel_end(st);
  return PASN_OK;
}

int generic_occurrence_only(const void* feat, const pasn_weights& w, const pasn_dims& d, void* occ, void* ws,
                            size_t ws_bytes, cudaStream_t st) {
  if (d.dtype == PASN_F16) return PASN_ERR_UNSUPPORTED;   // the CUDA-core path is the fp32 / bf16 correctness path
  if (ws_bytes < generic_workspace_bytes(d)) return PASN_ERR_WORKSPACE;
  const int nb_max = fwd_chunk(d);
  const int D2 = d.D / 2;
  const bool rnd = d.dtype == PASN_BF16;
  float* H = reinterpret_cast<float*>(ws);
  float* G2 = H + (size_t)2 * nb_max * d.D * d.S;
  const size_t elt = dtype_bytes(d.dtype);
  for (int n0 = 0; n0 < d.N; n0 += nb_max) {
    const int nb = (d.N - n0 < nb_max) ? d.N - n0 : nb_max;
    const char* x = reinterpret_cast<const char*>(feat) + (size_t)n0 * d.C * d.S * elt;
    int rc;
    if ((rc = conv1x1(x, true, d, nb, w.occ_w1, w.occ_b1, d.D, d.C, H, nullptr, nullptr, ACT_RELU, rnd, st))) return rc;
    if ((rc = conv1x1(H, false, d, nb, w.occ_w2, w.occ_b2, D2, d.D, G2, nullptr, nullptr, ACT_RELU, rnd, st))) return rc;
    float* o32 = nullptr;
    __nv_bfloat16* o16 = nullptr;
    if (d.dtype == PASN_F32) o32 = reinterpret_cast<float*>(occ) + (size_t)n0 * d.P * d.S;
    else o16 = reinterpret_cast<__nv_bfloat16*>(occ) + (size_t)n0 * d.P * d.S;
    if ((rc = conv1x1(G2, false, d, nb, w.occ_w3, nullptr, d.P, D2, o32, o16, nullptr, ACT_ABS, rnd, st))) return rc;
  }
  return PASN_OK;
}

// =================================================================================================================
// Backward (see the top of the file for the math)
// =================================================================================================================
namespace {

// gb[m] += sum over (batch, s) of G[b][m][s]
__global__ void __launch_bounds__(256) rowsum_kernel(const float* __restrict__ G, float* __restrict__ gb, int nb, int M, int S) {
  __shared__ float red[8];
  const int m = blockIdx.x;
  float a = 0.f;
  const long long total = (long long)nb * S;
  for (long long i = threadIdx.x; i < total; i += 256) {
    const long long b = i / S, s = i - b * S;
    a += G[(b * M + m) * S + s];
  }
  a = warp_sum(a);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i];
    gb[m] += t;
  }
}

// gOpre = (gO + gOcc) * sign(Opre), in place in gO
__global__ void sign_kernel(float* __restrict__ gO, const float* __restrict__ gOcc, const float* __restrict__ Opre, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float v = gO[i] + (gOcc ? gOcc[i] : 0.f);
  const float o = Opre[i];
  gO[i] = o > 0.f ? v : (o < 0.f ? -v : 0.f);
}

// Cosine / similarity / logits backward.  One block per prototype p, looping over the clips of the chunk:
//   gsim = gSim[n,p] - gDist[n,p] + sum_k gLogits[n,k] Wl[k,p];  gcos = gsim / 2
//   gFE[n,p,:] = (cosine's gradient) + gFEin[n,p,:], gV[p,:] += ..., gWl[k,p] += gLogits[n,k] * sim[n,p]  (gV, gWl may be
//   NULL: not wanted)
__global__ void __launch_bounds__(256) proto_bwd_kernel(const float* __restrict__ FE, const float* __restrict__ protos,
                                                        const float* __restrict__ last_layer, const float* __restrict__ gLogits,
                                                        const float* __restrict__ gSim, const float* __restrict__ gDist,
                                                        const float* __restrict__ gFEin, int nb, int P, int D, int K,
                                                        float* __restrict__ gFE, float* __restrict__ gV, float* __restrict__ gWl) {
  __shared__ float red[3][8];
  __shared__ float bc[3];
  const int p = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* v = protos + (size_t)p * D;
  constexpr float eps = 1e-8f;
  auto block_sum3 = [&](float a, float b, float c) {
    a = warp_sum(a); b = warp_sum(b); c = warp_sum(c);
    __syncthreads();
    if (lane == 0) { red[0][warp] = a; red[1][warp] = b; red[2][warp] = c; }
    __syncthreads();
    if (tid < 3) {
      float t = 0.f;
      for (int i = 0; i < 8; ++i) t += red[tid][i];
      bc[tid] = t;
    }
    __syncthreads();
  };
  float vv_part = 0.f;
  for (int d = tid; d < D; d += 256) vv_part = fmaf(v[d], v[d], vv_part);
  block_sum3(vv_part, 0.f, 0.f);
  const float vnorm = sqrtf(bc[0]);
  const float nv = fmaxf(vnorm, eps);
  const bool v_clamped = !(vnorm > eps);
  for (int n = 0; n < nb; ++n) {
    const float* f = FE + ((size_t)n * P + p) * D;
    float ff = 0.f, dot = 0.f;
    for (int d = tid; d < D; d += 256) {
      ff = fmaf(f[d], f[d], ff);
      dot = fmaf(f[d], v[d], dot);
    }
    block_sum3(ff, dot, 0.f);
    const float fnorm = sqrtf(bc[0]);
    const float nf = fmaxf(fnorm, eps);
    const bool f_clamped = !(fnorm > eps);
    const float cosv = bc[1] / (nf * nv);
    const float sim = (cosv + 1.0f) * 0.5f;
    float gs = gSim ? gSim[(size_t)n * P + p] : 0.f;
    if (gDist) gs -= gDist[(size_t)n * P + p];
    if (gLogits)
      for (int k = 0; k < K; ++k) gs = fmaf(gLogits[(size_t)n * K + k], last_layer[(size_t)k * P + p], gs);
    const float gcos = 0.5f * gs;
    // the block owns column p of gWl: no other block writes it, so each clip adds its terms in place (any K)
    if (gLogits && gWl)
      for (int k = tid; k < K; k += 256) gWl[(size_t)k * P + p] = fmaf(gLogits[(size_t)n * K + k], sim, gWl[(size_t)k * P + p]);
    // cos = <f, v> / (nf nv); nf, nv constants when clamped
    const float inv = 1.0f / (nf * nv);
    const float cf = f_clamped ? 0.f : cosv / (nf * nf);
    const float cv = v_clamped ? 0.f : cosv / (nv * nv);
    const size_t row = ((size_t)n * P + p) * D;
    // roundings spelled out: the compiler keeps a loop copy per `gV` case and would contract each its own way, so gFE
    // would depend on whether gV is wanted
    for (int d = tid; d < D; d += 256) {
      float gf = __fmul_rn(gcos, fmaf(v[d], inv, -__fmul_rn(cf, f[d])));
      if (gFEin) gf = __fadd_rn(gf, gFEin[row + d]);
      gFE[row + d] = gf;
      if (gV) gV[(size_t)p * D + d] = fmaf(gcos, fmaf(f[d], inv, -__fmul_rn(cv, v[d])), gV[(size_t)p * D + d]);
    }
  }
}

// per-clip workspace of the backward (fp32); chunks bounded to ~384 MB
size_t bwd_per_clip(const pasn_dims& d) {
  const size_t DS = (size_t)d.D * d.S, D2S = (size_t)(d.D / 2) * d.S, PS = (size_t)d.P * d.S, PD = (size_t)d.P * d.D;
  return (3 * DS + D2S + 2 * PS + 2 * PD + PS + 2 * DS + D2S + DS) * 4;   // H1 F G1 | G2 | Opre O | FE gFE | gO | gF gH1 | gG2 | gG1
}
int bwd_chunk(const pasn_dims& d) { return chunk_clips(d, bwd_per_clip(d), (size_t)384 << 20); }

}  // namespace

size_t generic_backward_workspace_bytes(const pasn_dims& d) { return align_up(bwd_per_clip(d) * bwd_chunk(d), 256) + 256; }

int generic_head_backward(const void* feat, const pasn_weights& w, const pasn_dims& d, const pasn_upstream& up,
                          const pasn_grads& g, float* gX, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (ws_bytes < generic_backward_workspace_bytes(d)) return PASN_ERR_WORKSPACE;
  const float *gLogits = up.grad_logits, *gSim = up.grad_similarity, *gDist = up.grad_distance, *gOcc = up.grad_occurrence,
              *gFEin = up.grad_features;
  const int nbm = bwd_chunk(d);
  const int D = d.D, D2 = d.D / 2, S = d.S, P = d.P, C = d.C, K = d.K;
  const size_t DS = (size_t)D * S, D2S = (size_t)D2 * S, PS = (size_t)P * S, PD = (size_t)P * D;
  float* q = reinterpret_cast<float*>(ws);
  auto take = [&](size_t per_clip) { float* r = q; q += per_clip * nbm; return r; };
  float *H1 = take(DS), *F = take(DS), *G1 = take(DS), *G2 = take(D2S), *Opre = take(PS), *O = take(PS), *FE = take(PD),
        *gFE = take(PD), *gO = take(PS), *gF = take(DS), *gH1 = take(DS), *gG2 = take(D2S), *gG1 = take(DS);
  const bool xbf = d.dtype == PASN_BF16;
  const size_t elt = dtype_bytes(d.dtype);
  // strides of the feature map seen as B[k = channel][n = voxel] per clip
  const long long x_sk = d.layout == PASN_LAYOUT_NSC ? 1 : S, x_sn = d.layout == PASN_LAYOUT_NSC ? C : 1;

  const BwdNeeds need = bwd_needs(g, gX);
  // gW[o][c] += sum_b sum_s gY[b][o][s] * X[b][c][s]  (gW NULL: not wanted)
  auto wgrad = [&](const float* gY, int O_, const void* X, bool x_is_input, int Cin, float* gW, int nb) -> int {
    if (!gW) return PASN_OK;
    GemmArgs a{};
    a.A = gY; a.B = X; a.C = gW; a.accumulate = 1; a.reduce_batch = 1; a.nbatch = nb;
    a.M = O_; a.N = Cin; a.K = S;
    a.a_sb = (long long)O_ * S; a.a_sm = S; a.a_sk = 1;
    a.b_sb = (long long)Cin * S;
    if (x_is_input) { a.b_sk = x_sn; a.b_sn = x_sk; } else { a.b_sk = 1; a.b_sn = S; }   // B[k = s][n = c]
    a.c_sb = 0; a.c_sm = Cin; a.c_sn = 1;
    return launch_gemm(a, x_is_input && xbf, st);
  };
  // gXin[b][c][s] (+)= sum_o W[o][c] gY[b][o][s], masked by relu output `mask` (same shape) when given
  auto dgrad = [&](const float* W, int O_, int Cin, const float* gY, float* gXin, const float* mask, int accumulate, int nb) -> int {
    GemmArgs a{};
    a.A = W; a.B = gY; a.C = gXin; a.mask = mask; a.accumulate = accumulate; a.nbatch = nb;
    a.M = Cin; a.N = S; a.K = O_;
    a.a_sb = 0; a.a_sm = 1; a.a_sk = Cin;            // A[m = c][k = o] = W[o][c]
    a.b_sb = (long long)O_ * S; a.b_sk = S; a.b_sn = 1;
    a.c_sb = (long long)Cin * S; a.c_sm = S; a.c_sn = 1;
    return launch_gemm(a, false, st);
  };
  auto rowsum = [&](const float* G, float* gb, int M, int nb) -> int {
    if (!gb) return PASN_OK;
    rowsum_kernel<<<M, 256, 0, st>>>(G, gb, nb, M, S);
    PASN_LAUNCH_CHECK();
    count_launch();
    return PASN_OK;
  };

  for (int n0 = 0; n0 < d.N; n0 += nbm) {
    const int nb = (d.N - n0 < nbm) ? d.N - n0 : nbm;
    const char* x = reinterpret_cast<const char*>(feat) + (size_t)n0 * C * S * elt;
    int rc;
    // ---- recompute the forward intermediates of this chunk (unrounded weights: the fp32 formulation)
    if ((rc = conv1x1(x, true, d, nb, w.addon_w1, w.addon_b1, D, C, H1, nullptr, nullptr, ACT_RELU, false, st))) return rc;
    if ((rc = conv1x1(H1, false, d, nb, w.addon_w2, w.addon_b2, D, D, F, nullptr, nullptr, ACT_NONE, false, st))) return rc;
    if ((rc = conv1x1(x, true, d, nb, w.occ_w1, w.occ_b1, D, C, G1, nullptr, nullptr, ACT_RELU, false, st))) return rc;
    if ((rc = conv1x1(G1, false, d, nb, w.occ_w2, w.occ_b2, D2, D, G2, nullptr, nullptr, ACT_RELU, false, st))) return rc;
    if ((rc = conv1x1(G2, false, d, nb, w.occ_w3, nullptr, P, D2, Opre, nullptr, O, ACT_NONE, false, st))) return rc;
    if ((rc = pool(O, F, FE, d, nb, st))) return rc;
    // ---- prototype stage backward
    proto_bwd_kernel<<<P, 256, 0, st>>>(FE, w.prototypes, w.last_layer, gLogits ? gLogits + (size_t)n0 * K : nullptr,
                                        gSim ? gSim + (size_t)n0 * P : nullptr, gDist ? gDist + (size_t)n0 * P : nullptr,
                                        gFEin ? gFEin + (size_t)n0 * PD : nullptr, nb, P, D, K, gFE, g.prototypes, g.last_layer);
    PASN_LAUNCH_CHECK();
    count_launch();
    if (need.gOpre) {  // gO[b][p][s] = sum_d gFE[b][p][d] F[b][d][s]
      GemmArgs a{};
      a.A = gFE; a.B = F; a.C = gO; a.nbatch = nb;
      a.M = P; a.N = S; a.K = D;
      a.a_sb = (long long)PD; a.a_sm = D; a.a_sk = 1;
      a.b_sb = (long long)DS; a.b_sk = S; a.b_sn = 1;
      a.c_sb = (long long)PS; a.c_sm = S; a.c_sn = 1;
      if ((rc = launch_gemm(a, false, st))) return rc;
    }
    if (need.gF) {  // gF[b][d][s] = sum_p gFE[b][p][d] O[b][p][s]
      GemmArgs a{};
      a.A = gFE; a.B = O; a.C = gF; a.nbatch = nb;
      a.M = D; a.N = S; a.K = P;
      a.a_sb = (long long)PD; a.a_sm = 1; a.a_sk = D;
      a.b_sb = (long long)PS; a.b_sk = S; a.b_sn = 1;
      a.c_sb = (long long)DS; a.c_sm = S; a.c_sn = 1;
      if ((rc = launch_gemm(a, false, st))) return rc;
    }
    if (need.gOpre) {
      const long long n = (long long)nb * PS;
      sign_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(gO, gOcc ? gOcc + (size_t)n0 * PS : nullptr, Opre, n);
      PASN_LAUNCH_CHECK();
      count_launch();
    }
    // ---- add-on branch: F = W2 H1 + b2, H1 = relu(W1 x + b1)
    if ((rc = wgrad(gF, D, H1, false, D, g.addon_w2, nb))) return rc;
    if ((rc = rowsum(gF, g.addon_b2, D, nb))) return rc;
    if (need.gH1 && (rc = dgrad(w.addon_w2, D, D, gF, gH1, H1, 0, nb))) return rc;
    if ((rc = wgrad(gH1, D, x, true, C, g.addon_w1, nb))) return rc;
    if ((rc = rowsum(gH1, g.addon_b1, D, nb))) return rc;
    // ---- occurrence branch: Opre = W5 G2, G2 = relu(W4 G1 + b4), G1 = relu(W3 x + b3)
    if ((rc = wgrad(gO, P, G2, false, D2, g.occ_w3, nb))) return rc;
    if (need.gG2 && (rc = dgrad(w.occ_w3, P, D2, gO, gG2, G2, 0, nb))) return rc;
    if ((rc = wgrad(gG2, D2, G1, false, D, g.occ_w2, nb))) return rc;
    if ((rc = rowsum(gG2, g.occ_b2, D2, nb))) return rc;
    if (need.gG1 && (rc = dgrad(w.occ_w2, D2, D, gG2, gG1, G1, 0, nb))) return rc;
    if ((rc = wgrad(gG1, D, x, true, C, g.occ_w1, nb))) return rc;
    if ((rc = rowsum(gG1, g.occ_b1, D, nb))) return rc;
    // ---- feature-map gradient (fp32, [N][C][S])
    if (gX) {
      float* gx = gX + (size_t)n0 * C * S;
      if ((rc = dgrad(w.addon_w1, D, C, gH1, gx, nullptr, 0, nb))) return rc;
      if ((rc = dgrad(w.occ_w1, D, C, gG1, gx, nullptr, 1, nb))) return rc;
    }
  }
  return PASN_OK;
}

int generic_last_layer_backward(const float* gL, const float* sim, int N, int P, int K, float* gWl, cudaStream_t st) {
  GemmArgs a{};
  a.A = gL; a.B = sim; a.C = gWl; a.accumulate = 1; a.nbatch = 1;
  a.M = K; a.N = P; a.K = N;
  a.a_sm = 1; a.a_sk = K;   // A[m = k][kk = n] = gL[n][k]
  a.b_sk = P; a.b_sn = 1;
  a.c_sm = P; a.c_sn = 1;
  return launch_gemm(a, false, st);
}

}  // namespace pasn
