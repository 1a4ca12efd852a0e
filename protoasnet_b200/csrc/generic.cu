// Generic prototype-head path: CUDA-core FFMA kernels, fp32 accumulate, any shape / dtype / layout.
// This is the fp32 correctness mode (1e-5 parity; TF32/bf16 tensor cores would not meet it) and the
// path for shapes the fused tcgen05 kernel does not cover.  Op order follows the reference exactly:
//   add-on  conv->ReLU->conv              src/models/Video_XProtoNet.py:27-39, :85
//   occ     conv->ReLU->conv->ReLU->conv->abs   :42-62, :106-109
//   pooling sum_s occ[p,s] * fmap[d,s]    :87
//   cosine / (.+1)/2 / logits             :90-96   (proto_stage.cu)
#include "common.cuh"

namespace pasn {

enum { ACT_NONE = 0, ACT_RELU = 1, ACT_ABS = 2 };

struct GemmArgs {
  const void* A; const void* B; const float* bias; float* C; __nv_bfloat16* C2;
  int M, N, K;
  long long a_sb, a_sm, a_sk;  // element strides: batch, row(m), k
  long long b_sb, b_sk, b_sn;
  long long c_sb, c_sm, c_sn;
  int act;
  int round_a_bf16;     // round A (weights) to bf16 on load
  int round_bias_bf16;
};

constexpr int BM = 64, BN = 64, BK = 16;

// C[b][m][n] = act(sum_k A[b][m][k] * B[b][k][n] + bias[m]); 256 threads, 4x4 outputs per thread.
template <typename TA, typename TB>
__global__ void __launch_bounds__(256) strided_gemm_kernel(GemmArgs g) {
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Bs[BK][BN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const long long b = blockIdx.z;
  const TA* A = reinterpret_cast<const TA*>(g.A) + b * g.a_sb;
  const TB* B = reinterpret_cast<const TB*>(g.B) + b * g.b_sb;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const bool a_k_contig = (g.a_sk == 1);
  const bool b_n_contig = (g.b_sn == 1);

  for (int k0 = 0; k0 < g.K; k0 += BK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int m, k;
      if (a_k_contig) { k = tid & 15; m = (tid >> 4) + 16 * i; }
      else            { m = tid & 63; k = (tid >> 6) + 4 * i; }
      float v = 0.f;
      if (m0 + m < g.M && k0 + k < g.K) {
        v = to_f32<TA>(A[(long long)(m0 + m) * g.a_sm + (long long)(k0 + k) * g.a_sk]);
        if (g.round_a_bf16) v = round_bf16(v);
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
      float4 a4 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      float4 b4 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      float a[4] = {a4.x, a4.y, a4.z, a4.w};
      float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }

  float* C = g.C ? g.C + b * g.c_sb : nullptr;
  __nv_bfloat16* C2 = g.C2 ? g.C2 + b * g.c_sb : nullptr;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int m = m0 + ty * 4 + i;
    if (m >= g.M) continue;
    float bv = 0.f;
    if (g.bias) { bv = g.bias[m]; if (g.round_bias_bf16) bv = round_bf16(bv); }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int n = n0 + tx * 4 + j;
      if (n >= g.N) continue;
      float v = acc[i][j] + bv;
      if (g.act == ACT_RELU) v = fmaxf(v, 0.f);
      else if (g.act == ACT_ABS) v = fabsf(v);
      long long off = (long long)m * g.c_sm + (long long)n * g.c_sn;
      if (C) C[off] = v;
      if (C2) C2[off] = __float2bfloat16_rn(v);
    }
  }
}

template <typename TA, typename TB>
static int launch_gemm(const GemmArgs& g, int batch, cudaStream_t st) {
  if (batch <= 0 || g.M <= 0 || g.N <= 0) return PASN_OK;
  dim3 grid(ceil_div(g.N, BN), ceil_div(g.M, BM), batch);
  strided_gemm_kernel<TA, TB><<<grid, 256, 0, st>>>(g);
  PASN_LAUNCH_CHECK();
  count_launch();
  return PASN_OK;
}

// conv1x1: Y[n][o][s] = act(W[o][:] . X[n][:][s] + b[o]); X is either the user's feature map (dtype/layout from dims)
// or an fp32 NCS intermediate.
static int conv1x1(const void* X, bool x_is_input, const pasn_dims& d, int nb, const float* W, const float* bias,
                   int O, int Cin, float* Y, __nv_bfloat16* Y2, int act, cudaStream_t st) {
  GemmArgs g{};
  g.A = W; g.B = X; g.bias = bias; g.C = Y; g.C2 = Y2;
  g.M = O; g.N = d.S; g.K = Cin;
  g.a_sb = 0; g.a_sm = Cin; g.a_sk = 1;
  g.b_sb = (long long)Cin * d.S;
  if (x_is_input && d.layout == PASN_LAYOUT_NSC) { g.b_sk = 1; g.b_sn = Cin; }
  else { g.b_sk = d.S; g.b_sn = 1; }
  g.c_sb = (long long)O * d.S; g.c_sm = d.S; g.c_sn = 1;
  g.act = act;
  g.round_a_bf16 = g.round_bias_bf16 = (d.dtype == PASN_BF16);
  if (x_is_input && d.dtype == PASN_BF16) return launch_gemm<float, __nv_bfloat16>(g, nb, st);
  return launch_gemm<float, float>(g, nb, st);
}

// per-chunk workspace layout (fp32): H [nb,D,S] | F [nb,D,S] | G2 [nb,D/2,S] | O [nb,P,S] | FE [nb,P,D]
static int chunk_clips(const pasn_dims& d) {
  // bound the scratch to ~256 MB
  size_t per_clip = ((size_t)2 * d.D * d.S + (size_t)(d.D / 2) * d.S + (size_t)d.P * d.S + (size_t)d.P * d.D) * 4;
  size_t cap = (size_t)256 << 20;
  long long c = (long long)(cap / (per_clip ? per_clip : 1));
  if (c < 1) c = 1;
  if (c > d.N) c = d.N > 0 ? d.N : 1;
  return (int)c;
}

size_t generic_workspace_bytes(const pasn_dims& d) {
  int nb = chunk_clips(d);
  size_t per_clip = ((size_t)2 * d.D * d.S + (size_t)(d.D / 2) * d.S + (size_t)d.P * d.S + (size_t)d.P * d.D) * 4;
  return align_up(per_clip * nb, 256) + 256;
}

int generic_head_forward(const void* feat, const pasn_weights& w, const pasn_dims& d, float* logits, float* sim,
                         void* occ, float* feats, float* dist, const pasn_push_args* push, void* ws, size_t ws_bytes,
                         cudaStream_t st) {
  if (d.dtype == PASN_F16) return PASN_ERR_UNSUPPORTED;   // the CUDA-core path is the fp32 / bf16 correctness path
  if (ws_bytes < generic_workspace_bytes(d)) return PASN_ERR_WORKSPACE;
  const int nb_max = chunk_clips(d);
  const int D2 = d.D / 2;
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
    if ((rc = conv1x1(x, true, d, nb, w.addon_w1, w.addon_b1, d.D, d.C, H, nullptr, ACT_RELU, st))) return rc;
    if ((rc = conv1x1(H, false, d, nb, w.addon_w2, w.addon_b2, d.D, d.D, F, nullptr, ACT_NONE, st))) return rc;
    // occurrence branch (H reused for the first hidden layer)
    if ((rc = conv1x1(x, true, d, nb, w.occ_w1, w.occ_b1, d.D, d.C, H, nullptr, ACT_RELU, st))) return rc;
    if ((rc = conv1x1(H, false, d, nb, w.occ_w2, w.occ_b2, D2, d.D, G2, nullptr, ACT_RELU, st))) return rc;
    float* o32 = O;
    __nv_bfloat16* o16 = nullptr;
    if (occ) {
      if (d.dtype == PASN_F32) o32 = reinterpret_cast<float*>(occ) + (size_t)n0 * d.P * d.S;
      else o16 = reinterpret_cast<__nv_bfloat16*>(occ) + (size_t)n0 * d.P * d.S;
    }
    if ((rc = conv1x1(G2, false, d, nb, w.occ_w3, nullptr, d.P, D2, o32, o16, ACT_ABS, st))) return rc;
    // pooling: FE[n][p][d] = sum_s O[n][p][s] * F[n][d][s]
    GemmArgs g{};
    float* fe = feats ? feats + (size_t)n0 * d.P * d.D : FE;
    g.A = o32; g.B = F; g.bias = nullptr; g.C = fe; g.C2 = nullptr;
    g.M = d.P; g.N = d.D; g.K = d.S;
    g.a_sb = (long long)d.P * d.S; g.a_sm = d.S; g.a_sk = 1;
    g.b_sb = (long long)d.D * d.S; g.b_sk = 1; g.b_sn = d.S;
    g.c_sb = (long long)d.P * d.D; g.c_sm = d.D; g.c_sn = 1;
    g.act = ACT_NONE;
    if ((rc = launch_gemm<float, float>(g, nb, st))) return rc;
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
  const int nb_max = chunk_clips(d);
  const int D2 = d.D / 2;
  float* H = reinterpret_cast<float*>(ws);
  float* G2 = H + (size_t)2 * nb_max * d.D * d.S;
  const size_t elt = dtype_bytes(d.dtype);
  for (int n0 = 0; n0 < d.N; n0 += nb_max) {
    const int nb = (d.N - n0 < nb_max) ? d.N - n0 : nb_max;
    const char* x = reinterpret_cast<const char*>(feat) + (size_t)n0 * d.C * d.S * elt;
    int rc;
    if ((rc = conv1x1(x, true, d, nb, w.occ_w1, w.occ_b1, d.D, d.C, H, nullptr, ACT_RELU, st))) return rc;
    if ((rc = conv1x1(H, false, d, nb, w.occ_w2, w.occ_b2, D2, d.D, G2, nullptr, ACT_RELU, st))) return rc;
    float* o32 = nullptr;
    __nv_bfloat16* o16 = nullptr;
    if (d.dtype == PASN_F32) o32 = reinterpret_cast<float*>(occ) + (size_t)n0 * d.P * d.S;
    else o16 = reinterpret_cast<__nv_bfloat16*>(occ) + (size_t)n0 * d.P * d.S;
    if ((rc = conv1x1(G2, false, d, nb, w.occ_w3, nullptr, d.P, D2, o32, o16, ACT_ABS, st))) return rc;
  }
  return PASN_OK;
}

}  // namespace pasn
