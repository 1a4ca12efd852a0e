// Backward of the prototype head (SURVEY.md section 8(f) row 2): gradients of
//     logits, similarity, occurrence_map  =  head(feature map; W1,b1,W2,b2,W3,b3,W4,b4,W5, prototypes, last_layer)
// with respect to the feature map and every parameter, so that training (reference: src/agents/XProtoNet_Base.py:397,
// src/agents/Video_XProtoNet_e2e.py:138 call loss.backward() through Video_XProtoNet.forward, src/models/Video_XProtoNet.py:82-98)
// can run through this library instead of a PyTorch composite.
//
// First correct path, like generic.cu for the forward: CUDA-core FFMA GEMMs, fp32 throughout, forward intermediates
// recomputed per chunk of clips (nothing is saved by the forward).  Sub-gradients follow PyTorch: relu'(0) = 0,
// d|x|/dx at 0 = 0, CosineSimilarity clamps each norm at eps = 1e-8 (a clamped norm is a constant).
//   H1 = relu(W1 x + b1), F = W2 H1 + b2, G1 = relu(W3 x + b3), G2 = relu(W4 G1 + b4), Opre = W5 G2, O = |Opre|
//   FE[p,:] = sum_s O[p,s] F[:,s];  cos = <FE/nf, v/nv>;  sim = (cos+1)/2;  logits = sim Wl^T
// bf16 feature maps are read exactly (converted to fp32); weights are used unrounded: this is the gradient of the fp32
// formulation, which is also what the reference's autograd computes.
#include "common.cuh"

namespace pasn {

namespace {

struct BGemm {
  const void* A; const void* B; float* C; const float* mask;   // mask: same indexing as C, result zeroed where mask <= 0
  int M, N, K;
  long long a_sb, a_sm, a_sk;
  long long b_sb, b_sk, b_sn;
  long long c_sb, c_sm, c_sn;
  int accumulate;     // C += result
  int reduce_batch;   // sum the products of all `nbatch` batches into one C (weight gradients)
  int nbatch;
  const float* bias;  // optional, per row m
  int act;            // 0 none, 1 relu, 2 keep pre-activation in C and |.| in C_abs
  float* C_abs;
};

constexpr int TM = 64, TN = 64, TK = 16;

template <typename TA, typename TB>
__global__ void __launch_bounds__(256) bgemm_kernel(BGemm g) {
  __shared__ __align__(16) float As[TK][TM + 4];
  __shared__ __align__(16) float Bs[TK][TN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
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
    for (int k0 = 0; k0 < g.K; k0 += TK) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int m, k;
        if (a_k_contig) { k = tid & 15; m = (tid >> 4) + 16 * i; }
        else            { m = tid & 63; k = (tid >> 6) + 4 * i; }
        float v = 0.f;
        if (m0 + m < g.M && k0 + k < g.K) v = to_f32<TA>(A[(long long)(m0 + m) * g.a_sm + (long long)(k0 + k) * g.a_sk]);
        As[k][m] = v;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int n, k;
        if (b_n_contig) { n = tid & 63; k = (tid >> 6) + 4 * i; }
        else            { k = tid & 15; n = (tid >> 4) + 16 * i; }
        float v = 0.f;
        if (n0 + n < g.N && k0 + k < g.K) v = to_f32<TB>(B[(long long)(k0 + k) * g.b_sk + (long long)(n0 + n) * g.b_sn]);
        Bs[k][n] = v;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < TK; ++kk) {
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
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= g.M) continue;
    const float bv = g.bias ? g.bias[m] : 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= g.N) continue;
      const long long off = cb + (long long)m * g.c_sm + (long long)n * g.c_sn;
      float v = acc[i][j] + bv;
      if (g.act == 1) v = fmaxf(v, 0.f);
      if (g.mask && !(g.mask[off] > 0.f)) v = 0.f;
      if (g.accumulate) v += g.C[off];
      g.C[off] = v;
      if (g.act == 2) g.C_abs[off] = fabsf(v);
    }
  }
}

template <typename TA, typename TB>
int launch_bgemm(const BGemm& g, cudaStream_t st) {
  if (g.nbatch <= 0 || g.M <= 0 || g.N <= 0) return PASN_OK;
  dim3 grid(ceil_div(g.N, TN), ceil_div(g.M, TM), g.reduce_batch ? 1 : g.nbatch);
  bgemm_kernel<TA, TB><<<grid, 256, 0, st>>>(g);
  PASN_LAUNCH_CHECK();
  count_launch();
  return PASN_OK;
}

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
//   gsim = gSim[n,p] + sum_k gLogits[n,k] Wl[k,p];  gcos = gsim / 2
//   gFE[n,p,:], gV[p,:] += ..., gWl[k,p] += gLogits[n,k] * sim[n,p]
__global__ void __launch_bounds__(256) proto_bwd_kernel(const float* __restrict__ FE, const float* __restrict__ protos,
                                                        const float* __restrict__ last_layer, const float* __restrict__ gLogits,
                                                        const float* __restrict__ gSim, int nb, int P, int D, int K,
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
  float gwl = 0.f;   // thread k < K accumulates gWl[k, p]
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
    if (gLogits)
      for (int k = 0; k < K; ++k) gs = fmaf(gLogits[(size_t)n * K + k], last_layer[(size_t)k * P + p], gs);
    const float gcos = 0.5f * gs;
    if (gLogits && tid < K) gwl = fmaf(gLogits[(size_t)n * K + tid], sim, gwl);
    // cos = <f, v> / (nf nv); nf, nv constants when clamped
    const float inv = 1.0f / (nf * nv);
    const float cf = f_clamped ? 0.f : cosv / (nf * nf);
    const float cv = v_clamped ? 0.f : cosv / (nv * nv);
    for (int d = tid; d < D; d += 256) {
      gFE[((size_t)n * P + p) * D + d] = gcos * (v[d] * inv - cf * f[d]);
      gV[(size_t)p * D + d] += gcos * (f[d] * inv - cv * v[d]);
    }
  }
  if (gLogits && tid < K) gWl[(size_t)tid * P + p] += gwl;
}

struct Scratch {
  float *H1, *F, *G1, *G2, *Opre, *O, *FE, *gFE, *gO, *gF, *gH1, *gG2, *gG1;
};

size_t per_clip_floats(const pasn_dims& d) {
  const size_t DS = (size_t)d.D * d.S, D2S = (size_t)(d.D / 2) * d.S, PS = (size_t)d.P * d.S, PD = (size_t)d.P * d.D;
  return 3 * DS + D2S + 2 * PS + 2 * PD + PS + 2 * DS + D2S + DS;   // H1 F G1 | G2 | Opre O | FE gFE | gO | gF gH1 | gG2 | gG1
}

int bwd_chunk(const pasn_dims& d) {
  const size_t cap = (size_t)384 << 20;
  long long c = (long long)(cap / (per_clip_floats(d) * 4));
  if (c < 1) c = 1;
  if (c > d.N) c = d.N > 0 ? d.N : 1;
  return (int)c;
}

}  // namespace

size_t backward_workspace_bytes(const pasn_dims& d) {
  if (tiled_backward_supported(d)) return tiled_backward_workspace_bytes(d);
  return align_up(per_clip_floats(d) * 4 * bwd_chunk(d), 256) + 256;
}

int head_backward(const void* feat, const pasn_weights& w, const pasn_dims& d, const float* gLogits, const float* gSim,
                  const float* gOcc, const pasn_grads& g, float* gX, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (d.D % 2 != 0) return PASN_ERR_UNSUPPORTED;
  if (tiled_backward_supported(d)) return tiled_head_backward(feat, w, d, gLogits, gSim, gOcc, g, gX, ws, ws_bytes, st);
  if (ws_bytes < backward_workspace_bytes(d)) return PASN_ERR_WORKSPACE;
  const int nbm = bwd_chunk(d);
  const int D = d.D, D2 = d.D / 2, S = d.S, P = d.P, C = d.C, K = d.K;
  const size_t DS = (size_t)D * S, D2S = (size_t)D2 * S, PS = (size_t)P * S, PD = (size_t)P * D;
  Scratch s;
  float* q = reinterpret_cast<float*>(ws);
  s.H1 = q; q += DS * nbm;   s.F = q; q += DS * nbm;    s.G1 = q; q += DS * nbm;   s.G2 = q; q += D2S * nbm;
  s.Opre = q; q += PS * nbm; s.O = q; q += PS * nbm;    s.FE = q; q += PD * nbm;   s.gFE = q; q += PD * nbm;
  s.gO = q; q += PS * nbm;   s.gF = q; q += DS * nbm;   s.gH1 = q; q += DS * nbm;  s.gG2 = q; q += D2S * nbm;
  s.gG1 = q;
  if (d.dtype == PASN_F16) return PASN_ERR_UNSUPPORTED;   // fp16 feature maps: tensor-core backward only
  const bool xbf = d.dtype == PASN_BF16;
  const size_t elt = dtype_bytes(d.dtype);
  // strides of the feature map seen as B[k = channel][n = voxel] per clip
  const long long x_sk = d.layout == PASN_LAYOUT_NSC ? 1 : S, x_sn = d.layout == PASN_LAYOUT_NSC ? C : 1;

  auto gemm = [&](const BGemm& a, bool b_is_x) -> int {
    return (b_is_x && xbf) ? launch_bgemm<float, __nv_bfloat16>(a, st) : launch_bgemm<float, float>(a, st);
  };
  // Y[b][o][s] = act(W[o][:] X[b][:][s] + bias[o])
  auto conv = [&](const float* W, const float* bias, int O_, int Cin, const void* X, bool x_is_input, float* Y, int act,
                  float* Yabs, int nb) -> int {
    BGemm a{};
    a.A = W; a.B = X; a.C = Y; a.C_abs = Yabs; a.bias = bias; a.act = act;
    a.M = O_; a.N = S; a.K = Cin; a.nbatch = nb;
    a.a_sb = 0; a.a_sm = Cin; a.a_sk = 1;
    a.b_sb = (long long)Cin * S;
    if (x_is_input) { a.b_sk = x_sk; a.b_sn = x_sn; } else { a.b_sk = S; a.b_sn = 1; }
    a.c_sb = (long long)O_ * S; a.c_sm = S; a.c_sn = 1;
    return gemm(a, x_is_input);
  };
  // gW[o][c] += sum_b sum_s gY[b][o][s] * X[b][c][s]
  auto wgrad = [&](const float* gY, int O_, const void* X, bool x_is_input, int Cin, float* gW, int nb) -> int {
    BGemm a{};
    a.A = gY; a.B = X; a.C = gW; a.accumulate = 1; a.reduce_batch = 1; a.nbatch = nb;
    a.M = O_; a.N = Cin; a.K = S;
    a.a_sb = (long long)O_ * S; a.a_sm = S; a.a_sk = 1;
    a.b_sb = (long long)Cin * S;
    if (x_is_input) { a.b_sk = x_sn; a.b_sn = x_sk; } else { a.b_sk = 1; a.b_sn = S; }   // B[k = s][n = c]
    a.c_sb = 0; a.c_sm = Cin; a.c_sn = 1;
    return gemm(a, x_is_input);
  };
  // gXin[b][c][s] (+)= sum_o W[o][c] gY[b][o][s], masked by relu output `mask` (same shape) when given
  auto dgrad = [&](const float* W, int O_, int Cin, const float* gY, float* gXin, const float* mask, int accumulate, int nb) -> int {
    BGemm a{};
    a.A = W; a.B = gY; a.C = gXin; a.mask = mask; a.accumulate = accumulate; a.nbatch = nb;
    a.M = Cin; a.N = S; a.K = O_;
    a.a_sb = 0; a.a_sm = 1; a.a_sk = Cin;            // A[m = c][k = o] = W[o][c]
    a.b_sb = (long long)O_ * S; a.b_sk = S; a.b_sn = 1;
    a.c_sb = (long long)Cin * S; a.c_sm = S; a.c_sn = 1;
    return launch_bgemm<float, float>(a, st);
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
    // ---- recompute the forward intermediates of this chunk
    if ((rc = conv(w.addon_w1, w.addon_b1, D, C, x, true, s.H1, 1, nullptr, nb))) return rc;
    if ((rc = conv(w.addon_w2, w.addon_b2, D, D, s.H1, false, s.F, 0, nullptr, nb))) return rc;
    if ((rc = conv(w.occ_w1, w.occ_b1, D, C, x, true, s.G1, 1, nullptr, nb))) return rc;
    if ((rc = conv(w.occ_w2, w.occ_b2, D2, D, s.G1, false, s.G2, 1, nullptr, nb))) return rc;
    if ((rc = conv(w.occ_w3, nullptr, P, D2, s.G2, false, s.Opre, 2, s.O, nb))) return rc;
    {  // FE[b][p][d] = sum_s O[b][p][s] F[b][d][s]
      BGemm a{};
      a.A = s.O; a.B = s.F; a.C = s.FE; a.nbatch = nb;
      a.M = P; a.N = D; a.K = S;
      a.a_sb = (long long)PS; a.a_sm = S; a.a_sk = 1;
      a.b_sb = (long long)DS; a.b_sk = 1; a.b_sn = S;
      a.c_sb = (long long)PD; a.c_sm = D; a.c_sn = 1;
      if ((rc = launch_bgemm<float, float>(a, st))) return rc;
    }
    // ---- prototype stage backward
    proto_bwd_kernel<<<P, 256, 0, st>>>(s.FE, w.prototypes, w.last_layer, gLogits ? gLogits + (size_t)n0 * K : nullptr,
                                        gSim ? gSim + (size_t)n0 * P : nullptr, nb, P, D, K, s.gFE, g.prototypes, g.last_layer);
    PASN_LAUNCH_CHECK();
    count_launch();
    {  // gO[b][p][s] = sum_d gFE[b][p][d] F[b][d][s]
      BGemm a{};
      a.A = s.gFE; a.B = s.F; a.C = s.gO; a.nbatch = nb;
      a.M = P; a.N = S; a.K = D;
      a.a_sb = (long long)PD; a.a_sm = D; a.a_sk = 1;
      a.b_sb = (long long)DS; a.b_sk = S; a.b_sn = 1;
      a.c_sb = (long long)PS; a.c_sm = S; a.c_sn = 1;
      if ((rc = launch_bgemm<float, float>(a, st))) return rc;
    }
    {  // gF[b][d][s] = sum_p gFE[b][p][d] O[b][p][s]
      BGemm a{};
      a.A = s.gFE; a.B = s.O; a.C = s.gF; a.nbatch = nb;
      a.M = D; a.N = S; a.K = P;
      a.a_sb = (long long)PD; a.a_sm = 1; a.a_sk = D;
      a.b_sb = (long long)PS; a.b_sk = S; a.b_sn = 1;
      a.c_sb = (long long)DS; a.c_sm = S; a.c_sn = 1;
      if ((rc = launch_bgemm<float, float>(a, st))) return rc;
    }
    {
      const long long n = (long long)nb * PS;
      sign_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(s.gO, gOcc ? gOcc + (size_t)n0 * PS : nullptr, s.Opre, n);
      PASN_LAUNCH_CHECK();
      count_launch();
    }
    // ---- add-on branch: F = W2 H1 + b2, H1 = relu(W1 x + b1)
    if ((rc = wgrad(s.gF, D, s.H1, false, D, g.addon_w2, nb))) return rc;
    if ((rc = rowsum(s.gF, g.addon_b2, D, nb))) return rc;
    if ((rc = dgrad(w.addon_w2, D, D, s.gF, s.gH1, s.H1, 0, nb))) return rc;
    if ((rc = wgrad(s.gH1, D, x, true, C, g.addon_w1, nb))) return rc;
    if ((rc = rowsum(s.gH1, g.addon_b1, D, nb))) return rc;
    // ---- occurrence branch: Opre = W5 G2, G2 = relu(W4 G1 + b4), G1 = relu(W3 x + b3)
    if ((rc = wgrad(s.gO, P, s.G2, false, D2, g.occ_w3, nb))) return rc;
    if ((rc = dgrad(w.occ_w3, P, D2, s.gO, s.gG2, s.G2, 0, nb))) return rc;
    if ((rc = wgrad(s.gG2, D2, s.G1, false, D, g.occ_w2, nb))) return rc;
    if ((rc = rowsum(s.gG2, g.occ_b2, D2, nb))) return rc;
    if ((rc = dgrad(w.occ_w2, D2, D, s.gG2, s.gG1, s.G1, 0, nb))) return rc;
    if ((rc = wgrad(s.gG1, D, x, true, C, g.occ_w1, nb))) return rc;
    if ((rc = rowsum(s.gG1, g.occ_b1, D, nb))) return rc;
    // ---- feature-map gradient (fp32, [N][C][S])
    if (gX) {
      float* gx = gX + (size_t)n0 * C * S;
      if ((rc = dgrad(w.addon_w1, D, C, s.gH1, gx, nullptr, 0, nb))) return rc;
      if ((rc = dgrad(w.occ_w1, D, C, s.gG1, gx, nullptr, 1, nb))) return rc;
    }
  }
  return PASN_OK;
}

}  // namespace pasn
