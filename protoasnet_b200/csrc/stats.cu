// Loss / metric consumers of the head outputs, computed on the device without a host round trip (SURVEY.md 8(f) row 3).
//
// Reference arithmetic being restated:
//   ClusterRoiFeat.compute      src/loss/loss.py:114-138   -sum_n max_{j in class y_n} sim[n,j]
//   SeparationRoiFeat.compute   src/loss/loss.py:158-187   sum_n sum_{k != y_n, k not abstention} max_{j in class k} sim[n,j]
//   L_norm.compute (p = 1 | 2, dim = trailing spatial dims)  src/loss/loss.py:236-250   sum_{n,p} ||occ[n,p,:]||_p
//   prototype diversity counters  src/agents/Video_XProtoNet_e2e.py:158-173 (torch.sort on the CPU + np.add.at every
//       step): count[j] += [j among the top-a most similar class prototypes of clip n], same with top-b for the
//       abstention prototypes; simscore_cumsum[j] += sum_n sim[n,j]
// Sums over the batch are accumulated in double (one atomic per block), so the result does not depend on the grid in
// any digit a float32 loss would show.  `reduction` ('mean' divides the batch sum by N) is applied by the caller.
#include "common.cuh"

namespace pasn {

namespace {

constexpr int ST_THREADS = 128;

// One thread per clip.  class_arg[n,k] = argmax_j sim[n, k*ppc + j] (global prototype index), class_max[n,k] its value.
__global__ void __launch_bounds__(ST_THREADS) sim_stats_kernel(const float* __restrict__ sim, const int64_t* __restrict__ labels,
                                                               int N, int P, int K, int abstain, int n_specific, int top_a,
                                                               int top_b, float* __restrict__ class_max,
                                                               int32_t* __restrict__ class_arg, double* __restrict__ sums,
                                                               unsigned long long* __restrict__ counts,
                                                               double* __restrict__ simsum) {
  __shared__ double red[2][ST_THREADS / 32];
  const int n = blockIdx.x * ST_THREADS + threadIdx.x;
  const int ppc = P / K;
  double cl = 0.0, sp = 0.0;
  if (n < N) {
    const float* s = sim + (size_t)n * P;
    const int y = labels ? (int)labels[n] : -1;
    for (int k = 0; k < K; ++k) {
      float best = s[k * ppc];
      int arg = k * ppc;
      for (int j = 1; j < ppc; ++j) {
        const float v = s[k * ppc + j];
        if (v > best) { best = v; arg = k * ppc + j; }     // first maximum wins, like torch.max
      }
      if (class_max) class_max[(size_t)n * K + k] = best;
      if (class_arg) class_arg[(size_t)n * K + k] = arg;
      if (labels) {
        if (k == y) cl -= (double)best;
        else if (!(abstain && k == K - 1)) sp += (double)best;
      }
    }
    if (counts) {
      // top-a of the class-specific prototypes [0, n_specific), top-b of the rest: repeated arg-max with a taken mask
      unsigned long long taken = 0ull;   // P <= 64 (checked by the host)
      for (int part = 0; part < 2; ++part) {
        const int lo = part ? n_specific : 0, hi = part ? P : n_specific;
        const int top = part ? top_b : top_a;
        for (int t = 0; t < top && t < hi - lo; ++t) {
          int arg = -1;
          float best = 0.f;
          for (int j = lo; j < hi; ++j) {
            if ((taken >> j) & 1ull) continue;
            if (arg < 0 || s[j] > best) { best = s[j]; arg = j; }
          }
          taken |= 1ull << arg;
          atomicAdd(&counts[arg], 1ull);
        }
      }
    }
  }
  if (sums) {
    cl = warp_sum_d(cl);
    sp = warp_sum_d(sp);
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = cl; red[1][threadIdx.x >> 5] = sp; }
    __syncthreads();
    if (threadIdx.x == 0) {
      double a = 0.0, b = 0.0;
      for (int i = 0; i < ST_THREADS / 32; ++i) { a += red[0][i]; b += red[1][i]; }
      atomicAdd(&sums[0], a);
      atomicAdd(&sums[1], b);
    }
  }
  if (simsum) {   // column sums: thread j of block 0..: loop over this block's rows
    __syncthreads();
    const int n0 = blockIdx.x * ST_THREADS, n1 = min(N, n0 + ST_THREADS);
    for (int j = threadIdx.x; j < P; j += ST_THREADS) {
      double a = 0.0;
      for (int r = n0; r < n1; ++r) a += (double)sim[(size_t)r * P + j];
      atomicAdd(&simsum[j], a);
    }
  }
}

// one warp per (n, p) row of the occurrence map: sums[0] += (sum_s |o|^p)^(1/p)
template <typename T>
__global__ void __launch_bounds__(256) occ_lnorm_kernel(const T* __restrict__ occ, long long rows, int S, int p,
                                                        double* __restrict__ sums, float* __restrict__ row_norm) {
  __shared__ double red[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + warp;
  double contrib = 0.0;
  if (row < rows) {
    const T* o = occ + row * S;
    float a = 0.f;
    for (int s = lane; s < S; s += 32) {
      const float v = fabsf(to_f32<T>(o[s]));
      a += p == 1 ? v : v * v;
    }
    a = warp_sum(a);
    const float nrm = p == 1 ? a : sqrtf(a);
    if (lane == 0 && row_norm) row_norm[row] = nrm;
    contrib = (double)nrm;
  }
  if (lane == 0) red[warp] = contrib;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += red[i];
    atomicAdd(&sums[0], t);
  }
}

}  // namespace

int launch_sim_stats(const float* sim, const int64_t* labels, int N, int P, int K, int abstain, int n_specific, int top_a,
                     int top_b, float* class_max, int32_t* class_arg, double* sums, unsigned long long* counts, double* simsum,
                     cudaStream_t st) {
  if (N <= 0) return PASN_OK;
  if (K <= 0 || P % K != 0 || (counts && (P > 64 || n_specific < 0 || n_specific > P))) return PASN_ERR_INVALID;
  sim_stats_kernel<<<ceil_div(N, ST_THREADS), ST_THREADS, 0, st>>>(sim, labels, N, P, K, abstain, n_specific, top_a, top_b,
                                                                    class_max, class_arg, sums, counts, simsum);
  PASN_LAUNCH_CHECK();
  count_launch();
  return PASN_OK;
}

int launch_occ_lnorm(const void* occ, int dtype, long long rows, int S, int p, double* sums, float* row_norm, cudaStream_t st) {
  if (rows <= 0) return PASN_OK;
  if (p != 1 && p != 2) return PASN_ERR_INVALID;
  const unsigned grid = (unsigned)((rows + 7) / 8);
  if (dtype == PASN_F16)
    occ_lnorm_kernel<__half><<<grid, 256, 0, st>>>(reinterpret_cast<const __half*>(occ), rows, S, p, sums, row_norm);
  else if (dtype == PASN_BF16)
    occ_lnorm_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(occ), rows, S, p, sums, row_norm);
  else
    occ_lnorm_kernel<float><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(occ), rows, S, p, sums, row_norm);
  PASN_LAUNCH_CHECK();
  count_launch();
  return PASN_OK;
}

}  // namespace pasn
