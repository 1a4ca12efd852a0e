// Tiled tcgen05 GEMM with TMA tensor-map loads and stores: the building block of the "tiled" tensor-core path that serves
// the shapes the fused token kernel does not (D != 256, S < 128, P > 48, fp32-exact mode): every 1x1(x1) convolution of
// the head, the occurrence-weighted pooling contraction and the W2 stage are instances of
//     OUT[b][m][n] = act( sum_pass sum_k A[b][m][a_off[pass] + k] * B[b][n][b_off[pass] + k]  + bias[n] + rowvec[m]*colvec[n] )
// with bf16 operands, fp32 accumulation in TMEM, and up to four operand passes: the hi/lo split for fp32 inputs,
// x*w = (xh + xl)(wh + wl) with xh = bf16(x), xl = bf16(x - xh) -- 16 significant bits per operand at bf16's full range, all
// four partial products kept.  (kind::f16 does not take an fp16 operand next to a bf16 one -- tried, the launch faults --
// so the lo planes cannot carry fp16's 11 bits.)  ab_f16 runs one pass with BOTH operands fp16 instead: the first layer of an
// fp16 feature map against fp16 weight planes.  Every other GEMM stays bf16 x bf16, so no launch can mix the two types.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace pasn {
namespace tcg {

enum { ACT_NONE = 0, ACT_RELU = 1, ACT_ABS = 2 };
enum { OUT_NONE = 0, OUT_BF16 = 1, OUT_BF16_HILO = 2, OUT_F32 = 3, OUT_F16 = 4 };   // HILO: bf16 hi plane | bf16 lo plane

struct Output {
  void* ptr;          // base of the [batch][M][ld] array (element (b, m, n) at ptr + (b*bs + m*ld + n) * elt)
  int mode;           // OUT_*
  long long ld, bs;   // row / batch stride in elements
  int lo_off;         // OUT_BF16_HILO: column offset of the lo half (the hi half starts at column 0)
  int ncols;          // columns of this output (0: N); columns beyond it are computed but not stored
  int absval;         // store |value| (only on the LAST output in use: the values are made absolute in place)
  int trans_S;        // > 0: rows are tokens (clip = m / trans_S, voxel = m % trans_S) and the output is channel-major per clip,
                      // element (m, n) at ptr + (m / trans_S) * bs + n * ld + m % trans_S  (plain stores, coalesced along m)
};

// optional element-wise epilogue input: element (b, m, n) at ptr[b*bs + m*ld + n*cs]  (cs = 0 means 1; cs > 1 with
// ld = 1 reads a transposed array, coalesced along m)
struct Aux {
  const void* ptr;
  long long ld, bs, cs;
};

struct Gemm {
  // A: K-major [a_batched ? batch : 1][M][ka] (row stride lda, k contiguous) or, a_mn_major, [batch?][K][ka] with m contiguous
  const void* A; long long lda, a_bs; int a_batched; int ka; int a_mn_major;
  int a_rows;                    // a_mn_major: K rows A really has per batch item (0: K); rows beyond read as zero
  // B: K-major [b_batched ? batch : 1][N][kb] (row stride ldb) or, b_mn_major, [batch?][K][nb] with n contiguous
  const void* B; long long ldb, b_bs; int b_batched; int kb; int b_mn_major;
  int b_rows;                    // rows B really has per batch item (0: N, or K when b_mn_major); rows beyond read as zero
  int M, N, K, batch;            // K per pass
  int k_rows_per_batch;          // split-K (both operands MN-major): batch item b covers K rows [b*k_rows_per_batch, +K) of the
                                 // same un-batched operands and writes its own partial output
  int npass; int a_off[4], b_off[4];   // column offset of each pass' operand plane
  int bn;                        // tile width: 64, 128 or 256
  const float* bias;             // [N] or null
  const float* rowparts; int nparts; const float* colvec;   // rank-1 term (sum_t rowparts[(b*M+m)*nparts + t]) * colvec[n], or null
  Aux addin;                     // fp32: value += addin            (applied in this order, before act)
  Aux signin;                    // bf16: value *= sign(signin), sign(0) = 0
  Aux mask;                      // bf16: value = mask > 0 ? value : 0
  int act;
  Output out[2];
  float* psum;                   // optional [batch*M][2*tiles_n]: row sums of the outputs per column half-tile ...
  int psum_rounded;              // ... of the bf16-rounded values (what a bf16 consumer of the outputs will read) or of the fp32
                                 // values (an OUT_F16 output feeds no GEMM: the fp16 chain pools its bf16 copy)
  int pair;                      // 1: CTA pairs (cta_group::2): 256 x bn tiles, each CTA of a 2-CTA cluster loads its 128 rows of A
                                 // and half of the B tile -- a third less L2 -> SM traffic per flop (bn >= 128 only; else ignored)
  // optional per-row statistics of the final fp32 values (the prototype stage's reductions folded into the GEMM that produces
  // the pooled features, so that those need not be written and read back): rowstat[(b*M + m) * 2*tiles_n + t][0..3] =
  // (sum_n v^2, sum_n v * w, sum_n w^2, 0) with w = dotvec[(m % dot_mod) * dot_ld + n] over the columns of column half-tile t
  float* rowstat; const float* dotvec; long long dot_ld; int dot_mod;
  // optional block-diagonal batching of small per-item GEMMs (both operands MN-major and batched, one pass, K <= 64): `group` items
  // share one 128-row tile -- item j's `group_rows` rows sit at rows [j*group_rows, +group_rows) and its K rows are the tile's
  // j-th k-block (the other rows of that k-block's A tile are zero: the boxes are loaded at negative / out-of-range m
  // coordinates, which the TMA unit zero-fills).  Pass M = group * group_rows, batch = ceil(group_items / group), a_bs / b_bs per
  // ITEM; only with row statistics and no outputs.  (The per-clip pooling of few prototypes: 40 of a tile's 128 rows otherwise.)
  int group, group_rows, group_items;
  long long stat_rows;           // rows of rowstat that exist (0: batch * M): rows past it are not written
  int dot_early;                 // dotvec is not written by the kernel in front on the stream: it may be read before that one has completed
  int ab_f16;                    // 1: A and B are fp16 (kind::f16 with F16 x F16; npass must be 1), 0: both bf16.  Placed in the tail
                                 // padding of the struct: sizeof(Gemm) is unchanged (448)
};

void set_trace(void* dev_buf);   // debug: 64 rows of 64 int64 globaltimer stamps of CTA 0, one row per launch (null = off)
int launch(const Gemm& g, cudaStream_t st);   // 0 or a negative pasn_status
bool available();                             // driver entry point for tensor-map encoding found

}  // namespace tcg
}  // namespace pasn
