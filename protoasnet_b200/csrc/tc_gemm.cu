// Persistent, warp-specialised tcgen05 GEMM (see tc_gemm.cuh for the operation).
//
//   warp 0      TMA producer: cp.async.bulk.tensor (tensor maps, SWIZZLE_128B) into a 3-stage ring of
//               [A 128x64 | B bn x 64] bf16 operand tiles; out-of-range rows / k are zero-filled by the TMA unit
//   warp 1      MMA issuer: one elected thread, tcgen05.mma kind::f16 M128 x N(bn) x K16, fp32 accumulators in TMEM,
//               two accumulator buffers of 256 columns so the epilogue of tile i overlaps the MMAs of tile i+1
//   warp 2      TMEM allocation
//   warps 4-11  epilogue: warp w reads TMEM lanes 32*(w%4).. (its 32 rows) of column half w/4, applies
//               bias / rank-1 term / ReLU / abs, converts, and leaves the rows either through a private swizzled
//               staging slab + TMA store (16-byte aligned outputs) or with plain stores (small unaligned outputs)
//
// PAIR = true runs the same roles on 2-CTA clusters (cta_group::2): a pair owns a 256 x bn tile, each CTA loads its 128
// rows of A and bn/2 rows of B (TMA completions of both CTAs land on the leader's "full" barrier), one thread of the
// leader issues M = 256 MMAs that read both CTAs' shared memory and write both CTAs' TMEM, tcgen05.commit multicasts the
// "stage free" / "accumulator full" arrivals to both CTAs, and the non-leader's epilogue warps hand the accumulator back
// with remote arrivals.  Per flop a pair pulls 2/3 of the bytes from L2 that two independent CTAs would (the chain's big
// GEMMs are bound by the ~6300 B/clk L2 -> SM fabric, not by the tensor pipe: profiles/README.md).
//
// Every mbarrier wait is bounded: a protocol fault becomes an error code in *err, not a hung GPU.
#include <cuda.h>

#include "sm100_prims.cuh"
#include "tc_gemm.cuh"

namespace pasn {
namespace tcg {
using namespace sm100;

namespace {

constexpr int BM = 128, BK = 64, STAGES = 3, MAX_STAGES = 8;
// the operand ring is 3 x 48 KB; a stage only takes what its tiles need (A 16 KB + 128 B per row of the B tile this CTA
// loads), so narrower tiles and CTA pairs get a deeper ring out of the same bytes -- what matters is the number of bytes
// in flight against the L2 round trip, not the stage count
constexpr uint32_t A_BYTES = BM * BK * 2, B_BYTES_MAX = 256 * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES_MAX;   // 48 KB
constexpr int EPI_WARPS = 8, EPI_WARP0 = 4, THREADS = 32 * (EPI_WARP0 + EPI_WARPS);
constexpr uint32_t SLAB_BYTES = 4096;                             // 32 rows x 128 bytes
constexpr uint32_t SM_STG = STAGES * STAGE_BYTES;                 // 147456: staging slabs, 2 per epilogue warp
constexpr uint32_t SM_VEC = SM_STG + EPI_WARPS * 2 * SLAB_BYTES;  // 212992: per-warp bias / colvec slices (2 groups x 2 x 64 floats)
constexpr uint32_t SM_BAR = SM_VEC + EPI_WARPS * 1024;            // 221184
constexpr uint32_t SM_MISC = SM_BAR + 24 * 8;
constexpr uint32_t SMEM_BYTES = SM_MISC + 64;
enum { B_FULL = 0, B_EMPTY = MAX_STAGES, B_ACCFULL = 2 * MAX_STAGES, B_ACCEMPTY = 2 * MAX_STAGES + 2, B_WARM = 2 * MAX_STAGES + 4 };

struct alignas(64) KParams {
  CUtensorMap tmA, tmB, tmO[4];   // out0 (hi), out0 lo, out1 (hi), out1 lo
  Gemm g;
  int out_tma[2];
  int tall;   // 1: a tile has two 128-row (per CTA) sub-tiles that share each B stage; they take the two accumulator buffers
  int tiles_m, tiles_n, nkb;
  int* err;
  long long* trace;   // optional: 64 globaltimer stamps of CTA 0 (tools/trace_gemm.py)
};

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
      : "memory");
}
// CTA-pair form: the completion bytes are counted on the barrier at the same offset in the leader (even) CTA of the pair
__device__ __forceinline__ void tma_load_3d_2sm(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar) & 0xFEFFFFFFu)
      : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%1, %2, %3}], [%4];" ::"l"(map), "r"(c0),
               "r"(c1), "r"(c2), "r"(src)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) { asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory"); }

static __device__ __noinline__ bool wait_slow(uint64_t* bar, uint32_t parity, int* err, int code) {
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000ll) {
      *reinterpret_cast<volatile int*>(err) = code;
      return false;
    }
  }
  return true;
}
__device__ __forceinline__ long long gtimer_ns() {
  long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define TCG_TRACE(slot) do { if (kp.trace != nullptr && blockIdx.x == 0) kp.trace[slot] = gtimer_ns(); } while (0)
#define TCG_TRACE1(slot) do { if (kp.trace != nullptr && blockIdx.x == 1) kp.trace[slot] = gtimer_ns(); } while (0)
__device__ __forceinline__ bool bwait(uint64_t* bar, uint32_t parity, int* err, int code) {
  if (mbar_try_wait(bar, parity)) return true;
  return wait_slow(bar, parity, err, code);
}


}  // namespace

// EPI says how much of the epilogue is compiled in (a bit per feature).  The generic epilogue (EPI_FULL) is ~10 k
// instructions of unrolled 64-element loops behind launch-uniform branches; a tile's path through it jumps from one cold
// instruction-cache line to the next (ncu: 20-30 % of the short GEMMs' issue slots lost to stall_no_inst).  The shapes that
// carry the chains get their own lean instantiations; launch() picks the first one that covers what the descriptor asks for.
enum {
  E_BIT_AUX = 1,      // element-wise epilogue inputs (addin / signin / mask: the backward)
  E_BIT_PSUM = 2,     // row sums per column half-tile
  E_BIT_STAT = 4,     // row statistics
  E_BIT_DIRECT = 8,   // plain stores (unaligned / channel-major outputs), two outputs split between the warp groups
  E_BIT_OUT = 16,     // any output at all
  E_BIT_ABSOUT = 32,  // |value| on the second output
  E_BIT_F16 = 64,     // fp16 outputs (OUT_F16): only in the instantiation that needs them, the others keep their code
  EPI_FULL = 63,
  EPI_F16 = EPI_FULL | E_BIT_F16,
  EPI_LEAN = E_BIT_OUT,                   // bias / rank-1 term / activation, TMA-stored outputs
  EPI_STAT = E_BIT_STAT,                  // no output, row statistics only
  EPI_DIRECT = E_BIT_OUT | E_BIT_DIRECT,
  EPI_PSUM = E_BIT_OUT | E_BIT_PSUM,
  EPI_AUX = E_BIT_OUT | E_BIT_AUX,
};
template <bool PAIR, int EPI>   // PAIR: CTA pairs, else one CTA per tile
__global__ void __launch_bounds__(THREADS, 1) tc_gemm_kernel(const __grid_constant__ KParams kp) {
  constexpr bool E_AUX = (EPI & E_BIT_AUX) != 0, E_PSUM = (EPI & E_BIT_PSUM) != 0, E_STAT = (EPI & E_BIT_STAT) != 0,
                 E_DIRECT = (EPI & E_BIT_DIRECT) != 0, E_OUT = (EPI & E_BIT_OUT) != 0, E_ABSOUT = (EPI & E_BIT_ABSOUT) != 0,
                 E_SPLIT = E_DIRECT, E_F16 = (EPI & E_BIT_F16) != 0;
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM_BAR);
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(smem + SM_MISC);
  const Gemm& g = kp.g;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if ((smem_u32(smem) & 1023u) != 0) {
    if (tid == 0) *reinterpret_cast<volatile int*>(kp.err) = 700;
    return;
  }
  if (tid == 0) TCG_TRACE(0);
  const uint32_t crank = PAIR ? cluster_ctarank() : 0u;         // rank in the cluster
  const uint32_t rank = crank & 1u;                             // rank in the pair: 0 = leader
  if (tid == 0) {
    for (int i = 0; i < MAX_STAGES; ++i) { mbar_init(&bars[B_FULL + i], 1); mbar_init(&bars[B_EMPTY + i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&bars[B_ACCFULL + i], 1); mbar_init(&bars[B_ACCEMPTY + i], PAIR ? 2 * EPI_WARPS : EPI_WARPS); }
    mbar_init(&bars[B_WARM], 1);
    fence_mbar_init();
    prefetch_tmap(&kp.tmA);
    prefetch_tmap(&kp.tmB);
  }
  if (warp == 2) { if constexpr (PAIR) tmem_alloc2(tmem_ptr_s, 512); else tmem_alloc(tmem_ptr_s, 512); }
  tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) cluster_sync_all();   // both CTAs' barriers exist before any remote arrival / multicast commit
  tc_fence_after();
  // programmatic dependent launch: the chain's GEMMs follow each other on one stream; the next launch may set itself up
  // (barriers, TMEM, tensor-map prefetch) while this grid drains, and nothing here touches global memory before the
  // grid in front of it has completed
  if (tid == 0) TCG_TRACE(1);   // set-up done
  griddep_launch_dependents();
  // (the producer thread waits below, after warming up its first loads; epilogue warps that may read the statistics' vectors
  // early do so first)
  const bool stat_early = g.rowstat != nullptr && g.dot_early != 0;
  if (warp != 0 && !(stat_early && warp >= EPI_WARP0)) griddep_wait();
  const uint32_t tbase = *tmem_ptr_s;
  const uint32_t sbase = smem_u32(smem);
  const int bn = g.bn;
  const int bnl = PAIR ? bn / 2 : bn;                           // rows of the B tile this CTA loads
  const int tiles_per_batch = kp.tiles_m * kp.tiles_n;
  const int ntiles = g.batch * tiles_per_batch;
  constexpr int CL = PAIR ? 2 : 1;                                          // CTAs per cluster = per tile
  const int tile0 = (int)(blockIdx.x / CL);                                 // persistent walk of this CTA / pair
  const int tstep = (int)(gridDim.x / CL);
  constexpr int BMC = CL * BM;                                              // rows of one sub-tile (one MMA) across the cluster
  const int nu = kp.tall ? 2 : 1;                                           // sub-tiles per tile (long-K GEMMs: see launch())
  const int BMT = BMC * nu;                                                 // rows of a (cluster) tile
  const uint16_t pair_mask = (uint16_t)(3u << (crank & ~1u));               // the two CTAs of this pair
  const uint32_t a_stage = A_BYTES * (uint32_t)nu;                          // A boxes of a stage (one per sub-tile)
  const uint32_t stage_bytes = a_stage + (uint32_t)bnl * 128u;              // multiple of 1024: swizzle atoms stay aligned
  const uint32_t nst_fit = (STAGES * STAGE_BYTES) / stage_bytes;
  const uint32_t nst = nst_fit < (uint32_t)MAX_STAGES ? nst_fit : (uint32_t)MAX_STAGES;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      uint32_t s = 0, ph = 0;
      bool ok = true;
      const uint32_t stage_tx = stage_bytes * (PAIR ? 2u : 1u);   // both CTAs' bytes land on the leader's barrier
      auto tma_load = [&](uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
        if constexpr (PAIR) tma_load_3d_2sm(dst, map, c0, c1, c2, bar);
        else tma_load_3d(dst, map, c0, c1, c2, bar);
      };
      if (tile0 < ntiles) {
        // The first load of a launch takes ~2.7 us (tensor-map fetch, translation, cold lines) against ~1 us later on: touch
        // the first boxes of both operands while the grid in front is still draining.  What lands may be stale (A is being
        // written by that grid) and is thrown away; the real loads below overwrite the stage.
        const int b = tile0 / tiles_per_batch, r = tile0 - b * tiles_per_batch;
        const int m0 = (r / kp.tiles_n) * BMT + (int)rank * BM, n0 = (r % kp.tiles_n) * bn + (int)rank * bnl;
        const bool split_k = g.k_rows_per_batch > 0;
        const int krow = split_k ? b * g.k_rows_per_batch : 0;
        const uint32_t a_tx = g.a_mn_major ? 8192u : A_BYTES, b_tx = g.b_mn_major ? 8192u : (uint32_t)bnl * 128u;
        mbar_arrive_expect_tx(&bars[B_WARM], a_tx + b_tx);
        if (!g.a_mn_major) tma_load_3d(sbase, &kp.tmA, g.a_off[0], m0, g.a_batched ? b : 0, &bars[B_WARM]);
        else tma_load_3d(sbase, &kp.tmA, g.a_off[0] + m0, krow, (g.a_batched && !split_k) ? b : 0, &bars[B_WARM]);
        if (!g.b_mn_major) tma_load_3d(sbase + A_BYTES, &kp.tmB, g.b_off[0], n0, g.b_batched ? b : 0, &bars[B_WARM]);
        else tma_load_3d(sbase + A_BYTES, &kp.tmB, g.b_off[0] + n0, krow, (g.b_batched && !split_k) ? b : 0, &bars[B_WARM]);
      }
      griddep_wait();
      TCG_TRACE(2);   // the grid in front has completed
      if (tile0 < ntiles) ok = bwait(&bars[B_WARM], 0, kp.err, 702);
      for (int t = tile0; t < ntiles && ok; t += tstep) {
        const int b = t / tiles_per_batch, r = t - b * tiles_per_batch;
        const int m0 = (r / kp.tiles_n) * BMT + (int)rank * BM, n0 = (r % kp.tiles_n) * bn + (int)rank * bnl;
        const bool split_k = g.k_rows_per_batch > 0;
        const int krow0 = split_k ? b * g.k_rows_per_batch : 0;
        for (int pass = 0; pass < g.npass && ok; ++pass) {
          for (int kb = 0; kb < kp.nkb; ++kb) {
            if (!(ok = bwait(&bars[B_EMPTY + s], ph ^ 1, kp.err, 701))) break;
            const uint32_t dst = sbase + s * stage_bytes;
            if (t == tile0 && pass == 0 && kb == 0) TCG_TRACE(6);   // first load goes out
            if (rank == 0) mbar_arrive_expect_tx(&bars[B_FULL + s], stage_tx);
            const int krow = krow0 + kb * BK;   // K coordinate of MN-major operands (rows)
            for (int u = 0; u < nu; ++u) {
              const int mu = m0 + u * BMC;
              const uint32_t da = dst + (uint32_t)u * A_BYTES;
              if (!g.a_mn_major) {
                tma_load(da, &kp.tmA, g.a_off[pass] + kb * BK, mu, g.a_batched ? b : 0, &bars[B_FULL + s]);
              } else if (g.group > 1) {   // block-diagonal: item b*group + kb, its rows shifted to [kb*group_rows, ...)
                for (int j = 0; j < 2; ++j)
                  tma_load(da + j * 8192, &kp.tmA, g.a_off[pass] + 64 * j - g.group_rows * kb, 0, b * g.group + kb, &bars[B_FULL + s]);
              } else {
                for (int j = 0; j < 2; ++j)
                  tma_load(da + j * 8192, &kp.tmA, g.a_off[pass] + mu + 64 * j, krow, (g.a_batched && !split_k) ? b : 0,
                           &bars[B_FULL + s]);
              }
            }
            if (!g.b_mn_major) {
              tma_load(dst + a_stage, &kp.tmB, g.b_off[pass] + kb * BK, n0, g.b_batched ? b : 0, &bars[B_FULL + s]);
            } else if (g.group > 1) {
              for (int j = 0; j < bnl / 64; ++j)
                tma_load(dst + a_stage + j * 8192, &kp.tmB, g.b_off[pass] + n0 + 64 * j, 0, b * g.group + kb, &bars[B_FULL + s]);
            } else {
              for (int j = 0; j < bnl / 64; ++j)
                tma_load(dst + a_stage + j * 8192, &kp.tmB, g.b_off[pass] + n0 + 64 * j, krow,
                         (g.b_batched && !split_k) ? b : 0, &bars[B_FULL + s]);
            }
            s = s + 1 == nst ? 0 : s + 1;
            ph ^= (s == 0) ? 1u : 0u;
          }
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA of a pair)
    if (elect_one()) {
      const uint32_t ab_bf16 = g.ab_f16 ? 0u : 1u;   // one element type for both operands (launch() checks npass == 1)
      const uint32_t id = make_idesc_16(BMC, (uint32_t)bn, ab_bf16, ab_bf16, g.a_mn_major ? 1u : 0u, g.b_mn_major ? 1u : 0u);
      auto mma = [&](uint32_t d, uint32_t alo, uint32_t ahi, uint32_t blo, uint32_t bhi, uint32_t acc) {
        if constexpr (PAIR) mma_ss2_x(d, alo, ahi, blo, bhi, id, acc);
        else mma_ss_x(d, alo, ahi, blo, bhi, id, acc);
      };
      auto commit = [&](uint32_t bar_saddr) {          // to this pair
        if constexpr (PAIR) mma_commit2_a(bar_saddr, pair_mask);
        else mma_commit_a(bar_saddr);
      };
      const uint32_t a_lbo = g.a_mn_major ? 8192u : 16u, a_kstep = g.a_mn_major ? 128u : 2u;
      constexpr uint32_t HI = desc_hi(1024, SWZ_128B);
      const uint32_t b_lbo = g.b_mn_major ? 8192u : 16u, b_kstep = g.b_mn_major ? 128u : 2u;
      const uint32_t bar0 = smem_u32(bars);
      uint32_t s = 0, ph = 0;
      bool ok = true;
      int i = 0;
      // i counts sub-tiles (= accumulator hand-overs); a tall tile takes both buffers at once
      for (int t = tile0; t < ntiles && ok; t += tstep, i += nu) {
        const uint32_t buf = i & 1;
        if (!(ok = bwait(&bars[B_ACCEMPTY + buf], ((i >> 1) & 1) ^ 1, kp.err, 711))) break;
        if (nu == 2 && !(ok = bwait(&bars[B_ACCEMPTY + 1], ((i >> 1) & 1) ^ 1, kp.err, 713))) break;
        tc_fence_after();
        const uint32_t d = tbase + 256u * buf;
        for (int pass = 0; pass < g.npass && ok; ++pass) {
          for (int kb = 0; kb < kp.nkb; ++kb) {
            if (!(ok = bwait(&bars[B_FULL + s], ph, kp.err, 712))) break;
            if (i == 0 && pass == 0 && kb == 0) TCG_TRACE(3);   // first operand stage has landed
            if (pass == 0 && kb == 0 && i < 16) TCG_TRACE(48 + i);   // ... and each tile's first one
            tc_fence_after();
            const uint32_t sa = sbase + s * stage_bytes;
            const uint32_t alo = desc_lo(sa, a_lbo), blo = desc_lo(sa + a_stage, b_lbo);
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4) mma(d, alo + k4 * a_kstep, HI, blo + k4 * b_kstep, HI, (pass | kb | k4) ? 1u : 0u);
            if (nu == 2) {   // second sub-tile: its own A box, the same B stage, the other accumulator buffer
              const uint32_t alo1 = desc_lo(sa + A_BYTES, a_lbo);
#pragma unroll
              for (int k4 = 0; k4 < 4; ++k4)
                mma(tbase + 256u, alo1 + k4 * a_kstep, HI, blo + k4 * b_kstep, HI, (pass | kb | k4) ? 1u : 0u);
            }
            commit(bar0 + 8u * (B_EMPTY + s));
            s = s + 1 == nst ? 0 : s + 1;
            ph ^= (s == 0) ? 1u : 0u;
          }
        }
        if (ok) {
          if (i == 0) TCG_TRACE(4);   // first tile's MMAs issued
          commit(bar0 + 8u * (B_ACCFULL + buf));
          if (nu == 2) commit(bar0 + 8u * (B_ACCFULL + 1));
        }
      }
    }
  } else if (warp >= EPI_WARP0) {
    // ------------------------------------------------------------------ epilogue
    const int w = warp - EPI_WARP0, q = w & 3, hw = w >> 2;
    const uint32_t tl = tbase + ((uint32_t)(q * 32) << 16);
    const uint32_t slab0 = sbase + SM_STG + (uint32_t)w * 2u * SLAB_BYTES;
    float* vecs_w = reinterpret_cast<float*>(smem + SM_VEC + w * 1024);   // per group: [0,64) bias slice, [64,128) colvec slice
    // The per-element work below is what bounds the wide, short-K GEMMs of the chain (8 warps share 4 issue slots: every
    // instruction per accumulator element costs ~1/4 cycle per element of the tile), so everything that is uniform
    // over the launch is decided by branches around the element loops, never by selects inside them.
    const bool has_vec = g.bias != nullptr || (g.rowparts != nullptr && g.colvec != nullptr);
    const bool has_aux = E_AUX && (g.addin.ptr != nullptr || g.signin.ptr != nullptr || g.mask.ptr != nullptr);
    float* const psum_p = E_PSUM ? g.psum : nullptr;
    float* const rowstat_p = E_STAT ? g.rowstat : nullptr;
    const int nh = bn >= 128 ? 2 : 1;            // column halves in use (a 64-wide tile is one 64-column group: half 0 only)
    // a 64-wide tile with two outputs: the second warp group, otherwise idle, reads the same columns and takes output 1
    // (the channel-major plain stores of the occurrence map run next to the TMA store of the token-major copy)
    const bool split_out = E_SPLIT && nh == 1 && g.out[0].mode != OUT_NONE && g.out[1].mode != OUT_NONE;
    const int h = split_out ? 0 : hw;            // column half this warp reads
    const int half_cols = bn / nh;
    const int ngroups = half_cols / 64;
    uint32_t nstores = 0;   // TMA stores issued by this warp so far (slab = nstores & 1)
    // row statistics with the vectors' slices cached in the staging slabs (see below)
    const bool stat_cached = !PAIR && rowstat_p != nullptr && !kp.out_tma[0] && !kp.out_tma[1] && kp.tiles_m == 1 &&
                             (g.M <= 64 || (g.M <= BM && ngroups == 1)) &&   // second column group in the idle row groups' slabs
                             nh == 2 && (g.N & 63) == 0 && (g.dot_ld & 3) == 0 && (reinterpret_cast<uintptr_t>(g.dotvec) & 15) == 0;
    int stat_key0 = -1, stat_key1 = -1;
    // slice of the vectors for this warp's rows and one column group -> slab(s); the row pairs are walked from a different
    // start in every CTA and warp: all CTAs read the same few KB, in step they queue up on the same L2 lines (19 us measured)
    auto stat_fill = [&](int cg, int col0) {
      float* stg = reinterpret_cast<float*>(smem + SM_STG + (uint32_t)(w + 2 * cg) * 2u * SLAB_BYTES);
      const int rot = (int)((blockIdx.x * 5u + (uint32_t)w * 3u + (uint32_t)cg * 7u) & 15u);
      __syncwarp();
#pragma unroll 8
      for (int it0 = 0; it0 < 16; ++it0) {
        const int it = (it0 + rot) & 15;
        const int r = 2 * it + (lane >> 4), j = lane & 15;
        const int rr = q * 32 + r;
        float4 w4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rr < g.M) w4 = __ldg(reinterpret_cast<const float4*>(g.dotvec + (long long)(rr % g.dot_mod) * g.dot_ld + col0) + j);
        *reinterpret_cast<float4*>(stg + r * 64 + ((j ^ (r & 7)) << 2)) = w4;
      }
      __syncwarp();
    };
    if (stat_cached && q * 32 < g.M && tile0 < ntiles) {   // the first tile's slices, while its operands are still on their way
      const int n00 = ((tile0 % tiles_per_batch) % kp.tiles_n) * bn + hw * half_cols;
      stat_fill(0, n00);
      stat_key0 = n00;
      if (ngroups > 1) { stat_fill(1, n00 + 64); stat_key1 = n00 + 64; }
    }
    if (stat_early) griddep_wait();
    bool ok = true;
    int i = 0;
    // one 64-column group of one output leaves through the staging slab(s) + TMA store(s)
    auto store_tma = [&](const Output& o, int mi, const float (&v)[64], int col0, int row0, int b) {
      const int nbox = (o.mode == OUT_BF16 || (E_F16 && o.mode == OUT_F16)) ? 1 : 2;
#pragma unroll
      for (int bx = 0; bx < 2; ++bx) {
        if (bx >= nbox) break;
        if (lane == 0) bulk_wait_read<1>();   // the slab used two stores ago has been read out
        __syncwarp();
        const uint32_t slab = slab0 + (nstores & 1u) * SLAB_BYTES;
        const uint32_t rowaddr = slab + (uint32_t)lane * 128u;
        if (o.mode == OUT_F32) {
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const uint32_t a = rowaddr + (uint32_t)((c ^ (lane & 7)) << 4);
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v[32 * bx + 4 * c]),
                         "f"(v[32 * bx + 4 * c + 1]), "f"(v[32 * bx + 4 * c + 2]), "f"(v[32 * bx + 4 * c + 3])
                         : "memory");
          }
        } else if (E_F16 && o.mode == OUT_F16) {
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            uint32_t pk[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const __half2 h2 = __floats2half2_rn(v[8 * c + 2 * j], v[8 * c + 2 * j + 1]);
              pk[j] = *reinterpret_cast<const uint32_t*>(&h2);
            }
            const uint32_t a = rowaddr + (uint32_t)((c ^ (lane & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3]) : "memory");
          }
        } else if (o.mode == OUT_BF16_HILO && bx == 1) {
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            uint32_t pk[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float a0 = v[8 * c + 2 * j], a1 = v[8 * c + 2 * j + 1];
              pk[j] = pack_bf16x2(a0 - round_bf16(a0), a1 - round_bf16(a1));
            }
            const uint32_t a = rowaddr + (uint32_t)((c ^ (lane & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3]) : "memory");
          }
        } else {
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            uint32_t pk[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) pk[j] = pack_bf16x2(v[8 * c + 2 * j], v[8 * c + 2 * j + 1]);
            const uint32_t a = rowaddr + (uint32_t)((c ^ (lane & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3]) : "memory");
          }
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          const int c0 = o.mode == OUT_F32 ? col0 + 32 * bx : col0;
          const CUtensorMap* map = &kp.tmO[2 * mi + ((o.mode == OUT_BF16_HILO && bx == 1) ? 1 : 0)];
          tma_store_3d(map, slab, c0, row0, b);
          bulk_commit();
        }
        ++nstores;
      }
    };
    // plain stores (unaligned or channel-major outputs).  One tight loop per output mode: with the mode / bounds decided per
    // element the compiler emitted ~20 instructions per value and this path bounded the GEMMs that use it.
    auto store_direct = [&](const Output& o, const float (&v)[64], int col0, int row, int b, bool row_ok) {
      if (!row_ok) return;
      const int ncols = o.ncols ? o.ncols : g.N;
      int nv = ncols - col0;            // valid columns of this group
      if (nv <= 0) return;
      if (nv > 64) nv = 64;
      // row-major rows, or (trans_S) channel-major per clip with the token index running along the rows of this tile
      const long long base = o.trans_S > 0 ? (long long)(row / o.trans_S) * o.bs + (row % o.trans_S)
                                           : (long long)b * o.bs + (long long)row * o.ld;
      const long long cstep = o.trans_S > 0 ? o.ld : 1;
      if (o.mode == OUT_F32) {
        float* p = reinterpret_cast<float*>(o.ptr) + base + (long long)col0 * cstep;
        if (nv == 64) {
#pragma unroll
          for (int j = 0; j < 64; ++j) p[j * cstep] = v[j];
        } else {
#pragma unroll
          for (int j = 0; j < 64; ++j)
            if (j < nv) p[j * cstep] = v[j];
        }
      } else if (E_F16 && o.mode == OUT_F16) {
        __half* p = reinterpret_cast<__half*>(o.ptr) + base + (long long)col0 * cstep;
#pragma unroll
        for (int j = 0; j < 64; ++j)
          if (j < nv) p[j * cstep] = __float2half_rn(v[j]);
      } else {
        __nv_bfloat16* p = reinterpret_cast<__nv_bfloat16*>(o.ptr) + base + (long long)col0 * cstep;
        const bool lo = o.mode == OUT_BF16_HILO;
        if (!lo) {
          if (nv == 64) {
#pragma unroll
            for (int j = 0; j < 64; ++j) p[j * cstep] = __float2bfloat16_rn(v[j]);
          } else {
#pragma unroll
            for (int j = 0; j < 64; ++j)
              if (j < nv) p[j * cstep] = __float2bfloat16_rn(v[j]);
          }
        } else {
          __nv_bfloat16* q = p + o.lo_off;
#pragma unroll
          for (int j = 0; j < 64; ++j) {
            if (j < nv) {
              const __nv_bfloat16 hi = __float2bfloat16_rn(v[j]);
              p[j * cstep] = hi;
              q[j * cstep] = __float2bfloat16_rn(v[j] - __bfloat162float(hi));
            }
          }
        }
      }
    };
    // hand an accumulator buffer back to the MMA issuer (of the leader CTA)
    auto acc_release = [&](uint32_t buf) {
      if constexpr (PAIR) {
        if (rank != 0) { mbar_arrive_cluster(mapa_u32(smem_u32(&bars[B_ACCEMPTY + buf]), crank & ~1u)); return; }
      }
      mbar_arrive(&bars[B_ACCEMPTY + buf]);
    };
    for (int tv = 0; ok; ++tv, ++i) {       // sub-tiles in the issuer's order: tile tile0 + (tv / nu) * tstep, sub-tile tv % nu
      const int t = tile0 + (tv / nu) * tstep;
      if (t >= ntiles) break;
      const int b = t / tiles_per_batch, r = t - b * tiles_per_batch;
      const int tn = r % kp.tiles_n;
      const int m0 = (r / kp.tiles_n) * BMT + (tv % nu) * BMC + (int)rank * BM, n0 = tn * bn;
      const uint32_t buf = i & 1;
      const int row = m0 + q * 32 + lane;
      const bool row_ok = row < g.M && (g.stat_rows == 0 || (long long)b * g.M + row < g.stat_rows);
      float rowterm = 0.f;
      if (g.rowparts != nullptr && row_ok) {
        const float* rp = g.rowparts + ((size_t)b * g.M + row) * g.nparts;
        for (int j = 0; j < g.nparts; ++j) rowterm += rp[j];
      }
      float psum = 0.f, st_ff = 0.f, st_dot = 0.f, st_vv = 0.f;
      if (has_vec && h < nh && m0 + q * 32 < g.M) {   // bias / colvec slices of this warp's groups -> per-warp smem, before the accumulator is due
        __syncwarp();
        for (int cg = 0; cg < ngroups; ++cg) {
          const int colb = n0 + h * half_cols + 64 * cg;
          float* vecs = vecs_w + 128 * cg;
          for (int j = lane; j < 64; j += 32) {
            const int col = colb + j;
            vecs[j] = (g.bias != nullptr && col < g.N) ? g.bias[col] : 0.f;
            vecs[64 + j] = (g.colvec != nullptr && col < g.N) ? g.colvec[col] : 0.f;
          }
        }
        __syncwarp();
      }
      if (!(ok = bwait(&bars[B_ACCFULL + buf], (i >> 1) & 1, kp.err, 721))) break;
      if (w == 0 && lane == 0) { if (tv == 0) TCG_TRACE(5); TCG_TRACE(7); if (tv < 16) TCG_TRACE(16 + tv); }   // first / last / each accumulator handed over
      tc_fence_after();
      if (h >= nh || m0 + q * 32 >= g.M) {
        // nothing to read for this warp (unused column half, or all 32 rows past M: the per-clip GEMMs with M = P = 40 only
        // need two of the four row groups): release the accumulator, keep the psum table dense
        __syncwarp();
        if (lane == 0) acc_release(buf);
        if (psum_p != nullptr && row_ok) psum_p[((size_t)b * g.M + row) * (2 * kp.tiles_n) + 2 * tn + hw] = 0.f;
        if (rowstat_p != nullptr && row_ok)
          *reinterpret_cast<float4*>(rowstat_p + (((size_t)b * g.M + row) * (2 * kp.tiles_n) + 2 * tn + hw) * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
        continue;
      }
      for (int cg = 0; cg < ngroups; ++cg) {
        const int cl = h * half_cols + 64 * cg;       // column inside the tile
        const int col0 = n0 + cl;
        const float* vecs = vecs_w + 128 * cg;
        float v[64];
        {
          uint32_t ra[32], rb[32];
          tmem_ld_x32(tl + 256u * buf + (uint32_t)cl, ra);
          tmem_ld_x32(tl + 256u * buf + (uint32_t)cl + 32u, rb);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) { v[j] = __uint_as_float(ra[j]); v[32 + j] = __uint_as_float(rb[j]); }
        }
        if (cg == ngroups - 1) {   // all TMEM reads of this tile are done: hand the accumulator back early
          tc_fence_before();
          __syncwarp();
          if (lane == 0) acc_release(buf);
        }
        if (has_vec) {
#pragma unroll
          for (int j4 = 0; j4 < 16; ++j4) {
            const float4 bb = *reinterpret_cast<const float4*>(vecs + 4 * j4);
            const float4 cc = *reinterpret_cast<const float4*>(vecs + 64 + 4 * j4);
            v[4 * j4 + 0] = fmaf(rowterm, cc.x, v[4 * j4 + 0] + bb.x);
            v[4 * j4 + 1] = fmaf(rowterm, cc.y, v[4 * j4 + 1] + bb.y);
            v[4 * j4 + 2] = fmaf(rowterm, cc.z, v[4 * j4 + 2] + bb.z);
            v[4 * j4 + 3] = fmaf(rowterm, cc.w, v[4 * j4 + 3] + bb.w);
          }
        }
        if (g.act == ACT_RELU) {
#pragma unroll
          for (int j = 0; j < 64; ++j) v[j] = fmaxf(v[j], 0.f);
        } else if (g.act == ACT_ABS) {
#pragma unroll
          for (int j = 0; j < 64; ++j) v[j] = fabsf(v[j]);
        }
        if (has_aux) {
          // element-wise epilogue inputs (backward: + upstream gradient, * sign of the |.| argument, ReLU mask)
          if (row_ok) {
            const float* ad = g.addin.ptr ? reinterpret_cast<const float*>(g.addin.ptr) + (long long)b * g.addin.bs + (long long)row * g.addin.ld : nullptr;
            const __nv_bfloat16* sg = g.signin.ptr ? reinterpret_cast<const __nv_bfloat16*>(g.signin.ptr) + (long long)b * g.signin.bs + (long long)row * g.signin.ld : nullptr;
            const __nv_bfloat16* mk = g.mask.ptr ? reinterpret_cast<const __nv_bfloat16*>(g.mask.ptr) + (long long)b * g.mask.bs + (long long)row * g.mask.ld : nullptr;
            const long long acs = g.addin.cs ? g.addin.cs : 1, scs = g.signin.cs ? g.signin.cs : 1, mcs = g.mask.cs ? g.mask.cs : 1;
            if (ad) {   // fp32, read along the rows (coalesced over the lanes when the array is transposed: ld = 1)
#pragma unroll
              for (int j = 0; j < 64; ++j)
                if (col0 + j < g.N) v[j] += __ldg(ad + (col0 + j) * acs);
            }
            // bf16 inputs with the tile's own orientation: this thread's 64 columns are 128 contiguous bytes, read as
            // 16-byte vectors wherever a whole vector lies inside the row (scalar reads for a ragged tail / strided arrays)
            auto apply_bf16 = [&](const __nv_bfloat16* src, long long cs, bool is_sign) {
              const bool vec_ok = cs == 1 && ((reinterpret_cast<uintptr_t>(src + col0) & 15) == 0);
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                const int c8 = col0 + 8 * q;
                if (c8 >= g.N) break;
                uint32_t wds[4];
                if (vec_ok && c8 + 8 <= g.N) {
                  const uint4 u = __ldg(reinterpret_cast<const uint4*>(src + c8));
                  wds[0] = u.x; wds[1] = u.y; wds[2] = u.z; wds[3] = u.w;
                } else {
#pragma unroll
                  for (int e = 0; e < 4; ++e) {
                    const int ca = c8 + 2 * e, cb = ca + 1;
                    const uint32_t lo = ca < g.N ? (uint32_t)__bfloat16_as_ushort(src[ca * cs]) : 0u;
                    const uint32_t hi = cb < g.N ? (uint32_t)__bfloat16_as_ushort(src[cb * cs]) : 0u;
                    wds[e] = lo | (hi << 16);
                  }
                }
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                  // bf16 -> fp32 is a 16-bit shift; only sign and zero-ness matter here
                  const float x = __uint_as_float((e & 1) ? (wds[e >> 1] & 0xFFFF0000u) : (wds[e >> 1] << 16));
                  float& y = v[8 * q + e];
                  if (is_sign) y = x > 0.f ? y : (x < 0.f ? -y : 0.f);
                  else y = x > 0.f ? y : 0.f;
                }
              }
            };
            if (sg) apply_bf16(sg, scs, true);
            if (mk) apply_bf16(mk, mcs, false);
          }
        }
        if (stat_cached) {
          // Few rows per batch item (the per-clip pooling GEMMs with M = P <= 64): every tile of this CTA pairs the same rows
          // with the same vectors, and the warps of the two upper row groups are idle -- their staging slabs hold this
          // warp's second column group.  The 32 x 64 slices are read once per CTA (whole 256-byte rows, chunks swizzled by
          // the row: conflict-free on both sides) instead of once per tile by every SM from the same few L2 lines.
          float* stg = reinterpret_cast<float*>(smem + SM_STG + (uint32_t)(w + 2 * cg) * 2u * SLAB_BYTES);
          if ((cg ? stat_key1 : stat_key0) != col0) {
            stat_fill(cg, col0);
            if (cg) stat_key1 = col0; else stat_key0 = col0;
          }
#pragma unroll
          for (int j4 = 0; j4 < 16; ++j4) {
            const float4 w4 = *reinterpret_cast<const float4*>(stg + lane * 64 + ((j4 ^ (lane & 7)) << 2));
            st_ff = fmaf(v[4 * j4], v[4 * j4], st_ff);         st_dot = fmaf(v[4 * j4], w4.x, st_dot);
            st_ff = fmaf(v[4 * j4 + 1], v[4 * j4 + 1], st_ff); st_dot = fmaf(v[4 * j4 + 1], w4.y, st_dot);
            st_ff = fmaf(v[4 * j4 + 2], v[4 * j4 + 2], st_ff); st_dot = fmaf(v[4 * j4 + 2], w4.z, st_dot);
            st_ff = fmaf(v[4 * j4 + 3], v[4 * j4 + 3], st_ff); st_dot = fmaf(v[4 * j4 + 3], w4.w, st_dot);
            st_vv = fmaf(w4.x, w4.x, fmaf(w4.y, w4.y, fmaf(w4.z, w4.z, fmaf(w4.w, w4.w, st_vv))));
          }
        } else if (rowstat_p != nullptr && row_ok) {   // ||row||^2 and <row, vector of this row's prototype> over this group's columns
          const float* vr = g.dotvec + (long long)(row % g.dot_mod) * g.dot_ld + col0;
          if (col0 + 64 <= g.N && ((reinterpret_cast<uintptr_t>(vr) & 15) == 0)) {
#pragma unroll
            for (int j4 = 0; j4 < 16; ++j4) {
              const float4 w4 = __ldg(reinterpret_cast<const float4*>(vr) + j4);
              st_ff = fmaf(v[4 * j4], v[4 * j4], st_ff);         st_dot = fmaf(v[4 * j4], w4.x, st_dot);
              st_ff = fmaf(v[4 * j4 + 1], v[4 * j4 + 1], st_ff); st_dot = fmaf(v[4 * j4 + 1], w4.y, st_dot);
              st_ff = fmaf(v[4 * j4 + 2], v[4 * j4 + 2], st_ff); st_dot = fmaf(v[4 * j4 + 2], w4.z, st_dot);
              st_ff = fmaf(v[4 * j4 + 3], v[4 * j4 + 3], st_ff); st_dot = fmaf(v[4 * j4 + 3], w4.w, st_dot);
              st_vv = fmaf(w4.x, w4.x, fmaf(w4.y, w4.y, fmaf(w4.z, w4.z, fmaf(w4.w, w4.w, st_vv))));
            }
          } else {
#pragma unroll
            for (int j = 0; j < 64; ++j)
              if (col0 + j < g.N) { const float wv = __ldg(vr + j); st_ff = fmaf(v[j], v[j], st_ff); st_dot = fmaf(v[j], wv, st_dot); st_vv = fmaf(wv, wv, st_vv); }
          }
        }
        if (psum_p != nullptr) {
          if (col0 + 64 <= g.N) {
            if (g.psum_rounded) {
#pragma unroll
              for (int j = 0; j < 64; ++j) psum += round_bf16(v[j]);
            } else {
#pragma unroll
              for (int j = 0; j < 64; ++j) psum += v[j];
            }
          } else {
            const bool rounded = g.psum_rounded != 0;
#pragma unroll
            for (int j = 0; j < 64; ++j) psum += (col0 + j < g.N) ? (rounded ? round_bf16(v[j]) : v[j]) : 0.f;
          }
        }
#pragma unroll
        for (int mi = 0; mi < 2; ++mi) {
          const Output& o = g.out[mi];
          if (!E_OUT || o.mode == OUT_NONE || (split_out && mi != hw)) continue;
          if (E_ABSOUT && o.absval) {   // |value| next to an output that keeps the sign: only the first output may be the signed one
#pragma unroll
            for (int j = 0; j < 64; ++j) v[j] = fabsf(v[j]);
          }
          if (!E_DIRECT || kp.out_tma[mi]) store_tma(o, mi, v, col0, m0 + q * 32, b);
          else store_direct(o, v, col0, row, b, row_ok);
        }
      }
      if (w == 0 && lane == 0 && tv < 16) TCG_TRACE(32 + tv);   // this tile's rows are out of the registers
      if (psum_p != nullptr && row_ok) psum_p[((size_t)b * g.M + row) * (2 * kp.tiles_n) + 2 * tn + hw] = (split_out && hw == 1) ? 0.f : psum;
      if (rowstat_p != nullptr && row_ok)
        *reinterpret_cast<float4*>(rowstat_p + (((size_t)b * g.M + row) * (2 * kp.tiles_n) + 2 * tn + hw) * 4) =
            (split_out && hw == 1) ? make_float4(0.f, 0.f, 0.f, 0.f) : make_float4(st_ff, st_dot, st_vv, 0.f);
    }
    if (w == 0 && lane == 0) { TCG_TRACE(8); TCG_TRACE1(13); }   // last tile's rows are out of the registers
    if (w == 4 && lane == 0) TCG_TRACE(12);
    if (lane == 0) bulk_wait<0>();   // outstanding TMA stores must complete before the CTA's smem goes away
    __syncwarp();
    if (w == 0 && lane == 0) { TCG_TRACE(9); TCG_TRACE1(14); }
  }
  tc_fence_before();
  __syncthreads();
  if (tid == 0) TCG_TRACE(11);
  if constexpr (PAIR) cluster_sync_all();   // the partner may still read this CTA's shared memory / signal its barriers
  if (warp == 2) { if constexpr (PAIR) tmem_dealloc2(tbase, 512); else tmem_dealloc(tbase, 512); }
  if (tid == 0) TCG_TRACE(10);
}

// -------------------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------------------
namespace {
typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeFn encode_fn() {
  static EncodeFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return reinterpret_cast<EncodeFn>(p);
  }();
  return fn;
}
// 3-D map over [d2][d1][d0] (d0 innermost), strides in bytes, box {b0, b1, 1}
bool make_map(CUtensorMap* m, CUtensorMapDataType dt, int elt, const void* base, unsigned long long d0, unsigned long long d1,
              unsigned long long d2, unsigned long long s1_bytes, unsigned long long s2_bytes, unsigned b0, unsigned b1) {
  EncodeFn fn = encode_fn();
  if (!fn) return false;
  if (((uintptr_t)base & 15) != 0 || (s1_bytes & 15) != 0 || (s2_bytes & 15) != 0) return false;
  cuuint64_t dims[3] = {d0, d1, d2 ? d2 : 1};
  cuuint64_t strides[2] = {s1_bytes, s2_bytes ? s2_bytes : s1_bytes * d1};
  cuuint32_t box[3] = {b0, b1, 1};
  cuuint32_t es[3] = {1, 1, 1};
  (void)elt;
  return fn(m, dt, 3, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
bool out_aligned(const Output& o) {
  const int elt = o.mode == OUT_F32 ? 4 : 2;
  if (((uintptr_t)o.ptr & 15) != 0 || ((o.ld * elt) & 15) != 0 || ((o.bs * elt) & 15) != 0) return false;
  if (o.mode == OUT_BF16_HILO && ((o.lo_off * elt) & 15) != 0) return false;
  return true;
}
}  // namespace

bool available() { return encode_fn() != nullptr; }

static long long* g_trace = nullptr;
static int g_trace_slot = 0;
void set_trace(void* dev_buf) { g_trace = reinterpret_cast<long long*>(dev_buf); g_trace_slot = 0; }



int launch(const Gemm& g, cudaStream_t st) {
  if (g.M <= 0 || g.N <= 0 || g.K <= 0 || g.batch <= 0) return PASN_OK;
  if (g.npass < 1 || g.npass > 4 || (g.bn != 64 && g.bn != 128 && g.bn != 256)) return PASN_ERR_INVALID;
  if (g.ab_f16 && g.npass != 1) return PASN_ERR_INVALID;   // fp16 operands have no lo planes
  const bool f16_out = g.out[0].mode == OUT_F16 || g.out[1].mode == OUT_F16;
  static bool attr_done = false;
  if (!attr_done) {
    const void* fns[] = {(const void*)tc_gemm_kernel<false, EPI_FULL>, (const void*)tc_gemm_kernel<true, EPI_FULL>,
                         (const void*)tc_gemm_kernel<false, EPI_F16>, (const void*)tc_gemm_kernel<true, EPI_F16>,
                         (const void*)tc_gemm_kernel<false, EPI_LEAN>, (const void*)tc_gemm_kernel<true, EPI_LEAN>,
                         (const void*)tc_gemm_kernel<false, EPI_STAT>, (const void*)tc_gemm_kernel<true, EPI_STAT>,
                         (const void*)tc_gemm_kernel<false, EPI_DIRECT>, (const void*)tc_gemm_kernel<true, EPI_DIRECT>,
                         (const void*)tc_gemm_kernel<false, EPI_PSUM>, (const void*)tc_gemm_kernel<true, EPI_PSUM>,
                         (const void*)tc_gemm_kernel<false, EPI_AUX>, (const void*)tc_gemm_kernel<true, EPI_AUX>};
    for (const void* f : fns)
      if (cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES) != cudaSuccess) return PASN_ERR_CUDA;
    attr_done = true;
  }
  // pairs pay off when the main loop is long (big K: +10 % on square GEMMs, tools/bench_gemm.py), from 8 k-block passes per
  // tile.  (With the generic epilogue the K = 512 GEMMs of the chain lost 4 us of 64 to pairs -- the partner CTA's last rows
  // left 1.5-1.9 us after the leader's, tools/trace_gemm.py; with the lean epilogues pairs win there too: config 2 at
  // N = 1024 0.194 -> 0.187 ms, config 5 at N = 32 0.822 -> 0.806 ms.)
  const int kpasses = ceil_div(g.K, BK) * g.npass;
  const bool pair = g.pair != 0 && kpasses >= 8 && g.bn >= 128 && g.M > BM;
  const int cl = pair ? 2 : 1;
  // tall tiles for long main loops: two sub-tiles per CTA share every B stage (and take both accumulator buffers, so the
  // epilogue no longer overlaps the MMAs -- negligible when K is long): a quarter less L2 -> SM traffic per flop
  const bool tall = pair && g.M > cl * BM && kpasses >= 40;   // (24 k-block passes: 285 vs 267 us, slower)
  int* fault = fault_word();   // bounded waits report into the host-mapped sticky fault word
  if (fault == nullptr) return PASN_ERR_CUDA;
  KParams kp;
  kp.g = g;
  kp.err = fault;
  kp.trace = nullptr;
  if (g_trace != nullptr && g_trace_slot < 64) kp.trace = g_trace + 64 * g_trace_slot++;   // debug: a row of stamps per launch
  kp.tall = tall ? 1 : 0;

  kp.tiles_m = ceil_div(g.M, cl * BM * (tall ? 2 : 1));
  kp.tiles_n = ceil_div(g.N, g.bn);
  kp.nkb = ceil_div(g.K, BK);
  if (g.group > 1) {
    if (!(g.a_mn_major && g.b_mn_major && g.a_batched && g.b_batched) || g.npass != 1 || g.K > BK || g.k_rows_per_batch > 0 ||
        g.M > BM || g.group * g.group_rows != g.M || g.group_items <= 0 || g.out[0].mode != OUT_NONE || g.out[1].mode != OUT_NONE ||
        g.rowstat == nullptr || pair)
      return PASN_ERR_INVALID;
    kp.nkb = g.group;   // one k-block per item of the group
  }
  const bool split_k = g.k_rows_per_batch > 0;
  if (split_k && !(g.a_mn_major && g.b_mn_major)) return PASN_ERR_INVALID;
  const CUtensorMapDataType ab_dt = g.ab_f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  if (!g.a_mn_major) {
    if (!make_map(&kp.tmA, ab_dt, 2, g.A, (unsigned long long)g.ka, (unsigned long long)g.M,
                  g.a_batched ? g.batch : 1, (unsigned long long)g.lda * 2, (unsigned long long)g.a_bs * 2, BK, BM))
      return PASN_ERR_ALIGN;
  } else {   // [batch][K rows][ka columns], m contiguous: boxes of 64 m x 64 k
    if (!make_map(&kp.tmA, ab_dt, 2, g.A, (unsigned long long)g.ka,
                  (unsigned long long)(g.a_rows ? g.a_rows : g.K), (g.a_batched && !split_k) ? (g.group > 1 ? g.group_items : g.batch) : 1,
                  (unsigned long long)g.lda * 2, (unsigned long long)g.a_bs * 2, 64, BK))
      return PASN_ERR_ALIGN;
  }
  if (!g.b_mn_major) {
    if (!make_map(&kp.tmB, ab_dt, 2, g.B, (unsigned long long)g.kb,
                  (unsigned long long)(g.b_rows ? g.b_rows : g.N), g.b_batched ? g.batch : 1, (unsigned long long)g.ldb * 2, (unsigned long long)g.b_bs * 2, BK, (unsigned)(pair ? g.bn / 2 : g.bn)))
      return PASN_ERR_ALIGN;
  } else {   // [batch][K rows][kb columns], n contiguous: boxes of 64 n x 64 k
    if (!make_map(&kp.tmB, ab_dt, 2, g.B, (unsigned long long)g.kb,
                  (unsigned long long)(g.b_rows ? g.b_rows : g.K), (g.b_batched && !split_k) ? (g.group > 1 ? g.group_items : g.batch) : 1, (unsigned long long)g.ldb * 2, (unsigned long long)g.b_bs * 2, 64, BK))
      return PASN_ERR_ALIGN;
  }
  for (int mi = 0; mi < 2; ++mi) {
    const Output& o = g.out[mi];
    kp.out_tma[mi] = 0;
    kp.tmO[2 * mi] = kp.tmA;
    kp.tmO[2 * mi + 1] = kp.tmA;
    if (o.mode == OUT_NONE || o.trans_S > 0 || !out_aligned(o)) continue;
    const bool f32 = o.mode == OUT_F32;
    const CUtensorMapDataType dt = f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                       : (o.mode == OUT_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
    const int elt = f32 ? 4 : 2;
    const unsigned long long ncols = o.ncols ? o.ncols : g.N;
    bool okm = make_map(&kp.tmO[2 * mi], dt, elt, o.ptr, ncols, (unsigned long long)g.M, g.batch,
                        (unsigned long long)o.ld * elt, (unsigned long long)o.bs * elt, f32 ? 32 : 64, 32);
    if (okm && o.mode == OUT_BF16_HILO)
      okm = make_map(&kp.tmO[2 * mi + 1], dt, elt, reinterpret_cast<const char*>(o.ptr) + (size_t)o.lo_off * 2,
                     ncols, (unsigned long long)g.M, g.batch, (unsigned long long)o.ld * elt,
                     (unsigned long long)o.bs * elt, 64, 32);
    kp.out_tma[mi] = okm ? 1 : 0;
  }
  static const int num_sms = [] {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    return n;
  }();
  const long long ntiles = (long long)g.batch * kp.tiles_m * kp.tiles_n;
  {
    const int ncl = (int)(ntiles < num_sms / cl ? ntiles : num_sms / cl);   // clusters of 1 or 2 (pair) CTAs
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(cl * ncl); cfg.blockDim = dim3(THREADS); cfg.dynamicSmemBytes = SMEM_BYTES; cfg.stream = st;
    cudaLaunchAttribute at[2];
    int na = 0;
    if (cl > 1) {
      at[na].id = cudaLaunchAttributeClusterDimension;
      at[na].val.clusterDim.x = cl; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1;
      ++na;
    }
    at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
    cfg.attrs = at; cfg.numAttrs = na;
    // the leanest epilogue that can do what this launch asks for
    int need = 0;
    for (int mi = 0; mi < 2; ++mi) {
      if (g.out[mi].mode == OUT_NONE) continue;
      need |= E_BIT_OUT;
      if (!kp.out_tma[mi]) need |= E_BIT_DIRECT;
      if (g.out[mi].absval) need |= E_BIT_ABSOUT;
    }
    if (g.bn == 64 && g.out[0].mode != OUT_NONE && g.out[1].mode != OUT_NONE) need |= E_BIT_DIRECT;   // split between the warp groups
    if (g.addin.ptr || g.signin.ptr || g.mask.ptr) need |= E_BIT_AUX;
    if (g.psum) need |= E_BIT_PSUM;
    if (g.rowstat) need |= E_BIT_STAT;
    // (EPI_AUX: fwd+bwd of 256 clips 1.09-1.10 -> 1.06-1.07 ms; at 64 clips the step is launch-bound and moves with the box)
    static const int variants[] = {EPI_LEAN, EPI_STAT, EPI_DIRECT, EPI_PSUM, EPI_AUX};
    int epi = f16_out ? EPI_F16 : EPI_FULL;   // (fp16 outputs: the fp16 chain's occurrence-map stores only)
    if (!f16_out)
      for (int v : variants)
        if ((v & need) == need) { epi = v; break; }
    cudaError_t e;
#define TCG_LAUNCH(EPI_) (pair ? cudaLaunchKernelEx(&cfg, tc_gemm_kernel<true, EPI_>, kp) : cudaLaunchKernelEx(&cfg, tc_gemm_kernel<false, EPI_>, kp))
    if (epi == EPI_LEAN) e = TCG_LAUNCH(EPI_LEAN);
    else if (epi == EPI_STAT) e = TCG_LAUNCH(EPI_STAT);
    else if (epi == EPI_DIRECT) e = TCG_LAUNCH(EPI_DIRECT);
    else if (epi == EPI_PSUM) e = TCG_LAUNCH(EPI_PSUM);
    else if (epi == EPI_AUX) e = TCG_LAUNCH(EPI_AUX);
    else if (epi == EPI_F16) e = TCG_LAUNCH(EPI_F16);
    else e = TCG_LAUNCH(EPI_FULL);
#undef TCG_LAUNCH
    if (e != cudaSuccess) return PASN_ERR_CUDA;
  }
  PASN_LAUNCH_CHECK();
  count_launch();
  return PASN_OK;
}

}  // namespace tcg
}  // namespace pasn
