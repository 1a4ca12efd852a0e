// K1 of the fused prototype head: the token kernel (see head_sm100.cu for K2, packing and the host side, and for the
// reference computation being replaced: src/models/Video_XProtoNet.py:82-98).  Measurements in profiles/README.md.
//
//   * add-on branch transposed.  acc_A^T[d, voxel] = W1 X^T  (weights are the A operand, the X tile the B operand), so
//     H1^T = relu(. + b1) is converted to bf16 IN PLACE in TMEM (lane = channel d, bias is a per-lane scalar) and feeds
//     the pooling MMA  FEpartial^T[d,(slot,p)] = H1^T O  as its TMEM A operand.  H1 never goes through shared memory.
//   * the CTA needs 187 KB of shared memory, which keeps 60 KB of L1.  The NCDHW gather is done with cp.async (8-byte
//     LDGSTS, three 16 KB chunks in flight per SM): 22 B/clk/SM measured against 11 B/clk/SM for an
//     ld.global -> st.shared version (whose register loads all shared one scoreboard, i.e. one unit in flight) and
//     13 B/clk/SM for cp.async when only 28 KB of L1 were left.
//   * per tile, layer 1 issues both accumulators chunk by chunk from one gathered X chunk: acc_G = X W3^T into TMEM
//     columns [0,256), acc_A^T into [256,512).  The serial chain G1 -> G2 -> O -> pooling follows; its MMAs come from a
//     second issuing thread, so its waits on the epilogue stay off the layer-1 issuer's path.
//
// Warp roles (16 warps): 0 layer-1 MMA issuer, 1 weight producer (cp.async.bulk), 2 tail MMA issuer (G2, O, pooling),
// 3 occurrence-map store + column sums, 4-7 X gather, 8-15 epilogue (TMEM lane quadrant = warp % 4, two per quadrant).
#include "head_sm100_shared.cuh"

namespace pasn {
using namespace sm100;
using namespace k1;

namespace {

constexpr int XSLOTS = 4, WSLOTS = 3, XDEPTH = XSLOTS - 1;   // XDEPTH chunks of cp.async in flight per producer warp
constexpr uint32_t XSLOT_BYTES = 16384, WSLOT_BYTES = 32768;
constexpr int K1_WARPS = 16, K1_THREADS = K1_WARPS * 32;
constexpr int W_MMA = 0, W_WPROD = 1, W_TAIL = 2, W_OCC = 3, W_X0 = 4, W_EPI0 = 8;
// shared-memory map (offsets from a 1024-byte aligned base); total < 195 KB so that 60 KB stay L1
constexpr uint32_t SM_X = 0;
constexpr uint32_t SM_W = SM_X + XSLOTS * XSLOT_BYTES;            // 65536
constexpr uint32_t SM_OS = SM_W + WSLOTS * WSLOT_BYTES;           // 163840
constexpr uint32_t OS_BYTES_MAX = TILE_M * 2 * PP_MAX * 2;        // 24576
constexpr uint32_t SM_BIAS = SM_OS + OS_BYTES_MAX;                // 188416  b3[256] b1[256] b4[128] fp32
constexpr uint32_t SM_BAR = SM_BIAS + (DD + DD + DH) * 4;         // 190976
constexpr uint32_t SM_MISC = SM_BAR + 36 * 8;                     // 191232
constexpr uint32_t K1_SMEM = SM_MISC + 64;                        // 191296
static_assert(K1_SMEM <= 195 * 1024, "keep the 196 KB carve-out (60 KB of L1 for the cp.async gather)");

enum {
  B_XFULL = 0, B_XEMPTY = XSLOTS, B_WFULL = 2 * XSLOTS, B_WEMPTY = 2 * XSLOTS + WSLOTS, B_GDONE = 2 * XSLOTS + 2 * WSLOTS, B_ADONE, B_G1READY, B_G2DONE, B_G2READY, B_ODONE,
  B_OSREADY, B_OSEMPTY, B_H1TREADY, B_FEDONE0, B_FEDONE1, B_GBFREE, B_ABFREE, B_W4RDY, B_W4BRDY, B_W5RDY, B_COUNT
};
static_assert(B_COUNT <= 36, "barrier table");

// TMEM columns (512 x 128 lanes)
//   GB [  0,256)  acc_G fp32 (lane = voxel) -> G1 bf16 at [0,64) + [192,256) -> acc_G2 fp32 [64,192) -> G2 bf16 at
//                 [64,96) + [128,160) -> acc_O fp32 [0,64)
//   AB [256,512)  acc_A^T fp32, two channel halves [256,384) and [384,512) (lane = d % 128, column = voxel) ->
//                 H1^T bf16 at [256,320) (half 0, packed upwards) and [448,512) (half 1, packed downwards) ->
//                 FEpartial^T fp32 at [320, 320 + 2*PP) (lane = d % 128), one channel half after the other
constexpr uint32_t COL_AT = 256, COL_H1T0 = 256, COL_H1T1 = 448, COL_FE = 320;

}  // namespace

// Everything that is fixed per launch is a template parameter: the kernel is ~7 k instructions for five warp roles, and code
// of input kinds that do not run still spreads the ones that do over more instruction-cache lines
// (ncu: 8 % of the issue slots lost to instruction fetch before; bf16 NCDHW instantiation 8256 -> ~5.5 k instructions).
// IN: 0 = bf16 [N,C,S], 1 = bf16 channels_last [N,S,C], 2 = fp32 [N,C,S] (rounded to bf16 on the fly), 3 = fp16 [N,C,S],
// 4 = fp16 channels_last.  fp16 maps are gathered byte for byte like bf16 ones; only the layer-1 MMAs (fp16 x fp16 against
// fp16 weight images: kind::f16 takes no mixed fp16 / bf16 operands) and the map store differ.
template <int PP, bool TRACE, int IN>
__global__ void __launch_bounds__(K1_THREADS, 1) head_tokens2_kernel(const K1Params p) {
  constexpr bool nsc = IN == 1 || IN == 4, f32_in = IN == 2, f16_in = IN == 3 || IN == 4;
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM_BAR);
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(smem + SM_MISC);
  volatile int* abort_s = reinterpret_cast<volatile int*>(smem + SM_MISC + 8);
  float* sb3 = reinterpret_cast<float*>(smem + SM_BIAS);
  float* sb1 = sb3 + DD;
  float* sb4 = sb1 + DD;

  constexpr int NPOOL = 2 * PP;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int c_begin = blockIdx.x * p.clips_per_cta;
  int ncl = p.N - c_begin;
  if (ncl > p.clips_per_cta) ncl = p.clips_per_cta;
  if (ncl <= 0) return;
  const int S = p.S;
  const int ntok = ncl * S;
  const int ntiles = (ntok + TILE_M - 1) / TILE_M;
  const PackedLayout PL = packed_layout(p.C);
  Ctx ctx{p.err, abort_s, p.fault};

  if ((smem_u32(smem) & 1023u) != 0) {  // swizzled layouts need the 1024-byte alignment we asked for
    if (tid == 0) atomicCAS(p.err, 0, 900);
    return;
  }

  if (tid == 0) {
    *abort_s = 0;
    for (int i = 0; i < XSLOTS; ++i) { mbar_init(&bars[B_XFULL + i], 4); mbar_init(&bars[B_XEMPTY + i], 1); }
    for (int i = 0; i < WSLOTS; ++i) { mbar_init(&bars[B_WFULL + i], 1); mbar_init(&bars[B_WEMPTY + i], 1); }
    mbar_init(&bars[B_GDONE], 1);
    mbar_init(&bars[B_ADONE], 1);
    mbar_init(&bars[B_G1READY], 8);
    mbar_init(&bars[B_G2DONE], 1);
    mbar_init(&bars[B_G2READY], 8);
    mbar_init(&bars[B_ODONE], 1);
    mbar_init(&bars[B_OSREADY], 8);
    mbar_init(&bars[B_OSEMPTY], 2);   // pooling MMAs retired + occurrence warp (map store and column sums)
    mbar_init(&bars[B_H1TREADY], 8);
    mbar_init(&bars[B_FEDONE0], 1);
    mbar_init(&bars[B_FEDONE1], 1);
    mbar_init(&bars[B_GBFREE], 8);
    mbar_init(&bars[B_ABFREE], 8);    // both channel halves drained their FEpartial^T columns
    mbar_init(&bars[B_W4RDY], 1);
    mbar_init(&bars[B_W4BRDY], 1);
    mbar_init(&bars[B_W5RDY], 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(tmem_ptr_s, 512);
  {
    const float* gb = reinterpret_cast<const float*>(p.packed + PL.off_bias);
    for (int i = tid; i < DD + DD + DH; i += K1_THREADS) sb3[i] = gb[i];
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  griddep_launch_dependents();   // K2 may start launching (its CTAs only fit on an SM once one of ours has exited)
  if constexpr (TRACE) {
    if (tid == 0 && p.trace != nullptr && blockIdx.x == 0) {
      long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      p.trace[768 + 0] = t;
    }
  }
  const uint32_t tbase = *tmem_ptr_s;
  const uint32_t x_base = smem_u32(smem + SM_X), w_base = smem_u32(smem + SM_W), os_base = smem_u32(smem + SM_OS);
  const int nkc = p.nkc;

  if (warp == W_MMA) {
    // ------------------------------------------------------------------ MMA issuer (one elected thread)
    // The tensor pipe only queues about three MMAs ahead of the issuing thread (probe_rate.cu: a block of 4 N=256 MMAs
    // tolerates ~250 cycles of issuer-side work before the pipe runs dry, a block of N=128 MMAs none), so everything
    // between two issue blocks is kept to a few dozen straight-line instructions:
    //   * the whole loop runs inside `if (elect_one())`, so ptxas knows one thread is active and feeds the uniform
    //     registers tcgen05 wants with plain R2UR (under `if (lane == 0)` every operand went through an
    //     ELECT / R2UR.BROADCAST loop, ~16 instructions per MMA);
    //   * descriptors are (lo, hi) halves advanced by 32-bit adds, ring slots / phases are kept incrementally;
    //   * the full barriers of the next X chunk and weight stage are probed (test_wait) right after the current ones
    //     were consumed, so the probe's round trip overlaps the issue; the bounded spin is out of line;
    //   * no clock reads unless TRACE.
    if (elect_one()) {
      auto stamp = [&](int tile, int slot) {
        if constexpr (TRACE) K1_TRACE(0, tile, slot);
      };
      // X tile: MN-major (voxels contiguous) for NCDHW input, K-major (channels contiguous) for channels_last input
      const uint32_t x_mn = nsc ? 0u : 1u;
      // A = X tile, B = W3 chunk (K-major) / A = W1 half chunk (K-major), B = X tile; fp16 maps: both operands fp16
      const uint32_t idesc_g = f16_in ? make_idesc_16(128, 256, 0, 0, x_mn, 0) : make_idesc_bf16(128, 256, x_mn, 0);
      const uint32_t idesc_a = f16_in ? make_idesc_16(128, 128, 0, 0, 0, x_mn) : make_idesc_bf16(128, 128, 0, x_mn);
      const uint32_t xk = nsc ? 2u : 128u;                          // descriptor advance per K step of 16 channels
      constexpr uint32_t HI_SW128 = desc_hi(1024, SWZ_128B);   // X tile (MN-major) and weight images (K-major): SBO 1024
      const uint32_t tb = tbase;
      const uint32_t x_lo0 = desc_lo(x_base, nsc ? 16u : 8192u), w_lo0 = desc_lo(w_base, 16);
      const uint32_t bar0 = smem_u32(bars);
      auto baddr = [&](int b) -> uint32_t { return bar0 + 8u * (uint32_t)b; };
      const uint32_t njobs = (uint32_t)ntiles * (uint32_t)nkc;
      uint32_t xs = 0, xph = 0, xcount = 0;   // X ring: slot and phase parity of the next job, jobs taken so far
      uint32_t ws = 0, wph = 0;               // weight ring
      bool xr = false, wr = false;            // "already seen full" for the next job / stage (probed early)
      bool ok = true;
      long long xwait = 0, wwait = 0;         // TRACE only: cycles blocked on X chunks / weight stages

      // wait for the next X job (slot returned in s), advance the ring, probe the job after it
      auto take_x = [&](uint32_t& s) -> bool {
        s = xs;
        bool r = true;
        if (!xr) {
          long long t0 = 0;
          if constexpr (TRACE) t0 = clock64();
          r = bwait(&bars[B_XFULL + xs], xph, ctx, 102);
          if constexpr (TRACE) xwait += clock64() - t0;
        }
        ++xcount;
        xs = xs + 1 == XSLOTS ? 0 : xs + 1;
        xph ^= (xs == 0) ? 1u : 0u;
        xr = xcount < njobs && mbar_test_wait(&bars[B_XFULL + xs], xph);
        return r;
      };
      auto take_w = [&](uint32_t& s) -> bool {
        s = ws;
        bool r = true;
        if (!wr) {
          long long t0 = 0;
          if constexpr (TRACE) t0 = clock64();
          r = bwait(&bars[B_WFULL + ws], wph, ctx, 103);
          if constexpr (TRACE) wwait += clock64() - t0;
        }
        ws = ws + 1 == WSLOTS ? 0 : ws + 1;
        wph ^= (ws == 0) ? 1u : 0u;
        wr = mbar_test_wait(&bars[B_WFULL + ws], wph);
        return r;
      };
      auto issue_g = [&](int kc, uint32_t sx, uint32_t sw) {   // 4 MMAs: one 64-channel chunk into acc_G (X slot freed by issue_a)
        const uint32_t alo = x_lo0 + sx * (XSLOT_BYTES >> 4), blo = w_lo0 + sw * (WSLOT_BYTES >> 4);
        mma_ss_x(tb, alo, HI_SW128, blo, HI_SW128, idesc_g, kc ? 1u : 0u);
#pragma unroll
        for (int k4 = 1; k4 < 4; ++k4) mma_ss_x(tb, alo + k4 * xk, HI_SW128, blo + k4 * 2, HI_SW128, idesc_g, 1u);
        mma_commit_a(baddr(B_WEMPTY) + 8u * sw);
      };
      auto issue_a = [&](int kc, uint32_t sx, uint32_t sw) {   // 8 MMAs: one chunk into both channel halves of acc_A^T
        const uint32_t blo = x_lo0 + sx * (XSLOT_BYTES >> 4), alo = w_lo0 + sw * (WSLOT_BYTES >> 4);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          mma_ss_x(tb + COL_AT + 128u * h, alo + h * 1024, HI_SW128, blo, HI_SW128, idesc_a, kc ? 1u : 0u);
#pragma unroll
          for (int k4 = 1; k4 < 4; ++k4)
            mma_ss_x(tb + COL_AT + 128u * h, alo + h * 1024 + k4 * 2, HI_SW128, blo + k4 * xk, HI_SW128, idesc_a, 1u);
        }
        mma_commit_a(baddr(B_WEMPTY) + 8u * sw);
        mma_commit_a(baddr(B_XEMPTY) + 8u * sx);
      };
      auto chunk_g = [&](int kc, uint32_t sx) -> bool {
        uint32_t sw;
        if (!take_w(sw)) return false;
        issue_g(kc, sx, sw);
        return true;
      };
      auto chunk_a = [&](int kc, uint32_t sx) -> bool {
        uint32_t sw;
        if (!take_w(sw)) return false;
        issue_a(kc, sx, sw);
        return true;
      };
      // Weight stages that belong to the tail issuer (W4a, W4b, W5) sit at fixed positions of the stream.  This thread
      // sees every stage in order, so it is the one that waits for them to land (a parity wait by the tail issuer
      // could alias when the slot's previous occupant has not even arrived yet) and then hands them over.
      auto pass_w = [&](int n, int rdy_bar) -> bool {
        for (int i = 0; i < n; ++i) {
          if (!wr && !bwait(&bars[B_WFULL + ws], wph, ctx, 112)) return false;
          ws = ws + 1 == WSLOTS ? 0 : ws + 1;
          wph ^= (ws == 0) ? 1u : 0u;
          wr = false;
        }
        mbar_arrive(&bars[rdy_bar]);
        return true;
      };
      auto chunk_time = [&](int tile, int slot, long long t0) {
        if constexpr (TRACE) {
          if (p.trace != nullptr && blockIdx.x == 0 && tile < 16 && slot < 16) p.trace[(2 * 16 + tile) * 16 + slot] = clock64() - t0;
        }
      };

      for (int tile = 0; tile < ntiles && ok; ++tile) {
        const uint32_t tp = tile & 1;
        stamp(tile, 0);
        if (!(ok = bwait(&bars[B_GBFREE], tp ^ 1, ctx, 101))) break;   // G-branch columns of the previous tile consumed
        tc_fence_after();
        stamp(tile, 1);
        if (!(ok = bwait(&bars[B_ABFREE], tp ^ 1, ctx, 111))) break;   // previous tile's pooling drained
        tc_fence_after();
        stamp(tile, 3);
        // (G, A) blocks per chunk, except that the last `skew` chunks issue their G blocks first: acc_G is then
        // complete -- and G1's conversion can start -- while the add-on blocks of those chunks are still running
        // (their X slots stay held a little longer; at the end of a tile the ring has nothing urgent to prefetch)
        // skew <= XSLOTS - (XDEPTH - 1): a chunk is only published once the XDEPTH - 1 chunks after it were issued,
        // and those need free slots while this thread still holds `skew` of them
        constexpr int SKEW = XSLOTS - (XDEPTH - 1) < 3 ? XSLOTS - (XDEPTH - 1) : 3;
        // (only for channels_last input: the NCDHW gather is the slower one and does not like waiting for two chunks
        // before the add-on block of the first -- measured 159.6 vs 157.3 us -- while channels_last gains 2-4 %)
        const int skew = !nsc ? 0 : (nkc < SKEW ? nkc : SKEW), k_skew = nkc - skew;
        for (int kc = 0; kc < k_skew && ok; ++kc) {
          long long tc0 = 0;
          if constexpr (TRACE) tc0 = clock64();
          uint32_t sx;
          ok = take_x(sx) && chunk_g(kc, sx) && chunk_a(kc, sx);
          chunk_time(tile, kc, tc0);
        }
        uint32_t sxs[3] = {0, 0, 0};
        for (int j = 0; j < skew && ok; ++j) ok = take_x(sxs[j]) && chunk_g(k_skew + j, sxs[j]);
        if (!ok) break;
        mma_commit_a(baddr(B_GDONE));
        stamp(tile, 2);
        for (int j = 0; j < skew && ok; ++j) ok = chunk_a(k_skew + j, sxs[j]);
        if (!ok) break;
        mma_commit_a(baddr(B_ADONE));
        stamp(tile, 6);
        // the two halves of W4 are handed over one by one: the first eight G2 MMAs only need the first (the stages of
        // the chain are requested late -- their ring slots free when the last layer-1 blocks retire -- and land ~0.5 k cycles apart)
        ok = pass_w(1, B_W4RDY) && pass_w(1, B_W4BRDY) && pass_w(1, B_W5RDY);
        if constexpr (TRACE) {
          if (p.trace != nullptr && blockIdx.x == 0 && tile < 16) {
            p.trace[(0 * 16 + tile) * 16 + 11] = xwait;
            p.trace[(0 * 16 + tile) * 16 + 12] = wwait;
          }
          xwait = wwait = 0;
        }
      }
    }
  } else if (warp == W_TAIL) {
    // ------------------------------------------------------------------ tail MMA issuer (one elected thread)
    // The serial chain of a tile -- G2 = G1 W4^T, O = G2 W5^T, pooling halves -- waits on the epilogue between every
    // step.  A second issuing thread keeps those waits off the layer-1 issuer's path: the tensor pipe interleaves the two
    // streams, and all ordering between them goes through the mbarriers anyway.  Its weight stages sit at fixed
    // positions of the shared ring (the layer-1 issuer steps over them).
    if (elect_one()) {
      const uint32_t idesc_g2 = make_idesc_bf16(128, 128, 0, 0);
      const uint32_t idesc_o = make_idesc_bf16(128, 64, 0, 0);
      const uint32_t idesc_pool = make_idesc_bf16(128, NPOOL, 0, 1);  // A = H1^T in TMEM, B = Os (MN-major, no swizzle)
      constexpr uint32_t lbo_os = (uint32_t)(NPOOL / 8) * 128u;
      constexpr uint32_t HI_SW128 = desc_hi(1024, SWZ_128B), HI_OS = desc_hi(128, SWZ_NONE);
      const uint32_t tb = tbase;
      const uint32_t w_lo0 = desc_lo(w_base, 16), os_lo0 = desc_lo(os_base, lbo_os);
      const uint32_t bar0 = smem_u32(bars);
      auto baddr = [&](int b) -> uint32_t { return bar0 + 8u * (uint32_t)b; };
      const uint32_t stages_per_tile = 2u * (uint32_t)nkc + 3u;
      const uint32_t off_w4 = 2u * (uint32_t)nkc, off_w5 = off_w4 + 2u;   // after the tile's layer-1 stages
      bool ok = true;
      // stages are handed over by the layer-1 issuer (B_W4RDY / B_W5RDY) once they have landed

      for (int tile = 0; tile < ntiles && ok; ++tile) {
        const uint32_t tp = tile & 1;
        const uint32_t base = (uint32_t)tile * stages_per_tile;
        // ---- G2 = G1 W4^T : A from TMEM (cols [0,64) + [192,256)), D = [64,192)
        if (!(ok = bwait(&bars[B_G1READY], tp, ctx, 104))) break;
        if constexpr (TRACE) K1_TRACE(0, tile, 9);
        if (!(ok = bwait(&bars[B_W4RDY], tp, ctx, 113))) break;
        if constexpr (TRACE) K1_TRACE(0, tile, 10);
        tc_fence_after();
#pragma unroll
        for (int st = 0; st < 2; ++st) {
          if (st == 1 && !(ok = bwait(&bars[B_W4BRDY], tp, ctx, 115))) break;
          const uint32_t sw = (base + off_w4 + st) % WSLOTS;
          const uint32_t blo = w_lo0 + sw * (WSLOT_BYTES >> 4);
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            mma_ts_x(tb + 64u, tb + (st ? 192u : 0u) + 8u * kk, blo + (kk >> 2) * 1024 + (kk & 3) * 2, HI_SW128, idesc_g2,
                     (st | kk) ? 1u : 0u);
          mma_commit_a(baddr(B_WEMPTY) + 8u * sw);
        }
        if (!ok) break;
        mma_commit_a(baddr(B_G2DONE));
        if constexpr (TRACE) K1_TRACE(0, tile, 4);
        // ---- O = G2 W5^T : A from TMEM (cols [64,96) + [128,160)), D = [0,64)
        if (!(ok = bwait(&bars[B_G2READY], tp, ctx, 106) && bwait(&bars[B_W5RDY], tp, ctx, 114))) break;
        tc_fence_after();
        {
          const uint32_t sw = (base + off_w5) % WSLOTS;
          const uint32_t blo = w_lo0 + sw * (WSLOT_BYTES >> 4);
#pragma unroll
          for (int ks = 0; ks < 8; ++ks) {
            const uint32_t a_col = ks < 4 ? 64u + 8u * ks : 128u + 8u * (ks - 4);
            mma_ts_x(tb, tb + a_col, blo + (ks >> 2) * 512 + (ks & 3) * 2, HI_SW128, idesc_o, ks ? 1u : 0u);
          }
          mma_commit_a(baddr(B_WEMPTY) + 8u * sw);
          mma_commit_a(baddr(B_ODONE));
        }
        if constexpr (TRACE) K1_TRACE(0, tile, 5);
        // ---- pooling FEpartial^T = H1^T O, one channel half after the other (they share the FEpartial^T columns)
#pragma unroll
        for (int step = 0; step < 2; ++step) {
          // half 0 lands in [320, 320+NPOOL), half 1 in the idle G-branch columns [0, NPOOL): issued back to back
          if (step == 0 && !(ok = bwait(&bars[B_H1TREADY], tp, ctx, 108) && bwait(&bars[B_OSREADY], tp, ctx, 109))) break;
          tc_fence_after();
          const uint32_t a0 = step ? COL_H1T1 : COL_H1T0;
          const uint32_t d0 = step ? 0u : COL_FE;
#pragma unroll
          for (int ks = 0; ks < 8; ++ks)
            mma_ts_x(tb + d0, tb + a0 + 8u * ks, os_lo0 + ks * (2 * lbo_os / 16), HI_OS, idesc_pool, ks ? 1u : 0u);
          if (step == 0) mma_commit_a(baddr(B_FEDONE0));
          else { mma_commit_a(baddr(B_FEDONE1)); mma_commit_a(baddr(B_OSEMPTY)); }
          if constexpr (TRACE) K1_TRACE(0, tile, 7 + step);
        }
      }
    }
  } else if (warp == W_WPROD) {
    // ------------------------------------------------------------------ weight producer (one thread)
    // stage order = consumption order of the issuer: (W3[k], W1[k]) pairs, for the last `skew` chunks all W3 before
    // all W1 (skewed issue order), then W4a, W4b, W5.
    if (lane == 0) {
      uint32_t wst = 0;
      bool ok = true;
      auto put = [&](size_t src, uint32_t bytes) -> bool {
        const uint32_t ws = wst % WSLOTS, wph = (wst / WSLOTS) & 1;
        ++wst;
        if (!bwait(&bars[B_WEMPTY + ws], wph ^ 1, ctx, 201)) return false;
        mbar_arrive_expect_tx(&bars[B_WFULL + ws], bytes);
        for (uint32_t o = 0; o < bytes; o += 16384)
          bulk_g2s(w_base + ws * WSLOT_BYTES + o, p.packed + src + o, 16384, &bars[B_WFULL + ws]);
        return true;
      };
      for (int tile = 0; tile < ntiles && ok; ++tile) {
        constexpr int SKEW = XSLOTS - (XDEPTH - 1) < 3 ? XSLOTS - (XDEPTH - 1) : 3;
        const int skew = !nsc ? 0 : (nkc < SKEW ? nkc : SKEW), k_skew = nkc - skew;
        for (int kc = 0; kc < k_skew && ok; ++kc)
          ok = put(PL.off_l1 + (size_t)(2 * kc) * 32768, 32768) && put(PL.off_l1 + (size_t)(2 * kc + 1) * 32768, 32768);
        for (int kc = k_skew; kc < nkc && ok; ++kc) ok = put(PL.off_l1 + (size_t)(2 * kc) * 32768, 32768);
        for (int kc = k_skew; kc < nkc && ok; ++kc) ok = put(PL.off_l1 + (size_t)(2 * kc + 1) * 32768, 32768);
        ok = ok && put(PL.off_w4, 32768) && put(PL.off_w4 + 32768, 32768) && put(PL.off_w5, 16384);
      }
    }
  } else if (warp >= W_X0 && warp < W_X0 + 4) {
    // ------------------------------------------------------------------ X producers: NCDHW gather -> MN-major SW128
    // Four warps, each owning 16 of the 64 channels of a chunk; lane l owns voxels 4l..4l+3 of the tile, so one
    // warp-wide 8-byte cp.async is a coalesced 256-byte run of one channel row, written straight into the swizzled
    // operand layout (zero fill past the clip range).  XDEPTH chunks are in flight per warp; a chunk is published
    // (wait_group, cross-proxy fence, one arrive per warp) once the chunks issued after it are on their way.  The
    // 16-byte L1-bypassing form needs an alignment NCDHW rows (392-byte pitch) only have for every other channel; TMA
    // needs 16-byte global strides.  Job g is chunk g % nkc of tile g / nkc.
    const int xw = warp - W_X0;
    const uint32_t njobs = (uint32_t)ntiles * (uint32_t)nkc;
    bool ok = true;
    if (nsc) {
      // channels_last feature map [N][S][C]: a voxel's 64 channels of a chunk are 128 contiguous, 16-byte aligned bytes,
      // i.e. one row of the K-major SWIZZLE_128B operand image.  16-byte L1-bypassing cp.async: eight lanes per voxel row,
      // four rows per warp instruction, 32 rows per warp.  Voxels of consecutive clips are contiguous in this layout.
      uint32_t pub = 0;
      auto publish = [&]() {
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars[B_XFULL + (pub % XSLOTS)]);
        ++pub;
      };
      const int sub = lane & 7, r4 = lane >> 3;
      for (uint32_t g = 0; g < njobs; ++g) {
        const uint32_t xs = g % XSLOTS, xph = (g / XSLOTS) & 1;
        if (!bwait(&bars[B_XEMPTY + xs], xph ^ 1, ctx, 301)) { ok = false; break; }
        const int tile = (int)(g / (uint32_t)nkc);
        const int kc = (int)(g - (uint32_t)tile * (uint32_t)nkc);
        const uint32_t dst0 = x_base + xs * XSLOT_BYTES;
        const __nv_bfloat16* src0 = p.feat + ((size_t)c_begin * S + (size_t)tile * TILE_M) * p.C + kc * 64 + sub * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int row = xw * 32 + j * 4 + r4;
          const bool valid = tile * TILE_M + row < ntok;
          cp_async_16(dst0 + off_kmajor_sw128(row, sub * 8), src0 + (size_t)(valid ? row : 0) * p.C, valid ? 16u : 0u);
        }
        cp_async_commit();
        if (pub + (XDEPTH - 1) <= g) {
          cp_async_wait<XDEPTH - 1>();
          publish();
        }
      }
      if (ok) {
        cp_async_wait<0>();
        while (pub < njobs) publish();
      }
    } else if (!f32_in) {
      const uint64_t pol_first = l2_policy_evict_first();
      uint32_t pub = 0;
      auto publish = [&]() {
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars[B_XFULL + (pub % XSLOTS)]);
        ++pub;
      };
      for (uint32_t g = 0; g < njobs; ++g) {
        const uint32_t xs = g % XSLOTS, xph = (g / XSLOTS) & 1;
        if (!bwait(&bars[B_XEMPTY + xs], xph ^ 1, ctx, 301)) { ok = false; break; }
        const int tile = (int)(g / (uint32_t)nkc);
        const int kc = (int)(g - (uint32_t)tile * (uint32_t)nkc);
        const int t = tile * TILE_M + 4 * lane;
        const bool valid = t < ntok;
        const int clipl = valid ? t / S : 0;
        const int s = valid ? t - clipl * S : 0;
        // virtual clip -> (real clip, voxel group): rows of the feature map keep the real pitch SR
        const int vc = c_begin + clipl, rc = vc / p.G, vg = vc - rc * p.G;
        const __nv_bfloat16* src = p.feat + ((size_t)rc * p.C + kc * 64 + xw * 16) * p.SR + (size_t)vg * S + s;
        const uint32_t dst0 = x_base + xs * XSLOT_BYTES;
#pragma unroll
        for (int j = 0; j < 16; ++j)
          cp_async_8_hint(dst0 + off_mnmajor_sw128(4 * lane, xw * 16 + j, 8192), src + (size_t)j * p.SR, valid ? 8u : 0u, pol_first);
        cp_async_commit();
        if (pub + (XDEPTH - 1) <= g) {
          cp_async_wait<XDEPTH - 1>();
          publish();
        }
      }
      if (ok) {
        cp_async_wait<0>();
        while (pub < njobs) publish();
      }
    } else {
      // fp32 feature maps ("bf16 compute" mode, opt-in): 16-byte loads of 4 voxels, rounded to bf16 on the way into
      // smem.  Units are 8 channel rows (u = 2*job + half) so the raw loads of the next unit fit in registers.
      float4 qa[8], qb[8];
      const uint32_t nunits = 2 * njobs;
      auto load32 = [&](uint32_t u, float4* q) {
        const uint32_t g = u >> 1, h = u & 1;
        const int tile = (int)(g / (uint32_t)nkc);
        const int kc = (int)(g - (uint32_t)tile * (uint32_t)nkc);
        const int t = tile * TILE_M + 4 * lane;
        const bool valid = t < ntok;
        const int clipl = valid ? t / S : 0;
        const int s = valid ? t - clipl * S : 0;
        const int vc = c_begin + clipl, rc = vc / p.G, vg = vc - rc * p.G;
        const float* src = p.feat32 + ((size_t)rc * p.C + kc * 64 + xw * 16 + 8 * h) * p.SR + (size_t)vg * S + s;
#pragma unroll
        for (int j = 0; j < 8; ++j) q[j] = valid ? ldg_nc_na_v4f(src + (size_t)j * p.SR) : make_float4(0.f, 0.f, 0.f, 0.f);
      };
      auto store32 = [&](uint32_t u, const float4* q) -> bool {
        const uint32_t g = u >> 1, h = u & 1;
        const uint32_t xs = g % XSLOTS, xph = (g / XSLOTS) & 1;
        if (h == 0 && !bwait(&bars[B_XEMPTY + xs], xph ^ 1, ctx, 301)) return false;
        const uint32_t dst0 = x_base + xs * XSLOT_BYTES;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          st_shared_v2(dst0 + off_mnmajor_sw128(4 * lane, xw * 16 + 8 * h + j, 8192),
                       make_uint2(pack_bf16x2(q[j].x, q[j].y), pack_bf16x2(q[j].z, q[j].w)));
        if (h == 1) {
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(&bars[B_XFULL + xs]);
        }
        return true;
      };
      if (nunits > 0) load32(0, qa);
      for (uint32_t u = 0; u < nunits && ok; u += 2) {
        load32(u + 1, qb);
        if (!(ok = store32(u, qa))) break;
        if (u + 2 < nunits) load32(u + 2, qa);
        ok = store32(u + 1, qb);
      }
    }
  } else if (warp == W_OCC) {
    // ------------------------------------------------------------------ occurrence warp: Os (smem) -> occurrence map
    // [N][P][S], then the column sums of Os (bias term of W2: sum_s O[p,s]) into Osum [N][P]
    float acc0 = 0.f, acc1 = 0.f;  // running sums of the current clip: p = lane, p = lane + 32
    bool ok = true;
    const unsigned char* os = smem + SM_OS;
    for (int tile = 0; tile < ntiles && ok; ++tile) {
      if (!(ok = bwait(&bars[B_OSREADY], tile & 1, ctx, 402))) break;
      const int first_clip = (tile * TILE_M) / S;
      if (p.occ != nullptr || p.occ32 != nullptr) {
#pragma unroll 1
        for (int grp = 0; grp < 4; ++grp) {
          const int tok = grp * 32 + lane;
          const int t = tile * TILE_M + tok;
          if (t < ntok) {
            const int clipl = t / S, s = t - clipl * S, slot = clipl - first_clip;
            const int vc = c_begin + clipl, rc = vc / p.G, vg = vc - rc * p.G;
            const size_t o0 = ((size_t)rc * p.P) * p.SR + (size_t)vg * S + s;
            const unsigned char* src = os + off_mnmajor_nosw(slot * PP, tok, NPOOL);
            if constexpr (f16_in) {   // O is bf16 in Os; the map leaves in the feature map's type
              __half* orow = reinterpret_cast<__half*>(p.occ) + o0;
#pragma unroll 8
              for (int pp = 0; pp < p.P; ++pp)
                orow[(size_t)pp * p.SR] = __float2half_rn(__bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(src + (pp >> 3) * 128 + (pp & 7) * 2)));
            } else if (!f32_in) {
              __nv_bfloat16* orow = p.occ + o0;
#pragma unroll 8
              for (int pp = 0; pp < p.P; ++pp)
                orow[(size_t)pp * p.SR] = *reinterpret_cast<const __nv_bfloat16*>(src + (pp >> 3) * 128 + (pp & 7) * 2);
            } else {
              float* orow = p.occ32 + o0;
#pragma unroll 8
              for (int pp = 0; pp < p.P; ++pp)
                orow[(size_t)pp * p.SR] = __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(src + (pp >> 3) * 128 + (pp & 7) * 2));
            }
          }
        }
      }
      float s0[2] = {0.f, 0.f}, s1[2] = {0.f, 0.f};  // [slot]
#pragma unroll 1
      for (int slot = 0; slot < 2; ++slot) {
        const int n0 = slot * PP + lane, n1 = n0 + 32;
        if (lane < PP) {
          float a = 0.f;
#pragma unroll 8
          for (int tok = 0; tok < TILE_M; ++tok)
            a += __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(os + off_mnmajor_nosw(n0, tok, NPOOL)));
          s0[slot] = a;
        }
        if (lane + 32 < PP) {
          float a = 0.f;
#pragma unroll 8
          for (int tok = 0; tok < TILE_M; ++tok)
            a += __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(os + off_mnmajor_nosw(n1, tok, NPOOL)));
          s1[slot] = a;
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_OSEMPTY]);
      const int last_tok = min(tile * TILE_M + TILE_M - 1, ntok - 1);
      const int last_clip = last_tok / S;
      acc0 += s0[0]; acc1 += s1[0];
      if (last_clip > first_clip) {
        if (lane < p.P) p.osum[(size_t)(c_begin + first_clip) * p.P + lane] = acc0;
        if (lane + 32 < p.P) p.osum[(size_t)(c_begin + first_clip) * p.P + lane + 32] = acc1;
        acc0 = s0[1]; acc1 = s1[1];
      }
      if ((last_tok + 1) % S == 0) {
        if (lane < p.P) p.osum[(size_t)(c_begin + last_clip) * p.P + lane] = acc0;
        if (lane + 32 < p.P) p.osum[(size_t)(c_begin + last_clip) * p.P + lane + 32] = acc1;
        acc0 = acc1 = 0.f;
      }
    }
  } else if (warp >= W_EPI0) {
    // ------------------------------------------------------------------ epilogue warps 8..15
    const int q = warp & 3, hh = (warp - W_EPI0) >> 2;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    const uint32_t tl = tbase + lane_base;
    const int tok = q * 32 + lane;          // voxel row of the tile (G branch) / channel d % 128 (A branch)
    const int d = 128 * hh + tok;           // channel owned in the A branch and in the drain
    const float b1d = sb1[d];
    const bool tr = TRACE && warp == W_EPI0 && lane == 0;
    float facc[PP];
#pragma unroll
    for (int i = 0; i < PP; ++i) facc[i] = 0.f;
    bool ok = true;
    const uint64_t pol_last = l2_policy_evict_last();

    for (int tile = 0; tile < ntiles && ok; ++tile) {
      const uint32_t tp = tile & 1;
      const int t = tile * TILE_M + tok;
      const bool valid = t < ntok;
      const int first_clip = (tile * TILE_M) / S;
      const int clipl = valid ? t / S : first_clip;
      const int slot = clipl - first_clip;

      // ---- E1: acc_G -> G1 = relu(. + b3) bf16, in place.  Warp hh=0 walks its four 32-column chunks upwards and packs
      //      channels 0..127 into cols [0,64); warp hh=1 walks downwards and packs channels 128..255 into [192,256).
      if (tr) K1_TRACE(1, tile, 0);
      if (!(ok = bwait(&bars[B_GDONE], tp, ctx, 501))) break;
      tc_fence_after();
      if (tr) K1_TRACE(1, tile, 1);
      {
        uint32_t ra[32], rb[32], pk[16];
        const int c0 = hh ? 3 : 0, dc = hh ? -1 : 1;
        const uint32_t src = 128u * hh, dst = hh ? 192u : 0u;
        tmem_ld_x32(tl + src + 32 * c0, ra);
        tmem_ld_wait();
        tmem_ld_x32(tl + src + 32 * (c0 + dc), rb);
        bias_relu_pack(ra, sb3 + src + 32 * c0, pk);
        tmem_st_x16(tl + dst + 16 * c0, pk);
        tmem_ld_wait();
        tmem_ld_x32(tl + src + 32 * (c0 + 2 * dc), ra);
        bias_relu_pack(rb, sb3 + src + 32 * (c0 + dc), pk);
        tmem_st_x16(tl + dst + 16 * (c0 + dc), pk);
        tmem_ld_wait();
        tmem_ld_x32(tl + src + 32 * (c0 + 3 * dc), rb);
        bias_relu_pack(ra, sb3 + src + 32 * (c0 + 2 * dc), pk);
        tmem_st_x16(tl + dst + 16 * (c0 + 2 * dc), pk);
        tmem_ld_wait();
        bias_relu_pack(rb, sb3 + src + 32 * (c0 + 3 * dc), pk);
        tmem_st_x16(tl + dst + 16 * (c0 + 3 * dc), pk);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_G1READY]);
      if (tr) K1_TRACE(1, tile, 2);

      // ---- E2: acc_A^T half hh (128 voxel columns of this warp's 32 channel lanes) -> H1^T = relu(. + b1[d]) bf16, in
      //      place, while the G2 MMAs run.  hh = 0 packs upwards into [256,320), hh = 1 downwards into [448,512): every
      //      store lands on columns whose fp32 content this warp has already loaded, and [320,448) is left free for FEpartial^T.
      if (!(ok = bwait(&bars[B_ADONE], tp, ctx, 507))) break;
      tc_fence_after();
      if (tr) K1_TRACE(1, tile, 7);
      {
        uint32_t ra[32], rb[32], pk[16];
        const int c0 = hh ? 3 : 0, dc = hh ? -1 : 1;
        const uint32_t src = COL_AT + 128u * hh, dst = hh ? COL_H1T1 : COL_H1T0;
        auto cvt = [&](const uint32_t (&r)[32]) {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            pk[j] = pack_bf16x2_relu(__uint_as_float(r[2 * j]) + b1d, __uint_as_float(r[2 * j + 1]) + b1d);
        };
        tmem_ld_x32(tl + src + 32 * c0, ra);
        tmem_ld_wait();
        tmem_ld_x32(tl + src + 32 * (c0 + dc), rb);
        cvt(ra);
        tmem_st_x16(tl + dst + 16 * c0, pk);
        tmem_ld_wait();
        tmem_ld_x32(tl + src + 32 * (c0 + 2 * dc), ra);
        cvt(rb);
        tmem_st_x16(tl + dst + 16 * (c0 + dc), pk);
        tmem_ld_wait();
        tmem_ld_x32(tl + src + 32 * (c0 + 3 * dc), rb);
        cvt(ra);
        tmem_st_x16(tl + dst + 16 * (c0 + 2 * dc), pk);
        tmem_ld_wait();
        cvt(rb);
        tmem_st_x16(tl + dst + 16 * (c0 + 3 * dc), pk);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_H1TREADY]);
      if (tr) K1_TRACE(1, tile, 8);

      // ---- E3: acc_G2 (cols [64,192)) -> G2 = relu(. + b4) bf16 in place at [64+64hh, +32)
      if (!(ok = bwait(&bars[B_G2DONE], tp, ctx, 503))) break;
      tc_fence_after();
      if (tr) K1_TRACE(1, tile, 3);
      {
        uint32_t ra[32], rb[32], pk[16];
        const uint32_t col = 64u + 64u * hh;
        tmem_ld_x32(tl + col, ra);
        tmem_ld_wait();
        tmem_ld_x32(tl + col + 32, rb);
        bias_relu_pack(ra, sb4 + 64 * hh, pk);
        tmem_st_x16(tl + col, pk);
        tmem_ld_wait();
        bias_relu_pack(rb, sb4 + 64 * hh + 32, pk);
        tmem_st_x16(tl + col + 16, pk);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_G2READY]);
      if (tr) K1_TRACE(1, tile, 4);

      // ---- E4: acc_O -> O = |.| bf16 -> Os (pooling B operand, slot-in-N layout; other slot and invalid rows zero)
      if (!(ok = bwait(&bars[B_ODONE], tp, ctx, 504))) break;
      tc_fence_after();
      if (tr) K1_TRACE(1, tile, 5);
      {
        uint32_t r[32];
        tmem_ld_x32(tl + 32 * hh, r);
        tmem_ld_wait();
        // every G-branch column of this tile has been consumed: the next tile's G phase may overwrite [0,256)
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars[B_GBFREE]);
        if (!(ok = bwait(&bars[B_OSEMPTY], tp ^ 1, ctx, 505))) break;
        const int p0 = 32 * hh;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          if (p0 + 8 * g < PP) {
            uint32_t w4[4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
              w4[j] = valid ? pack_bf16x2(fabsf(__uint_as_float(r[8 * g + 2 * j])), fabsf(__uint_as_float(r[8 * g + 2 * j + 1])))
                            : 0u;
            const int n_data = slot * PP + p0 + 8 * g, n_zero = (1 - slot) * PP + p0 + 8 * g;
            *reinterpret_cast<uint4*>(smem + SM_OS + off_mnmajor_nosw(n_data, tok, NPOOL)) =
                make_uint4(w4[0], w4[1], w4[2], w4[3]);
            *reinterpret_cast<uint4*>(smem + SM_OS + off_mnmajor_nosw(n_zero, tok, NPOOL)) = make_uint4(0, 0, 0, 0);
          }
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_OSREADY]);
      if (tr) K1_TRACE(1, tile, 6);

      // ---- E5: drain FEpartial^T of this warp's channel half (lane = d % 128) into per-clip register accumulators;
      //      finished clips leave as bf16 hi/lo rows of the K2 operand images
      if (!(ok = bwait(&bars[hh ? B_FEDONE1 : B_FEDONE0], tp, ctx, 506))) break;
      tc_fence_after();
      if (tr) K1_TRACE(1, tile, 9);
      {
        const int last_tok = min(tile * TILE_M + TILE_M - 1, ntok - 1);
        const int last_clip = last_tok / S;
        const bool boundary = last_clip > first_clip;
        const bool ends = ((last_tok + 1) % S) == 0;
        const uint32_t fe = tl + (hh ? 0u : COL_FE);   // half 1 sits in the G-branch columns
        uint32_t nb[PP];  // slot-1 partial = start of the next clip (only meaningful when `boundary`)
        {
          uint32_t a[PP];
#pragma unroll
          for (int g = 0; g < PP / 8; ++g) tmem_ld_x8(fe + 8 * g, *reinterpret_cast<uint32_t(*)[8]>(&a[8 * g]));
          if (boundary) {
#pragma unroll
            for (int g = 0; g < PP / 8; ++g) tmem_ld_x8(fe + PP + 8 * g, *reinterpret_cast<uint32_t(*)[8]>(&nb[8 * g]));
          }
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < PP; ++j) facc[j] += __uint_as_float(a[j]);
        }
        // FEpartial^T columns read: once both halves are, the next tile's layer-1 MMAs may overwrite them
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars[B_ABFREE]);
        if (tr) K1_TRACE(1, tile, 10);
#pragma unroll 1
        for (int rep = 0; rep < 2; ++rep) {
          const bool flush = rep == 0 ? boundary : ends;
          if (!flush) continue;
          const int clip = c_begin + (rep == 0 ? first_clip : last_clip);
          const int tile2 = clip / p.cpt;
          const int rowb = (clip - tile2 * p.cpt) * PP;
          uint8_t* img = p.feimg + (size_t)tile2 * FE_TILE_BYTES + (size_t)(d >> 6) * 16384;
          // K2's A operand K-major (row = (clip,p), k = d contiguous): the 32 lanes of a warp hold 32 consecutive d of
          // one row, i.e. 64 bytes inside one 128-byte swizzle row -> one line per warp store (hi at +0, lo at +64 KB);
          // evict_last: K2 reads them right after this kernel
#pragma unroll
          for (int j = 0; j < PP; ++j) {
            const float v = facc[j];
            const __nv_bfloat16 h = __float2bfloat16_rn(v);
            const __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
            const uint32_t off = off_kmajor_sw128(rowb + j, d & 63);
            st_global_u16_hint(img + off, __bfloat16_as_ushort(h), pol_last);
            st_global_u16_hint(img + 65536 + off, __bfloat16_as_ushort(l), pol_last);
          }
          if (rep == 0) {
#pragma unroll
            for (int j = 0; j < PP; ++j) facc[j] = __uint_as_float(nb[j]);
          } else {
#pragma unroll
            for (int j = 0; j < PP; ++j) facc[j] = 0.f;
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tbase, 512);
  if constexpr (TRACE) {   // wall-clock end of CTA 0 (ns), next to K2's stamps (tools/trace_k2.py)
    if (tid == 0 && p.trace != nullptr && blockIdx.x == 0) {
      long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      p.trace[768 + 1] = t;
    }
  }
}

template <int PP, bool TRACE, int IN>
static int launch_inst(const K1Params& k1, int grid, cudaStream_t st) {
  static bool attr_done = false;
  if (!attr_done) {
    if (cudaFuncSetAttribute(head_tokens2_kernel<PP, TRACE, IN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K1_SMEM) != cudaSuccess)
      return PASN_ERR_CUDA;
    attr_done = true;
  }
  head_tokens2_kernel<PP, TRACE, IN><<<grid, K1_THREADS, K1_SMEM, st>>>(k1);
  PASN_LAUNCH_CHECK();
  return PASN_OK;
}
template <int PP>
static int launch_one(const K1Params& k1, int grid, cudaStream_t st) {
  // The instrumented instantiation (clock reads on the issue path) only runs while a trace buffer is installed.  The
  // trace exists for bf16 maps; fp32 and fp16 maps always run the plain kernel.
  const bool tr = k1.trace != nullptr;
  if (k1.f32_in) return launch_inst<PP, false, 2>(k1, grid, st);
  if (k1.f16_in) return k1.nsc ? launch_inst<PP, false, 4>(k1, grid, st) : launch_inst<PP, false, 3>(k1, grid, st);
  if (k1.nsc) return tr ? launch_inst<PP, true, 1>(k1, grid, st) : launch_inst<PP, false, 1>(k1, grid, st);
  return tr ? launch_inst<PP, true, 0>(k1, grid, st) : launch_inst<PP, false, 0>(k1, grid, st);
}

int launch_k1(const K1Params& k1, int ppad, int grid, cudaStream_t st) {
  if (ppad <= 16) return launch_one<16>(k1, grid, st);
  if (ppad <= 32) return launch_one<32>(k1, grid, st);
  if (ppad <= 40) return launch_one<40>(k1, grid, st);
  return launch_one<48>(k1, grid, st);
}

}  // namespace pasn
