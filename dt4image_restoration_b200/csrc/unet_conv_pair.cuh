// 3x3 convolution as CTA-PAIR implicit GEMM: tcgen05.mma.cta_group::2 (M = 256 across two SMs of a cluster).
//
// Same tiling and pipeline as conv3x3_umma_kernel (unet_conv.cuh), but two CTAs of a 2-CTA cluster work on two pixel
// tiles with the SAME output-channel tile in lock step, and every MMA covers both of them:
//   * each CTA TMA-loads the halo tile of its own pixel tile (the A rows it contributes: 128 per M-block) and only
//     HALF of every weight blob (BN/2 rows of B) - the tensor cores of the pair read the two halves from both shared
//     memories, so weight traffic L2 -> SM and the per-CTA B operand reads are halved (verified and measured with
//     tools/mma2_bench.cu: D rows split by CTA, B = [half of CTA 0 ; half of CTA 1], 43 clk per N=64 MMA instead of 52);
//   * the leader CTA (cluster rank 0) issues all MMAs (two issuing warps, one per M-block, as in the single-CTA
//     kernel) and multicasts its tcgen05.commit arrivals to the empty / accumulator-full barriers of both CTAs;
//   * both CTAs' TMA loads (`cp.async.bulk.tensor...cta_group::2`, the weights through a 2-D tensor map over the packed
//     blobs because the 1-D bulk copy has no pair form) complete their bytes on the LEADER's full barrier, for which the
//     leader's producer expects the bytes of both CTAs (first version: a forwarder warp in the peer relayed its
//     completions with remote arrives - 2.70 ms per U-Net at BN=128 instead of 2.67 single-CTA);
//   * the peer's epilogue warps hand their accumulator stage back with a remote arrive on the leader's acc_empty.
// Accumulators: every CTA's TMEM holds its own 128 rows x BN columns per M-block, double buffered, exactly as before.
// Used for the layers with the plain bf16 epilogue and BN in {64, 128} whose weights do not stay resident in a single
// CTA (build_conv in unet.cu).
#pragma once
#include <cooperative_groups.h>
#include "unet_conv.cuh"

namespace pnp {
namespace cgp = cooperative_groups;

__device__ __forceinline__ void tmem_alloc2(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish2() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// arrival on the barrier at the same shared-memory offset in BOTH CTAs once this thread's MMAs have completed
__device__ __forceinline__ void tc_commit2(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(uint16_t(3))
               : "memory");
}
__device__ __forceinline__ void umma2_bf16_ss(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                              uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}\n" ::"r"(tmem_d),
      "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// shared::cluster address of the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t cluster_addr(const void* p, uint32_t rank) {
  uint32_t ra;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(smem_u32(p)), "r"(rank));
  return ra;
}
// TMA loads of a CTA pair: the destination is this CTA's shared memory, the bytes complete on `mbar_cluster`, which may be
// the peer's barrier
__device__ __forceinline__ void tma_load_4d_pair(void* smem_dst, const CUtensorMap* m, uint32_t mbar_cluster, int c0, int c1,
                                                 int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(mbar_cluster), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* m, uint32_t mbar_cluster, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(mbar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
// arrive on the mbarrier at the same offset in the shared memory of cluster rank `rank`.  Relaxed: the only thing the
// waiter depends on are this warp's TMEM reads, which tcgen05.wait::ld + tcgen05.fence::before_thread_sync have ordered;
// a release at cluster scope would first drain the global stores of the previous tile (measured: +30 % on thin layers).
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [ra];\n\t}\n" ::"r"(smem_u32(bar)),
      "r"(rank)
      : "memory");
}

template <int KC, int BN>
struct PairCfg {
  static constexpr int ROWB = KC * 2;
  static constexpr int A_BYTES = kHalo * kHalo * ROWB;
  static constexpr int A_STAGE = (A_BYTES + 1023) / 1024 * 1024;
  static constexpr int B_FULL = BN * ROWB;                      // one packed (slice, tap, n-tile) blob in global memory
  static constexpr int B_BYTES = B_FULL / 2;                    // the half this CTA keeps (BN/2 rows)
  static constexpr int B_STAGE = (B_BYTES + 1023) / 1024 * 1024;
  static constexpr int NACC = 2;
  static constexpr int TMEM_COLS = 2 * BN * NACC;
  static constexpr int MAX_RING = 16;
  static constexpr int BAR_BYTES = (4 * MAX_RING + 2 * NACC + 2) * 8 + 16 + kEpiSmemFloats * 4;
  static_assert(TMEM_COLS >= 32 && TMEM_COLS <= 512 && (TMEM_COLS & (TMEM_COLS - 1)) == 0, "TMEM cols");
  static_assert((BN / 2) % 8 == 0, "half blobs must be whole 8-row groups");
};

// ConvParams as for conv3x3_umma_kernel, except: total_tiles = PAIR tiles = ceil(pixel tiles / 2) * n_tiles, grid = 2 x pairs.
// pair tile u -> (nt = u % n_tiles, pixel-tile pair = u / n_tiles); CTA rank r owns pixel tile 2*pair + r (the last pair
// of an odd pixel-tile count computes tile 2*pair twice and stores it once).
template <int KC, int BN>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kConvThreads, 1)
conv3x3_pair_kernel(const ConvParams p, const __grid_constant__ CUtensorMap tmA0,
                    const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmW) {
  using Cfg = PairCfg<KC, BN>;
  constexpr int ROWB = Cfg::ROWB;
  constexpr int NACC = Cfg::NACC;
  const int SA = p.sa, SB = p.sb;
  const int nchunks = p.nchunks0 + p.nchunks1;
  const int b_region = p.wres ? nchunks * 9 * Cfg::B_BYTES : SB * Cfg::B_STAGE;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* a_smem = smem;
  uint8_t* b_smem = smem + SA * Cfg::A_STAGE;
  uint64_t* bars = reinterpret_cast<uint64_t*>(b_smem + ((b_region + 1023) & ~1023));
  uint64_t* a_full = bars;
  uint64_t* a_empty = a_full + Cfg::MAX_RING;
  uint64_t* b_full = a_empty + Cfg::MAX_RING;
  uint64_t* b_empty = b_full + Cfg::MAX_RING;
  uint64_t* acc_full = b_empty + Cfg::MAX_RING;
  uint64_t* acc_empty = acc_full + NACC;
  uint64_t* w_full = acc_empty + NACC;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_full + 2);
  float* epi_s = reinterpret_cast<float*>(tmem_slot + 4);

  cgp::cluster_group cluster = cgp::this_cluster();
  const uint32_t rank = cluster.block_rank();
  const bool leader = rank == 0;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int pixel_tiles = p.B * p.tiles_y * p.tiles_x;
  const int total_pairs = p.total_tiles;                 // pair tiles (host)
  const int pair_id = int(blockIdx.x) >> 1, n_pairs = int(gridDim.x) >> 1;

  grid_dep_launch();
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA0);
    tma_prefetch_desc(&tmA1);
    tma_prefetch_desc(&tmW);
  }
  if (warp == 1 && lane == 0) {
    // only the leader's full barriers are used: one arrival (its producer's expect_tx of BOTH CTAs' bytes)
    for (int i = 0; i < SA; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], kNumMmaWarps); }
    for (int i = 0; i < SB; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], kNumMmaWarps); }
    for (int i = 0; i < NACC; ++i) { mbar_init(&acc_full[i], kNumMmaWarps); mbar_init(&acc_empty[i], 2 * kNumEpiWarps); }
    mbar_init(w_full, 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc2(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish2();
  }
  if (warp >= kEpiWarp0) {
    const int t = threadIdx.x - kEpiWarp0 * 32;
    for (int i = t; i < p.Cout; i += kNumEpiWarps * 32) epi_s[i] = __ldg(p.bias + i);
  }
  tc_fence_before();
  cluster.sync();                     // barriers of BOTH CTAs are initialised before anyone arrives remotely
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // this CTA's pixel tile of pair tile u (and whether it is the duplicate of an odd tail)
  auto my_tile = [&](int u, int& nt, int& tx, int& ty, int& img, bool& dup) {
    const int uu = p.rev ? total_pairs - 1 - u : u;
    nt = uu % p.n_tiles;
    int pt = 2 * (uu / p.n_tiles) + int(rank);
    dup = pt >= pixel_tiles;
    if (dup) pt = pixel_tiles - 1;
    tx = pt % p.tiles_x; pt /= p.tiles_x;
    ty = pt % p.tiles_y;
    img = pt / p.tiles_y;
  };

  if (warp == 0) {
    // ===================================== TMA producer (both CTAs) =========================
    if (lane == 0) {
      int sa = 0, pa = 0, sb = 0, pb = 0;
      const int row_half = int(rank) * (BN / 2);                       // this CTA's rows inside every blob
      if (p.wres && pair_id < total_pairs) {
        // n_tiles == 1: blob (c, tap) starts at row (c*9 + tap) * BN of the weight map; keep our half of each
        const uint32_t wbar = cluster_addr(w_full, 0);
        if (leader) mbar_arrive_expect_tx(w_full, 2u * uint32_t(nchunks) * 9 * Cfg::B_BYTES);
        for (int i = 0; i < nchunks * 9; ++i)
          tma_load_2d_pair(b_smem + size_t(i) * Cfg::B_BYTES, &tmW, wbar, 0, i * BN + row_half);
      }
      grid_dep_wait();
      for (int u = pair_id; u < total_pairs; u += n_pairs) {
        int nt, tx, ty, img; bool dup;
        my_tile(u, nt, tx, ty, img, dup);
        for (int c = 0; c < nchunks; ++c) {
          mbar_wait(&a_empty[sa], pa ^ 1);
          if (leader) mbar_arrive_expect_tx(&a_full[sa], 2u * Cfg::A_BYTES);
          const bool seg0 = c < p.nchunks0;
          tma_load_4d_pair(a_smem + sa * Cfg::A_STAGE, seg0 ? &tmA0 : &tmA1, cluster_addr(&a_full[sa], 0),
                           (seg0 ? c : c - p.nchunks0) * KC, tx * kTile - 1, ty * kTile - 1, img);
          if (++sa == SA) { sa = 0; pa ^= 1; }
          if (p.wres) continue;
          const int row0 = (c * 9 * p.n_tiles + nt) * BN + row_half;
          for (int tap = 0; tap < 9; ++tap) {
            mbar_wait(&b_empty[sb], pb ^ 1);
            if (leader) mbar_arrive_expect_tx(&b_full[sb], 2u * Cfg::B_BYTES);
            tma_load_2d_pair(b_smem + sb * Cfg::B_STAGE, &tmW, cluster_addr(&b_full[sb], 0), 0,
                             row0 + tap * p.n_tiles * BN);
            if (++sb == SB) { sb = 0; pb ^= 1; }
          }
        }
      }
    }
  } else if (leader && (warp == 1 || warp == 3)) {
    // ===================================== MMA issuers (leader CTA) =========================
    const int mb = warp == 3 ? 1 : 0;
    constexpr uint32_t idesc = umma_idesc_bf16(256, BN);
    constexpr uint32_t kLayout = (ROWB == 128) ? 2u : 4u;
    constexpr uint32_t a_hi = (uint32_t(kHalo * ROWB) >> 4) | (1u << 14) | (kLayout << 29);
    constexpr uint32_t b_hi = (uint32_t(8 * ROWB) >> 4) | (1u << 14) | (kLayout << 29);
    int sa = 0, pa = 0, sb = 0, pb = 0;
    int it = 0;
    if (p.wres && pair_id < total_pairs) mbar_wait(w_full, 0);
    for (int u = pair_id; u < total_pairs; u += n_pairs, ++it) {
      const int as = it % NACC;
      const uint32_t aph = (it / NACC) & 1;
      mbar_wait(&acc_empty[as], aph ^ 1);
      const uint32_t d0 = tmem_base + as * (2 * BN) + mb * BN;
      for (int c = 0; c < nchunks; ++c) {
        mbar_wait(&a_full[sa], pa);
        tc_fence_after();
        const uint32_t a_lo0 = ((smem_u32(a_smem + sa * Cfg::A_STAGE) + uint32_t(mb * 8 * ROWB)) >> 4) | (1u << 16);
        if (p.wres) {
          const uint32_t b_lo0 = (smem_u32(b_smem + c * 9 * Cfg::B_BYTES) >> 4) | (1u << 16);
          if (elect_one()) {
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
              const uint32_t a_tap = a_lo0 + uint32_t(((tap / 3) * kHalo + (tap % 3)) * ROWB) / 16;
              const uint32_t b_tap = b_lo0 + uint32_t(tap * Cfg::B_BYTES) / 16;
#pragma unroll
              for (int k = 0; k < KC / 16; ++k)
                umma2_bf16_ss(d0, a_tap + k * 2, a_hi, b_tap + k * 2, b_hi, idesc, (c | tap | k) != 0 ? 1u : 0u);
            }
          }
          __syncwarp();
        } else {
#pragma unroll 1
          for (int tap = 0; tap < 9; ++tap) {
            mbar_wait(&b_full[sb], pb);
            tc_fence_after();
            const uint32_t b_tap = (smem_u32(b_smem + sb * Cfg::B_STAGE) >> 4) | (1u << 16);
            const uint32_t a_tap = a_lo0 + uint32_t(((tap / 3) * kHalo + (tap % 3)) * ROWB) / 16;
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < KC / 16; ++k)
                umma2_bf16_ss(d0, a_tap + k * 2, a_hi, b_tap + k * 2, b_hi, idesc, (c | tap | k) != 0 ? 1u : 0u);
              tc_commit2(&b_empty[sb]);
            }
            __syncwarp();
            if (++sb == SB) { sb = 0; pb ^= 1; }
          }
        }
        if (elect_one()) tc_commit2(&a_empty[sa]);
        __syncwarp();
        if (++sa == SA) { sa = 0; pa ^= 1; }
      }
      if (elect_one()) tc_commit2(&acc_full[as]);
      __syncwarp();
    }
  } else if (warp >= kEpiWarp0) {
    // ===================================== epilogue (both CTAs) =============================
    const int q = warp & 3;
    const int mb = (warp - kEpiWarp0) >> 2;
    const int m = q * 32 + lane;
    const int prow = m >> 3, pcol = (m & 7) + mb * 8;
    int it = 0;
    for (int u = pair_id; u < total_pairs; u += n_pairs, ++it) {
      int nt, tx, ty, img; bool dup;
      my_tile(u, nt, tx, ty, img, dup);
      const int as = it % NACC;
      const uint32_t aph = (it / NACC) & 1;
      const int y = ty * kTile + prow, x = tx * kTile + pcol;
      mbar_wait(&acc_full[as], aph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + as * (2 * BN) + mb * BN;
#pragma unroll 1
      for (int cc = 0; cc < BN / 32; ++cc) {
        uint32_t r[32];
        tmem_ld_32x32(taddr + cc * 32, r);
        tmem_ld_wait();
        if (cc == BN / 32 - 1) {       // stage drained: both CTAs report to the leader's acc_empty
          tc_fence_before();
          __syncwarp();
          if (lane == 0) { if (leader) mbar_arrive(&acc_empty[as]); else mbar_arrive_remote(&acc_empty[as], 0); }
        }
        epilogue_bf16_chunk(p, r, epi_s + nt * BN + cc * 32, nt * BN + cc * 32, img, y, x, lane, !dup);
      }
    }
  }

  tc_fence_before();
  cluster.sync();                     // nobody leaves (or frees TMEM) while the peer may still be read or signalled
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc2(tmem_base, Cfg::TMEM_COLS);
  }
}

}  // namespace pnp
