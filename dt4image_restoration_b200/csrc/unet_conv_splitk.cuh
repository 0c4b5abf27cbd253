// Split-K variant of the 3x3 implicit-GEMM convolution for launches with FEW output tiles (batch 1-4 at the deep
// U-Net levels: reference evaluation/noise.py:75-98 run the way the reference's evaluation runs it, one image at a time).
//
// Why: conv3x3_umma_kernel / conv3x3_pair_kernel give one CTA a 16x16 pixel tile x 64..128 output channels and let it
// stream ALL K = 9*Cin weights of those channels.  With one image at 16x16 .. 64x64 that is 4-16 CTAs, each pulling
// 1-2 MB through one SM's L2 port (~70-100 GB/s with the ring depth that fits): 15-40 us per layer, 0.25 of the
// 0.34 ms denoiser pass at B=1.  Here the same work is cut along N (32 output channels per CTA) AND along K (a cluster
// of S CTAs, each reducing its own 64-channel slices), so ~128 CTAs each fetch one or two (halo tile 41 KB + weights
// 36 KB) stages at once and issue 72 MMAs per slice; the S partial accumulators (256 pixels x 32 channels fp32) are then
// summed through distributed shared memory in a fixed order (rank 0..S-1: deterministic), each CTA finishing 256/S pixels
// (bias + LeakyReLU + bf16, optional fused MaxPool2d(2) of reference noise.py:23).
//
// The weights are the layer's ordinary packed blobs (pack_weights_kernel, KC = 64): rows of a blob are output channels,
// the 128-byte swizzle depends on (row mod 8) only, so 32 consecutive rows of a BN = 64/128 blob ARE a BN = 32 blob.
#pragma once
#include "unet_conv.cuh"

namespace pnp {

constexpr int kSkBN = 32;
constexpr int kSkKC = 64;
constexpr int kSkRowB = kSkKC * 2;                                       // bytes per pixel / weight row
constexpr int kSkABytes = kHalo * kHalo * kSkRowB;                       // TMA box bytes (41472)
constexpr int kSkAStage = (kSkABytes + 1023) / 1024 * 1024;
constexpr int kSkBTap = kSkBN * kSkRowB;                                 // one tap's [32 x 64] weight block (4 KB)
constexpr int kSkBStage = 9 * kSkBTap;
constexpr int kSkStage = kSkAStage + kSkBStage;
constexpr int kSkStages = 2;                                             // p.sk_stages = min(slices per CTA, 2)
constexpr int kSkPartialBytes = 256 * kSkBN * 4;                         // aliases stage 0 once every MMA has completed
constexpr int sk_smem_bytes(int stages) { return 1024 + stages * kSkStage + 128; }
constexpr int kSkSmem = sk_smem_bytes(kSkStages);                        // opt-in maximum
constexpr int kSkTmemCols = 64;                                          // 2 M-blocks x 32 fp32 columns
static_assert(kSkPartialBytes <= kSkStage, "partial accumulator must fit into a pipeline stage");

__device__ __forceinline__ uint32_t sk_mapa(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ float4 sk_ld_cluster_f4(uint32_t caddr) {
  float4 v;
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(caddr));
  return v;
}
__device__ __forceinline__ uint32_t sk_max_bf16x2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("max.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t sk_cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void sk_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release;\n\tbarrier.cluster.wait.acquire;" ::: "memory");
}

// grid = units * S CTAs, cluster (S,1,1); unit = (image, tile y, tile x, 32-channel block), p.sk_split = S,
// p.sk_cpc = 64-channel slices per CTA (S * sk_cpc = nchunks0 + nchunks1).
__global__ void __launch_bounds__(kConvThreads, 1)      // (.., 2) = 80 registers was measured slower: 0.2245 vs 0.2148 ms at B=1
conv3x3_splitk_kernel(const ConvParams p, const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.sk_stages * kSkStage);
  uint64_t* full = bars;                 // [2] halo tile + nine weight blocks of a slice have landed
  uint64_t* empty = bars + 2;            // [2] both issuers' MMAs have read the stage
  uint64_t* acc_full = bars + 4;         // both M-block accumulators complete
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int S = p.sk_split, cpc = p.sk_cpc;
  const uint32_t rank = sk_cluster_rank();
  int unit = int(blockIdx.x) / S;
  const int n_sub = p.Cout / kSkBN;
  const int ns = unit % n_sub; unit /= n_sub;
  const int tx = unit % p.tiles_x; unit /= p.tiles_x;
  const int ty = unit % p.tiles_y;
  const int img = unit / p.tiles_y;

  grid_dep_launch();
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmA0); tma_prefetch_desc(&tmA1); }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kSkStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], kNumMmaWarps); }
    mbar_init(acc_full, kNumMmaWarps);
    fence_mbar_init();
  }
  if (warp == 2) { tmem_alloc(tmem_slot, kSkTmemCols); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================================== producer =====================================
    if (lane == 0) {
      for (int i = 0; i < cpc; ++i) {
        const int st = i & 1;
        if (i >= kSkStages) mbar_wait(&empty[st], ((i >> 1) - 1) & 1);
        uint8_t* a_dst = smem + st * kSkStage;
        uint8_t* b_dst = a_dst + kSkAStage;
        mbar_arrive_expect_tx(&full[st], kSkABytes + kSkBStage);
        const int c = int(rank) * cpc + i;
        const uint8_t* wsrc = p.wpk + (size_t(c) * 9 * p.Cout + size_t(ns) * kSkBN) * kSkRowB;
        for (int tap = 0; tap < 9; ++tap)
          bulk_load_1d(b_dst + tap * kSkBTap, wsrc + size_t(tap) * p.Cout * kSkRowB, kSkBTap, &full[st]);
        if (i == 0) grid_dep_wait();          // weights are constants; the activations come from the previous kernel
        const bool seg0 = c < p.nchunks0;
        tma_load_4d(a_dst, seg0 ? &tmA0 : &tmA1, &full[st], (seg0 ? c : c - p.nchunks0) * kSkKC, tx * kTile - 1,
                    ty * kTile - 1, img);
      }
    }
  } else if (warp == 1 || warp == 3) {
    // ===================================== MMA issuers (one per M=128 pixel block) =====================================
    const int mb = warp == 3 ? 1 : 0;
    constexpr uint32_t idesc = umma_idesc_bf16(128, kSkBN);
    constexpr uint32_t a_hi = (uint32_t(kHalo * kSkRowB) >> 4) | (1u << 14) | (2u << 29);
    constexpr uint32_t b_hi = (uint32_t(8 * kSkRowB) >> 4) | (1u << 14) | (2u << 29);
    const uint32_t d0 = tmem_base + mb * kSkBN;
    for (int i = 0; i < cpc; ++i) {
      const int st = i & 1;
      mbar_wait(&full[st], (i >> 1) & 1);
      tc_fence_after();
      const uint32_t a_lo0 = ((smem_u32(smem + st * kSkStage) + uint32_t(mb * 8 * kSkRowB)) >> 4) | (1u << 16);
      const uint32_t b_lo0 = (smem_u32(smem + st * kSkStage + kSkAStage) >> 4) | (1u << 16);
      if (elect_one()) {
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
          const uint32_t a_tap = a_lo0 + uint32_t(((tap / 3) * kHalo + (tap % 3)) * kSkRowB) / 16;
          const uint32_t b_tap = b_lo0 + uint32_t(tap * kSkBTap) / 16;
#pragma unroll
          for (int k = 0; k < kSkKC / 16; ++k)
            umma_bf16_ss2(d0, a_tap + k * 2, a_hi, b_tap + k * 2, b_hi, idesc, (i | tap | k) != 0 ? 1u : 0u);
        }
        tc_commit(&empty[st]);
        if (i == cpc - 1) tc_commit(acc_full);
      }
      __syncwarp();
    }
  } else if (warp >= kEpiWarp0) {
    // ===================================== partial accumulator -> shared memory =====================================
    const int q = warp & 3, mb = (warp - kEpiWarp0) >> 2;
    const int id = mb * 128 + q * 32 + lane;             // pixel id inside the tile: M-block, then row-major 16 x 8
    mbar_wait(acc_full, 0);
    tc_fence_after();
    uint32_t r[32];
    tmem_ld_32x32(tmem_base + (uint32_t(q * 32) << 16) + mb * kSkBN, r);
    tmem_ld_wait();
    uint8_t* prow = smem + size_t(id) * 128;
#pragma unroll
    for (int c = 0; c < 8; ++c)                          // 16-byte chunk c sits at position c ^ (id & 7): conflict-free
      *reinterpret_cast<uint4*>(prow + ((c ^ (lane & 7)) << 4)) = make_uint4(r[4 * c], r[4 * c + 1], r[4 * c + 2], r[4 * c + 3]);
  }
  tc_fence_before();
  sk_cluster_sync();                                     // every CTA's partial sums are in its shared memory

  if (warp >= kEpiWarp0) {
    // ===================================== cluster reduction + epilogue =====================================
    // this CTA finishes pixel ids [rank * P, (rank + 1) * P): whole 2x2 blocks, one block per warp pass
    // (lane = 8 * pixel-in-block + 16-byte chunk of the 32 fp32 channels)
    const int P = 256 / S, nblk = P / 4;
    const int k = lane >> 3, c = lane & 7;
    const uint32_t part = smem_u32(smem);
    const float4 bia = __ldg(reinterpret_cast<const float4*>(p.bias + ns * kSkBN) + c);
    const int Hp = p.H >> 1, Wp = p.W >> 1;
    for (int b = warp - kEpiWarp0; b < nblk; b += kNumEpiWarps) {
      const int id = int(rank) * P + (b >> 2) * 16 + (b & 3) * 2 + (k & 1) + (k >> 1) * 8;
      const uint32_t off = uint32_t(id) * 128u + (uint32_t(c ^ (id & 7)) << 4);
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int s = 0; s < S; ++s) {
        const float4 v = sk_ld_cluster_f4(sk_mapa(part + off, uint32_t(s)));
        a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
      }
      a.x += bia.x; a.y += bia.y; a.z += bia.z; a.w += bia.w;
      a.x = fmaxf(a.x, a.x * p.slope); a.y = fmaxf(a.y, a.y * p.slope);
      a.z = fmaxf(a.z, a.z * p.slope); a.w = fmaxf(a.w, a.w * p.slope);
      uint2 o = make_uint2(pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w));
      const int m = id & 127;
      const int y = ty * kTile + (m >> 3), x = tx * kTile + (m & 7) + (id >> 7) * 8;
      if (y < p.H && x < p.W)
        *reinterpret_cast<uint2*>(p.out + ((size_t(img) * p.H + y) * p.W + x) * p.Cout + ns * kSkBN + 4 * c) = o;
      if (p.pool_out) {
        uint32_t h0 = o.x, h1 = o.y;                       // MaxPool2d(2): the block's four pixels sit in lanes ^8 and ^16
#pragma unroll
        for (int sh = 8; sh <= 16; sh <<= 1) {
          h0 = sk_max_bf16x2(h0, __shfl_xor_sync(0xffffffffu, h0, sh));
          h1 = sk_max_bf16x2(h1, __shfl_xor_sync(0xffffffffu, h1, sh));
        }
        if (k == 0 && (y >> 1) < Hp && (x >> 1) < Wp)
          *reinterpret_cast<uint2*>(p.pool_out + ((size_t(img) * Hp + (y >> 1)) * Wp + (x >> 1)) * p.Cout + ns * kSkBN + 4 * c) =
              make_uint2(h0, h1);
      }
    }
  }
  sk_cluster_sync();                                     // nobody leaves while a peer still reads its partial sums
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kSkTmemCols);
  }
}

}  // namespace pnp
