// 3x3 convolution with 32 output channels: "kw-stacked" implicit GEMM (N = 3 taps x 32 channels = 96).
//
// Why a second kernel: tcgen05.mma with M=128, N=32 spends 40-49 cycles on a 16-cycle MMA because every MMA re-reads
// its 4 KB A operand from shared memory (measured, tools/mma_bench.cu: N=32 -> 33 % of the math rate, N=96 -> 81 %).
// The 32-channel layers of the U-Net (reference evaluation/noise.py:104,112 - inc and up4, 5 of the 26 tensor-core
// convs but 30 % of the time) are therefore shared-memory bound in conv3x3_umma_kernel.  Here the three horizontal
// taps are stacked along N instead:
//     P[(y, x'), (kw, co)] = sum_{kh, ci} in[y + kh - 1, x' - 1][ci] * W[co][ci][kh][kw]        (N = 96, 3 x fewer A reads)
//     out[y, x][co]        = P[(y, x), (0, co)] + P[(y, x + 1), (1, co)] + P[(y, x + 2), (2, co)]
// The second line is done by the epilogue with two warp shuffles per value: TMEM lane = 8*y + (x' % 8), so the
// neighbours x'+1, x'+2 are the next two lanes as long as the output column is one of the first 6 of its 8-wide
// M-block window.  Tile = 16 rows x 12 columns (two M-blocks whose windows start 6 columns apart), halo 18 x 14.
// Everything else (TMA halo ring, resident weights, two MMA-issuing warps, TMEM double buffering, fused bias /
// LeakyReLU / max-pool) follows conv3x3_umma_kernel.
#pragma once
#include "unet_conv.cuh"

namespace pnp {

constexpr int kKwsTileW = 12, kKwsTileH = 16;
constexpr int kKwsHaloW = kKwsTileW + 2, kKwsHaloH = kKwsTileH + 2;
constexpr int kKwsN = 96;

struct KwsCfg {
  static constexpr int KC = 32, ROWB = 64;
  static constexpr int A_BYTES = kKwsHaloW * kKwsHaloH * ROWB;            // 16128
  static constexpr int A_STAGE = (A_BYTES + 1023) / 1024 * 1024;          // 16384
  static constexpr int B_BYTES = kKwsN * ROWB;                            // one (chunk, kh) blob: 96 rows x 64 B
  static constexpr int NACC = 2;
  static constexpr int ACC_COLS = 2 * kKwsN;                              // two M-blocks per stage
  static constexpr int TMEM_COLS = 512;
  static constexpr int MAX_RING = 16;
  static constexpr int BAR_BYTES = (4 * MAX_RING + 2 * NACC + 2) * 8 + 16 + kEpiSmemFloats * 4;
};

__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

// ConvParams is shared with conv3x3_umma_kernel; here tiles_x = ceil(W/12), tiles_y = ceil(H/16), n_tiles = 1,
// wres = 1 (the layer's weights, at most 96 x 32 x 9 bf16 = 54 KB, always stay resident), Cout = 32.
__global__ void __launch_bounds__(kConvThreads, 1)
conv3x3_kws_kernel(const ConvParams p, const __grid_constant__ CUtensorMap tmA0,
                   const __grid_constant__ CUtensorMap tmA1) {
  using Cfg = KwsCfg;
  constexpr int ROWB = Cfg::ROWB, NACC = Cfg::NACC, KC = Cfg::KC;
  const int SA = p.sa;
  const int nchunks = p.nchunks0 + p.nchunks1;
  const int b_region = nchunks * 3 * Cfg::B_BYTES;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* a_smem = smem;
  uint8_t* b_smem = smem + SA * Cfg::A_STAGE;
  uint64_t* bars = reinterpret_cast<uint64_t*>(b_smem + ((b_region + 1023) & ~1023));
  uint64_t* a_full = bars;
  uint64_t* a_empty = a_full + Cfg::MAX_RING;
  uint64_t* acc_full = a_empty + 3 * Cfg::MAX_RING;       // same barrier block layout as the plain kernel
  uint64_t* acc_empty = acc_full + NACC;
  uint64_t* w_full = acc_empty + NACC;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_full + 2);
  float* epi_s = reinterpret_cast<float*>(tmem_slot + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int total_tiles = p.B * p.tiles_y * p.tiles_x;

  grid_dep_launch();
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA0);
    tma_prefetch_desc(&tmA1);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < SA; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], kNumMmaWarps); }
    for (int i = 0; i < NACC; ++i) { mbar_init(&acc_full[i], kNumMmaWarps); mbar_init(&acc_empty[i], kNumEpiWarps); }
    mbar_init(w_full, 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  if (warp >= kEpiWarp0) {
    const int t = threadIdx.x - kEpiWarp0 * 32;
    if (t < 32) epi_s[t] = __ldg(p.bias + t);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================================== TMA producer =====================================
    if (lane == 0 && int(blockIdx.x) < total_tiles) {
      int sa = 0, pa = 0;
      const uint32_t wbytes = uint32_t(b_region);
      mbar_arrive_expect_tx(w_full, wbytes);
      for (uint32_t off = 0; off < wbytes; off += 3 * Cfg::B_BYTES)
        bulk_load_1d(b_smem + off, p.wpk + off, 3 * Cfg::B_BYTES, w_full);
      grid_dep_wait();          // weights are constants; the activations below come from the previous kernel
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const TileCoord tc = decode_tile(p, tile);
        for (int c = 0; c < nchunks; ++c) {
          const bool seg0 = c < p.nchunks0;
          mbar_wait(&a_empty[sa], pa ^ 1);
          mbar_arrive_expect_tx(&a_full[sa], Cfg::A_BYTES);
          tma_load_4d(a_smem + sa * Cfg::A_STAGE, seg0 ? &tmA0 : &tmA1, &a_full[sa],
                      (seg0 ? c : c - p.nchunks0) * KC, tc.tx * kKwsTileW - 1, tc.ty * kKwsTileH - 1, tc.img);
          if (++sa == SA) { sa = 0; pa ^= 1; }
        }
      }
    }
  } else if (warp == 1 || warp == 3) {
    // ===================================== MMA issuers (one per M-block) ====================
    const int mb = warp == 3 ? 1 : 0;
    constexpr uint32_t idesc = umma_idesc_bf16(128, kKwsN);
    constexpr uint32_t kLayout = 4u;                                           // SWIZZLE_64B
    constexpr uint32_t a_hi = (uint32_t(kKwsHaloW * ROWB) >> 4) | (1u << 14) | (kLayout << 29);   // next output row
    constexpr uint32_t b_hi = (uint32_t(8 * ROWB) >> 4) | (1u << 14) | (kLayout << 29);
    int sa = 0, pa = 0, it = 0;
    if (int(blockIdx.x) < total_tiles) mbar_wait(w_full, 0);
    const uint32_t b_base = (smem_u32(b_smem) >> 4) | (1u << 16);
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const int as = it % NACC;
      const uint32_t aph = (it / NACC) & 1;
      mbar_wait(&acc_empty[as], aph ^ 1);
      const uint32_t d0 = tmem_base + as * Cfg::ACC_COLS + mb * kKwsN;
      for (int c = 0; c < nchunks; ++c) {
        mbar_wait(&a_full[sa], pa);
        tc_fence_after();
        // this M-block's window: halo columns 6*mb .. 6*mb+7, rows kh .. kh+15 (8-pixel groups one halo row apart)
        const uint32_t a_lo0 = ((smem_u32(a_smem + sa * Cfg::A_STAGE) + uint32_t(mb * 6 * ROWB)) >> 4) | (1u << 16);
        const uint32_t b_lo0 = b_base + uint32_t(c * 3 * Cfg::B_BYTES) / 16;
        if (elect_one()) {
#pragma unroll
          for (int kh = 0; kh < 3; ++kh) {
#pragma unroll
            for (int k = 0; k < KC / 16; ++k)
              umma_bf16_ss2(d0, a_lo0 + uint32_t(kh * kKwsHaloW * ROWB) / 16 + k * 2, a_hi,
                            b_lo0 + uint32_t(kh * Cfg::B_BYTES) / 16 + k * 2, b_hi, idesc, (c | kh | k) != 0 ? 1u : 0u);
          }
          tc_commit(&a_empty[sa]);
        }
        __syncwarp();
        if (++sa == SA) { sa = 0; pa ^= 1; }
      }
      if (elect_one()) tc_commit(&acc_full[as]);
      __syncwarp();
    }
  } else if (warp >= kEpiWarp0) {
    // ===================================== epilogue =========================================
    const int q = warp & 3;
    const int mb = (warp - kEpiWarp0) >> 2;
    const int yl = q * 4 + (lane >> 3);        // output row inside the tile
    const int i8 = lane & 7;                   // column inside the 8-wide window; outputs exist for i8 < 6
    const int r4 = lane & 3;
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const TileCoord tc = decode_tile(p, tile);
      const int as = it % NACC;
      const uint32_t aph = (it / NACC) & 1;
      const int y = tc.ty * kKwsTileH + yl, x = tc.tx * kKwsTileW + mb * 6 + i8;
      const size_t pix = (size_t(tc.img) * p.H + y) * p.W + x;
      mbar_wait(&acc_full[as], aph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + as * Cfg::ACC_COLS + mb * kKwsN;
      uint4 o[4];
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t r0[16], r1[16], r2[16];
        tmem_ld_32x16(taddr + half * 16, r0);
        tmem_ld_32x16(taddr + 32 + half * 16, r1);
        tmem_ld_32x16(taddr + 64 + half * 16, r2);
        tmem_ld_wait();
        if (half == 1) {                       // accumulator stage drained
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc_empty[as]);
        }
        // out(x) = D_kw0(x) + D_kw1(x + 1) + D_kw2(x + 2) + bias.  (Packed fp32x2 adds / max-form LeakyReLU as in the other
        // conv kernels were measured here and lost 3-5 %: the shuffled values do not arrive in register pairs.)
        float s[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          const float p1 = __shfl_down_sync(0xffffffffu, __uint_as_float(r1[c]), 1);
          const float p2 = __shfl_down_sync(0xffffffffu, __uint_as_float(r2[c]), 2);
          float v = (__uint_as_float(r0[c]) + p1) + p2 + epi_s[half * 16 + c];
          s[c] = v > 0.f ? v : v * p.slope;
        }
#pragma unroll
        for (int g = 0; g < 2; ++g)
          o[half * 2 + g] = make_uint4(pack_bf16x2(s[g * 8], s[g * 8 + 1]), pack_bf16x2(s[g * 8 + 2], s[g * 8 + 3]),
                                       pack_bf16x2(s[g * 8 + 4], s[g * 8 + 5]), pack_bf16x2(s[g * 8 + 6], s[g * 8 + 7]));
      }
      if (p.pool_out) {
        // 2x2 max-pool partners: x+1 = lane^1 (x and i8 have the same parity, i8+1 <= 5 for even i8 < 6), y+1 = lane^8
        uint4 mx[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          mx[g] = bf16x8_max(o[g], shfl_xor_u4(o[g], 1));
          mx[g] = bf16x8_max(mx[g], shfl_xor_u4(mx[g], 8));
        }
        const int Hp = p.H >> 1, Wp = p.W >> 1;
        if (((lane & 9) == 0) && i8 < 6 && (y >> 1) < Hp && (x >> 1) < Wp) {
          uint4* pd = reinterpret_cast<uint4*>(p.pool_out + ((size_t(tc.img) * Hp + (y >> 1)) * Wp + (x >> 1)) * 32);
#pragma unroll
          for (int g = 0; g < 4; ++g) pd[g] = mx[g];
        }
      }
      quad_transpose(o, lane);
      // lane 4g+r now holds 16-byte chunk r of the pixels of lanes 4g .. 4g+3
      if (y < p.H) {
        uint8_t* obase = reinterpret_cast<uint8_t*>(p.out + (pix - r4) * 32) + r4 * 16;
        const int x0 = x - r4, i0 = i8 - r4;
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (i0 + j < 6 && x0 + j < p.W) *reinterpret_cast<uint4*>(obase + size_t(j) * 64) = o[j];
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

}  // namespace pnp
