// 3x3 stride-1 zero-pad-1 convolution + bias + LeakyReLU as an implicit GEMM on the 5th-gen tensor cores.
//
// Replaces the reference's nn.Conv2d + LeakyReLU(0.2) pairs (reference evaluation/noise.py:75-98) for
// every conv whose Cin is a multiple of 32 (26 of the 28 convs; the 2->32 first conv and the 1x1 output
// conv are handled elsewhere / in this kernel's FINAL epilogue).
//
// Mapping (B200-first, not a GEMM library call):
//   * activations are NHWC bf16; one CTA owns a 16x16 output-pixel tile of one image and BN output channels;
//   * for every KC-channel slice of the input, ONE TMA box load brings the 18x18 halo tile into shared
//     memory (rows = pixels, KC*2 bytes each, hardware 64B/128B swizzle, out-of-image pixels zero-filled =
//     the conv's zero padding).  All 9 filter taps are then issued as tcgen05.mma instructions whose
//     A-operand descriptors simply point at a shifted window of that same halo tile (start address moved by
//     (kh*18+kw) rows, 8-row groups 18 rows apart), so each input byte is read from L2 once per 9 taps;
//   * the 16x16 tile is two M=128 MMAs (16 rows x 8 columns each), accumulators live in TMEM
//     (2 x BN fp32 columns, double buffered so the epilogue of tile i overlaps the MMAs of tile i+1);
//   * weights are pre-packed on the device at plan creation into ready-to-use swizzled [BN x KC] K-major
//     blobs, one per (channel slice, tap, n-tile), fetched with 1-D bulk copies into a 4-8 deep ring;
//   * warp roles: warp0 = TMA producer, warps 1 and 3 = MMA issuers (one per M-block, one elected lane each),
//     warp2 = TMEM allocator, warps 4..11 = epilogue (tcgen05.ld -> bias -> LeakyReLU -> bf16 -> global), synchronised only through
//     mbarriers;
//   * the concat of the `up` blocks (reference noise.py:59) is never materialised: the K loop walks two
//     tensor maps (skip tensor, then upsampled tensor);
//   * FINAL epilogue (last conv of up4): the 1x1 output conv (noise.py:64-71), the global residual
//     `noisy[:, :1] + residual` (noise.py:132-133) and the clamp (noise.py:164) are applied in fp32 on the
//     un-rounded accumulators and written as fp32.
#pragma once
#include "common.cuh"

namespace pnp {

constexpr int kTile = 16;                 // output tile edge (pixels)
constexpr int kHalo = kTile + 2;          // halo tile edge
constexpr int kConvThreads = 384;         // 12 warps
constexpr int kEpiWarp0 = 4;              // first epilogue warp
constexpr int kNumEpiWarps = 8;
constexpr int kNumMmaWarps = 2;           // warps 1 and 3: M-block 0 / 1 of every tile

struct ConvParams {
  int B, H, W;              // images, spatial size (input == output size)
  int tiles_x, tiles_y;     // ceil(W/16), ceil(H/16)
  int n_tiles;              // Cout / BN
  int nchunks0, nchunks1;   // KC-channel slices taken from tensor map 0 / 1
  int Cout;
  int sa, sb;               // ring depths: halo tiles / weight tiles (sb unused when wres)
  int wres;                 // 1: all weights of this CTA's n-tile stay resident in smem (loaded once)
  int sk_split, sk_cpc;     // split-K kernel (unet_conv_splitk.cuh): cluster size S and 64-channel slices per CTA
  int sk_stages;            //   pipeline stages in shared memory: min(sk_cpc, 2)
  int rev;                  // 1: walk the tiles in descending order (the plan alternates the direction layer by layer so
                            // that a layer starts with the images its producer wrote last, which are still in L2)
  int total_tiles;
  uint32_t mg_n, mg_x, mg_y; // floor(2^32/d)+1 for d = n_tiles, tiles_x, tiles_y (tile index decomposition without IDIV)
  const uint8_t* wpk;       // packed weights, blob index ((chunk*9 + tap)*n_tiles + nt), BN*KC*2 bytes each
  const float* bias;        // [Cout]
  __nv_bfloat16* out;       // NHWC [B,H,W,Cout]                      (EPI_BF16)
  __nv_bfloat16* pool_out;  // optional NHWC [B,H/2,W/2,Cout]: MaxPool2d(2) of `out` fused into the epilogue (EPI_BF16)
  const float* wout;        // [32] 1x1 output conv weights          (EPI_FINAL)
  const float* bout;        // 1x1 output conv bias (device scalar)
  const float* noisy;       // [B,H,W] fp32 denoiser input (channel 0)
  float* x_out;             // [B,H,W] fp32 clamp(noisy + residual, 0, 1)
  float* preclamp;          // optional [B,H,W] fp32 noisy + residual
  const uint8_t* active;    // optional [B]: 0 = leave x_out / preclamp of this image untouched (early exit, env.py:79-81)
  float slope;              // LeakyReLU negative slope (0.2)
};

enum { EPI_BF16 = 0, EPI_FINAL = 1 };

constexpr int kEpiSmemFloats = 512 + 32 + 4;   // bias[Cout <= 512], 1x1 output conv weights[32], its bias

// n / d for n*d < 2^32 with the host-computed magic m = floor(2^32/d) + 1 (d == 1 has no 32-bit magic).
__host__ __device__ inline uint32_t conv_magic(uint32_t d) { return d <= 1 ? 0u : uint32_t((uint64_t(1) << 32) / d) + 1u; }
__device__ __forceinline__ uint32_t fast_div(uint32_t n, uint32_t d, uint32_t m) { return d == 1 ? n : __umulhi(n, m); }

struct TileCoord { int nt, tx, ty, img; };
__device__ __forceinline__ TileCoord decode_tile(const ConvParams& p, int tile) {
  uint32_t t = uint32_t(p.rev ? p.total_tiles - 1 - tile : tile);
  uint32_t q = fast_div(t, p.n_tiles, p.mg_n);
  TileCoord c;
  c.nt = int(t - q * p.n_tiles); t = q;
  q = fast_div(t, p.tiles_x, p.mg_x);
  c.tx = int(t - q * p.tiles_x); t = q;
  q = fast_div(t, p.tiles_y, p.mg_y);
  c.ty = int(t - q * p.tiles_y);
  c.img = int(q);
  return c;
}

// 4x4 transpose of 16-byte elements across each aligned group of 4 lanes: in v[j] = chunk j of this lane's pixel,
// out v[i] = this lane's chunk index (lane & 3) of pixel (4*(lane/4) + i).  16 SHFL; lets 4 lanes store 64 contiguous
// bytes per pixel instead of every lane storing 16 bytes into its own line.
__device__ __forceinline__ uint4 bf16x8_max(uint4 a, uint4 b) {
  uint4 r;
  const __nv_bfloat162* pa = reinterpret_cast<const __nv_bfloat162*>(&a);
  const __nv_bfloat162* pb = reinterpret_cast<const __nv_bfloat162*>(&b);
  __nv_bfloat162* pr = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) pr[i] = __hmax2(pa[i], pb[i]);
  return r;
}
__device__ __forceinline__ uint4 shfl_xor_u4(uint4 v, int m) {
  v.x = __shfl_xor_sync(0xffffffffu, v.x, m); v.y = __shfl_xor_sync(0xffffffffu, v.y, m);
  v.z = __shfl_xor_sync(0xffffffffu, v.z, m); v.w = __shfl_xor_sync(0xffffffffu, v.w, m);
  return v;
}
__device__ __forceinline__ void quad_transpose(uint4 (&v)[4], int lane) {
  const bool b0 = lane & 1, b1 = lane & 2;
#pragma unroll
  for (int j = 0; j < 4; j += 2) {
    const uint4 r = shfl_xor_u4(b0 ? v[j] : v[j + 1], 1);
    if (b0) v[j] = r; else v[j + 1] = r;
  }
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const uint4 r = shfl_xor_u4(b1 ? v[j] : v[j + 2], 2);
    if (b1) v[j] = r; else v[j + 2] = r;
  }
}

// bf16 epilogue of one 32-channel chunk (conv3x3_umma_kernel, conv3x3_pair_kernel).  r = the fp32 accumulators of
// channels ch0 .. ch0+31 of this lane's pixel (img, y, x), bias = their biases.  The warp holds 4 rows x 8 columns of
// pixels, lane = 8 * row + column with the first row even: lane ^ 1 is the right neighbour, lane ^ 8 the one below.
// Writes bias + LeakyReLU as bf16 to p.out and, when p.pool_out is set, its MaxPool2d(2) (reference noise.py:23).
// store = false computes without storing (a duplicated tile); the shuffles stay warp-uniform.
__device__ __forceinline__ void epilogue_bf16_chunk(const ConvParams& p, const uint32_t (&r)[32], const float* bias, int ch0,
                                                    int img, int y, int x, int lane, bool store) {
  uint4 o[4];
  const float2 sl2 = make_float2(p.slope, p.slope);
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    const float4 ba = *reinterpret_cast<const float4*>(bias + i);
    const float4 bb = *reinterpret_cast<const float4*>(bias + i + 4);
    // bias + LeakyReLU on packed fp32 pairs: max(v, slope v) == LeakyReLU(v) for 0 < slope < 1
    const float2 a0 = __fadd2_rn(make_float2(__uint_as_float(r[i]), __uint_as_float(r[i + 1])), make_float2(ba.x, ba.y));
    const float2 a1 = __fadd2_rn(make_float2(__uint_as_float(r[i + 2]), __uint_as_float(r[i + 3])), make_float2(ba.z, ba.w));
    const float2 a2 = __fadd2_rn(make_float2(__uint_as_float(r[i + 4]), __uint_as_float(r[i + 5])), make_float2(bb.x, bb.y));
    const float2 a3 = __fadd2_rn(make_float2(__uint_as_float(r[i + 6]), __uint_as_float(r[i + 7])), make_float2(bb.z, bb.w));
    const float2 m0 = __fmul2_rn(a0, sl2), m1 = __fmul2_rn(a1, sl2), m2 = __fmul2_rn(a2, sl2), m3 = __fmul2_rn(a3, sl2);
    const float v0 = fmaxf(a0.x, m0.x), v1 = fmaxf(a0.y, m0.y), v2 = fmaxf(a1.x, m1.x), v3 = fmaxf(a1.y, m1.y);
    const float v4 = fmaxf(a2.x, m2.x), v5 = fmaxf(a2.y, m2.y), v6 = fmaxf(a3.x, m3.x), v7 = fmaxf(a3.y, m3.y);
    o[i / 8] = make_uint4(pack_bf16x2(v0, v1), pack_bf16x2(v2, v3), pack_bf16x2(v4, v5), pack_bf16x2(v6, v7));
  }
  // after the quad transpose this lane holds 16-byte chunk r4 of the pixels x0 .. x0+3 (x0 a multiple of 4) of row y
  quad_transpose(o, lane);
  const int r4 = lane & 3, x0 = x - r4;
  if (store && y < p.H) {
    uint8_t* obase = reinterpret_cast<uint8_t*>(p.out + ((size_t(img) * p.H + y) * p.W + x0) * p.Cout + ch0) + r4 * 16;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (x0 + i < p.W) *reinterpret_cast<uint4*>(obase + size_t(i) * p.Cout * 2) = o[i];
  }
  if (p.pool_out) {
    // MaxPool2d(2) on the transposed registers: the horizontal maxima need no shuffle; the row below (y even) lives in
    // lane ^ 8.  8 SHFL; four lanes store 64 contiguous bytes per pooled pixel.
    uint4 h0 = bf16x8_max(o[0], o[1]), h1 = bf16x8_max(o[2], o[3]);
    h0 = bf16x8_max(h0, shfl_xor_u4(h0, 8));
    h1 = bf16x8_max(h1, shfl_xor_u4(h1, 8));
    const int Hp = p.H >> 1, Wp = p.W >> 1;
    if (store && ((lane & 8) == 0) && (y >> 1) < Hp) {
      uint8_t* pd = reinterpret_cast<uint8_t*>(p.pool_out + ((size_t(img) * Hp + (y >> 1)) * Wp + (x0 >> 1)) * p.Cout + ch0) +
                    r4 * 16;
      if ((x0 >> 1) < Wp) *reinterpret_cast<uint4*>(pd) = h0;
      if ((x0 >> 1) + 1 < Wp) *reinterpret_cast<uint4*>(pd + size_t(p.Cout) * 2) = h1;
    }
  }
}

template <int KC, int BN>
struct ConvCfg {
  static constexpr int ROWB = KC * 2;                                    // bytes per pixel row in smem
  static constexpr int A_BYTES = kHalo * kHalo * ROWB;                   // TMA box bytes
  static constexpr int A_STAGE = (A_BYTES + 1023) / 1024 * 1024;
  static constexpr int B_BYTES = BN * ROWB;
  static constexpr int B_STAGE = (B_BYTES + 1023) / 1024 * 1024;
  static constexpr int NACC = (BN == 32) ? 4 : 2;                           // TMEM accumulator stages
  static constexpr int TMEM_COLS = 2 * BN * NACC;                        // 2 M-blocks x BN x stages
  static constexpr int MAX_RING = 16;                                    // upper bound for sa, sb
  static constexpr int BAR_BYTES = (4 * MAX_RING + 2 * NACC + 2) * 8 + 16 + kEpiSmemFloats * 4;
  // dynamic smem = 1024 (alignment slack) + sa*A_STAGE + (wres ? nchunks*9*B_BYTES : sb*B_STAGE) + BAR_BYTES
  static_assert(TMEM_COLS >= 32 && TMEM_COLS <= 512 && (TMEM_COLS & (TMEM_COLS - 1)) == 0, "TMEM cols");
};

template <int KC, int BN, int EPI>
__global__ void __launch_bounds__(kConvThreads, 1)
conv3x3_umma_kernel(const ConvParams p, const __grid_constant__ CUtensorMap tmA0,
                    const __grid_constant__ CUtensorMap tmA1) {
  using Cfg = ConvCfg<KC, BN>;
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
  float* epi_s = reinterpret_cast<float*>(tmem_slot + 4);   // bias[Cout] | wout[32] | bout   (kEpiSmemFloats)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int total_tiles = p.B * p.tiles_y * p.tiles_x * p.n_tiles;

  grid_dep_launch();
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA0);
    tma_prefetch_desc(&tmA1);
  }
  if (warp == 1 && lane == 0) {
    // two MMA-issuing warps (one per M-block): every "consumed" barrier gets one tcgen05.commit arrival from each
    for (int i = 0; i < SA; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], kNumMmaWarps); }
    for (int i = 0; i < SB; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], kNumMmaWarps); }
    for (int i = 0; i < NACC; ++i) { mbar_init(&acc_full[i], kNumMmaWarps); mbar_init(&acc_empty[i], kNumEpiWarps); }
    mbar_init(w_full, 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  if (warp >= kEpiWarp0) {   // epilogue constants: read from shared memory per tile, not through L1 from global
    const int t = threadIdx.x - kEpiWarp0 * 32;
    for (int i = t; i < p.Cout; i += kNumEpiWarps * 32) epi_s[i] = __ldg(p.bias + i);
    if (EPI == EPI_FINAL && t < 33) epi_s[512 + t] = t < 32 ? __ldg(p.wout + t) : __ldg(p.bout);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================================== TMA producer =====================================
    if (lane == 0) {
      int sa = 0, pa = 0, sb = 0, pb = 0;
      if (p.wres && int(blockIdx.x) < total_tiles) {
        // n_tiles == 1 here: the layer's packed weights are one contiguous run of nchunks*9 blobs
        const uint32_t wbytes = uint32_t(nchunks) * 9 * Cfg::B_BYTES;
        mbar_arrive_expect_tx(w_full, wbytes);
        for (uint32_t off = 0; off < wbytes; off += 9 * Cfg::B_BYTES)
          bulk_load_1d(b_smem + off, p.wpk + off, 9 * Cfg::B_BYTES, w_full);
      }
      grid_dep_wait();          // weights are constants; the activations below come from the previous kernel
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const TileCoord tc = decode_tile(p, tile);
        const int nt = tc.nt, tx = tc.tx, ty = tc.ty, img = tc.img;
        for (int c = 0; c < nchunks; ++c) {
          mbar_wait(&a_empty[sa], pa ^ 1);
          mbar_arrive_expect_tx(&a_full[sa], Cfg::A_BYTES);
          const bool seg0 = c < p.nchunks0;
          tma_load_4d(a_smem + sa * Cfg::A_STAGE, seg0 ? &tmA0 : &tmA1, &a_full[sa],
                      (seg0 ? c : c - p.nchunks0) * KC, tx * kTile - 1, ty * kTile - 1, img);
          if (++sa == SA) { sa = 0; pa ^= 1; }
          if (p.wres) continue;
          const uint8_t* wsrc = p.wpk + (size_t(c) * 9 * p.n_tiles + nt) * Cfg::B_BYTES;
          for (int tap = 0; tap < 9; ++tap) {
            mbar_wait(&b_empty[sb], pb ^ 1);
            mbar_arrive_expect_tx(&b_full[sb], Cfg::B_BYTES);
            bulk_load_1d(b_smem + sb * Cfg::B_STAGE, wsrc + size_t(tap) * p.n_tiles * Cfg::B_BYTES, Cfg::B_BYTES,
                         &b_full[sb]);
            if (++sb == SB) { sb = 0; pb ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1 || warp == 3) {
    // ===================================== MMA issuers ======================================
    // Two issuing warps, one per M=128 pixel block of the tile (warp 1: left 8 columns, warp 3: right 8 columns), each
    // with its own accumulator.  Measured on B200 (tools/mma_bench2.cu): the tensor pipe runs only ~1 MMA ahead of an
    // issuing thread, so every barrier wait / commit between MMA groups of ONE issuer idles the pipe for ~100-170
    // cycles (30 % of a deep layer); with two independent issuers one warp's wait is covered by the other's MMAs
    // (64.1 clk per M128xN128xK16 MMA = the math rate, and 40 instead of 49 clk at N=32).
    // Each warp walks the loop warp-uniformly (descriptors stay in uniform registers); one elected lane issues.
    const int mb = warp == 3 ? 1 : 0;
    constexpr uint32_t idesc = umma_idesc_bf16(128, BN);
    // high words of the smem descriptors are loop invariant: SBO | version | layout
    constexpr uint32_t kLayout = (ROWB == 128) ? 2u : 4u;
    constexpr uint32_t a_hi = (uint32_t(kHalo * ROWB) >> 4) | (1u << 14) | (kLayout << 29);
    constexpr uint32_t b_hi = (uint32_t(8 * ROWB) >> 4) | (1u << 14) | (kLayout << 29);
    int sa = 0, pa = 0, sb = 0, pb = 0;
    int it = 0;
    if (p.wres && int(blockIdx.x) < total_tiles) mbar_wait(w_full, 0);
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const int as = it % NACC;
      const uint32_t aph = (it / NACC) & 1;
      mbar_wait(&acc_empty[as], aph ^ 1);
      const uint32_t d0 = tmem_base + as * (2 * BN) + mb * BN;
      for (int c = 0; c < nchunks; ++c) {
        mbar_wait(&a_full[sa], pa);
        tc_fence_after();
        // descriptor low word: (addr >> 4) | LBO(=1) << 16 ; smem addresses are < 256 KB so no masking is needed
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
                umma_bf16_ss2(d0, a_tap + k * 2, a_hi, b_tap + k * 2, b_hi, idesc, (c | tap | k) != 0 ? 1u : 0u);
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
                umma_bf16_ss2(d0, a_tap + k * 2, a_hi, b_tap + k * 2, b_hi, idesc, (c | tap | k) != 0 ? 1u : 0u);
              tc_commit(&b_empty[sb]);   // weight slot free once both warps' MMAs have read it
            }
            __syncwarp();
            if (++sb == SB) { sb = 0; pb ^= 1; }
          }
        }
        if (elect_one()) tc_commit(&a_empty[sa]);     // halo slot free
        __syncwarp();
        if (++sa == SA) { sa = 0; pa ^= 1; }
      }
      if (elect_one()) tc_commit(&acc_full[as]);      // this M-block's accumulator complete -> epilogue
      __syncwarp();
    }
  } else if (warp >= kEpiWarp0) {
    // ===================================== epilogue =========================================
    const int q = warp & 3;                    // TMEM lane quarter this warp may access
    const int mb = (warp - kEpiWarp0) >> 2;    // which M-block (left / right 8 columns of the tile)
    const int m = q * 32 + lane;               // row of the M=128 accumulator = pixel within the 16x8 block
    const int prow = m >> 3, pcol = (m & 7) + mb * 8;
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const TileCoord tc = decode_tile(p, tile);
      const int nt = tc.nt;
      const int as = it % NACC;
      const uint32_t aph = (it / NACC) & 1;
      const int y = tc.ty * kTile + prow, x = tc.tx * kTile + pcol;
      const size_t pix = (size_t(tc.img) * p.H + y) * p.W + x;
      // FINAL epilogue: the residual input is fetched BEFORE the wait for the accumulator (its latency then overlaps the
      // MMAs instead of sitting between the last FMA and the store)
      float noisy_px = 0.f;
      if constexpr (EPI == EPI_FINAL) { if ((y < p.H) && (x < p.W)) noisy_px = __ldg(p.noisy + pix); }
      mbar_wait(&acc_full[as], aph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + as * (2 * BN) + mb * BN;
      if constexpr (EPI == EPI_BF16) {
#pragma unroll 1
        for (int cc = 0; cc < BN / 32; ++cc) {
          uint32_t r[32];
          tmem_ld_32x32(taddr + cc * 32, r);
          tmem_ld_wait();
          if (cc == BN / 32 - 1) {     // accumulator stage drained: hand it back before the math and the stores
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[as]);
          }
          epilogue_bf16_chunk(p, r, epi_s + nt * BN + cc * 32, nt * BN + cc * 32, tc.img, y, x, lane, true);
        }
      } else {
        static_assert(EPI == EPI_BF16 || BN == 32, "FINAL epilogue needs all 32 channels in one thread");
        uint32_t r[32];
        tmem_ld_32x32(taddr, r);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[as]);
        float s = epi_s[512 + 32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float v = __uint_as_float(r[i]) + epi_s[i];
          v = v > 0.f ? v : v * p.slope;
          s = fmaf(v, epi_s[512 + i], s);
        }
        if ((y < p.H) && (x < p.W) && !(p.active && p.active[tc.img] == 0)) {
          const float o = noisy_px + s;
          if (p.preclamp) p.preclamp[pix] = o;
          p.x_out[pix] = fminf(fmaxf(o, 0.f), 1.f);
        }
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
