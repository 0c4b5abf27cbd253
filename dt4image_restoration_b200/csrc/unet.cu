// U-Net denoiser (reference evaluation/noise.py:101-164) as a launch plan over hand-written sm_100a kernels.
//
//   conv_first_kernel   : noise-level-map concat (noise.py:161-162) + 2->32 3x3 conv + LeakyReLU, fp32 math
//                         on CUDA cores (K = 18 is not tensor-core work), NHWC bf16 out
//   conv3x3_umma_kernel : every other 3x3 conv (unet_conv.cuh), incl. the fused 1x1 output conv + global
//                         residual + clamp in the FINAL epilogue
//   upsample2x_kernel   : nn.Upsample(x2, bilinear, align_corners=True) + zero pad to the skip size
//                         (noise.py:39,46-53), NHWC bf16; the channel concat (noise.py:59) is never
//                         materialised - the consuming conv walks two tensor maps
//   pack_weights_kernel : reference state_dict fp32 [Cout][Cin][3][3] -> bf16 swizzled K-major UMMA blobs
#include <algorithm>
#include <mutex>
#include <vector>
#include <string>
#include <cstring>
#include "common.cuh"
#include "unet_conv.cuh"
#include "unet_conv_kws.cuh"
#include "unet_conv_pair.cuh"
#include "unet_conv_splitk.cuh"
#include "pnp_internal.h"

namespace pnp {

// ------------------------------------------------------------------------------------------------
// auxiliary kernels
// ------------------------------------------------------------------------------------------------
// First conv (noise.py:161-162 concat + 2->32 3x3 conv + LeakyReLU) in fp32 on CUDA cores.
// The weights travel as a __grid_constant__ kernel parameter, i.e. they live in the constant bank and feed FFMA
// directly (no shared-memory loads).  One thread per PAIR of vertically adjacent output pixels, all 32 output channels:
// the pair shares 12 input loads and every weight fetch.  The noise-level channel is constant inside the image, so its
// nine taps collapse to sigma * (sum of the taps that fall inside the image): nine pre-summed cases (row position
// first/inner/last x column position first/inner/last), the inner one served from the constant bank.
struct FirstConvW {
  float w[9][32];         // image channel, [tap][co]
  float b[32];
  float ws[9][32];        // [3 * rowcase + colcase][co]: sum of the sigma-channel taps inside the image; case 4 = inner
};

// A thread walks `ppt` row pairs downwards (grid.y = ceil(ceil(H/2) / ppt)) with the next pair's rows loaded ahead.

__global__ void __launch_bounds__(256) conv_first_kernel(const float* __restrict__ v, const float* __restrict__ sigma,
                                                         const __grid_constant__ FirstConvW cw,
                                                         __nv_bfloat16* __restrict__ out, int B, int H, int W,
                                                         float slope, int rev, int ppt) {
  grid_dep_launch();
  grid_dep_wait();
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int pairs = (H + 1) / 2;
  const int pair0 = ppt * (rev ? int(gridDim.y) - 1 - int(blockIdx.y) : int(blockIdx.y));
  const int pair1 = pair0 + ppt < pairs ? pair0 + ppt : pairs;
  const int b = rev ? B - 1 - int(blockIdx.z) : int(blockIdx.z);
  if (x >= W) return;
  const float sg = __ldg(sigma + b);
  const float* vb = v + size_t(b) * H * W + x;
  const bool xl = x > 0, xr = x + 1 < W;
  const int cx = xl ? (xr ? 1 : 2) : 0;
  auto load_row = [&](int yy, float (&r)[3]) {     // row yy, columns x-1 .. x+1 (zero outside the image)
    const bool ok = (yy >= 0) && (yy < H);
    const float* row = vb + ptrdiff_t(yy) * W;
    r[0] = (ok && xl) ? __ldg(row - 1) : 0.f;
    r[1] = ok ? __ldg(row) : 0.f;
    r[2] = (ok && xr) ? __ldg(row + 1) : 0.f;
  };
  float in[4][3], nx[2][3];                        // window rows y0-1 .. y0+2 and the two rows the next pair adds
#pragma unroll
  for (int r = 0; r < 4; ++r) load_row(2 * pair0 - 1 + r, in[r]);
#pragma unroll 1
  for (int pair = pair0; pair < pair1; ++pair) {
    const int y0 = 2 * pair;
    load_row(y0 + 3, nx[0]);                       // in flight while this pair is computed
    load_row(y0 + 4, nx[1]);
    const int cs0 = (y0 == 0 ? 0 : (y0 == H - 1 ? 6 : 3)) + cx;
    const int cs1 = (y0 + 1 == H - 1 ? 6 : 3) + cx;
    float acc0[32], acc1[32];
    if (cs0 == 4 && cs1 == 4) {
#pragma unroll
      for (int co = 0; co < 32; ++co) acc0[co] = acc1[co] = fmaf(sg, cw.ws[4][co], cw.b[co]);
    } else {
#pragma unroll
      for (int co = 0; co < 32; ++co) {
        acc0[co] = fmaf(sg, cw.ws[cs0][co], cw.b[co]);
        acc1[co] = fmaf(sg, cw.ws[cs1][co], cw.b[co]);
      }
    }
#pragma unroll
    for (int t = 0; t < 9; ++t) {
#pragma unroll
      for (int co = 0; co < 32; ++co) {
        const float wv = cw.w[t][co];
        acc0[co] = fmaf(wv, in[t / 3][t % 3], acc0[co]);
        acc1[co] = fmaf(wv, in[t / 3 + 1][t % 3], acc1[co]);
      }
    }
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      if (p == 1 && y0 + 1 >= H) break;
      const float* acc = p ? acc1 : acc0;
      uint32_t o[16];
#pragma unroll
      for (int co = 0; co < 32; co += 2) {
        const float a0 = fmaxf(acc[co], acc[co] * slope);            // LeakyReLU for 0 < slope < 1
        const float a1 = fmaxf(acc[co + 1], acc[co + 1] * slope);
        o[co / 2] = pack_bf16x2(a0, a1);
      }
      uint4* dst = reinterpret_cast<uint4*>(out + ((size_t(b) * H + y0 + p) * W + x) * 32);
      dst[0] = make_uint4(o[0], o[1], o[2], o[3]);
      dst[1] = make_uint4(o[4], o[5], o[6], o[7]);
      dst[2] = make_uint4(o[8], o[9], o[10], o[11]);
      dst[3] = make_uint4(o[12], o[13], o[14], o[15]);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      in[0][c] = in[2][c]; in[1][c] = in[3][c]; in[2][c] = nx[0][c]; in[3][c] = nx[1][c];
    }
  }
}


// in [B,h,w,C] -> out [B,Ho,Wo,C]: bilinear x2 (align_corners=True) placed at offset (py,px), zeros elsewhere.
// grid (ceil(Wo*C8/256), ceil(Ho/4), B); each thread produces 8 channels of 4 vertically adjacent output pixels
// (16 independent 16-byte loads in flight).
constexpr int kUpsRows = 4;
__global__ void __launch_bounds__(256) upsample2x_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, int B,
                                                         int h, int w, int Ho, int Wo, int C8, int py, int px,
                                                         float sy, float sx) {
  grid_dep_launch();
  grid_dep_wait();
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= Wo * C8) return;
  const int c = e % C8, xo = e / C8;
  const int b = blockIdx.z;
  const int ux = xo - px;
  const bool xin = ux >= 0 && ux < 2 * w;
  const float fx = sx * float(ux);
  const int x0 = xin ? int(fx) : 0;
  const int x1 = x0 + (x0 < w - 1 ? 1 : 0);
  const float lx = fx - float(x0), hx = 1.f - lx;
  const size_t base = size_t(b) * h * w;
  uint4 q[kUpsRows][4];
  float ly[kUpsRows];
  bool ok[kUpsRows];
#pragma unroll
  for (int r = 0; r < kUpsRows; ++r) {
    const int yo = blockIdx.y * kUpsRows + r;
    const int uy = yo - py;
    ok[r] = xin && yo < Ho && uy >= 0 && uy < 2 * h;
    const float fy = sy * float(uy);
    const int y0 = ok[r] ? int(fy) : 0;
    const int y1 = y0 + (y0 < h - 1 ? 1 : 0);
    ly[r] = fy - float(y0);
    q[r][0] = __ldg(in + (base + size_t(y0) * w + x0) * C8 + c);
    q[r][1] = __ldg(in + (base + size_t(y0) * w + x1) * C8 + c);
    q[r][2] = __ldg(in + (base + size_t(y1) * w + x0) * C8 + c);
    q[r][3] = __ldg(in + (base + size_t(y1) * w + x1) * C8 + c);
  }
#pragma unroll
  for (int r = 0; r < kUpsRows; ++r) {
    const int yo = blockIdx.y * kUpsRows + r;
    if (yo >= Ho) break;
    uint4 res = make_uint4(0, 0, 0, 0);
    if (ok[r]) {
      const float hy = 1.f - ly[r];
      const __nv_bfloat162* a = reinterpret_cast<const __nv_bfloat162*>(&q[r][0]);
      const __nv_bfloat162* bq = reinterpret_cast<const __nv_bfloat162*>(&q[r][1]);
      const __nv_bfloat162* cq = reinterpret_cast<const __nv_bfloat162*>(&q[r][2]);
      const __nv_bfloat162* d = reinterpret_cast<const __nv_bfloat162*>(&q[r][3]);
      uint32_t* o = reinterpret_cast<uint32_t*>(&res);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 f00 = __bfloat1622float2(a[k]), f01 = __bfloat1622float2(bq[k]);
        const float2 f10 = __bfloat1622float2(cq[k]), f11 = __bfloat1622float2(d[k]);
        const float vx = hy * (hx * f00.x + lx * f01.x) + ly[r] * (hx * f10.x + lx * f11.x);
        const float vy = hy * (hx * f00.y + lx * f01.y) + ly[r] * (hx * f10.y + lx * f11.y);
        o[k] = pack_bf16x2(vx, vy);
      }
    }
    out[(size_t(b) * Ho + yo) * Wo * C8 + e] = res;
  }
}

// Fast path of the x2 bilinear upsample (align_corners=True) for the exact-doubling case (Ho == 2h, Wo == 2w, no pad).
// With scale s = (h-1)/(2h-1) the source index of output row uy is uy/2 - uy/(2(2h-1)), i.e. for uy > 0
//     floor(s*uy) = uy/2 - 1 (uy even),  (uy-1)/2 (uy odd)
// so the output rows (2m+1, 2m+2) both interpolate the source rows (m, m+1), and likewise for columns: one thread
// loads the 2x2 source block (m..m+1, n..n+1) of 8 channels (4 x 16 B) and produces the 2x2 output block
// (rows 2m+1..2m+2, cols 2n+1..2n+2) - one load and ~28 instructions per 16-byte output instead of 4 loads and ~100
// (the general kernel is instruction-issue bound: 0.24 ms for 537 MB written at 256^2 x 64 ch x B=64).
// Blocks m = -1 and m = h-1 (n = -1, n = w-1) produce the first / last output row (column) with clamped sources.
// The interpolation weights are taken from the same fp32 formula as the general kernel / the reference
// (lambda = s*u - floor index), so both paths agree to rounding.
// grid (ceil((w+1)*C8/256), h+1, B)
// int -> float for -1 <= k < 2^22 on the FMA pipe (exact; I2FP and the runtime division below ran on the quarter-rate XU
// pipe, which ncu showed 82 % busy: profiles/r02_ncu_full_upsample.txt)
__device__ __forceinline__ float small_int_to_float(int k) { return __int_as_float(0x4B000000 + (k + 1)) - 8388609.0f; }

// A thread walks `walk` source row blocks downwards (grid.y = ceil((h + 1) / walk)): the x-interpolated bottom row of one
// block is the top row of the next (half the loads), the next row's loads are in flight while a block is written, and a
// launch has ~8x fewer, longer-lived CTAs.

__global__ void __launch_bounds__(256) upsample2x_fast_kernel(const uint4* __restrict__ in, uint4* __restrict__ out,
                                                              int h, int w, int C8, float sy, float sx, int nimg,
                                                              int rev, int c8_shift, int walk) {
  grid_dep_launch();
  grid_dep_wait();
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (w + 1) * C8) return;
  const int c = e & (C8 - 1), n = (e >> c8_shift) - 1;          // C8 is a power of two; source column block n = -1 .. w-1
  const int by = rev ? int(gridDim.y) - 1 - int(blockIdx.y) : int(blockIdx.y);
  const int m0 = by * walk - 1;                                  // first source row block of this walk (m = -1 .. h-1)
  const int m1 = (m0 + walk < h) ? m0 + walk : h;                // one past the last
  const int b = rev ? nimg - 1 - int(blockIdx.z) : int(blockIdx.z);
  const int xa = n < 0 ? 0 : n, xb = n + 1 < w ? n + 1 : w - 1;
  const uint4* src = in + size_t(b) * h * w * C8 + c;
  const int Ho = 2 * h, Wo = 2 * w;
  float lx[2];
#pragma unroll
  for (int j = 0; j < 2; ++j) lx[j] = sx * small_int_to_float(2 * n + 1 + j) - small_int_to_float(n);
  // x-interpolated source row for the two output columns, 4 channel pairs each
  auto xlerp = [&](const uint4& qa, const uint4& qb, float2 (&t)[2][4]) {
    const uint32_t* a = reinterpret_cast<const uint32_t*>(&qa);
    const uint32_t* bb = reinterpret_cast<const uint32_t*>(&qb);
#pragma unroll
    for (int k = 0; k < 4; ++k) {                 // channel pair k (bf16x2 -> packed fp32x2 arithmetic)
      const float2 fa = make_float2(__uint_as_float(a[k] << 16), __uint_as_float(a[k] & 0xffff0000u));
      const float2 fb = make_float2(__uint_as_float(bb[k] << 16), __uint_as_float(bb[k] & 0xffff0000u));
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const float2 l2 = make_float2(lx[j], lx[j]), h2 = make_float2(1.f - lx[j], 1.f - lx[j]);
        t[j][k] = __ffma2_rn(fb, l2, __fmul2_rn(fa, h2));
      }
    }
  };
  auto row_ptr = [&](int y) { return src + size_t(y < 0 ? 0 : (y < h ? y : h - 1)) * w * C8; };
  float2 top[2][4], bot[2][4];
  {
    const uint4* r = row_ptr(m0);
    xlerp(__ldg(r + size_t(xa) * C8), __ldg(r + size_t(xb) * C8), top);
  }
  const uint4* rn = row_ptr(m0 + 1);
  uint4 qa = __ldg(rn + size_t(xa) * C8), qb = __ldg(rn + size_t(xb) * C8);
#pragma unroll 1
  for (int m = m0; m < m1; ++m) {
    xlerp(qa, qb, bot);
    if (m + 1 < m1) {                             // the row after next is in flight while this block is written
      rn = row_ptr(m + 2);
      qa = __ldg(rn + size_t(xa) * C8); qb = __ldg(rn + size_t(xb) * C8);
    }
    // interpolation weights of the two output rows relative to source index m (same fp32 formula as the general kernel)
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int yo = 2 * m + 1 + i;
      if (yo < 0 || yo >= Ho) continue;
      const float ly = sy * small_int_to_float(yo) - small_int_to_float(m);
      const float2 ll = make_float2(ly, ly), hh = make_float2(1.f - ly, 1.f - ly);
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int xo = 2 * n + 1 + j;
        if (xo < 0 || xo >= Wo) continue;
        uint4 res;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 v = __ffma2_rn(bot[j][k], ll, __fmul2_rn(top[j][k], hh));
          reinterpret_cast<uint32_t*>(&res)[k] = pack_bf16x2(v.x, v.y);
        }
        out[((size_t(b) * Ho + yo) * Wo + xo) * C8 + c] = res;
      }
    }
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int k = 0; k < 4; ++k) top[j][k] = bot[j][k];
  }
}

// fp32 [Cout][Cin][3][3] -> swizzled bf16 blobs (layout documented in unet_conv.cuh / DESIGN.md).
__global__ void pack_weights_kernel(const float* __restrict__ w, uint8_t* __restrict__ out, int Cin, int Cout, int KC,
                                    int BN) {
  const int n_tiles = Cout / BN;
  const int ROWB = KC * 2;
  const int swz_mask = (ROWB == 128) ? 7 : 3;
  const size_t total = size_t(Cout) * Cin * 9;
  for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
    const int tap = int(i % 9);
    const int ci = int((i / 9) % Cin);
    const int co = int(i / (size_t(9) * Cin));
    const int chunk = ci / KC, kk = ci % KC;
    const int nt = co / BN, n = co % BN;
    const uint32_t off = uint32_t(n * ROWB + (kk / 8) * 16);
    const uint32_t phys = off ^ (((off >> 7) & swz_mask) << 4);
    const size_t blob = (size_t(chunk) * 9 + tap) * n_tiles + nt;
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(out + blob * size_t(BN) * ROWB + phys) + (kk % 8);
    *dst = __float2bfloat16_rn(w[i]);
  }
}

// Weights of a 32-output-channel layer for conv3x3_kws_kernel: blob (chunk, kh) = [96 rows (kw, co)][32 ci] bf16,
// K-major, SWIZZLE_64B.
__global__ void pack_weights_kws_kernel(const float* __restrict__ w, uint8_t* __restrict__ out, int Cin) {
  const size_t total = size_t(32) * Cin * 9;
  for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
    const int tap = int(i % 9), kh = tap / 3, kw = tap % 3;
    const int ci = int((i / 9) % Cin);
    const int co = int(i / (size_t(9) * Cin));
    const int chunk = ci / 32, kk = ci % 32;
    const int n = kw * 32 + co;
    const uint32_t off = uint32_t(n * 64 + (kk / 8) * 16);
    const uint32_t phys = off ^ (((off >> 7) & 3) << 4);
    const size_t blob = size_t(chunk) * 3 + kh;
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(out + blob * size_t(KwsCfg::B_BYTES) + phys) + (kk % 8);
    *dst = __float2bfloat16_rn(w[i]);
  }
}

// ------------------------------------------------------------------------------------------------
// host side: tensor maps, conv launches
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static int g_num_sms = 148;
static const int kSkGain = 3;       // measured on B200 (B = 1..32, 128^2 and 256^2): 3 and 4 tie, 2 and 6 lose a little
static int g_splitk_mode = -1;      // -1 auto (few-tile launches), 0 never, 1 every eligible conv (tests)
int unet_set_splitk(int mode) {
  const int old = g_splitk_mode;
  if (mode >= -1 && mode <= 1) g_splitk_mode = mode;
  return old;
}

static const int kConvSmemMax = 227 * 1024;          // opt-in maximum per CTA on sm_100
static const int kConvSmemBudget = 222 * 1024;       // what the ring sizing may use

template <int KC, int BN, int EPI>
static int set_conv_attr() {
  return int(cudaFuncSetAttribute(conv3x3_umma_kernel<KC, BN, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  kConvSmemMax));
}

int unet_global_init() {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || fn == nullptr) {
    set_error("cuTensorMapEncodeTiled driver entry point not available");
    return e != cudaSuccess ? int(e) : 999;
  }
  g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
  int rc = 0;
  rc |= set_conv_attr<32, 32, EPI_BF16>();
  rc |= set_conv_attr<32, 32, EPI_FINAL>();
  rc |= set_conv_attr<32, 64, EPI_BF16>();
  rc |= set_conv_attr<64, 64, EPI_BF16>();
  rc |= set_conv_attr<64, 128, EPI_BF16>();
  rc |= int(cudaFuncSetAttribute(conv3x3_pair_kernel<32, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, kConvSmemMax));
  rc |= int(cudaFuncSetAttribute(conv3x3_pair_kernel<64, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, kConvSmemMax));
  rc |= int(cudaFuncSetAttribute(conv3x3_pair_kernel<64, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, kConvSmemMax));
  rc |= int(cudaFuncSetAttribute(conv3x3_kws_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kConvSmemMax));
  rc |= int(cudaFuncSetAttribute(conv3x3_splitk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSkSmem));
  if (rc) set_error("cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed");
  return rc;
}

int num_sms() { return g_num_sms; }

// NHWC bf16 activation tensor -> 4-D map (C, W, H, N), box (KC, 18, 18, 1), swizzle = KC*2 bytes.
static int make_act_map(CUtensorMap* m, const void* base, int B, int H, int W, int C, int KC, int box_w = kHalo,
                        int box_h = kHalo) {
  if (!g_encode) { set_error("pnp_init() has not been called"); return -3; }
  cuuint64_t dims[4] = {cuuint64_t(C), cuuint64_t(W), cuuint64_t(H), cuuint64_t(B)};
  cuuint64_t strides[3] = {cuuint64_t(C) * 2, cuuint64_t(W) * C * 2, cuuint64_t(H) * W * C * 2};
  cuuint32_t box[4] = {cuuint32_t(KC), cuuint32_t(box_w), cuuint32_t(box_h), 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, KC == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (code " + std::to_string(int(r)) + ")");
    return 1000 + int(r);
  }
  return 0;
}

struct ConvLaunch {
  ConvParams p;
  CUtensorMap tm0, tm1;
  CUtensorMap tmw;          // pair kernel: 2-D map over the layer's packed weight blobs (rows of KC channels)
  int KC, BN, EPI;
  int kws;                  // 1: conv3x3_kws_kernel (32 output channels, kw-stacked N = 96)
  int pair;                 // 1: conv3x3_pair_kernel (CTA pairs, tcgen05.mma.cta_group::2)
  int splitk;               // 1: conv3x3_splitk_kernel (few-tile launches: N and K cut across a cluster)
  int grid;
  int smem;
};

// barriers + epilogue constants of a conv CTA, sized for ConvCfg::NACC = 4 (BN = 32); what is left of the budget after
// them and the alignment slack goes to the rings
static const int kConvBarBytes = (4 * 16 + 2 * 4 + 2) * 8 + 16 + kEpiSmemFloats * 4;
static const int kConvRingBytes = kConvSmemBudget - 1024 - kConvBarBytes - 1024;
static int halo_stage_bytes(int KC) { return (kHalo * kHalo * KC * 2 + 1023) / 1024 * 1024; }

// A CTA keeps its weights resident when it has one n-tile and all of it (wbytes) fits next to >= 3 halo stages; otherwise
// they are streamed through as deep a ring as fits (latency of an L2 fetch ~1 us vs ~0.1-0.3 us of MMA work per tap).
static bool weights_fit(int KC, int n_tiles, long long wbytes) {
  return n_tiles == 1 && wbytes + 3 * halo_stage_bytes(KC) <= kConvRingBytes;
}

static void size_rings(ConvLaunch& L) {
  if (L.kws) {
    const int bar = KwsCfg::BAR_BYTES;
    const int avail = kConvSmemBudget - 1024 - bar - 1024;
    const int wtotal = (L.p.nchunks0 + L.p.nchunks1) * 3 * KwsCfg::B_BYTES;
    int sa = (avail - wtotal) / KwsCfg::A_STAGE;
    L.p.wres = 1; L.p.sb = 1;
    L.p.sa = sa > 8 ? 8 : sa;
    L.smem = 1024 + L.p.sa * KwsCfg::A_STAGE + ((wtotal + 1023) & ~1023) + bar;
    return;
  }
  const int ROWB = L.KC * 2;
  const int a_stage = halo_stage_bytes(L.KC);
  const int b_bytes = L.BN * ROWB / (L.pair ? 2 : 1);       // a CTA of a pair keeps half of every weight blob
  const int b_stage = (b_bytes + 1023) / 1024 * 1024;
  const int bar = kConvBarBytes;
  const int avail = kConvRingBytes;
  const int nchunks = L.p.nchunks0 + L.p.nchunks1;
  const int wtotal = nchunks * 9 * b_bytes;
  ConvParams& p = L.p;
  if (weights_fit(L.KC, p.n_tiles, wtotal)) {
    p.wres = 1;
    p.sb = 1;
    int sa = (avail - wtotal) / a_stage;
    p.sa = sa > 8 ? 8 : sa;
    L.smem = 1024 + p.sa * a_stage + ((wtotal + 1023) & ~1023) + bar;
  } else {
    p.wres = 0;
    // two halo stages are enough (one chunk = 72+ MMAs of lookahead); the shared memory goes to the weight ring, whose
    // depth hides the L2 latency of the streamed blobs (measured: 128->128 @64 91 -> 82 us with 2 instead of 3 stages)
    p.sa = 2;
    int sb = (avail - p.sa * a_stage) / b_stage;
    if (sb > 12) sb = 12;
    if (sb < 2) { p.sa = 2; sb = (avail - p.sa * a_stage) / b_stage; }
    p.sb = sb;
    L.smem = 1024 + p.sa * a_stage + p.sb * b_stage + bar;
  }
}

static int pick_bn(int Cout) { return Cout >= 128 ? 128 : Cout; }

// 32-output-channel layers whose input segments are multiples of 32 channels use the kw-stacked kernel when they have
// at least two 32-channel slices (measured: with a single slice the heavier epilogue of the stacked kernel - three
// TMEM reads and two shuffles per value - outweighs the cheaper MMAs; 96->32 gains 20 %).
static bool use_kws(int C0, int C1, int Cout) {
  return Cout == 32 && C0 > 0 && C0 % 32 == 0 && C1 % 32 == 0 && (C0 + C1) >= 64 && (C0 + C1) <= 96;
}

size_t conv_packed_bytes(int Cin, int Cout) { return size_t(Cin) * Cout * 9 * 2; }

static int build_conv(ConvLaunch& L, const __nv_bfloat16* in0, int C0, const __nv_bfloat16* in1, int C1,
                      const uint8_t* wpk, const float* bias, __nv_bfloat16* out, int B, int H, int W, int Cout,
                      int epi) {
  const bool kws = use_kws(C0, C1, Cout);
  const int KC = (!kws && C0 % 64 == 0 && C1 % 64 == 0) ? 64 : 32;
  if (C0 % KC || C1 % KC || C0 <= 0) { set_error("conv: channel counts must be multiples of 32"); return -4; }
  const int BN = pick_bn(Cout);
  if (Cout % BN) { set_error("conv: Cout must be 32, 64 or a multiple of 128"); return -4; }
  if (epi == EPI_FINAL && !(KC == 32 && BN == 32)) { set_error("conv: FINAL epilogue needs Cin=Cout=32"); return -4; }
  L = ConvLaunch{};
  L.KC = KC; L.BN = BN; L.EPI = epi; L.kws = kws ? 1 : 0;
  {
    // CTA-pair kernel (unet_conv_pair.cuh) for the layers whose weights do not stay resident in a single CTA (streamed
    // weights: -4..-12 % per layer, both in burst and in the power-capped sustained run); layers with resident weights
    // gain nothing from halving them.  PNP_CONV_PAIR=0 / 1 forces the single-CTA / pair kernel for every eligible layer.
    static const int pair_env = [] { const char* e = getenv("PNP_CONV_PAIR"); return e ? atoi(e) : -1; }();
    const bool eligible = !kws && epi == EPI_BF16 && (BN == 64 || BN == 128);
    const bool want = pair_env < 0 ? !weights_fit(KC, Cout / BN, (long long)(C0 + C1) * 9 * BN * 2) : pair_env == 1;
    L.pair = (eligible && want) ? 1 : 0;
  }
  ConvParams& p = L.p;
  {
    // Split-K kernel (unet_conv_splitk.cuh) when it puts at least kSkGain times as many CTAs to work as the ordinary
    // kernels would (one image, or a few, at the deep levels) and still runs as ONE wave.  S = the largest power of two
    // <= 8 that divides the 64-channel slices and keeps units * S within the SM count.
    const long long pix_tiles = (long long)B * ((W + kTile - 1) / kTile) * ((H + kTile - 1) / kTile);
    const bool eligible = !kws && epi == EPI_BF16 && KC == 64 && Cout % kSkBN == 0;
    const long long units = pix_tiles * (Cout / kSkBN);
    if (eligible && g_splitk_mode != 0 && (units <= g_num_sms || g_splitk_mode == 1) && units < (1ll << 24)) {
      const int nch = (C0 + C1) / kSkKC;
      int S = 8;
      while (S > 1 && (nch % S != 0 || units * S > g_num_sms)) S >>= 1;
      const long long reg_ctas = std::min<long long>(pix_tiles * (Cout / BN), g_num_sms);
      if (g_splitk_mode == 1 || units * S >= kSkGain * reg_ctas) {
        L.splitk = 1; L.pair = 0;
        p.sk_split = S; p.sk_cpc = nch / S; p.sk_stages = p.sk_cpc < kSkStages ? p.sk_cpc : kSkStages;
      }
    }
  }
  p.B = B; p.H = H; p.W = W;
  p.tiles_x = kws ? (W + kKwsTileW - 1) / kKwsTileW : (W + kTile - 1) / kTile;
  p.tiles_y = kws ? (H + kKwsTileH - 1) / kKwsTileH : (H + kTile - 1) / kTile;
  p.n_tiles = Cout / BN;
  p.nchunks0 = C0 / KC; p.nchunks1 = C1 / KC;
  p.Cout = Cout; p.wpk = wpk; p.bias = bias; p.out = out; p.slope = 0.2f;
  p.mg_n = conv_magic(uint32_t(p.n_tiles)); p.mg_x = conv_magic(uint32_t(p.tiles_x)); p.mg_y = conv_magic(uint32_t(p.tiles_y));
  {
    const long long tiles_all = (long long)B * p.tiles_x * p.tiles_y * p.n_tiles;
    const int dmax = std::max(p.n_tiles, std::max(p.tiles_x, p.tiles_y));
    if (tiles_all * dmax >= (1ll << 32) || Cout > 512) { set_error("conv: problem too large for the tile index arithmetic"); return -4; }
  }
  size_rings(L);
  const int bw = kws ? kKwsHaloW : kHalo, bh = kws ? kKwsHaloH : kHalo;
  int rc = make_act_map(&L.tm0, in0, B, H, W, C0, KC, bw, bh);
  if (rc) return rc;
  rc = C1 > 0 ? make_act_map(&L.tm1, in1, B, H, W, C1, KC, bw, bh) : make_act_map(&L.tm1, in0, B, H, W, C0, KC, bw, bh);
  if (rc) return rc;
  if (L.pair) {
    // rows = all blobs of the layer back to back (blob = BN rows of KC bf16, already swizzled: copied verbatim)
    const cuuint64_t rows = cuuint64_t(p.nchunks0 + p.nchunks1) * 9 * Cout;
    cuuint64_t dims[2] = {cuuint64_t(KC), rows};
    cuuint64_t strides[1] = {cuuint64_t(KC) * 2};
    cuuint32_t box[2] = {cuuint32_t(KC), cuuint32_t(BN / 2)};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = g_encode(&L.tmw, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<uint8_t*>(wpk), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (weights) failed (code " + std::to_string(int(r)) + ")"); return 1000 + int(r); }
  }
  long long tiles = (long long)B * p.tiles_x * p.tiles_y * p.n_tiles;
  if (L.pair) {     // pair tiles: two pixel tiles with the same n-tile; grid = 2 CTAs per pair
    const long long pix = (long long)B * p.tiles_x * p.tiles_y;
    tiles = (pix + 1) / 2 * p.n_tiles;
    p.total_tiles = int(tiles);
    const long long pairs = g_num_sms / 2;
    L.grid = 2 * int(tiles < pairs ? tiles : pairs);
  } else {
  p.total_tiles = int(tiles);
  L.grid = int(tiles < g_num_sms ? tiles : g_num_sms);
  }
  if (L.splitk) {
    L.grid = int((long long)B * p.tiles_x * p.tiles_y * (Cout / kSkBN) * p.sk_split);
    L.smem = sk_smem_bytes(p.sk_stages);
  }
  return 0;
}

// All kernels of the denoiser are launched with programmatic stream serialization (PDL): each one may begin while its
// predecessor drains (see grid_dep_launch / grid_dep_wait in common.cuh).
template <typename... KArgs, typename... Args>
static cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

template <int KC, int BN, int EPI>
static void launch_conv_t(const ConvLaunch& L, cudaStream_t st) {
  launch_k(conv3x3_umma_kernel<KC, BN, EPI>, dim3(L.grid), dim3(kConvThreads), size_t(L.smem), st, L.p, L.tm0, L.tm1);
}

static int launch_conv(const ConvLaunch& L, cudaStream_t st) {
  if (L.splitk) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(L.grid); cfg.blockDim = dim3(kConvThreads); cfg.dynamicSmemBytes = size_t(L.smem); cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = unsigned(L.p.sk_split); attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 2;
    return int(cudaLaunchKernelEx(&cfg, conv3x3_splitk_kernel, L.p, L.tm0, L.tm1));
  }
  if (L.pair) {
    if (L.KC == 32 && L.BN == 64)
      launch_k(conv3x3_pair_kernel<32, 64>, dim3(L.grid), dim3(kConvThreads), size_t(L.smem), st, L.p, L.tm0, L.tm1, L.tmw);
    else if (L.KC == 64 && L.BN == 64)
      launch_k(conv3x3_pair_kernel<64, 64>, dim3(L.grid), dim3(kConvThreads), size_t(L.smem), st, L.p, L.tm0, L.tm1, L.tmw);
    else if (L.KC == 64 && L.BN == 128)
      launch_k(conv3x3_pair_kernel<64, 128>, dim3(L.grid), dim3(kConvThreads), size_t(L.smem), st, L.p, L.tm0, L.tm1, L.tmw);
    else { set_error("conv: unsupported (KC,BN) combination for the pair kernel"); return -4; }
    return int(cudaGetLastError());
  }
  if (L.kws) {
    launch_k(conv3x3_kws_kernel, dim3(L.grid), dim3(kConvThreads), size_t(L.smem), st, L.p, L.tm0, L.tm1);
    return int(cudaGetLastError());
  }
  if (L.EPI == EPI_FINAL) launch_conv_t<32, 32, EPI_FINAL>(L, st);
  else if (L.KC == 32 && L.BN == 32) launch_conv_t<32, 32, EPI_BF16>(L, st);
  else if (L.KC == 32 && L.BN == 64) launch_conv_t<32, 64, EPI_BF16>(L, st);
  else if (L.KC == 64 && L.BN == 64) launch_conv_t<64, 64, EPI_BF16>(L, st);
  else if (L.KC == 64 && L.BN == 128) launch_conv_t<64, 128, EPI_BF16>(L, st);
  else { set_error("conv: unsupported (KC,BN) combination"); return -4; }
  return int(cudaGetLastError());
}

static int ew_grid(size_t total) {
  size_t g = (total + 255) / 256;
  const size_t cap = size_t(g_num_sms) * 16;
  return int(g < cap ? (g ? g : 1) : cap);
}

int pack_conv_weights(const float* w_fp32, uint8_t* out, int Cin, int Cout, int KC, cudaStream_t st, bool kws) {
  if (kws) {
    pack_weights_kws_kernel<<<ew_grid(size_t(Cin) * Cout * 9), 256, 0, st>>>(w_fp32, out, Cin);
    return int(cudaGetLastError());
  }
  const int BN = pick_bn(Cout);
  pack_weights_kernel<<<ew_grid(size_t(Cin) * Cout * 9), 256, 0, st>>>(w_fp32, out, Cin, Cout, KC, BN);
  return int(cudaGetLastError());
}

// Single conv (test / bench entry): packs the weights into `wpk_scratch` and runs one launch.
int conv3x3_single(const __nv_bfloat16* in0, int C0, const __nv_bfloat16* in1, int C1, const float* w_fp32,
                   const float* bias, __nv_bfloat16* out, uint8_t* wpk_scratch, int B, int H, int W, int Cout,
                   cudaStream_t st) {
  ConvLaunch L;
  int rc = build_conv(L, in0, C0, in1, C1, wpk_scratch, bias, out, B, H, W, Cout, EPI_BF16);
  if (rc) return rc;
  rc = pack_conv_weights(w_fp32, wpk_scratch, C0 + C1, Cout, L.KC, st, L.kws != 0);
  if (rc) return rc;
  return launch_conv(L, st);
}

// ------------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------------
static const int kCh[5] = {32, 64, 128, 256, 512};

struct TensorSlot { size_t off; int C, H, W; };

enum { K_FIRST = 0, K_UMMA = 1, K_UPS = 3 };      // values reported by unet_profile (kinds[])

struct Op {
  int kind;
  int id;                   // conv: layer index 0..26; upsample: 200 + level
  int level;                // pyramid level the op writes
  int conv;                 // index into convs (K_UMMA)
  int rev;                  // sweep direction (alternates launch by launch, see ConvParams::rev)
};

struct UnetPlan {
  int B, H, W;
  int Hl[5], Wl[5];
  uint8_t* ws;              // caller-owned workspace
  size_t ws_bytes;
  const uint8_t* wts;       // caller-owned packed weights
  // activation slots (offsets into ws)
  TensorSlot tA[5], tB[5], skip[5], pooled[5], ups[4];
  std::vector<ConvLaunch> convs;   // tensor-core conv launches
  std::vector<Op> ops;             // execution order
  FirstConvW first;                // host copy of the 2->32 conv (passed by value as a kernel parameter)
};

// Flat fp32 parameter vector = the reference state_dict tensors concatenated in registration order
// (inc, down1..4, up1..4: conv-0/1/2 weight,bias; then outc weight,bias) - see oracle.unet_param_shapes().
struct LayerDesc { int cin, cout; size_t w_off, b_off; size_t pk_off; };
static const int kBlockCin[9] = {2, 32, 64, 128, 256, 768, 384, 192, 96};
static const int kBlockCout[9] = {32, 64, 128, 256, 512, 256, 128, 64, 32};

static void layer_table(LayerDesc (&L)[27], size_t& outc_w, size_t& outc_b, size_t& n_params, size_t& pk_bytes) {
  size_t off = 0, pk = 0;
  for (int blk = 0; blk < 9; ++blk)
    for (int i = 0; i < 3; ++i) {
      LayerDesc& d = L[blk * 3 + i];
      d.cin = (i == 0) ? kBlockCin[blk] : kBlockCout[blk];
      d.cout = kBlockCout[blk];
      d.w_off = off; off += size_t(d.cout) * d.cin * 9;
      d.b_off = off; off += d.cout;
      d.pk_off = pk;
      if (blk * 3 + i > 0) pk += (conv_packed_bytes(d.cin, d.cout) + 1023) / 1024 * 1024;
    }
  outc_w = off; off += 32;
  outc_b = off; off += 1;
  n_params = off;
  pk_bytes = pk;
}

// packed weight buffer layout: [bf16 UMMA blobs for layers 1..26][fp32 copy of the whole flat vector]
size_t unet_num_params() {
  LayerDesc L[27]; size_t a, b, n, pk;
  layer_table(L, a, b, n, pk);
  return n;
}
size_t unet_packed_bytes() {
  LayerDesc L[27]; size_t a, b, n, pk;
  layer_table(L, a, b, n, pk);
  return pk + (n * sizeof(float) + 1023) / 1024 * 1024;
}

int unet_pack(const float* flat_fp32, uint8_t* packed, cudaStream_t st) {
  LayerDesc L[27]; size_t ow, ob, n, pk;
  layer_table(L, ow, ob, n, pk);
  for (int i = 1; i < 27; ++i) {
    const int cin = L[i].cin, cout = L[i].cout;
    // segment split of the `up` blocks' first conv: skip channels first (noise.py:59)
    int c0 = cin, c1 = 0;
    if (i >= 15 && i % 3 == 0) { c0 = kBlockCout[i / 3]; c1 = cin - c0; }
    const bool kws = use_kws(c0, c1, cout);
    const int KC = (!kws && c0 % 64 == 0 && c1 % 64 == 0) ? 64 : 32;
    int rc = pack_conv_weights(flat_fp32 + L[i].w_off, packed + L[i].pk_off, cin, cout, KC, st, kws);
    if (rc) return rc;
  }
  return int(cudaMemcpyAsync(packed + pk, flat_fp32, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
}

static size_t plan_layout(UnetPlan* P) {
  size_t off = 0;
  auto take = [&](TensorSlot& s, int C, int H, int W) {
    s.off = off; s.C = C; s.H = H; s.W = W;
    off += (size_t(P->B) * H * W * C * 2 + 1023) / 1024 * 1024;
  };
  for (int l = 0; l < 5; ++l) {
    take(P->tA[l], kCh[l], P->Hl[l], P->Wl[l]);
    take(P->tB[l], kCh[l], P->Hl[l], P->Wl[l]);
    take(P->skip[l], kCh[l], P->Hl[l], P->Wl[l]);
    if (l > 0) take(P->pooled[l], kCh[l - 1], P->Hl[l], P->Wl[l]);
    if (l < 4) take(P->ups[l], kCh[l + 1], P->Hl[l], P->Wl[l]);
  }
  return off;
}

size_t unet_workspace_bytes(int B, int H, int W) {
  UnetPlan P{};
  P.B = B; P.H = H; P.W = W;
  for (int l = 0; l < 5; ++l) { P.Hl[l] = H >> l; P.Wl[l] = W >> l; }
  return plan_layout(&P);
}

// Execution schedule: the first conv, the down blocks, the up blocks, every launch over the whole (micro-)batch.  Running the
// shallow levels in chunks of images for L2 residency was measured on B200 (profiles/r01_*) and lost to the launch count.
int unet_plan_create(UnetPlan** out, const uint8_t* packed, uint8_t* workspace, size_t workspace_bytes, int B, int H,
                     int W) {
  if (B <= 0 || H < 16 || W < 16) { set_error("unet plan: need B>0 and H,W >= 16"); return -1; }
  UnetPlan* P = new UnetPlan();
  P->B = B; P->H = H; P->W = W;
  for (int l = 0; l < 5; ++l) { P->Hl[l] = H >> l; P->Wl[l] = W >> l; }
  const size_t need = plan_layout(P);
  if (workspace_bytes < need) { delete P; set_error("unet plan: workspace too small"); return -5; }
  if ((reinterpret_cast<uintptr_t>(workspace) & 1023) || (reinterpret_cast<uintptr_t>(packed) & 1023)) {
    delete P; set_error("unet plan: workspace / packed weights must be 1024-byte aligned"); return -6;
  }
  P->ws = workspace; P->ws_bytes = workspace_bytes; P->wts = packed;
  LayerDesc L[27]; size_t ow, ob, n, pk;
  layer_table(L, ow, ob, n, pk);
  const float* flat = reinterpret_cast<const float*>(packed + pk);
  auto T = [&](const TensorSlot& s) { return reinterpret_cast<__nv_bfloat16*>(P->ws + s.off); };
  int rc = 0;
  auto conv = [&](int li, const TensorSlot& in0, const TensorSlot* in1, const TensorSlot& o, int lvl,
                  const TensorSlot* pooled = nullptr) {
    if (rc) return;
    ConvLaunch cl;
    const int epi = (li == 26) ? EPI_FINAL : EPI_BF16;
    rc = build_conv(cl, T(in0), in0.C, in1 ? T(*in1) : nullptr, in1 ? in1->C : 0, packed + L[li].pk_off,
                    flat + L[li].b_off, T(o), B, P->Hl[lvl], P->Wl[lvl], L[li].cout, epi);
    if (rc) return;
    if (epi == EPI_FINAL) { cl.p.wout = flat + ow; cl.p.bout = flat + ob; }
    if (pooled) cl.p.pool_out = T(*pooled);
    P->convs.push_back(cl);
    P->ops.push_back(Op{K_UMMA, li, lvl, int(P->convs.size()) - 1});
  };
  {
    // first-layer weights to the host (plan creation may synchronise): fp32 [32][2][3][3] + bias[32]
    float hw[32 * 18 + 32];
    cudaError_t e = cudaMemcpy(hw, flat + L[0].w_off, sizeof(hw), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { delete P; set_error("unet plan: cannot read first-layer weights"); return int(e); }
    for (int co = 0; co < 32; ++co) {
      for (int k = 0; k < 9; ++k) P->first.w[k][co] = hw[co * 18 + k];
      P->first.b[co] = hw[32 * 18 + co];
      for (int cy = 0; cy < 3; ++cy)
        for (int cx = 0; cx < 3; ++cx) {
          float t = 0.f;                              // taps of the sigma channel that fall inside the image
          for (int k = 0; k < 9; ++k) {
            const int dy = k / 3 - 1, dx = k % 3 - 1;
            const bool in_y = !((cy == 0 && dy < 0) || (cy == 2 && dy > 0));
            const bool in_x = !((cx == 0 && dx < 0) || (cx == 2 && dx > 0));
            if (in_y && in_x) t += hw[co * 18 + 9 + k];
          }
          P->first.ws[cy * 3 + cx][co] = t;
        }
    }
  }
  // MaxPool2d(2) is fused into the epilogue of the conv that produces the skip tensor
  P->ops.push_back(Op{K_FIRST, 0, 0, -1});
  conv(1, P->tA[0], nullptr, P->tB[0], 0);
  conv(2, P->tB[0], nullptr, P->skip[0], 0, &P->pooled[1]);
  for (int l = 1; l <= 4; ++l) {
    conv(l * 3 + 0, P->pooled[l], nullptr, P->tA[l], l);
    conv(l * 3 + 1, P->tA[l], nullptr, P->tB[l], l);
    conv(l * 3 + 2, P->tB[l], nullptr, P->skip[l], l, l < 4 ? &P->pooled[l + 1] : nullptr);
  }
  for (int l = 3; l >= 0; --l) {                    // up1 .. up4
    const int blk = 5 + (3 - l);
    P->ops.push_back(Op{K_UPS, 200 + l, l, -1});
    conv(blk * 3 + 0, P->skip[l], &P->ups[l], P->tA[l], l);
    conv(blk * 3 + 1, P->tA[l], nullptr, P->tB[l], l);
    conv(blk * 3 + 2, P->tB[l], nullptr, P->tA[l], l);
  }
  if (rc) { delete P; return rc; }
  {
    // alternate the sweep direction launch by launch: a consumer starts with what its producer wrote last (L2 hits)
    int k = 0;
    for (Op& op : P->ops) {
      op.rev = k & 1;
      if (op.kind == K_UMMA) P->convs[op.conv].p.rev = op.rev;
      ++k;
    }
  }
  *out = P;
  return 0;
}

void unet_plan_destroy(UnetPlan* P) { delete P; }

// named activation lookup for layer-wise parity tests
int unet_plan_tensor(const UnetPlan* P, const char* name, size_t* off, int* C, int* H, int* W) {
  const TensorSlot* s = nullptr;
  const std::string n(name);
  // block outputs as laid out by unet_plan_create()
  if (n == "inc.conv-0") s = &P->tA[0];
  else if (n == "inc.conv-1") s = &P->tB[0];
  else if (n == "inc.conv-2") s = &P->skip[0];
  else {
    for (int l = 1; l <= 4 && !s; ++l) {
      const std::string d = "down" + std::to_string(l);
      if (n == d + ".pooled") s = &P->pooled[l];
      else if (n == d + ".conv-0") s = &P->tA[l];
      else if (n == d + ".conv-1") s = &P->tB[l];
      else if (n == d + ".conv-2") s = &P->skip[l];
    }
    for (int k = 1; k <= 4 && !s; ++k) {
      const int l = 4 - k;
      const std::string u = "up" + std::to_string(k);
      if (n == u + ".upsampled") s = &P->ups[l];
    }
  }
  if (!s) return -1;
  *off = s->off; *C = s->C; *H = s->H; *W = s->W;
  return 0;
}

struct ProfileCtx {
  std::vector<cudaEvent_t> ev;
  cudaStream_t st;
  void begin() {
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    ev.push_back(a); ev.push_back(b);
    cudaEventRecord(a, st);
  }
  void end() { cudaEventRecord(ev.back(), st); }
};

static int unet_forward_impl(UnetPlan* P, const float* v, const float* sigma, float* x_out, float* preclamp,
                             cudaStream_t st, ProfileCtx* prof, const uint8_t* active = nullptr) {
  LayerDesc L[27]; size_t ow, ob, n, pk;
  layer_table(L, ow, ob, n, pk);
  auto T = [&](const TensorSlot& s) { return reinterpret_cast<__nv_bfloat16*>(P->ws + s.off); };
  int rc = 0;
  for (const Op& op : P->ops) {
    if (prof) prof->begin();
    switch (op.kind) {
      case K_FIRST: {
        const int bd = P->W >= 256 ? 256 : ((P->W + 31) / 32) * 32;
        const int gx = (P->W + bd - 1) / bd, pairs = (P->H + 1) / 2;
        int ppt = 4;                                 // long walks only when the grid still fills the machine twice over
        while (ppt > 1 && size_t(gx) * ((pairs + ppt - 1) / ppt) * P->B < 4 * 148) ppt >>= 1;
        launch_k(conv_first_kernel, dim3(gx, (pairs + ppt - 1) / ppt, P->B), dim3(bd), 0, st, v, sigma, P->first,
                 T(P->tA[0]), P->B, P->H, P->W, 0.2f, op.rev, ppt);
        break;
      }
      case K_UMMA: {
        ConvLaunch& cl = P->convs[op.conv];
        if (cl.EPI == EPI_FINAL) { cl.p.noisy = v; cl.p.x_out = x_out; cl.p.preclamp = preclamp; cl.p.active = active; }
        rc = launch_conv(cl, st);
        break;
      }
      case K_UPS: {
        const int l = op.level;
        const TensorSlot& lo = (l == 3) ? P->skip[4] : P->tA[l + 1];   // previous block's output
        const int h = P->Hl[l + 1], w = P->Wl[l + 1], Ho = P->Hl[l], Wo = P->Wl[l];
        const int C8 = kCh[l + 1] / 8;
        const int dy = Ho - 2 * h, dx = Wo - 2 * w;
        const float sy = (2 * h > 1) ? float(h - 1) / float(2 * h - 1) : 0.f;
        const float sx = (2 * w > 1) ? float(w - 1) / float(2 * w - 1) : 0.f;
        if (dy == 0 && dx == 0 && h > 1 && w > 1)
        {
          const int gx = ((w + 1) * C8 + 255) / 256;
          int walk = 8;                              // long walks only while the grid still fills the machine
          while (walk > 1 && size_t(gx) * ((h + walk) / walk) * P->B < 4 * size_t(g_num_sms)) walk >>= 1;
          launch_k(upsample2x_fast_kernel, dim3(gx, (h + walk) / walk, P->B), dim3(256), 0, st,
                   reinterpret_cast<const uint4*>(T(lo)), reinterpret_cast<uint4*>(T(P->ups[l])), h, w,
                   C8, sy, sx, P->B, op.rev, (C8 == 64 ? 6 : (C8 == 32 ? 5 : (C8 == 16 ? 4 : 3))), walk);   // kCh / 8 = 8 .. 64
        }
        else
          launch_k(upsample2x_kernel, dim3((Wo * C8 + 255) / 256, (Ho + kUpsRows - 1) / kUpsRows, P->B), dim3(256), 0,
                   st, reinterpret_cast<const uint4*>(T(lo)), reinterpret_cast<uint4*>(T(P->ups[l])),
                   P->B, h, w, Ho, Wo, C8, dy / 2, dx / 2, sy, sx);
        break;
      }
    }
    if (prof) prof->end();
    if (rc) return rc;
  }
  return int(cudaGetLastError());
}

int unet_forward(UnetPlan* P, const float* v, const float* sigma, float* x_out, float* preclamp, cudaStream_t st,
                 const uint8_t* active) {
  return unet_forward_impl(P, v, sigma, x_out, preclamp, st, nullptr, active);
}

int unet_num_launches(const UnetPlan* P) { return int(P->ops.size()); }

// Profiling pass: one forward with a CUDA-event pair around every launch; SYNCHRONISES the stream.
// ms[i] = duration of launch i; kinds[i] in {0 first conv, 1 tcgen05 conv, 3 upsample};
// ids[i] = layer index 0..26 (convs), 200+level (upsamples).
int unet_profile(UnetPlan* P, const float* v, const float* sigma, float* x_out, cudaStream_t st, float* ms,
                 int* kinds, int* ids, int* n_inout) {
  ProfileCtx prof;
  prof.st = st;
  int rc = unet_forward_impl(P, v, sigma, x_out, nullptr, st, &prof);
  cudaError_t e = cudaStreamSynchronize(st);
  const int n = int(prof.ev.size() / 2);
  const int cap = *n_inout;
  for (int i = 0; i < n && i < cap; ++i) {
    float t = 0.f;
    cudaEventElapsedTime(&t, prof.ev[2 * i], prof.ev[2 * i + 1]);
    ms[i] = t; kinds[i] = P->ops[i].kind; ids[i] = P->ops[i].id;
  }
  for (cudaEvent_t evt : prof.ev) cudaEventDestroy(evt);
  *n_inout = n < cap ? n : cap;
  if (rc) return rc;
  return int(e);
}

}  // namespace pnp
