// SSIM metric (Wang et al. 2004, the form of pytorch-msssim / BasicSR), per image b:
//   X = clamp(x[b], 0, 1), Y = gt[b];  g = normalised 11-tap Gaussian, sigma 1.5, applied separably with VALID filtering;
//   mu_x = g*X, mu_y = g*Y, s_xx = g*(X.X) - mu_x^2, s_yy = g*(Y.Y) - mu_y^2, s_xy = g*(X.Y) - mu_x.mu_y;
//   map = ((2 mu_x mu_y + C1)(2 s_xy + C2)) / ((mu_x^2 + mu_y^2 + C1)(s_xx + s_yy + C2)),  C1 = 0.01^2, C2 = 0.03^2;
//   ssim[b] = mean of the (H-10) x (W-10) map.
//
// ssim_tile_kernel: one CTA per 64 x 28 block of the map of one image (grid = B x tiles, so any batch covers the chip).
//   1. stage the 74 x 38 input halo of X and Y in shared memory (float4 loads where the row is 16-byte aligned), shifted
//      by the tile's first pixel so that the moments do not cancel on flat regions;
//   2. horizontal 11-tap pass: a thread takes 8 output columns of one halo row, forms X.X, Y.Y, X.Y once per input pixel
//      in registers and filters the five quantities with packed FFMA2 (two output columns per instruction);
//   3. vertical 11-tap pass: warp q filters quantity q, each lane walks down two adjacent output columns with the rows in
//      registers, so every horizontally filtered value leaves shared memory once (an 11-tap read per output would move
//      ~220 B of shared memory per pixel and make the pass shared-memory bound), and writes the result in place;
//   4. the SSIM formula per output pixel, a fixed-order reduction, one fp32 partial sum per tile into the workspace.
// ssim_finalize_kernel (chained with programmatic dependent launch) sums each image's partials in an order fixed by the
// tile count and divides by (H-10)(W-10).  Tiling and summation order depend on (H, W) only: the value of an image is
// bitwise the same on every call and at any position of any batch.  No float atomics, no host synchronisation.
#include "common.cuh"
#include "pnp_internal.h"

namespace pnp {

constexpr int kTW = 64;                    // output columns per tile: 32 lanes x 2
constexpr int kTH = 28;                    // output rows per tile (3 CTAs of 160 threads fit an SM's shared memory)
constexpr int kHR = kTH + 10;              // halo rows
constexpr int kInStride = 76;              // 74 halo columns; a stride of 4 (mod 8) floats keeps the strip loads conflict-free
constexpr int kQuads = kInStride / 4;
constexpr int kThreads = 160;              // 5 warps: one per filtered quantity in the vertical pass
constexpr int kHItems = kHR * (kTW / 8);   // horizontal work items: halo row x strip of 8 output columns
constexpr size_t kSmemBytes = size_t(2 * kHR * kInStride + 5 * kHR * kTW) * sizeof(float);
constexpr float kC1 = 0.01f * 0.01f, kC2 = 0.03f * 0.03f;

// exp(-(k-5)^2 / (2 * 1.5^2)) / sum, rounded to fp32
__device__ constexpr float kG[11] = {1.028380124e-03f, 7.598758209e-03f, 3.600077331e-02f, 1.093606874e-01f,
                                     2.130055428e-01f, 2.660117149e-01f, 2.130055428e-01f, 1.093606874e-01f,
                                     3.600077331e-02f, 7.598758209e-03f, 1.028380124e-03f};

static __device__ __forceinline__ float2 gk2(int k) { return make_float2(kG[k], kG[k]); }

__global__ void __launch_bounds__(kThreads, 3)
ssim_tile_kernel(const float* __restrict__ x, const float* __restrict__ gt, long long gt_bstride,
                 float* __restrict__ partial, int H, int W, int tiles_x, int ntiles) {
  grid_dep_launch();
  extern __shared__ float4 smem4[];
  float* sx = reinterpret_cast<float*>(smem4);          // [kHR][kInStride]  X - kx
  float* sy = sx + kHR * kInStride;                     // [kHR][kInStride]  Y - ky
  float* hf = sy + kHR * kInStride;                     // [5][kHR][kTW]     filtered X', Y', X'X', Y'Y', X'Y'
  const int b = blockIdx.x / ntiles, tile = blockIdx.x - b * ntiles;
  const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
  const int r0 = ty * kTH, c0 = tx * kTW;
  const float* xb = x + size_t(b) * H * W;
  const float* gb = gt + size_t(b) * gt_bstride;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // The moments are taken about the tile's first pixel (kx, ky): the variances and the covariance do not change, but
  // E[X'X'] - E[X']^2 no longer cancels on flat regions (a constant image gives exactly 0 instead of rounding noise that
  // C2 = 9e-4 would amplify).
  const float kx = fminf(fmaxf(__ldg(xb + size_t(r0) * W + c0), 0.f), 1.f), ky = __ldg(gb + size_t(r0) * W + c0);

  // 1. halo of X' = X - kx and Y' = Y - ky; positions outside the image only feed outputs that are masked out below
#pragma unroll
  for (int k = 0; k < (kHR * kQuads + kThreads - 1) / kThreads; ++k) {
    const int it = threadIdx.x + k * kThreads;
    if (it < kHR * kQuads) {
      const int r = it / kQuads, q = it - r * kQuads;
      const int gr = r0 + r, gc = c0 + 4 * q;
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f), g = a;
      if (gr < H) {
        const float* xr = xb + size_t(gr) * W + gc;
        const float* yr = gb + size_t(gr) * W + gc;
        if (gc + 3 < W && ((reinterpret_cast<uintptr_t>(xr) | reinterpret_cast<uintptr_t>(yr)) & 15) == 0) {
          a = __ldg(reinterpret_cast<const float4*>(xr));
          g = __ldg(reinterpret_cast<const float4*>(yr));
        } else {
          if (gc + 0 < W) { a.x = __ldg(xr + 0); g.x = __ldg(yr + 0); }
          if (gc + 1 < W) { a.y = __ldg(xr + 1); g.y = __ldg(yr + 1); }
          if (gc + 2 < W) { a.z = __ldg(xr + 2); g.z = __ldg(yr + 2); }
          if (gc + 3 < W) { a.w = __ldg(xr + 3); g.w = __ldg(yr + 3); }
        }
      }
      a.x = fminf(fmaxf(a.x, 0.f), 1.f) - kx;
      a.y = fminf(fmaxf(a.y, 0.f), 1.f) - kx;
      a.z = fminf(fmaxf(a.z, 0.f), 1.f) - kx;
      a.w = fminf(fmaxf(a.w, 0.f), 1.f) - kx;
      g.x -= ky; g.y -= ky; g.z -= ky; g.w -= ky;
      reinterpret_cast<float4*>(sx + r * kInStride)[q] = a;
      reinterpret_cast<float4*>(sy + r * kInStride)[q] = g;
    }
  }
  __syncthreads();

  // 2. horizontal pass.  Lane bits: [1:0] strip & 3, [3:2] row & 3, [4] strip >> 2; each quarter warp then reads
  //    4 strips x 2 rows, which with kInStride = 4 (mod 8) covers the 32 banks once per LDS.128.
#pragma unroll 1
  for (int k = 0; k < (kHItems + kThreads - 1) / kThreads; ++k) {
    const int t = threadIdx.x + k * kThreads;
    const int s = (t & 3) | ((t >> 2) & 4);
    const int r = ((t >> 2) & 3) | ((t >> 5) << 2);
    if (r >= kHR) continue;
    float xs[18], ys[18];
    {
      const float4* px = reinterpret_cast<const float4*>(sx + r * kInStride + 8 * s);
      const float4* py = reinterpret_cast<const float4*>(sy + r * kInStride + 8 * s);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 a = px[j], c = py[j];
        xs[4 * j] = a.x; xs[4 * j + 1] = a.y; xs[4 * j + 2] = a.z; xs[4 * j + 3] = a.w;
        ys[4 * j] = c.x; ys[4 * j + 1] = c.y; ys[4 * j + 2] = c.z; ys[4 * j + 3] = c.w;
      }
      const float2 a = reinterpret_cast<const float2*>(px + 4)[0], c = reinterpret_cast<const float2*>(py + 4)[0];
      xs[16] = a.x; xs[17] = a.y;
      ys[16] = c.x; ys[17] = c.y;
    }
    float xx[18], yy[18], xy[18];                       // products, once per input pixel
#pragma unroll
    for (int m = 0; m < 9; ++m) {
      const float2 xv = make_float2(xs[2 * m], xs[2 * m + 1]), yv = make_float2(ys[2 * m], ys[2 * m + 1]);
      const float2 pxx = __fmul2_rn(xv, xv), pyy = __fmul2_rn(yv, yv), pxy = __fmul2_rn(xv, yv);
      xx[2 * m] = pxx.x; xx[2 * m + 1] = pxx.y;
      yy[2 * m] = pyy.x; yy[2 * m + 1] = pyy.y;
      xy[2 * m] = pxy.x; xy[2 * m + 1] = pxy.y;
    }
    float2 acc[5][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 g0 = gk2(0);
      acc[0][j] = __fmul2_rn(g0, make_float2(xs[2 * j], xs[2 * j + 1]));
      acc[1][j] = __fmul2_rn(g0, make_float2(ys[2 * j], ys[2 * j + 1]));
      acc[2][j] = __fmul2_rn(g0, make_float2(xx[2 * j], xx[2 * j + 1]));
      acc[3][j] = __fmul2_rn(g0, make_float2(yy[2 * j], yy[2 * j + 1]));
      acc[4][j] = __fmul2_rn(g0, make_float2(xy[2 * j], xy[2 * j + 1]));
    }
#pragma unroll
    for (int tap = 1; tap < 11; ++tap) {
      const float2 gt2 = gk2(tap);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int i = 2 * j + tap;
        acc[0][j] = __ffma2_rn(gt2, make_float2(xs[i], xs[i + 1]), acc[0][j]);
        acc[1][j] = __ffma2_rn(gt2, make_float2(ys[i], ys[i + 1]), acc[1][j]);
        acc[2][j] = __ffma2_rn(gt2, make_float2(xx[i], xx[i + 1]), acc[2][j]);
        acc[3][j] = __ffma2_rn(gt2, make_float2(yy[i], yy[i + 1]), acc[3][j]);
        acc[4][j] = __ffma2_rn(gt2, make_float2(xy[i], xy[i + 1]), acc[4][j]);
      }
    }
#pragma unroll
    for (int q = 0; q < 5; ++q) {
      float4* ph = reinterpret_cast<float4*>(hf + (q * kHR + r) * kTW + 8 * s);
      ph[0] = make_float4(acc[q][0].x, acc[q][0].y, acc[q][1].x, acc[q][1].y);
      ph[1] = make_float4(acc[q][2].x, acc[q][2].y, acc[q][3].x, acc[q][3].y);
    }
  }
  __syncthreads();

  // 3. vertical pass, in place: warp q, columns (2 lane, 2 lane + 1); row i of the result overwrites halo row i, which
  //    this lane has already read (rows i + 1 .. i + 10 are still in registers)
  {
    float2* col = reinterpret_cast<float2*>(hf + warp * kHR * kTW) + lane;
    constexpr int kRow = kTW / 2;                       // float2 per row
    float2 w[kHR];
#pragma unroll
    for (int r = 0; r < 10; ++r) w[r] = col[r * kRow];
#pragma unroll
    for (int i = 0; i < kTH; ++i) {
      w[i + 10] = col[(i + 10) * kRow];
      float2 a = __fmul2_rn(gk2(0), w[i]);
#pragma unroll
      for (int tap = 1; tap < 11; ++tap) a = __ffma2_rn(gk2(tap), w[i + tap], a);
      col[i * kRow] = a;
    }
  }
  __syncthreads();

  // 4. SSIM map over the valid outputs of the tile, summed in a fixed order
  float sum = 0.f;
  const int vc = (W - 10) - c0 - 2 * lane;              // valid columns of this lane's pair: >= 2 both, 1 the first
  const int vr = min(kTH, (H - 10) - r0);
  if (vc > 0) {
    const float2* f = reinterpret_cast<const float2*>(hf) + lane;
    constexpr int kQ = kHR * kTW / 2;                   // float2 per quantity plane
    const float2 two2 = make_float2(2.f, 2.f), kx2 = make_float2(kx, kx), ky2 = make_float2(ky, ky);
    const float2 c1 = make_float2(kC1, kC1), c2 = make_float2(kC2, kC2);
    for (int i = warp; i < vr; i += kThreads / 32) {
      const int o = i * (kTW / 2);
      const float2 dx = f[o], dy = f[kQ + o], exx = f[2 * kQ + o], eyy = f[3 * kQ + o], exy = f[4 * kQ + o];
      const float2 sxx = __ffma2_rn(dx, make_float2(-dx.x, -dx.y), exx);
      const float2 syy = __ffma2_rn(dy, make_float2(-dy.x, -dy.y), eyy);
      const float2 sxy = __ffma2_rn(dx, make_float2(-dy.x, -dy.y), exy);
      const float2 mx = __fadd2_rn(dx, kx2), my = __fadd2_rn(dy, ky2);
      const float2 mxx = __fmul2_rn(mx, mx), myy = __fmul2_rn(my, my), mxy = __fmul2_rn(mx, my);
      const float2 num = __fmul2_rn(__ffma2_rn(two2, mxy, c1), __ffma2_rn(two2, sxy, c2));
      const float2 den = __fmul2_rn(__fadd2_rn(__fadd2_rn(mxx, myy), c1), __fadd2_rn(__fadd2_rn(sxx, syy), c2));
      sum += num.x / den.x;
      if (vc > 1) sum += num.y / den.y;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  __shared__ float wsum[kThreads / 32];
  if (lane == 0) wsum[warp] = sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = wsum[0];
#pragma unroll
    for (int q = 1; q < kThreads / 32; ++q) s += wsum[q];
    partial[blockIdx.x] = s;
  }
}

// One warp per image: lane l sums partials l, l + 32, ... in order, then a fixed shuffle tree.
__global__ void __launch_bounds__(256) ssim_finalize_kernel(const float* __restrict__ partial, float* __restrict__ out,
                                                            int B, int ntiles, float count) {
  grid_dep_wait();
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  const float* p = partial + size_t(b) * ntiles;
  float s = 0.f;
  int t = lane;
  for (; t + 96 < ntiles; t += 128) {
    const float a0 = p[t], a1 = p[t + 32], a2 = p[t + 64], a3 = p[t + 96];
    s = (((s + a0) + a1) + a2) + a3;
  }
  for (; t < ntiles; t += 32) s += p[t];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[b] = s / count;
}

static void ssim_tiles(int H, int W, int* tiles_x, int* ntiles) {
  *tiles_x = (W - 10 + kTW - 1) / kTW;
  *ntiles = *tiles_x * ((H - 10 + kTH - 1) / kTH);
}

size_t ssim_workspace_bytes(int B, int H, int W) {
  if (B <= 0 || H < 11 || W < 11) return 0;
  int tx, nt;
  ssim_tiles(H, W, &tx, &nt);
  return (size_t(B) * nt * sizeof(float) + 15) & ~size_t(15);
}

int ssim_launch(const float* x, const float* gt, long long gt_bstride, float* out, void* workspace, int B, int H, int W,
                cudaStream_t st) {
  if (B <= 0 || H < 11 || W < 11) return -1;
  static const cudaError_t attr_rc =
      cudaFuncSetAttribute(ssim_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kSmemBytes));
  if (attr_rc != cudaSuccess) return int(attr_rc);
  int tiles_x, ntiles;
  ssim_tiles(H, W, &tiles_x, &ntiles);
  const long long grid = (long long)B * ntiles;
  if (grid > 0x7fffffffLL) return -2;
  float* partial = static_cast<float*>(workspace);
  ssim_tile_kernel<<<unsigned(grid), kThreads, kSmemBytes, st>>>(x, gt, gt_bstride, partial, H, W, tiles_x, ntiles);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return int(e);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(unsigned((B + 7) / 8));
  cfg.blockDim = dim3(256);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return int(cudaLaunchKernelEx(&cfg, ssim_finalize_kernel, static_cast<const float*>(partial), out, B, ntiles,
                                float((long long)(H - 10) * (W - 10))));
}

}  // namespace pnp
