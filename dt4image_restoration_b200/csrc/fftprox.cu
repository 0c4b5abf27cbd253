// Data-fidelity proximal step of PnP-ADMM for CS-MRI + dual update (reference evaluation/env.py:87-93):
//
//     z  = ifft( blend( fft(x + u) ) ),   blend(Z)[m] = (mu*Z[m] + y0[m]) / (1 + mu) under the mask, Z elsewhere
//     u' = u + x - z
//     v' = Re(z - u')                       (next denoiser input, env.py:85-86)
//
// `fft`/`ifft` are the reference's centred orthonormal transforms (evaluation/utils/transformations.py:6-19).
// For even H, W:  fft(w) = s * D . FFT2(D . w) / sqrt(HW)  with D[i,j] = (-1)^(i+j), s = (-1)^((H+W)/2), and the
// same for ifft, so the three shift passes of each transform collapse into sign flips on load/store and the
// only place s*D survives is as a factor on y0 inside the blend (see DESIGN.md).  The inverse transform is
// computed as conj(FFT(conj(.))) so a single forward FFT core serves both directions.
//
// Sizes that are not powers of two in 32..512 take the dense-DFT path of fftprox_any.cuh (any H, W in 2..1024).
// This file is the general (any power-of-two H, W in 32..512) three-launch path:
//   rows  : load D.(x+u)            -> row FFTs                      -> T (c64 workspace)
//   cols  : load 8..64 columns of T -> col FFT -> blend -> col FFT   -> T (in place)
//   rows  : load T                  -> row FFTs -> z, u', v'          (epilogue)
// T stays L2 resident for moderate batches.  256x256 and 128x128 have single-launch cluster kernels (fftprox_cl.cuh,
// fftprox_cl128.cuh) and all shapes a row-only kernel for column-only masks (fftprox_sep.cuh); the C-ABI selects.
#include "common.cuh"
#include "fft_core.cuh"
#include "pnp_internal.h"

namespace pnp {

__device__ float2 g_tw512[512];   // exp(-2*pi*i*k/512), filled by init_fft_tables()

void init_fft_tables() {
  static float2 h[512];
  for (int k = 0; k < 512; ++k) {
    const double a = -2.0 * 3.14159265358979323846 * double(k) / 512.0;
    h[k] = make_float2(float(cos(a)), float(sin(a)));
  }
  cudaMemcpyToSymbol(g_tw512, h, sizeof(h));
}

}  // namespace pnp
#include "fftprox_sep.cuh"
#include "fftprox_cl.cuh"
#include "fftprox_cl128.cuh"
#include "fftprox_any.cuh"
#include "measure.cuh"
namespace pnp {

enum { ROWS_LOAD_XU = 0, ROWS_LOAD_C = 1 };
enum { ROWS_STORE_C = 0, ROWS_STORE_PROX = 1 };

struct RowsParams {
  int H, W;
  int load_mode, store_mode;
  int load_sign;            // multiply loaded value by D[i,j]
  int load_conj;
  const float* x;           // [B,H,W]      (LOAD_XU, STORE_PROX)
  const float2* u;          // [B,H,W]
  const float2* src;        // [B,H,W]      (LOAD_C)
  float2* dst;              // [B,H,W]      (STORE_C)
  int store_sign, store_conj;
  float store_scale;
  float2* z_out;            // STORE_PROX
  float2* u_out;
  float* v_out;             // may be null
  const int* skip_flag;     // optional: != 0 -> the row-only kernel handles this batch, do nothing
  const uint8_t* active;    // optional [B], STORE_PROX only: 0 = leave the image's z, u, v untouched
};

template <int N>
__global__ void __launch_bounds__(256) fft_rows_kernel(const RowsParams p) {
  constexpr int G = FftPlan<N>::G;
  constexpr int P = fft_pitch(N);
  if (p.skip_flag && *p.skip_flag != 0) return;
  __shared__ float2 tw[kTwTotal];
  extern __shared__ float2 rows_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  fft_load_twiddles(tw, g_tw512);
  __syncthreads();
  const int b = blockIdx.y;
  const int row0 = (blockIdx.x * 8 + warp) * G;
  if (row0 >= p.H) return;
  float2* mine = rows_smem + warp * G * P;
  const size_t img = size_t(b) * p.H * p.W;
#pragma unroll 1
  for (int g = 0; g < G; ++g) {
    const int i = row0 + g;
    const size_t base = img + size_t(i) * N;
    for (int j = lane; j < N; j += 32) {
      float2 v;
      if (p.load_mode == ROWS_LOAD_XU) {
        const float2 uu = p.u[base + j];
        v = make_float2(p.x[base + j] + uu.x, uu.y);
      } else {
        v = p.src[base + j];
      }
      if (p.load_conj) v.y = -v.y;
      if (p.load_sign && ((i + j) & 1)) { v.x = -v.x; v.y = -v.y; }
      mine[g * P + fpad(j)] = v;
    }
  }
  __syncwarp();
  fft_warp_rows<N>(mine, P, tw, lane);
#pragma unroll 1
  for (int g = 0; g < G; ++g) {
    const int i = row0 + g;
    const size_t base = img + size_t(i) * N;
    // the epilogue's u, x loads are plain (u_out may alias u) and stay behind the preceding stores, so the loads of KB
    // elements are issued ahead of their stores by hand (load -> store -> load chains cost 25 % in the row-only kernels)
    constexpr int KB = (N / 32 < 4) ? N / 32 : 4;
    const bool prox_store = p.store_mode != ROWS_STORE_C;
    if (prox_store && p.active && p.active[b] == 0) continue;
    for (int j0 = lane; j0 < N; j0 += 32 * KB) {
      float2 uu[KB];
      float xx[KB];
      if (prox_store) {
#pragma unroll
        for (int q = 0; q < KB; ++q) {
          uu[q] = p.u[base + j0 + 32 * q];
          xx[q] = p.x[base + j0 + 32 * q];
        }
      }
#pragma unroll
      for (int q = 0; q < KB; ++q) {
        const int j = j0 + 32 * q;
        float2 v = mine[g * P + fpad(j)];
        v.x *= p.store_scale; v.y *= p.store_scale;
        if (p.store_conj) v.y = -v.y;
        if (p.store_sign && ((i + j) & 1)) { v.x = -v.x; v.y = -v.y; }
        if (!prox_store) {
          p.dst[base + j] = v;
        } else {
          const float2 un = make_float2(uu[q].x + xx[q] - v.x, uu[q].y - v.y);   // u' = u + x - z
          p.z_out[base + j] = v;
          p.u_out[base + j] = un;
          if (p.v_out) p.v_out[base + j] = v.x - un.x;                            // Re(z - u')
        }
      }
    }
  }
}

struct ColsParams {
  int H, W;
  float2* t;                // [B,H,W] in/out (or src -> dst)
  const float2* src;
  int blend;                // 1: blend with y0 then second FFT of the conjugate
  const float2* y0;         // [B,H,W]
  const uint8_t* mask;      // [mask_B,H,W]
  long long mask_bstride;   // 0 when one mask is shared by the batch
  const float* mu;          // [B] or [1]
  int mu_stride;
  float scale1;             // applied to the first FFT's output (1/sqrt(HW))
  float sgn;                // s = (-1)^((H+W)/2)
  int store_sign, store_conj;
  float store_scale;
  int load_sign, load_conj, load_neg;   // loaded value: conj if load_conj, times D[i,j] if load_sign, times -1 if load_neg
  const int* skip_flag;     // optional: != 0 -> do nothing (see RowsParams)
  const int* skip_unless_flag;   // optional: == 0 -> do nothing
};

// N = H (transform length), CTA owns NCOL = 8*G adjacent columns of one image.
template <int N>
__global__ void __launch_bounds__(256) fft_cols_kernel(const ColsParams p) {
  constexpr int G = FftPlan<N>::G;
  constexpr int NCOL = 8 * G;
  constexpr int P = fft_pitch(N) + ((fft_pitch(N) % 16 == 0) ? 4 : 0);   // de-conflict the transposed fill
  if (p.skip_flag && *p.skip_flag != 0) return;
  if (p.skip_unless_flag && *p.skip_unless_flag == 0) return;
  __shared__ float2 tw[kTwTotal];
  extern __shared__ float2 cols_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  fft_load_twiddles(tw, g_tw512);
  const int b = blockIdx.y;
  const int c0 = blockIdx.x * NCOL;
  const size_t img = size_t(b) * p.H * p.W;
  // load: consecutive threads walk the NCOL contiguous columns of a row
  for (int e = threadIdx.x; e < N * NCOL; e += blockDim.x) {
    const int c = e % NCOL, i = e / NCOL;
    float2 v = (c0 + c < p.W) ? p.src[img + size_t(i) * p.W + c0 + c] : make_float2(0.f, 0.f);
    if (p.load_conj) v.y = -v.y;
    if ((p.load_sign && ((i + c0 + c) & 1)) != (p.load_neg != 0)) { v.x = -v.x; v.y = -v.y; }
    cols_smem[c * P + fpad(i)] = v;
  }
  __syncthreads();
  float2* mine = cols_smem + warp * G * P;
  fft_warp_rows<N>(mine, P, tw, lane);
  if (p.blend) {
    __syncthreads();
    const float mu = p.mu[size_t(b) * p.mu_stride];
    const float inv1mu = 1.f / (1.f + mu);
    const uint8_t* mk = p.mask + size_t(b) * p.mask_bstride;
    for (int e = threadIdx.x; e < N * NCOL; e += blockDim.x) {
      const int c = e % NCOL, i = e / NCOL;
      if (c0 + c >= p.W) continue;
      const size_t g = size_t(i) * p.W + c0 + c;
      float2 Z = cols_smem[c * P + fpad(i)];
      Z.x *= p.scale1; Z.y *= p.scale1;
      if (mk[g]) {
        float2 y = p.y0[img + g];
        const float sg = ((i + c0 + c) & 1) ? -p.sgn : p.sgn;
        Z.x = (mu * Z.x + sg * y.x) * inv1mu;
        Z.y = (mu * Z.y + sg * y.y) * inv1mu;
      }
      cols_smem[c * P + fpad(i)] = make_float2(Z.x, -Z.y);   // conj -> forward FFT == inverse
    }
    __syncthreads();
    fft_warp_rows<N>(mine, P, tw, lane);
  }
  __syncthreads();
  for (int e = threadIdx.x; e < N * NCOL; e += blockDim.x) {
    const int c = e % NCOL, i = e / NCOL;
    if (c0 + c >= p.W) continue;
    float2 v = cols_smem[c * P + fpad(i)];
    v.x *= p.store_scale; v.y *= p.store_scale;
    if (p.store_conj) v.y = -v.y;
    if (p.store_sign && ((i + c0 + c) & 1)) { v.x = -v.x; v.y = -v.y; }
    p.t[img + size_t(i) * p.W + c0 + c] = v;
  }
}

template <int N> static void launch_rows(const RowsParams& p, int B, cudaStream_t st) {
  constexpr int G = FftPlan<N>::G;
  const size_t smem = size_t(8) * G * fft_pitch(N) * sizeof(float2);
  dim3 grid((p.H + 8 * G - 1) / (8 * G), B);
  fft_rows_kernel<N><<<grid, 256, smem, st>>>(p);
}
template <int N> static void launch_cols(const ColsParams& p, int B, cudaStream_t st) {
  constexpr int G = FftPlan<N>::G;
  constexpr int P = fft_pitch(N) + ((fft_pitch(N) % 16 == 0) ? 4 : 0);
  const size_t smem = size_t(8) * G * P * sizeof(float2);
  dim3 grid((p.W + 8 * G - 1) / (8 * G), B);
  fft_cols_kernel<N><<<grid, 256, smem, st>>>(p);
}

static int launch_cl(const ClParams& p, cudaStream_t st) { return launch_cl_t<16>(p, st); }

static int prox_prepare_cl(const float2* y0, const uint8_t* mask, long long mask_bstride, float2* y0R, uint16_t* mpack,
                           int B, cudaStream_t st, const int* skip_flag = nullptr) {
  prox_prepare_cl_kernel<<<dim3(kClN, B), 256, 0, st>>>(y0, mask, mask_bstride, y0R, mpack, mask_bstride ? B : 1, skip_flag);
  return int(cudaGetLastError());
}

static int prox_prepare_cl128(const float2* y0, const uint8_t* mask, long long mask_bstride, float2* y0R, uint16_t* mpack,
                              int B, cudaStream_t st, const int* skip_flag = nullptr) {
  prox_prepare_cl128_kernel<<<dim3(kC128N, B), kC128N, 0, st>>>(y0, mask, mask_bstride, y0R, mpack, mask_bstride ? B : 1,
                                                                 skip_flag);
  return int(cudaGetLastError());
}

static bool pow2_ok(int n) { return n == 32 || n == 64 || n == 128 || n == 256 || n == 512; }

#define DISPATCH_N(n, fn, ...)                         \
  switch (n) {                                         \
    case 32: fn<32>(__VA_ARGS__); break;               \
    case 64: fn<64>(__VA_ARGS__); break;               \
    case 128: fn<128>(__VA_ARGS__); break;             \
    case 256: fn<256>(__VA_ARGS__); break;             \
    default: fn<512>(__VA_ARGS__); break;              \
  }

int fft_shape_supported(int H, int W) { return pow2_ok(H) && pow2_ok(W); }
// every shape some kernel serves: the radix kernels above or the dense-DFT path (fftprox_any.cuh, 2..1024)
int fft_any_shape_supported(int H, int W) { return fft_shape_supported(H, W) || any_shape_supported(H, W); }

// Layout of the prepared buffers (pnp_prox_prepared_bytes), nb = B (per-image masks) or 1:
//   256x256 : y0p = [y0R: B*HW c64][Yt: B*HW c64]                      maskp = [packed rotated mask ..nb*HW][pad16][row mask][flag]
//   128x128 : y0p = [y0R][Yt][unused]                                  maskp = as 256x256
//   other   : y0p = [y0 copy: B*HW][Yt: B*HW][scratch: B*HW]           maskp = [mask copy: nb*HW][pad16][row mask][flag]
// (y0R / packed rotated mask: trajectory constants of the cluster kernels, fftprox_cl.cuh "Algebra")
// row mask = nb * sep_rowmask_stride(H, W) bytes (16 packed uint16 for 256x256, W plain bytes otherwise), flag = int32.
static size_t maskp_pack_off(int nb, int H, int W) { return (size_t(nb) * H * W + 15) / 16 * 16; }
static size_t maskp_flag_off(int nb, int H, int W) {
  return (maskp_pack_off(nb, H, W) + size_t(nb) * sep_rowmask_stride(H, W) + 15) / 16 * 16;
}
void prox_prepared_bytes(int B, int H, int W, size_t* y0p_bytes, size_t* maskp_bytes) {
  *y0p_bytes = size_t((H == 256 && W == 256) ? 2 : 3) * B * H * W * sizeof(float2);
  *maskp_bytes = maskp_flag_off(B, H, W) + 16;
}

static int prox_dual_general_impl(const float* x, const float2* u_in, const float2* y0, const uint8_t* mask,
                                  long long mask_bstride, const float* mu, int mu_stride, float2* z_out, float2* u_out,
                                  float* v_out, float2* work, int B, int H, int W, const int* skip_flag, cudaStream_t st,
                                  const uint8_t* active = nullptr);

// Full preparation: copies for the general kernels, the column-only-mask test (device flag), the row mask and
// Yt = Fc^-1 (s*D.y0) for the row-only kernels (fftprox_sep.cuh).  Once per trajectory.
int prox_prepare(const float2* y0, const uint8_t* mask, long long mask_bstride, float2* y0p, uint8_t* maskp, int B, int H,
                 int W, cudaStream_t st) {
  if (!fft_shape_supported(H, W)) return -2;
  const bool is256 = (H == 256 && W == 256);
  const int nb = mask_bstride ? B : 1;
  const size_t n = size_t(B) * H * W;
  uint16_t* mpack = reinterpret_cast<uint16_t*>(maskp + maskp_pack_off(nb, H, W));
  int* flag = reinterpret_cast<int*>(maskp + maskp_flag_off(nb, H, W));
  cudaMemsetAsync(flag, 1, sizeof(int), st);                        // bytes 01 01 01 01: non-zero = "column-only so far"
  sep_check_kernel<<<dim3(nb, kSepCheckSlices), 256, 0, st>>>(mask, mask_bstride, H, W, mpack, flag);
  // copies for the general kernels (the 256x256 transposes are skipped on the device when the masks are column-only)
  if (is256) {
    int rc = prox_prepare_cl(y0, mask, mask_bstride, y0p, reinterpret_cast<uint16_t*>(maskp), B, st, flag);
    if (rc) return rc;
  } else if (H == 128 && W == 128) {
    // 128x128: the cluster kernel serves EVERY mask (measured faster than the generic row-only kernel even for column-only
    // masks: 0.41-0.48 vs 0.34-0.42 of the HBM roofline, profiles/r02_config5_sweep_n1.txt), so it is always prepared
    int rc = prox_prepare_cl128(y0, mask, mask_bstride, y0p, reinterpret_cast<uint16_t*>(maskp), B, st, nullptr);
    if (rc) return rc;
    return int(cudaGetLastError());
  } else {
    cudaMemcpyAsync(y0p, y0, n * sizeof(float2), cudaMemcpyDeviceToDevice, st);
    cudaMemcpyAsync(maskp, mask, size_t(nb) * H * W, cudaMemcpyDeviceToDevice, st);
  }
  ColsParams c{};
  c.H = H; c.W = W; c.t = y0p + n; c.src = y0; c.blend = 0;
  c.load_sign = 1; c.load_conj = 1; c.load_neg = (((H + W) / 2) & 1) ? 1 : 0;
  c.store_conj = 1; c.store_scale = 1.0f / sqrtf(float(H));
  c.skip_unless_flag = flag;                                          // Yt is only read by the row-only kernels
  DISPATCH_N(H, launch_cols, c, B, st);
  return int(cudaGetLastError());
}

// The structure flag written by prox_prepare (device int32: != 0 = every mask of the batch depends on the column index only).
const int* prox_prepared_flag(const uint8_t* maskp, long long mask_bstride, int B, int H, int W) {
  return reinterpret_cast<const int*>(maskp + maskp_flag_off(mask_bstride ? B : 1, H, W));
}

// kind: -1 = unknown on the host (both kernels are launched, the device flag picks one), 0 = general masks (only the general
// kernel), 1 = column-only masks (only the row kernel).  0 / 1 must come from the flag itself (pnp_prox_prepared_kind_async).
int prox_dual_prepared(const float* x, const float2* u_in, const float2* y0p, const uint8_t* maskp,
                       long long mask_bstride, const float* mu, int mu_stride, float2* z_out, float2* u_out,
                       float* v_out, int B, int H, int W, int kind, cudaStream_t st, const uint8_t* active) {
  if (!fft_shape_supported(H, W)) return -2;
  const int nb = mask_bstride ? B : 1;
  const size_t n = size_t(B) * H * W;
  const int* flag = reinterpret_cast<const int*>(maskp + maskp_flag_off(nb, H, W));
  const uint8_t* rowmask = maskp + maskp_pack_off(nb, H, W);
  if (H == 256 && W == 256) {
    if (kind != 0) {
      SepParams sp{x, u_in, y0p + n, reinterpret_cast<const uint16_t*>(rowmask), mask_bstride ? 1 : 0, flag, mu, mu_stride,
                   z_out, u_out, v_out, B * H, B <= 96 ? 1 : 0, active};   // Yt row prefetch pays while latency-bound (r01_prox_prefetch_ab)
      int rc = launch_sep(sp, num_sms(), st);
      if (rc || kind == 1) return rc;
    }
    ClParams cp{x, u_in, y0p, reinterpret_cast<const uint16_t*>(maskp), mask_bstride ? 16 * kClN : 0, mu, mu_stride,
                z_out, u_out, v_out, B, flag, active};
    return launch_cl(cp, st);
  }
  if (H == 128 && W == 128) {                             // every mask at 128x128: the 4-CTA cluster kernel (see prox_prepare)
    ClParams cp{x, u_in, y0p, reinterpret_cast<const uint16_t*>(maskp), mask_bstride ? 8 * kC128N : 0, mu, mu_stride,
                z_out, u_out, v_out, B, nullptr, active};
    return launch_cl128(cp, st);
  }
  if (kind != 0) {
  SepGenParams gp{x, u_in, y0p + n, rowmask, mask_bstride ? 1 : 0, flag, mu, mu_stride, z_out, u_out, v_out, H, 0, active};
  switch (W) {
    case 32: gp.groups_total = B * H / FftPlan<32>::G; launch_sep_generic<32>(gp, num_sms(), st); break;
    case 64: gp.groups_total = B * H / FftPlan<64>::G; launch_sep_generic<64>(gp, num_sms(), st); break;
    case 128: gp.groups_total = B * H / FftPlan<128>::G; launch_sep_generic<128>(gp, num_sms(), st); break;
    case 256: gp.groups_total = B * H / FftPlan<256>::G; launch_sep_generic<256>(gp, num_sms(), st); break;
    default: gp.groups_total = B * H / FftPlan<512>::G; launch_sep_generic<512>(gp, num_sms(), st); break;
  }
  if (kind == 1) return int(cudaGetLastError());
  }
  // any other mask: the general three-launch path on the copies, gated by the same flag
  return prox_dual_general_impl(x, u_in, y0p, maskp, mask_bstride, mu, mu_stride, z_out, u_out, v_out,
                                const_cast<float2*>(y0p) + 2 * n, B, H, W, flag, st, active);
}

// General three-launch prox + dual update.  `work` is a c64 [B,H,W] scratch buffer.
int prox_dual_general(const float* x, const float2* u_in, const float2* y0, const uint8_t* mask,
                      long long mask_bstride, const float* mu, int mu_stride, float2* z_out, float2* u_out,
                      float* v_out, float2* work, int B, int H, int W, cudaStream_t st) {
  return prox_dual_general_impl(x, u_in, y0, mask, mask_bstride, mu, mu_stride, z_out, u_out, v_out, work, B, H, W,
                                nullptr, st);
}

static int prox_dual_general_impl(const float* x, const float2* u_in, const float2* y0, const uint8_t* mask,
                                  long long mask_bstride, const float* mu, int mu_stride, float2* z_out, float2* u_out,
                                  float* v_out, float2* work, int B, int H, int W, const int* skip_flag, cudaStream_t st,
                                  const uint8_t* active) {
  if (!fft_shape_supported(H, W))
    return (skip_flag == nullptr) ? prox_dual_any(x, u_in, y0, mask, mask_bstride, mu, mu_stride, z_out, u_out, v_out, work,
                                                   B, H, W, st, active)
                                  : -2;
  if (skip_flag == nullptr) {
    // single-launch cluster kernels (256x256, 128x128): y0R and the packed mask go to the workspace first
    if (H == 128 && W == 128) {
      float2* y0R = work;
      uint16_t* mpack = reinterpret_cast<uint16_t*>(work + size_t(B) * H * W);
      int rc = prox_prepare_cl128(y0, mask, mask_bstride, y0R, mpack, B, st);
      if (rc) return rc;
      ClParams cp{x, u_in, y0R, mpack, mask_bstride ? 8 * kC128N : 0, mu, mu_stride, z_out, u_out, v_out, B, nullptr, nullptr};
      return launch_cl128(cp, st);
    }
    if (H == 256 && W == 256) {
      float2* y0R = work;
      uint16_t* mpack = reinterpret_cast<uint16_t*>(work + size_t(B) * H * W);
      int rc = prox_prepare_cl(y0, mask, mask_bstride, y0R, mpack, B, st);
      if (rc) return rc;
      ClParams cp{x, u_in, y0R, mpack, mask_bstride ? 16 * kClN : 0, mu, mu_stride, z_out, u_out, v_out, B, nullptr, nullptr};
      return launch_cl(cp, st);
    }
  }
  const float inv = 1.0f / sqrtf(float(H) * float(W));
  RowsParams r1{};
  r1.H = H; r1.W = W; r1.load_mode = ROWS_LOAD_XU; r1.store_mode = ROWS_STORE_C; r1.load_sign = 1;
  r1.x = x; r1.u = u_in; r1.dst = work; r1.store_scale = 1.f; r1.skip_flag = skip_flag;
  DISPATCH_N(W, launch_rows, r1, B, st);
  ColsParams c{};
  c.H = H; c.W = W; c.t = work; c.src = work; c.blend = 1; c.y0 = y0; c.mask = mask; c.mask_bstride = mask_bstride;
  c.mu = mu; c.mu_stride = mu_stride; c.scale1 = inv; c.sgn = (((H + W) / 2) & 1) ? -1.f : 1.f;
  c.store_scale = 1.f; c.skip_flag = skip_flag;
  DISPATCH_N(H, launch_cols, c, B, st);
  RowsParams r2{};
  r2.H = H; r2.W = W; r2.load_mode = ROWS_LOAD_C; r2.store_mode = ROWS_STORE_PROX; r2.src = work;
  r2.x = x; r2.u = u_in; r2.store_scale = inv; r2.store_conj = 1; r2.store_sign = 1;
  r2.z_out = z_out; r2.u_out = u_out; r2.v_out = v_out; r2.skip_flag = skip_flag; r2.active = active;
  DISPATCH_N(W, launch_rows, r2, B, st);
  return int(cudaGetLastError());
}

// Stand-alone centred orthonormal 2-D transform (mirror of transformations.py fft / ifft). dst may equal src.
int fft2c_general(const float2* src, float2* dst, int B, int H, int W, int inverse, cudaStream_t st) {
  if (!fft_shape_supported(H, W)) return fft2c_any(src, dst, B, H, W, inverse, st);
  const float inv = 1.0f / sqrtf(float(H) * float(W));
  const float s = (((H + W) / 2) & 1) ? -1.f : 1.f;
  RowsParams r{};
  r.H = H; r.W = W; r.load_mode = ROWS_LOAD_C; r.store_mode = ROWS_STORE_C; r.load_sign = 1; r.load_conj = inverse;
  r.src = src; r.dst = dst; r.store_scale = 1.f;
  DISPATCH_N(W, launch_rows, r, B, st);
  ColsParams c{};
  c.H = H; c.W = W; c.t = dst; c.src = dst; c.blend = 0; c.store_scale = inv * s; c.store_sign = 1;
  c.store_conj = inverse;
  DISPATCH_N(H, launch_cols, c, B, st);
  return int(cudaGetLastError());
}

}  // namespace pnp

#ifdef PNP_PROX_PHASE_TIMING
// Debug build only (tools/prox_phases.py): read and clear the per-phase cycle sums of fftprox_cl_kernel.  Synchronises.
extern "C" int pnp_debug_prox_phases(unsigned long long* out16) {
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return int(e);
  e = cudaMemcpyFromSymbol(out16, pnp::g_f2_phase, 16 * sizeof(unsigned long long));
  if (e != cudaSuccess) return int(e);
  unsigned long long zero[16] = {};
  return int(cudaMemcpyToSymbol(pnp::g_f2_phase, zero, sizeof(zero)));
}
#endif
