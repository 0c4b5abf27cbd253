// Any-size path of the centred transforms and of the FFT-prox + dual update: H, W in 2..1024 that are NOT powers of two in
// 32..512 (those have the radix kernels).  The reference's `step` (evaluation/env.py:74-100) works at such sizes because
// torch.fft is mixed-radix (e.g. 130x130, 136x120, odd sizes); the drop-in therefore has to as well.
//
// Algebra.  With h = N / 2 (integer division) the reference's 1-D centred transform
//     fft_c(w) = fftshift(FFT(ifftshift(w))) / sqrt(N)          (evaluation/utils/transformations.py:6-12)
// is, for EVERY N (even or odd: ifftshift rolls by -h, fftshift by +h),
//     fft_c(w)[k] = 1/sqrt(N) * sum_m w[m] * omega^((m - h)(k - h)),   omega = exp(-2 pi i / N),
// and ifft_c (transformations.py:14-19) is the same sum with conj(omega): a dense N x N matrix whose entries are looked up
// in an N-entry table by the exponent (m - h)(k - h) mod N, walked incrementally (any_dft_lines, line_passes.cuh).
// O(N^2) per line instead of O(N log N): this is the compatibility path (a 130x130 image-iteration is ~35 MFLOP), not the
// throughput path; k-space coordinates need no rotation and the mask / y0 are read in place (no prepared constants).
//
// Three dense line passes (dense_lines_kernel) like the radix general path (fftprox.cu): rows -> work; columns: DFT,
// blend, inverse DFT in shared memory -> work; rows inverse + dual-update epilogue.  The blend and the epilogue below are
// shared with the radix ops of fftprox.cu, which add the centring signs.
#pragma once
#include "common.cuh"
#include "line_passes.cuh"

namespace pnp {

// One image's blend constants.
struct BlendImage {
  float mu, inv1mu;
  const uint8_t* mk;
};

// Column passes of the prox: blend(Z) = (mu Z + y) / (1 + mu) under the mask, Z elsewhere (env.py:88-90).
struct ProxBlendOp : LineOp {
  static constexpr bool kMiddle = true;
  const float2* y0;         // [B,H,W]
  const uint8_t* mask;      // [mask_B,H,W]
  long long mask_bstride;   // 0 when one mask is shared by the batch
  const float* mu;          // [B] or [1]
  int mu_stride;
  __device__ BlendImage middle_begin(int b) const {
    const float m = mu[size_t(b) * mu_stride];
    return {m, 1.f / (1.f + m), mask + size_t(b) * mask_bstride};
  }
  // y: y0 at the sample, times the centring sign where the transform leaves one
  __device__ static float2 blend(const BlendImage& m, float2 Z, float2 y) {
    return make_float2((m.mu * Z.x + y.x) * m.inv1mu, (m.mu * Z.y + y.y) * m.inv1mu);
  }
};

// Row-out stores of the prox: z, u' = u + x - z (env.py:93), v' = Re(z - u') (the next denoiser input).  u and x are
// plain loads (u_out may alias u), fetched by preload().
struct ProxDualOp : LineOp {
  const float* x;           // [B,H,W]
  const float2* u;          // [B,H,W]
  float2* z_out;
  float2* u_out;
  float* v_out;             // may be null
  const uint8_t* active;    // optional [B]: 0 = leave the image's z, u, v untouched
  struct Pre {
    float2 u;
    float x;
  };
  __device__ bool image_active(int b) const { return !(active && active[b] == 0); }
  __device__ Pre preload(const LineElem& e) const { return {u[e.g], x[e.g]}; }
  __device__ void store_dual(size_t g, float2 z, const Pre& p) const {
    const float2 un = make_float2(p.u.x + p.x - z.x, p.u.y - z.y);
    z_out[g] = z;
    u_out[g] = un;
    if (v_out) v_out[g] = z.x - un.x;
  }
};

// ---- dense ops: the transforms are centred and scaled inside any_dft_lines
struct ProxAnyRowsIn : LineOp {
  static constexpr bool kRows = true;
  const float* x;
  const float2* u;
  float2* work;
  float norm;               // 1 / sqrt(W)
  __device__ bool inverse() const { return false; }
  __device__ float scale(int) const { return norm; }
  __device__ float2 load(const LineElem& e) const {
    const float2 uu = u[e.g];
    return make_float2(x[e.g] + uu.x, uu.y);
  }
  __device__ void store(const LineElem& e, float2 v, Pre) const { work[e.g] = v; }
};

struct ProxAnyColsBlend : ProxBlendOp {
  static constexpr bool kRows = false;
  float2* work;
  float norm;               // 1 / sqrt(H)
  __device__ bool inverse() const { return false; }
  __device__ float scale(int) const { return norm; }
  __device__ float2 load(const LineElem& e) const { return work[e.g]; }
  __device__ float2 middle(const BlendImage& m, const LineElem& e, float2 Z) const {
    return m.mk[e.o] ? blend(m, Z, y0[e.g]) : Z;
  }
  __device__ void store(const LineElem& e, float2 v, Pre) const { work[e.g] = v; }
};

struct ProxAnyRowsOut : ProxDualOp {
  static constexpr bool kRows = true;
  const float2* work;
  float norm;               // 1 / sqrt(W)
  __device__ bool inverse() const { return true; }
  __device__ float scale(int) const { return norm; }
  __device__ float2 load(const LineElem& e) const { return work[e.g]; }
  __device__ void store(const LineElem& e, float2 v, const Pre& p) const { store_dual(e.g, v, p); }
};

template <bool ROWS> struct Fft2cAny : LineOp {
  static constexpr bool kRows = ROWS;
  const float2* src;
  float2* dst;
  float norm;               // 1 / sqrt(length)
  int inv;
  __device__ bool inverse() const { return inv != 0; }
  __device__ float scale(int) const { return norm; }
  __device__ float2 load(const LineElem& e) const { return src[e.g]; }
  __device__ void store(const LineElem& e, float2 v, Pre) const { dst[e.g] = v; }
};

// z = ifft_c(blend(fft_c(x + u))), u' = u + x - z, v' = Re(z - u') for any H, W in 2..1024; `work` = c64 [B,H,W] scratch.
static int prox_dual_any(const float* x, const float2* u_in, const float2* y0, const uint8_t* mask, long long mask_bstride,
                         const float* mu, int mu_stride, float2* z_out, float2* u_out, float* v_out, float2* work, int B,
                         int H, int W, cudaStream_t st, const uint8_t* active) {
  if (!any_shape_supported(H, W)) return -2;
  const float nw = 1.0f / sqrtf(float(W)), nh = 1.0f / sqrtf(float(H));
  int rc = dense_lines(ProxAnyRowsIn{{}, x, u_in, work, nw}, H, W, B, st);
  if (rc == 0) rc = dense_lines(ProxAnyColsBlend{{{}, y0, mask, mask_bstride, mu, mu_stride}, work, nh}, H, W, B, st);
  if (rc == 0) rc = dense_lines(ProxAnyRowsOut{{{}, x, u_in, z_out, u_out, v_out, active}, work, nw}, H, W, B, st);
  return rc;
}

// Stand-alone centred orthonormal 2-D transform for any H, W in 2..1024 (dst may equal src).
static int fft2c_any(const float2* src, float2* dst, int B, int H, int W, int inverse, cudaStream_t st) {
  if (!any_shape_supported(H, W)) return -2;
  int rc = dense_lines(Fft2cAny<true>{{}, src, dst, 1.0f / sqrtf(float(W)), inverse}, H, W, B, st);
  if (rc == 0) rc = dense_lines(Fft2cAny<false>{{}, dst, dst, 1.0f / sqrtf(float(H)), inverse}, H, W, B, st);
  return rc;
}

}  // namespace pnp
