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
// This file is the general (any power-of-two H, W in 32..512) three-launch path, the ops ProxRowsIn / ProxColsBlend /
// ProxRowsOut on the radix line passes of line_passes.cuh:
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
#include "line_passes.cuh"
#include "fftprox_any.cuh"
#include "measure.cuh"
namespace pnp {

// ---- radix ops of the general path (the centring signs D and s as in the header; blend and epilogue in fftprox_any.cuh)
// rows in: D.(x + u) -> row FFTs -> work
struct ProxRowsIn : LineOp {
  const float* x;
  const float2* u;
  float2* work;
  const int* skip_flag;     // optional: != 0 -> the row-only kernel handles this batch, do nothing
  __device__ bool skip() const { return skip_flag && *skip_flag != 0; }
  __device__ float2 load(const LineElem& e) const {
    const float2 uu = u[e.g];
    float2 v = make_float2(x[e.g] + uu.x, uu.y);
    if ((e.i + e.j) & 1) { v.x = -v.x; v.y = -v.y; }
    return v;
  }
  __device__ void store(const LineElem& e, float2 v, Pre) const { work[e.g] = v; }
};

// columns: col FFT -> / sqrt(HW) -> blend with s.D.y0 -> conj -> col FFT (the inverse, conjugated) -> work
struct ProxColsBlend : ProxBlendOp {
  float2* work;
  float norm;               // 1 / sqrt(HW)
  float sgn;                // s
  const int* skip_flag;
  __device__ bool skip() const { return skip_flag && *skip_flag != 0; }
  __device__ float2 load(const LineElem& e) const { return work[e.g]; }
  __device__ float2 middle(const BlendImage& m, const LineElem& e, float2 Z) const {
    Z.x *= norm; Z.y *= norm;
    if (m.mk[e.o]) {
      const float2 y = y0[e.g];
      const float sg = ((e.i + e.j) & 1) ? -sgn : sgn;
      Z = blend(m, Z, make_float2(sg * y.x, sg * y.y));
    }
    return make_float2(Z.x, -Z.y);   // conj -> forward FFT == inverse
  }
  __device__ void store(const LineElem& e, float2 v, Pre) const { work[e.g] = v; }
};

// rows out: row FFTs -> z = D.conj(.) / sqrt(HW) -> z, u', v'
struct ProxRowsOut : ProxDualOp {
  // left alone, ptxas gives the epilogue the registers of one CTA per SM at these lengths
  template <int N> static constexpr int kRowCtas = N == 32 ? 8 : N == 256 ? 6 : 0;
  const float2* work;
  float norm;               // 1 / sqrt(HW)
  const int* skip_flag;
  __device__ bool skip() const { return skip_flag && *skip_flag != 0; }
  __device__ float2 load(const LineElem& e) const { return work[e.g]; }
  __device__ void store(const LineElem& e, float2 v, const Pre& p) const {
    v.x *= norm; v.y *= norm;
    v.y = -v.y;
    if ((e.i + e.j) & 1) { v.x = -v.x; v.y = -v.y; }
    store_dual(e.g, v, p);
  }
};

// pnp_fft2c: rows D.w (conj(w) for the inverse) -> row FFTs -> dst; columns col FFT -> s.D / sqrt(HW) (conj) -> dst
struct Fft2cRows : LineOp {
  const float2* src;
  float2* dst;
  int inv;
  __device__ float2 load(const LineElem& e) const {
    float2 v = src[e.g];
    if (inv) v.y = -v.y;
    if ((e.i + e.j) & 1) { v.x = -v.x; v.y = -v.y; }
    return v;
  }
  __device__ void store(const LineElem& e, float2 v, Pre) const { dst[e.g] = v; }
};

struct Fft2cCols : LineOp {
  float2* dst;
  float norm;               // s / sqrt(HW)
  int inv;
  __device__ float2 load(const LineElem& e) const { return dst[e.g]; }
  __device__ void store(const LineElem& e, float2 v, Pre) const {
    v.x *= norm; v.y *= norm;
    if (inv) v.y = -v.y;
    if ((e.i + e.j) & 1) { v.x = -v.x; v.y = -v.y; }
    dst[e.g] = v;
  }
};

// prox_prepare: Yt = Fc^-1(s.D.y0) = conj(FFT_col(conj(s.D.y0))) / sqrt(H), read only by the row-only kernels
struct PrepareYt : LineOp {
  const float2* y0;
  float2* yt;
  float sgn;                // s
  float norm;               // 1 / sqrt(H)
  const int* flag;          // == 0 (not every mask is column-only) -> do nothing
  __device__ bool skip() const { return *flag == 0; }
  __device__ float2 load(const LineElem& e) const {
    float2 v = y0[e.g];
    v.y = -v.y;
    if ((((e.i + e.j) & 1) != 0) != (sgn < 0.f)) { v.x = -v.x; v.y = -v.y; }
    return v;
  }
  __device__ void store(const LineElem& e, float2 v, Pre) const {
    v.x *= norm; v.y *= norm;
    v.y = -v.y;
    yt[e.g] = v;
  }
};

// The three radix passes of the general path.  skip_flag: optional device flag, != 0 -> the row-only kernel handles this
// batch; active as in ClParams.
static int prox_radix3(const float* x, const float2* u_in, const float2* y0, const uint8_t* mask, long long mask_bstride,
                       const float* mu, int mu_stride, float2* z_out, float2* u_out, float* v_out, float2* work, int B, int H,
                       int W, const int* skip_flag, const uint8_t* active, cudaStream_t st) {
  const float inv = 1.0f / sqrtf(float(H) * float(W));
  int rc = radix_rows(ProxRowsIn{{}, x, u_in, work, skip_flag}, H, W, B, st);
  if (rc == 0)
    rc = radix_cols(ProxColsBlend{{{}, y0, mask, mask_bstride, mu, mu_stride}, work, inv, centre_sign(H, W), skip_flag},
                    H, W, B, st);
  if (rc == 0)
    rc = radix_rows(ProxRowsOut{{{}, x, u_in, z_out, u_out, v_out, active}, work, inv, skip_flag}, H, W, B, st);
  return rc;
}

// Shapes with a single-launch cluster kernel: 256x256 (fftprox_cl.cuh) and 128x128 (fftprox_cl128.cuh).
static bool cluster_shape(int H, int W) { return H == W && (H == kClN || H == kC128N); }

// The cluster kernel's trajectory constants y0R and packed rotated mask (fftprox_cl.cuh "Algebra") at a cluster shape.
static int prepare_cluster(const float2* y0, const uint8_t* mask, long long mask_bstride, float2* y0R, uint16_t* mpack,
                           int B, int H, const int* skip_flag, cudaStream_t st) {
  const int nb = mask_bstride ? B : 1;
  if (H == kClN)
    prox_prepare_cl_kernel<<<dim3(kClN, B), 256, 0, st>>>(y0, mask, mask_bstride, y0R, mpack, nb, skip_flag);
  else
    prox_prepare_cl128_kernel<<<dim3(kC128N, B), kC128N, 0, st>>>(y0, mask, mask_bstride, y0R, mpack, nb, skip_flag);
  return int(cudaGetLastError());
}

// One cluster-kernel prox + dual update on the constants of prepare_cluster.
static int launch_cluster(const float* x, const float2* u_in, const float2* y0R, const uint16_t* mpack, bool per_image_mask,
                          const float* mu, int mu_stride, float2* z_out, float2* u_out, float* v_out, int B, int H,
                          const int* skip_flag, const uint8_t* active, cudaStream_t st) {
  const long long mpack_bstride = !per_image_mask ? 0 : H == kClN ? 16 * kClN : 8 * kC128N;
  const ClParams cp{x, u_in, y0R, mpack, mpack_bstride, mu, mu_stride, z_out, u_out, v_out, B, skip_flag, active};
  return H == kClN ? launch_cl(cp, st) : launch_cl128(cp, st);
}

static bool pow2_ok(int n) { return n == 32 || n == 64 || n == 128 || n == 256 || n == 512; }

int fft_shape_supported(int H, int W) { return pow2_ok(H) && pow2_ok(W); }
// every shape some kernel serves: the radix passes or the dense-DFT pass (line_passes.cuh, 2..1024)
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
  if (cluster_shape(H, W)) {
    // the 256x256 constants are skipped on the device when the masks are column-only; 128x128: the cluster kernel serves
    // EVERY mask (measured faster than the generic row-only kernel even for column-only masks: 0.41-0.48 vs 0.34-0.42 of
    // the HBM roofline, profiles/r02_config5_sweep_n1.txt), so it is always prepared and needs no Yt
    int rc = prepare_cluster(y0, mask, mask_bstride, y0p, reinterpret_cast<uint16_t*>(maskp), B, H, is256 ? flag : nullptr,
                             st);
    if (rc || !is256) return rc;
  } else {                                                            // copies for the general kernels
    cudaMemcpyAsync(y0p, y0, n * sizeof(float2), cudaMemcpyDeviceToDevice, st);
    cudaMemcpyAsync(maskp, mask, size_t(nb) * H * W, cudaMemcpyDeviceToDevice, st);
  }
  return radix_cols(PrepareYt{{}, y0, y0p + n, centre_sign(H, W), 1.0f / sqrtf(float(H)), flag}, H, W, B, st);
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
    return launch_cluster(x, u_in, y0p, reinterpret_cast<const uint16_t*>(maskp), mask_bstride != 0, mu, mu_stride, z_out,
                          u_out, v_out, B, H, flag, active, st);
  }
  if (H == 128 && W == 128)                               // every mask at 128x128: the 4-CTA cluster kernel (see prox_prepare)
    return launch_cluster(x, u_in, y0p, reinterpret_cast<const uint16_t*>(maskp), mask_bstride != 0, mu, mu_stride, z_out,
                          u_out, v_out, B, H, nullptr, active, st);
  if (kind != 0) {
    SepGenParams gp{x, u_in, y0p + n, rowmask, mask_bstride ? 1 : 0, flag, mu, mu_stride, z_out, u_out, v_out, H, 0, active};
    with_pow2(W, [&](auto w) {
      gp.groups_total = B * H / FftPlan<decltype(w)::value>::G;
      launch_sep_generic<decltype(w)::value>(gp, num_sms(), st);
    });
    if (kind == 1) return int(cudaGetLastError());
  }
  // any other mask: the general three-launch path on the copies, gated by the same flag
  return prox_radix3(x, u_in, y0p, maskp, mask_bstride, mu, mu_stride, z_out, u_out, v_out, const_cast<float2*>(y0p) + 2 * n,
                     B, H, W, flag, active, st);
}

// Unprepared prox + dual update.  `work` is a c64 [B,H,W] scratch buffer; at 256x256 and 128x128 the cluster kernel's
// constants go there first.
int prox_dual_general(const float* x, const float2* u_in, const float2* y0, const uint8_t* mask,
                      long long mask_bstride, const float* mu, int mu_stride, float2* z_out, float2* u_out,
                      float* v_out, float2* work, int B, int H, int W, cudaStream_t st) {
  if (!fft_shape_supported(H, W))
    return prox_dual_any(x, u_in, y0, mask, mask_bstride, mu, mu_stride, z_out, u_out, v_out, work, B, H, W, st, nullptr);
  if (cluster_shape(H, W)) {
    uint16_t* mpack = reinterpret_cast<uint16_t*>(work + size_t(B) * H * W);
    int rc = prepare_cluster(y0, mask, mask_bstride, work, mpack, B, H, nullptr, st);
    if (rc) return rc;
    return launch_cluster(x, u_in, work, mpack, mask_bstride != 0, mu, mu_stride, z_out, u_out, v_out, B, H, nullptr, nullptr,
                          st);
  }
  return prox_radix3(x, u_in, y0, mask, mask_bstride, mu, mu_stride, z_out, u_out, v_out, work, B, H, W, nullptr, nullptr, st);
}

// Stand-alone centred orthonormal 2-D transform (mirror of transformations.py fft / ifft). dst may equal src.
int fft2c_general(const float2* src, float2* dst, int B, int H, int W, int inverse, cudaStream_t st) {
  if (!fft_shape_supported(H, W)) return fft2c_any(src, dst, B, H, W, inverse, st);
  const float inv = 1.0f / sqrtf(float(H) * float(W));
  int rc = radix_rows(Fft2cRows{{}, src, dst, inverse}, H, W, B, st);
  if (rc == 0) rc = radix_cols(Fft2cCols{{}, dst, inv * centre_sign(H, W), inverse}, H, W, B, st);
  return rc;
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
