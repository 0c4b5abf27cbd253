// Measurement simulator: undersampled, noisy k-space measurements of fully-sampled images, and seeded Cartesian and radial
// masks (pnp_simulate_measurements / pnp_cartesian_masks / pnp_radial_masks; the definitions are in include/pnp_b200.h).
// Per image b:
//
//     y0   = mask ? fft_c(gt) + sigma_n / 255 * (n_r + i n_i) : 0      (n_r, n_i: Philox4x32-10 + Box-Muller at (i, j))
//     ATy0 = ifft_c(y0),   x0 = (max(Re ATy0, 0), max(Im ATy0, 0))
//
// Three launches with the shape of the general prox path (fftprox.cu); the c64 intermediate T lives in x0 (every pass loads
// its whole lines into shared memory before it stores the same lines, so no workspace is needed):
//   rows : load D.gt (real)           -> row FFTs                                            -> T
//   cols : load columns of T -> col FFT -> s.D / sqrt(HW) = K -> noise, mask -> y0 (stored)
//          -> conj(D.y0) -> col FFT                                                          -> T
//   rows : load T -> row FFTs -> conj, s.D / sqrt(HW) = ATy0 -> x0 (and ATy0)
// with D[i,j] = (-1)^(i+j), s = (-1)^((H+W)/2) as in fftprox.cu.  Powers of two in 32..512 take the radix kernels below
// (fft_core.cuh); every other H, W in 2..1024 takes the dense-DFT kernel (any_dft_lines, fftprox_any.cuh), which computes
// the centred transforms directly.  The noise of a sample depends only on (seed, H, W, i, j), never on the mask or the batch
// position, and nothing is accumulated across CTAs, so every output is bitwise reproducible.
#pragma once
#include "common.cuh"
#include "fft_core.cuh"
#include "fftprox_any.cuh"

namespace pnp {

// Random123 Philox4x32-10 (Salmon et al., SC'11): 10 rounds, multipliers 0xD2511F53 / 0xCD9E8D57, key increments
// 0x9E3779B9 / 0xBB67AE85.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) { k.x += 0x9E3779B9u; k.y += 0xBB67AE85u; }
    const unsigned lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const unsigned lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
  }
  return c;
}

__device__ __forceinline__ uint2 seed_key(unsigned long long seed) {
  return make_uint2(unsigned(seed & 0xFFFFFFFFull), unsigned(seed >> 32));
}

// (n_r, n_i) of k-space sample p = i*W + j: Box-Muller on u = (w + 0.5) * 2^-32, so u is never 0 or 1 in exact arithmetic
// (fp32 may round u1 up to 1, which gives n = 0, never a NaN).
__device__ __forceinline__ float2 sample_noise(unsigned p, uint2 key) {
  const uint4 w = philox4x32_10(make_uint4(p, 0u, 0u, 0u), key);
  const float u1 = fmaf(__uint2float_rn(w.x), 0x1p-32f, 0x1p-33f);
  const float u2 = fmaf(__uint2float_rn(w.y), 0x1p-32f, 0x1p-33f);
  const float r = sqrtf(-2.f * logf(u1));
  float sn, cs;
  sincospif(2.f * u2, &sn, &cs);
  return make_float2(r * cs, r * sn);
}

// K -> y0 sample at (i, j): the noise is drawn only where the mask samples (it does not depend on the mask).
__device__ __forceinline__ float2 measure_sample(float2 K, bool sampled, int i, int j, int W, float sig, uint2 key) {
  if (!sampled) return make_float2(0.f, 0.f);
  const float2 n = sample_noise(unsigned(i * W + j), key);
  return make_float2(fmaf(sig, n.x, K.x), fmaf(sig, n.y, K.y));
}

struct SimParams {
  int H, W;
  const float* gt;              // [B or 1, H, W]
  long long gt_bstride;         // H*W, or 0 for one shared gt
  const uint8_t* mask;          // [B or 1, H, W]
  long long mask_bstride;
  const float* sigma;           // sigma_n[b * sigma_stride]
  int sigma_stride;
  const unsigned long long* seeds;   // [B]
  float2* y0;                   // [B, H, W]
  float2* x0;                   // [B, H, W]; holds T between the passes
  float2* aty0;                 // [B, H, W] or null
  float kscale;                 // radix: s / sqrt(HW)
  int gt_vec4;                  // radix rows pass: every image's gt is 16-byte aligned
};

// ---------------------------------------------------------------- radix path (H, W powers of two in 32..512)
// Pass 1: D.gt -> row FFTs -> T.  N = W; a warp owns G consecutive rows (G*N contiguous floats).
template <int N>
__global__ void __launch_bounds__(256) sim_rows_fwd_kernel(const SimParams p) {
  constexpr int G = FftPlan<N>::G;
  constexpr int P = fft_pitch(N);
  __shared__ float2 tw[kTwTotal];
  extern __shared__ float2 sim_rows_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  fft_load_twiddles(tw, g_tw512);
  __syncthreads();
  const int b = blockIdx.y;
  const int row0 = (blockIdx.x * 8 + warp) * G;
  if (row0 >= p.H) return;
  float2* mine = sim_rows_smem + warp * G * P;
  const float* g = p.gt + size_t(b) * p.gt_bstride + size_t(row0) * N;
  if (p.gt_vec4) {
    for (int q = lane; q < G * N / 4; q += 32) {
      const float4 v = reinterpret_cast<const float4*>(g)[q];
      const int r = (4 * q) / N, j = (4 * q) % N;
      const float s = ((row0 + r) & 1) ? -1.f : 1.f;     // D at the even column j
      float2* d = mine + r * P;
      d[fpad(j)] = make_float2(s * v.x, 0.f);
      d[fpad(j + 1)] = make_float2(-s * v.y, 0.f);
      d[fpad(j + 2)] = make_float2(s * v.z, 0.f);
      d[fpad(j + 3)] = make_float2(-s * v.w, 0.f);
    }
  } else {
    for (int e = lane; e < G * N; e += 32) {
      const int r = e / N, j = e % N;
      const float v = g[e];
      mine[r * P + fpad(j)] = make_float2(((row0 + r + j) & 1) ? -v : v, 0.f);
    }
  }
  __syncwarp();
  fft_warp_rows<N>(mine, P, tw, lane);
  float2* t = p.x0 + size_t(b) * p.H * N + size_t(row0) * N;
  for (int e = lane; e < G * N; e += 32) t[e] = mine[(e / N) * P + fpad(e % N)];
}

// Pass 2: columns of T -> col FFT -> K -> y0 -> conj(D.y0) -> col FFT -> T.  N = H; a CTA owns NCOL = 8*G adjacent
// columns of one image, so the loads and the y0 / T stores walk NCOL contiguous elements of a row.
template <int N>
__global__ void __launch_bounds__(256) sim_cols_kernel(const SimParams p) {
  constexpr int G = FftPlan<N>::G;
  constexpr int NCOL = 8 * G;
  constexpr int P = fft_pitch(N) + ((fft_pitch(N) % 16 == 0) ? 4 : 0);   // de-conflict the transposed fill
  __shared__ float2 tw[kTwTotal];
  extern __shared__ float2 sim_cols_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  fft_load_twiddles(tw, g_tw512);
  const int b = blockIdx.y, W = p.W;
  const int c0 = blockIdx.x * NCOL;
  float2* t = p.x0 + size_t(b) * N * W;
  for (int e = threadIdx.x; e < N * NCOL; e += blockDim.x) {
    const int c = e % NCOL, i = e / NCOL;
    sim_cols_smem[c * P + fpad(i)] = (c0 + c < W) ? t[size_t(i) * W + c0 + c] : make_float2(0.f, 0.f);
  }
  __syncthreads();
  float2* mine = sim_cols_smem + warp * G * P;
  fft_warp_rows<N>(mine, P, tw, lane);
  __syncthreads();
  const float sig = p.sigma[size_t(b) * p.sigma_stride] * (1.f / 255.f);
  const uint2 key = seed_key(p.seeds[b]);
  const uint8_t* mk = p.mask + size_t(b) * p.mask_bstride;
  float2* y0 = p.y0 + size_t(b) * N * W;
  for (int e = threadIdx.x; e < N * NCOL; e += blockDim.x) {
    const int c = e % NCOL, i = e / NCOL, j = c0 + c;
    if (j >= W) continue;
    const float d = ((i + j) & 1) ? -p.kscale : p.kscale;
    const float2 Z = sim_cols_smem[c * P + fpad(i)];
    const float2 y = measure_sample(make_float2(Z.x * d, Z.y * d), mk[size_t(i) * W + j] != 0, i, j, W, sig, key);
    y0[size_t(i) * W + j] = y;
    const float dy = ((i + j) & 1) ? -1.f : 1.f;
    sim_cols_smem[c * P + fpad(i)] = make_float2(dy * y.x, -dy * y.y);   // conj(D.y0): forward FFT == inverse
  }
  __syncthreads();
  fft_warp_rows<N>(mine, P, tw, lane);
  __syncthreads();
  for (int e = threadIdx.x; e < N * NCOL; e += blockDim.x) {
    const int c = e % NCOL, i = e / NCOL;
    if (c0 + c < W) t[size_t(i) * W + c0 + c] = sim_cols_smem[c * P + fpad(i)];
  }
}

// Pass 3: T -> row FFTs -> ATy0 = s.D.conj(.) / sqrt(HW) -> x0 = max(ATy0, 0) (and ATy0).  N = W.
template <int N>
__global__ void __launch_bounds__(256) sim_rows_inv_kernel(const SimParams p) {
  constexpr int G = FftPlan<N>::G;
  constexpr int P = fft_pitch(N);
  __shared__ float2 tw[kTwTotal];
  extern __shared__ float2 sim_rows_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  fft_load_twiddles(tw, g_tw512);
  __syncthreads();
  const int b = blockIdx.y;
  const int row0 = (blockIdx.x * 8 + warp) * G;
  if (row0 >= p.H) return;
  float2* mine = sim_rows_smem + warp * G * P;
  const size_t base = size_t(b) * p.H * N + size_t(row0) * N;
  for (int e = lane; e < G * N; e += 32) mine[(e / N) * P + fpad(e % N)] = p.x0[base + e];
  __syncwarp();
  fft_warp_rows<N>(mine, P, tw, lane);
  for (int e = lane; e < G * N; e += 32) {
    const int r = e / N, j = e % N;
    const float2 v = mine[r * P + fpad(j)];
    const float d = ((row0 + r + j) & 1) ? -p.kscale : p.kscale;
    const float2 a = make_float2(v.x * d, -v.y * d);
    if (p.aty0) p.aty0[base + e] = a;
    p.x0[base + e] = make_float2(fmaxf(a.x, 0.f), fmaxf(a.y, 0.f));
  }
}

// ---------------------------------------------------------------- dense-DFT path (every other H, W in 2..1024)
// PASS 0: gt rows -> fft_c along rows -> T;  PASS 1: columns of T -> fft_c -> y0 -> ifft_c -> T;
// PASS 2: rows of T -> ifft_c along rows -> x0, ATy0.  A CTA owns kAnyLines lines, as dft_any_kernel.
template <int PASS>
__global__ void __launch_bounds__(kAnyThreads) sim_any_kernel(const SimParams p) {
  extern __shared__ float2 sim_any_smem[];
  constexpr bool kRows = PASS != 1;
  const int W = p.W;
  const int N = kRows ? W : p.H;
  const int nlines = kRows ? p.H : W;
  const int P = any_pitch(N);
  float2* tw = sim_any_smem;
  float2* bufa = tw + N;
  float2* bufc = bufa + kAnyLines * P;
  const int b = blockIdx.y, l0 = blockIdx.x * kAnyLines;
  const int nl = min(kAnyLines, nlines - l0);
  const size_t img = size_t(b) * p.H * W;
  const float scale = rsqrtf(float(N));
  for (int k = threadIdx.x; k < N; k += kAnyThreads) {
    float s, c;
    sincospif(2.0f * float(k) / float(N), &s, &c);
    tw[k] = make_float2(c, PASS == 2 ? s : -s);
  }
  for (int e = threadIdx.x; e < kAnyLines * N; e += kAnyThreads) {
    int l, m;
    size_t g;
    if (kRows) { l = e / N; m = e % N; g = size_t(l0 + l) * W + m; }
    else       { l = e % kAnyLines; m = e / kAnyLines; g = size_t(m) * W + l0 + l; }
    if (l >= nl) continue;
    bufa[l * P + m] = (PASS == 0) ? make_float2(p.gt[size_t(b) * p.gt_bstride + g], 0.f) : p.x0[img + g];
  }
  __syncthreads();
  any_dft_lines(bufa, bufc, tw, N, P, nl, scale);
  __syncthreads();
  const float2* res = bufc;
  if (PASS == 1) {                                     // element (l, k) is k-space sample (row k, column l0 + l)
    const float sig = p.sigma[size_t(b) * p.sigma_stride] * (1.f / 255.f);
    const uint2 key = seed_key(p.seeds[b]);
    const uint8_t* mk = p.mask + size_t(b) * p.mask_bstride;
    for (int e = threadIdx.x; e < kAnyLines * N; e += kAnyThreads) {
      const int l = e % kAnyLines, k = e / kAnyLines;
      if (l >= nl) continue;
      const size_t g = size_t(k) * W + l0 + l;
      const float2 y = measure_sample(bufc[l * P + k], mk[g] != 0, k, l0 + l, W, sig, key);
      p.y0[img + g] = y;
      bufc[l * P + k] = y;
    }
    for (int k = threadIdx.x; k < N; k += kAnyThreads) tw[k].y = -tw[k].y;   // own entries only: no barrier needed before
    __syncthreads();
    any_dft_lines(bufc, bufa, tw, N, P, nl, scale);
    __syncthreads();
    res = bufa;
  }
  for (int e = threadIdx.x; e < kAnyLines * N; e += kAnyThreads) {
    int l, m;
    size_t g;
    if (kRows) { l = e / N; m = e % N; g = size_t(l0 + l) * W + m; }
    else       { l = e % kAnyLines; m = e / kAnyLines; g = size_t(m) * W + l0 + l; }
    if (l >= nl) continue;
    const float2 v = res[l * P + m];
    if (PASS != 2) {
      p.x0[img + g] = v;
    } else {
      if (p.aty0) p.aty0[img + g] = v;
      p.x0[img + g] = make_float2(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f));
    }
  }
}

// ---------------------------------------------------------------- Cartesian masks: one CTA per image
constexpr int kMaskThreads = 256;

__global__ void __launch_bounds__(kMaskThreads) cartesian_mask_kernel(const int* accel, int accel_stride,
                                                                      const unsigned long long* seeds, int acs_cols,
                                                                      uint8_t* out, int H, int W) {
  __shared__ unsigned long long rank_key[kAnyMaxN];
  __shared__ uint8_t col[kAnyMaxN];
  const int b = blockIdx.x;
  const int a = accel[size_t(b) * accel_stride];
  const int n_keep = (a >= 1) ? max(1, W / a) : W;     // accel < 1 samples every column
  const int n_acs = min(n_keep, acs_cols);
  const int c0 = W / 2 - n_acs / 2;
  const int extra = n_keep - n_acs;
  const uint2 key = seed_key(seeds[b]);
  // (key_j, j) as one 64-bit word, so the lexicographic order is the integer order; ACS columns get the largest word and
  // never precede a candidate
  for (int j = threadIdx.x; j < W; j += kMaskThreads) {
    const bool acs = j >= c0 && j < c0 + n_acs;
    rank_key[j] = acs ? ~0ull
                      : (((unsigned long long)philox4x32_10(make_uint4(unsigned(j), 1u, 0u, 0u), key).x << 32) | unsigned(j));
  }
  __syncthreads();
  for (int j = threadIdx.x; j < W; j += kMaskThreads) {
    const unsigned long long kj = rank_key[j];
    int rank = 0;
    for (int q = 0; q < W; ++q) rank += rank_key[q] < kj;
    col[j] = (kj == ~0ull || rank < extra) ? 1 : 0;
  }
  __syncthreads();
  // rows of the image as one flat run of H*W bytes: 16-byte stores between an unaligned head and tail
  const size_t n = size_t(H) * W;
  uint8_t* img = out + size_t(b) * n;
  const size_t head = min(size_t((16 - (reinterpret_cast<uintptr_t>(img) & 15)) & 15), n);
  const size_t nvec = (n - head) / 16;
  for (size_t e = threadIdx.x; e < head; e += kMaskThreads) img[e] = col[e % W];
  for (size_t q = threadIdx.x; q < nvec; q += kMaskThreads) {
    const size_t p0 = head + 16 * q;
    int j = int(p0 % W);
    unsigned w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      unsigned v = 0;
#pragma unroll
      for (int x = 0; x < 4; ++x) {
        v |= unsigned(col[j]) << (8 * x);
        if (++j == W) j = 0;
      }
      w[k] = v;
    }
    reinterpret_cast<uint4*>(img + p0)[0] = make_uint4(w[0], w[1], w[2], w[3]);
  }
  for (size_t e = head + 16 * nvec + threadIdx.x; e < n; e += kMaskThreads) img[e] = col[e % W];
}

// ---------------------------------------------------------------- golden-angle radial masks: one CTA per image
// Lines are drawn in order because the stopping rule reads the sampled count after every line.  The image is a bitmap in
// dynamic shared memory (one spare zero word past the end for the two-word reads of the write-out); a point sets its bit
// with atomicOr and is new when the old word lacked the bit, so a line's new pixels are counted exactly whatever the order
// of its points, and a pixel two t of one line round to is counted once.  sin / cos of kRadialThreads consecutive lines are
// computed together (one line per thread) into a table, instead of by every thread for every line: the FP64 pipe then does
// one sincos per line, and the table costs one extra barrier per kRadialThreads lines.
constexpr int kRadialThreads = 512;
constexpr int kRadialWarps = kRadialThreads / 32;
constexpr int kRadialPoints = 3;        // points per thread and line: 2R + 1 = 1453 <= 3 * 512 at 1024x1024 (R = 726)
__host__ __device__ constexpr size_t radial_smem_bytes(int H, int W) {
  return (size_t(H) * W / 32 + 2) * sizeof(unsigned);
}

__global__ void __launch_bounds__(kRadialThreads) radial_mask_kernel(const double* frac, int frac_stride,
                                                                     const unsigned long long* seeds, uint8_t* out,
                                                                     int* lines_out, int H, int W) {
  extern __shared__ unsigned radial_bits[];
  __shared__ double2 sc[kRadialThreads];                  // (sin, cos) of lines n0 .. n0 + kRadialThreads - 1
  __shared__ int warp_new[2][kRadialWarps];               // new pixels per warp, double-buffered by line parity
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_words = int(radial_smem_bytes(H, W) / sizeof(unsigned));
  for (int w = tid; w < n_words; w += kRadialThreads) radial_bits[w] = 0u;
  constexpr double kGolden = 0x1.f10d6bc8e0e35p+0;       // pi (sqrt 5 - 1) / 2 as NumPy computes it in float64
  const double phi = seeds ? __dmul_rn(double(philox4x32_10(make_uint4(0u, 2u, 0u, 0u), seed_key(seeds[b])).x),
                                       0x1.921fb54442d18p-31)      // pi * 2^-32: phi in [0, pi)
                           : 0.0;
  const double target = __dmul_rn(__dmul_rn(frac[size_t(b) * frac_stride], double(H)), double(W));   // NaN: no line
  const int s2 = H * H + W * W;
  int r = int(sqrt(double(s2)) * 0.5);                     // never above the smallest r with 4 r^2 >= s2
  while (4 * r * r < s2) ++r;
  const int R = r + 1, cap = 8 * max(H, W);
  const double cy = double(H / 2), cx = double(W / 2);
  double tv[kRadialPoints];                                // this thread's t: tid - R + k * kRadialThreads <= R
  int npts = 0;
#pragma unroll
  for (int k = 0; k < kRadialPoints; ++k) {
    tv[k] = double(tid - R + k * kRadialThreads);
    npts += tid - R + k * kRadialThreads <= R;
  }
  __syncthreads();                                         // the bitmap is zeroed
  int count = 0, n = 0;
  while (n < cap && double(count) < target) {             // the same values in every thread: a uniform loop
    if ((n & (kRadialThreads - 1)) == 0) {                 // the old table was last read before the previous barrier
      double s, c;
      sincos(__dadd_rn(__dmul_rn(double(n + tid), kGolden), phi), &s, &c);
      sc[tid] = make_double2(s, c);
      __syncthreads();
    }
    const double2 l = sc[n & (kRadialThreads - 1)];
    int fresh = 0;
#pragma unroll
    for (int k = 0; k < kRadialPoints; ++k) {
      // __double2int_rn is rint (half to even) and the conversion to int in one instruction (|value| < 2^11)
      const int y = __double2int_rn(__dadd_rn(cy, __dmul_rn(tv[k], l.x)));
      const int x = __double2int_rn(__dadd_rn(cx, __dmul_rn(tv[k], l.y)));
      if (k < npts && unsigned(y) < unsigned(H) && unsigned(x) < unsigned(W)) {
        const unsigned p = unsigned(y) * unsigned(W) + unsigned(x), bit = 1u << (p & 31);
        fresh += (atomicOr(&radial_bits[p >> 5], bit) & bit) == 0u;
      }
    }
    fresh = __reduce_add_sync(0xFFFFFFFFu, fresh);
    if (lane == 0) warp_new[n & 1][warp] = fresh;          // this slot was last read before the previous line's barrier
    __syncthreads();
#pragma unroll
    for (int w = 0; w < kRadialWarps; ++w) count += warp_new[n & 1][w];
    ++n;
  }
  if (lines_out && tid == 0) lines_out[b] = n;
  // the last barrier (the last line's, or the one after zeroing) orders every atomicOr before these reads.  Rows of the
  // image as one flat run of H*W bytes: 16-byte stores between an unaligned head and tail
  const size_t npx = size_t(H) * W;
  uint8_t* img = out + size_t(b) * npx;
  const size_t head = min(size_t((16 - (reinterpret_cast<uintptr_t>(img) & 15)) & 15), npx);
  const size_t nvec = (npx - head) / 16;
  for (size_t e = tid; e < head; e += kRadialThreads) img[e] = (radial_bits[e >> 5] >> (e & 31)) & 1u;
  for (size_t q = tid; q < nvec; q += kRadialThreads) {
    const size_t p0 = head + 16 * q;
    const unsigned w0 = radial_bits[p0 >> 5], w1 = radial_bits[(p0 >> 5) + 1];
    const unsigned bits = __funnelshift_r(w0, w1, unsigned(p0 & 31));   // pixels p0 .. p0 + 15 in the low 16 bits
    unsigned v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = (((bits >> (4 * k)) & 0xFu) * 0x00204081u) & 0x01010101u;   // 4 bits -> 4 bytes
    reinterpret_cast<uint4*>(img + p0)[0] = make_uint4(v[0], v[1], v[2], v[3]);
  }
  for (size_t e = head + 16 * nvec + tid; e < npx; e += kRadialThreads) img[e] = (radial_bits[e >> 5] >> (e & 31)) & 1u;
}

// ---------------------------------------------------------------- host side
// Launch `fn(q, nb)` over batch chunks of at most 65535 images (grid.y limit), q's pointers advanced to the chunk.
template <typename F>
static void for_batch_chunks(const SimParams& p, int B, F&& fn) {
  for (int b0 = 0; b0 < B; b0 += 65535) {
    SimParams q = p;
    const size_t off = size_t(b0) * p.H * p.W;
    q.gt += size_t(b0) * p.gt_bstride;
    q.mask += size_t(b0) * p.mask_bstride;
    q.sigma += size_t(b0) * p.sigma_stride;
    q.seeds += b0;
    q.y0 += off;
    q.x0 += off;
    if (q.aty0) q.aty0 += off;
    fn(q, (B - b0 < 65535) ? (B - b0) : 65535);
  }
}

template <int N> static void sim_launch_rows_fwd(const SimParams& p, int B, cudaStream_t st) {
  constexpr int G = FftPlan<N>::G;
  const size_t smem = size_t(8) * G * fft_pitch(N) * sizeof(float2);
  for_batch_chunks(p, B, [&](const SimParams& q, int nb) {
    sim_rows_fwd_kernel<N><<<dim3((p.H + 8 * G - 1) / (8 * G), nb), 256, smem, st>>>(q);
  });
}
template <int N> static void sim_launch_rows_inv(const SimParams& p, int B, cudaStream_t st) {
  constexpr int G = FftPlan<N>::G;
  const size_t smem = size_t(8) * G * fft_pitch(N) * sizeof(float2);
  for_batch_chunks(p, B, [&](const SimParams& q, int nb) {
    sim_rows_inv_kernel<N><<<dim3((p.H + 8 * G - 1) / (8 * G), nb), 256, smem, st>>>(q);
  });
}
template <int N> static void sim_launch_cols(const SimParams& p, int B, cudaStream_t st) {
  constexpr int G = FftPlan<N>::G;
  constexpr int P = fft_pitch(N) + ((fft_pitch(N) % 16 == 0) ? 4 : 0);
  const size_t smem = size_t(8) * G * P * sizeof(float2);
  for_batch_chunks(p, B, [&](const SimParams& q, int nb) {
    sim_cols_kernel<N><<<dim3((p.W + 8 * G - 1) / (8 * G), nb), 256, smem, st>>>(q);
  });
}

template <int PASS> static int sim_launch_any(const SimParams& p, int B, cudaStream_t st) {
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(sim_any_kernel<PASS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         int(any_smem_bytes(kAnyMaxN)));
    if (e != cudaSuccess) return int(e);
    attr_done = true;
  }
  const int N = (PASS != 1) ? p.W : p.H, nlines = (PASS != 1) ? p.H : p.W;
  for_batch_chunks(p, B, [&](const SimParams& q, int nb) {
    sim_any_kernel<PASS><<<dim3((nlines + kAnyLines - 1) / kAnyLines, nb), kAnyThreads, any_smem_bytes(N), st>>>(q);
  });
  return int(cudaGetLastError());
}

#define SIM_DISPATCH_N(n, fn, ...)                     \
  switch (n) {                                         \
    case 32: fn<32>(__VA_ARGS__); break;               \
    case 64: fn<64>(__VA_ARGS__); break;               \
    case 128: fn<128>(__VA_ARGS__); break;             \
    case 256: fn<256>(__VA_ARGS__); break;             \
    default: fn<512>(__VA_ARGS__); break;              \
  }

int simulate_measurements(const float* gt, long long gt_bstride, const uint8_t* mask, long long mask_bstride,
                          const float* sigma, int sigma_stride, const unsigned long long* seeds, float2* y0, float2* x0,
                          float2* aty0, int B, int H, int W, cudaStream_t st) {
  if (!any_shape_supported(H, W)) return -2;
  SimParams p{H, W, gt, gt_bstride, mask, mask_bstride, sigma, sigma_stride, seeds, y0, x0, aty0, 0.f, 0};
  if (!fft_shape_supported(H, W)) {
    int rc = sim_launch_any<0>(p, B, st);
    if (rc == 0) rc = sim_launch_any<1>(p, B, st);
    if (rc == 0) rc = sim_launch_any<2>(p, B, st);
    return rc;
  }
  p.kscale = ((((H + W) / 2) & 1) ? -1.f : 1.f) / sqrtf(float(H) * float(W));
  p.gt_vec4 = (reinterpret_cast<uintptr_t>(gt) % 16 == 0) && (gt_bstride % 4 == 0);
  SIM_DISPATCH_N(W, sim_launch_rows_fwd, p, B, st);
  SIM_DISPATCH_N(H, sim_launch_cols, p, B, st);
  SIM_DISPATCH_N(W, sim_launch_rows_inv, p, B, st);
  return int(cudaGetLastError());
}

int cartesian_masks(const int* accel, int accel_stride, const unsigned long long* seeds, int acs_cols, uint8_t* mask,
                    int B, int H, int W, cudaStream_t st) {
  if (!any_shape_supported(H, W)) return -2;
  cartesian_mask_kernel<<<B, kMaskThreads, 0, st>>>(accel, accel_stride, seeds, acs_cols, mask, H, W);
  return int(cudaGetLastError());
}

int radial_masks(const double* frac, int frac_stride, const unsigned long long* seeds, uint8_t* mask, int* lines_out,
                 int B, int H, int W, cudaStream_t st) {
  if (!any_shape_supported(H, W)) return -2;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(radial_mask_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         int(radial_smem_bytes(kAnyMaxN, kAnyMaxN)));
    if (e != cudaSuccess) return int(e);
    attr_done = true;
  }
  radial_mask_kernel<<<B, kRadialThreads, radial_smem_bytes(H, W), st>>>(frac, frac_stride, seeds, mask, lines_out, H, W);
  return int(cudaGetLastError());
}

#undef SIM_DISPATCH_N

}  // namespace pnp
