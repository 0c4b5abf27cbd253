// Measurement simulator: undersampled, noisy k-space measurements of fully-sampled images, and seeded Cartesian, radial and
// variable-density masks (pnp_simulate_measurements / pnp_cartesian_masks / pnp_radial_masks / pnp_variable_density_masks;
// the definitions are in include/pnp_b200.h).  Per image b:
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
// with D[i,j] = (-1)^(i+j), s = (-1)^((H+W)/2) as in fftprox.cu.  The passes are ops on the line passes of
// line_passes.cuh: powers of two in 32..512 take the radix passes (SimRowsFwd, SimCols, SimRowsInv); every other H, W in
// 2..1024 takes the dense-DFT pass (SimAnyRowsFwd, SimAnyCols, SimAnyRowsInv), which computes the centred transforms
// directly.  The noise of a sample depends only on (seed, H, W, i, j), never on the mask or the batch
// position, and nothing is accumulated across CTAs, so every output is bitwise reproducible.
#pragma once
#include "common.cuh"
#include "fft_core.cuh"
#include "line_passes.cuh"

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

// ---------------------------------------------------------------- ops of the three line passes (line_passes.cuh)
// Column passes: K -> y0 at k-space sample (i, j), stored; the y0 the second transform starts from.
struct SimSampleOp : LineOp {
  static constexpr bool kMiddle = true;
  const uint8_t* mask;          // [B or 1, H, W]
  long long mask_bstride;
  const float* sigma;           // sigma_n[b * sigma_stride]
  int sigma_stride;
  const unsigned long long* seeds;   // [B]
  float2* y0;                   // [B, H, W]
  int W;
  struct Mid {
    float sig;
    uint2 key;
    const uint8_t* mk;
  };
  __device__ Mid middle_begin(int b) const {
    return {sigma[size_t(b) * sigma_stride] * (1.f / 255.f), seed_key(seeds[b]), mask + size_t(b) * mask_bstride};
  }
  __device__ float2 sample(const Mid& m, const LineElem& e, float2 K) const {
    const float2 y = measure_sample(K, m.mk[e.o] != 0, e.i, e.j, W, m.sig, m.key);
    y0[e.g] = y;
    return y;
  }
};

// radix path (H, W powers of two in 32..512).  Pass 1: D.gt -> row FFTs -> T.
struct SimRowsFwd : LineOp {
  template <int N> static constexpr int kRowCtas = N == 128 ? 8 : 0;   // left alone, ptxas spills at N = 128
  const float* gt;              // [B or 1, H, W]
  long long gt_bstride;         // H*W, or 0 for one shared gt
  float2* t;                    // x0
  int gt_vec4;                  // every image's gt is 16-byte aligned
  // float4 loads: a warp's G rows are G*N contiguous floats
  template <int N> __device__ bool load_rows(float2* rows, int b, int row0, int lane) const {
    if (!gt_vec4) return false;
    constexpr int G = FftPlan<N>::G, P = fft_pitch(N);
    const float* g = gt + size_t(b) * gt_bstride + size_t(row0) * N;
    for (int q = lane; q < G * N / 4; q += 32) {
      const float4 v = reinterpret_cast<const float4*>(g)[q];
      const int r = (4 * q) / N, j = (4 * q) % N;
      const float s = ((row0 + r) & 1) ? -1.f : 1.f;     // D at the even column j
      float2* d = rows + r * P;
      d[fpad(j)] = make_float2(s * v.x, 0.f);
      d[fpad(j + 1)] = make_float2(-s * v.y, 0.f);
      d[fpad(j + 2)] = make_float2(s * v.z, 0.f);
      d[fpad(j + 3)] = make_float2(-s * v.w, 0.f);
    }
    return true;
  }
  __device__ float2 load(const LineElem& e) const {
    const float v = gt[size_t(e.b) * gt_bstride + e.o];
    return make_float2(((e.i + e.j) & 1) ? -v : v, 0.f);
  }
  __device__ void store(const LineElem& e, float2 v, Pre) const { t[e.g] = v; }
};

// Pass 2: columns of T -> col FFT -> K = s.D / sqrt(HW) -> y0 -> conj(D.y0) -> col FFT -> T.
struct SimCols : SimSampleOp {
  float2* t;
  float kscale;                 // s / sqrt(HW)
  __device__ float2 load(const LineElem& e) const { return t[e.g]; }
  __device__ float2 middle(const Mid& m, const LineElem& e, float2 Z) const {
    const float d = ((e.i + e.j) & 1) ? -kscale : kscale;
    const float2 y = sample(m, e, make_float2(Z.x * d, Z.y * d));
    const float dy = ((e.i + e.j) & 1) ? -1.f : 1.f;
    return make_float2(dy * y.x, -dy * y.y);   // conj(D.y0): forward FFT == inverse
  }
  __device__ void store(const LineElem& e, float2 v, Pre) const { t[e.g] = v; }
};

// Pass 3: T -> row FFTs -> ATy0 = s.D.conj(.) / sqrt(HW) -> x0 = max(ATy0, 0) (and ATy0).
struct SimRowsInv : LineOp {
  float2* x0;                   // [B, H, W]; holds T between the passes
  float2* aty0;                 // [B, H, W] or null
  float kscale;
  __device__ float2 load(const LineElem& e) const { return x0[e.g]; }
  __device__ void store(const LineElem& e, float2 v, Pre) const {
    const float d = ((e.i + e.j) & 1) ? -kscale : kscale;
    const float2 a = make_float2(v.x * d, -v.y * d);
    if (aty0) aty0[e.g] = a;
    x0[e.g] = make_float2(fmaxf(a.x, 0.f), fmaxf(a.y, 0.f));
  }
};

// dense-DFT path (every other H, W in 2..1024): gt rows -> fft_c along rows -> T; columns of T -> fft_c -> y0 -> ifft_c
// -> T; rows of T -> ifft_c along rows -> x0, ATy0.
struct SimAnyRowsFwd : LineOp {
  static constexpr bool kRows = true;
  const float* gt;
  long long gt_bstride;
  float2* t;
  __device__ bool inverse() const { return false; }
  __device__ float scale(int N) const { return rsqrtf(float(N)); }
  __device__ float2 load(const LineElem& e) const { return make_float2(gt[size_t(e.b) * gt_bstride + e.o], 0.f); }
  __device__ void store(const LineElem& e, float2 v, Pre) const { t[e.g] = v; }
};

struct SimAnyCols : SimSampleOp {
  static constexpr bool kRows = false;
  float2* t;
  __device__ bool inverse() const { return false; }
  __device__ float scale(int N) const { return rsqrtf(float(N)); }
  __device__ float2 load(const LineElem& e) const { return t[e.g]; }
  __device__ float2 middle(const Mid& m, const LineElem& e, float2 K) const { return sample(m, e, K); }
  __device__ void store(const LineElem& e, float2 v, Pre) const { t[e.g] = v; }
};

struct SimAnyRowsInv : LineOp {
  static constexpr bool kRows = true;
  float2* x0;
  float2* aty0;
  __device__ bool inverse() const { return true; }
  __device__ float scale(int N) const { return rsqrtf(float(N)); }
  __device__ float2 load(const LineElem& e) const { return x0[e.g]; }
  __device__ void store(const LineElem& e, float2 v, Pre) const {
    if (aty0) aty0[e.g] = v;
    x0[e.g] = make_float2(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f));
  }
};

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

// ---------------------------------------------------------------- variable-density random masks: one cluster per image
// Image b's mask is the ACS block plus the `extra` non-ACS pixels with the smallest 51-bit words (float_bits(key) << 20 | p):
// keys are positive floats, which order like their bits, and p < 2^20, so the integer order is the (key, p) order and the
// extra-th smallest word is a unique threshold.  It is found by radix selection over the cluster, 11 bits at a time
// (digits 50..40, 39..29, 28..18, 17..7, 6..0).  Each CTA owns a slice of `slice` consecutive pixels (a multiple of 32) and
// keeps its part of the mask as a bitmap in shared memory.  A pass counts the digit of the words whose higher bits equal the
// prefix P chosen so far into a shared histogram; one cluster barrier later every CTA sums the cluster's histograms
// through DSMEM (double-buffered by pass parity, so one barrier per pass) and picks the same bin and remaining rank.  The
// selection stops as soon as the chosen bin holds exactly the remaining rank; then a word is sampled iff (word >> L) <= P.
// A pass either recomputes the keys of the whole slice (and sets the bitmap bits of the words already below the prefix) or,
// once they fit, reads the slice's words of the current bin from a candidate list in shared memory: the recompute pass
// after which a CTA's share of the chosen bin is at most `cap` also writes that list.  Small slices fit from the first
// pass; large ones take two key computations per pixel and then passes over the list (an 11-bit bin of positive floats
// holds at most 1/8 of the slice in expectation, so cap >= slice / 8 is almost always enough; if not, a CTA recomputes
// once more, with the same code).  The key path uses only __dadd_rn / __dsub_rn / __dmul_rn / __ddiv_rn / __dsqrt_rn /
// __double2float_rn, so it is bit for bit the definition's, and integer counts make every mask independent of the cluster
// size and the batch position.
constexpr int kVdThreads = 512;
constexpr int kVdWarps = kVdThreads / 32;
constexpr int kVdDigit = 11;
constexpr int kVdBins = 1 << kVdDigit;                   // 4 per thread in the scan
constexpr int kVdMaxSlice = 131072;                      // pixels per CTA at most: 1024^2 on an 8-CTA cluster
__host__ __device__ constexpr size_t vd_bitmap_offset(int H, int W) {
  return 2 * kVdBins * sizeof(unsigned) + size_t(H + W) * sizeof(double);
}
__host__ __device__ constexpr size_t vd_cand_offset(int H, int W, int slice) {
  return (vd_bitmap_offset(H, W) + (size_t(slice) / 32 + 1) * sizeof(unsigned) + 7) / 8 * 8;
}
__host__ __device__ constexpr size_t vd_smem_bytes(int H, int W, int slice, int cap) {
  return vd_cand_offset(H, W, slice) + size_t(cap) * sizeof(unsigned long long);
}

__device__ __forceinline__ uint4 ld_dsmem_v4(const void* local, unsigned rank) {
  uint32_t a;
  uint4 v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(a) : "r"(smem_u32(local)), "r"(rank));
  asm volatile("ld.shared::cluster.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a)
               : "memory");
  return v;
}

// key = float32(u / w) at pixel p = i*W + j, with ky2 = ky*ky and kx2 = kx*kx of its row and column (definition in
// include/pnp_b200.h): every operation rounded on its own, no FMA.
__device__ __forceinline__ float vd_key(double ky2, double kx2, int power, unsigned p, uint2 seed_k) {
  const double r = __dsqrt_rn(__dmul_rn(0.5, __dadd_rn(ky2, kx2)));
  const double q = __dsub_rn(1.0, r);
  double w = 1.0;
  for (int k = 0; k < power; ++k) w = __dmul_rn(w, q);
  const unsigned w0 = philox4x32_10(make_uint4(p, 3u, 0u, 0u), seed_k).x;
  const double u = __dmul_rn(__dadd_rn(double(w0), 0.5), 0x1p-32);
  return __double2float_rn(__ddiv_rn(u, w));                // w = 0: +inf
}

__global__ void __launch_bounds__(kVdThreads) vd_mask_kernel(const int* accel, int accel_stride,
                                                             const unsigned long long* seeds, int acs_h, int acs_w,
                                                             int power, uint8_t* out, int H, int W, int slice, int cap) {
  extern __shared__ __align__(16) unsigned char vd_smem[];
  unsigned* hist = reinterpret_cast<unsigned*>(vd_smem);                      // [2][kVdBins], by pass parity
  double* sq = reinterpret_cast<double*>(vd_smem + 2 * kVdBins * sizeof(unsigned));   // ky^2 of the rows, kx^2 of the columns
  unsigned* bm = reinterpret_cast<unsigned*>(vd_smem + vd_bitmap_offset(H, W));      // the slice's mask, bit e = pixel s0 + e
  unsigned long long* cand = reinterpret_cast<unsigned long long*>(vd_smem + vd_cand_offset(H, W, slice));
  __shared__ unsigned warp_total[kVdWarps];
  __shared__ unsigned chosen[4];                           // bin, rank left in it, its population: cluster, this CTA
  __shared__ unsigned n_cand;
  unsigned cs, crank;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(cs));
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(crank));
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.x / int(cs);
  const int HW = H * W;
  const int s0 = min(HW, int(crank) * slice), s1 = min(HW, s0 + slice);
  const int nq = (s1 - s0 + 31) >> 5;                      // 32-pixel groups of the slice: bitmap words
  const int cy = H / 2, cx = W / 2, r0 = cy - acs_h / 2, c0 = cx - acs_w / 2;
  const int a = accel[size_t(b) * accel_stride];
  const int n_keep = a >= 1 ? max(1, HW / a) : HW;
  const int n_acs = acs_h * acs_w;
  const int extra = max(0, n_keep - n_acs);
  const uint2 seed_k = seed_key(seeds[b]);
  for (int t = tid; t < H + W; t += kVdThreads) {
    const int c = t < H ? cy : cx;
    const double k = __ddiv_rn(double((t < H ? t : t - H) - c), double(c));
    sq[t] = __dmul_rn(k, k);
  }
  if (tid == 0) n_cand = 0u;
  __syncthreads();

  // bits of group q (32 consecutive pixels of the slice, one group per thread): the ACS pixels, and each other pixel for
  // which take(word) holds (take is not called when keys = false)
  auto group = [&](int q, bool keys, auto&& take) -> unsigned {
    int p = s0 + (q << 5);
    int i = p / W, j = p - i * W;
    const int n = min(32, s1 - p);
    unsigned bits = 0u;
    for (int e = 0; e < n; ++e, ++p) {
      if (unsigned(i - r0) < unsigned(acs_h) && unsigned(j - c0) < unsigned(acs_w)) {
        bits |= 1u << e;
      } else if (keys) {
        const float key = vd_key(sq[i], sq[H + j], power, unsigned(p), seed_k);
        if (take((static_cast<unsigned long long>(__float_as_uint(key)) << 20) | unsigned(p))) bits |= 1u << e;
      }
      if (++j == W) { j = 0; ++i; }
    }
    return bits;
  };
  auto mark = [&](unsigned long long w) {                 // a listed word is sampled
    const unsigned e = unsigned(w & 0xFFFFFu) - unsigned(s0);
    atomicOr(&bm[e >> 5], 1u << (e & 31));
  };

  const bool all = extra == HW - n_acs;                    // every pixel is sampled (accel <= 1)
  const bool select = extra != 0 && !all;                  // the same in every CTA of the cluster
  if (!select) {                                           // no key, no DSMEM access
    for (int q = tid; q < nq; q += kVdThreads) {
      const unsigned bits = group(q, false, [](unsigned long long) { return false; });
      const int n = min(32, s1 - s0 - (q << 5));
      bm[q] = all ? (n == 32 ? ~0u : (1u << n) - 1u) : bits;
    }
  } else {
    int L = 51;                                            // the words in play have (w >> L) == P
    unsigned long long P = 0ull;
    unsigned k = unsigned(extra);                          // rank of the threshold among them
    bool listed = false;                                   // cand[] holds this CTA's words in play
    bool collect = s1 - s0 <= cap;                         // this pass writes cand[]
    for (int pass = 0;; ++pass) {
      unsigned* h = hist + (pass & 1) * kVdBins;           // peers last read this buffer before the previous barrier
      for (int d = tid; d < kVdBins; d += kVdThreads) h[d] = 0u;
      __syncthreads();
      const int Ln = max(L - kVdDigit, 0);
      const unsigned dmask = (1u << (L - Ln)) - 1u;
      if (listed) {
        for (unsigned c = tid; c < n_cand; c += kVdThreads) {
          const unsigned long long w = cand[c], t = w >> L;
          if (t < P) mark(w);
          else if (t == P) atomicAdd(&h[unsigned(w >> Ln) & dmask], 1u);
        }
      } else {
        for (int q = tid; q < nq; q += kVdThreads) {
          bm[q] = group(q, true, [&](unsigned long long w) {
            const unsigned long long t = w >> L;
            if (t == P) {
              atomicAdd(&h[unsigned(w >> Ln) & dmask], 1u);
              if (collect) {                               // warp-aggregated append
                const unsigned act = __activemask();
                const int leader = __ffs(act) - 1;
                unsigned base = 0u;
                if (lane == leader) base = atomicAdd(&n_cand, unsigned(__popc(act)));
                base = __shfl_sync(act, base, leader);
                cand[base + __popc(act & ((1u << lane) - 1u))] = w;
              }
            }
            return t < P;
          });
        }
      }
      asm volatile("barrier.cluster.arrive.release;\n\tbarrier.cluster.wait.acquire;" ::: "memory");
      // bins 4 tid .. 4 tid + 3 summed over the cluster; a block scan finds the bin that holds rank k
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      for (unsigned r = 0; r < cs; ++r) {
        const uint4 x = ld_dsmem_v4(h + 4 * tid, r);
        v = make_uint4(v.x + x.x, v.y + x.y, v.z + x.z, v.w + x.w);
      }
      const unsigned s = v.x + v.y + v.z + v.w;
      unsigned incl = s;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned y = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += y;
      }
      if (lane == 31) warp_total[warp] = incl;
      __syncthreads();
      unsigned before = incl - s;
      for (int w2 = 0; w2 < warp; ++w2) before += warp_total[w2];
      if (before < k && k <= before + s) {
        const unsigned c4[4] = {v.x, v.y, v.z, v.w};
        for (int m = 0; m < 4; ++m) {
          if (k <= before + c4[m]) {
            chosen[0] = unsigned(4 * tid + m);
            chosen[1] = k - before;
            chosen[2] = c4[m];
            chosen[3] = h[4 * tid + m];
            break;
          }
          before += c4[m];
        }
      }
      __syncthreads();
      P = (P << (L - Ln)) | chosen[0];
      L = Ln;
      k = chosen[1];
      listed |= collect;
      collect = !listed && chosen[3] <= unsigned(cap);
      if (chosen[2] == k || L == 0) break;                 // the whole bin is sampled (at L = 0 it holds one word)
    }
    asm volatile("barrier.cluster.arrive.release;" ::: "memory");    // the last DSMEM reads are done
    if (listed) {
      for (unsigned c = tid; c < n_cand; c += kVdThreads)
        if ((cand[c] >> L) <= P) mark(cand[c]);
    } else {
      for (int q = tid; q < nq; q += kVdThreads)
        bm[q] = group(q, true, [&](unsigned long long w) { return (w >> L) <= P; });
    }
  }
  __syncthreads();
  // the slice as one flat run of bytes: 16-byte stores between an unaligned head and tail (bits from two bitmap words)
  const int n = s1 - s0;
  uint8_t* img = out + size_t(b) * HW + s0;
  const int head = min(int((16 - (reinterpret_cast<uintptr_t>(img) & 15)) & 15), n);
  const int nvec = (n - head) / 16;
  for (int e = tid; e < head; e += kVdThreads) img[e] = (bm[e >> 5] >> (e & 31)) & 1u;
  for (int q = tid; q < nvec; q += kVdThreads) {
    const int p0 = head + 16 * q;
    const unsigned bits = __funnelshift_r(bm[p0 >> 5], bm[(p0 >> 5) + 1], unsigned(p0 & 31));
    unsigned v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = (((bits >> (4 * k)) & 0xFu) * 0x00204081u) & 0x01010101u;   // 4 bits -> 4 bytes
    reinterpret_cast<uint4*>(img + p0)[0] = make_uint4(v[0], v[1], v[2], v[3]);
  }
  for (int e = head + 16 * nvec + tid; e < n; e += kVdThreads) img[e] = (bm[e >> 5] >> (e & 31)) & 1u;
  if (select) asm volatile("barrier.cluster.wait.acquire;" ::: "memory");   // no peer reads this CTA's histograms any more
}

// ---------------------------------------------------------------- host side
int simulate_measurements(const float* gt, long long gt_bstride, const uint8_t* mask, long long mask_bstride,
                          const float* sigma, int sigma_stride, const unsigned long long* seeds, float2* y0, float2* x0,
                          float2* aty0, int B, int H, int W, cudaStream_t st) {
  if (!any_shape_supported(H, W)) return -2;
  const SimSampleOp smp{{}, mask, mask_bstride, sigma, sigma_stride, seeds, y0, W};
  if (!fft_shape_supported(H, W)) {
    int rc = dense_lines(SimAnyRowsFwd{{}, gt, gt_bstride, x0}, H, W, B, st);
    if (rc == 0) rc = dense_lines(SimAnyCols{smp, x0}, H, W, B, st);
    if (rc == 0) rc = dense_lines(SimAnyRowsInv{{}, x0, aty0}, H, W, B, st);
    return rc;
  }
  const float kscale = centre_sign(H, W) / sqrtf(float(H) * float(W));
  const int gt_vec4 = (reinterpret_cast<uintptr_t>(gt) % 16 == 0) && (gt_bstride % 4 == 0);
  int rc = radix_rows(SimRowsFwd{{}, gt, gt_bstride, x0, gt_vec4}, H, W, B, st);
  if (rc == 0) rc = radix_cols(SimCols{smp, x0, kscale}, H, W, B, st);
  if (rc == 0) rc = radix_rows(SimRowsInv{{}, x0, aty0, kscale}, H, W, B, st);
  return rc;
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

// Cluster size: enough CTAs that a slice is at most kVdMaxSlice pixels (8 at 1024^2), then more (up to 16, a non-portable
// size) while the batch leaves SMs idle and slices keep >= 4096 pixels; the masks do not depend on it.  The candidate list
// holds max(slice / 8, slice up to 4096) words.
int variable_density_masks(const int* accel, int accel_stride, const unsigned long long* seeds, int acs_h, int acs_w,
                           int power, uint8_t* mask, int B, int H, int W, cudaStream_t st) {
  if (!any_shape_supported(H, W)) return -2;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(vd_mask_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         int(vd_smem_bytes(kAnyMaxN, kAnyMaxN, kVdMaxSlice, kVdMaxSlice / 8)));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(vd_mask_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess) return int(e);
    attr_done = true;
  }
  const int hw = H * W;
  int cs = 1;
  while (cs < 16 && ((hw + cs - 1) / cs > kVdMaxSlice || ((long long)B * cs < num_sms() && hw / (2 * cs) >= 4096))) cs *= 2;
  const int slice = ((hw + cs - 1) / cs + 31) / 32 * 32;
  const int cap = max(slice / 8, min(slice, 4096));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(unsigned(B) * unsigned(cs));
  cfg.blockDim = dim3(kVdThreads);
  cfg.dynamicSmemBytes = vd_smem_bytes(H, W, slice, cap);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = unsigned(cs);
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return int(cudaLaunchKernelEx(&cfg, vd_mask_kernel, accel, accel_stride, seeds, acs_h, acs_w, power, mask, H, W, slice,
                                cap));
}

}  // namespace pnp
