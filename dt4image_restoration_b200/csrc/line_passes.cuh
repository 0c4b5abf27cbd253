// Line passes of the three-launch 2-D transforms: the general prox path and pnp_fft2c (fftprox.cu, fftprox_any.cuh),
// prox_prepare's Yt and the measurement simulator (measure.cuh).  Included by fftprox.cu after g_tw512.
//
// A pass transforms every row (or every column) of each image of a batch.  Each pass is written once per transform core
// - the radix row and column passes on fft_warp_rows (powers of two 32..512) and the dense pass on any_dft_lines (any
// length 2..1024) - as a kernel template over a per-caller op type, which supplies the loads, the stores and, for a column
// pass, a pointwise middle step followed by a second transform.  The op is a compile-time type: nothing branches at run
// time on which caller a kernel serves, and the kernel name says which pass ran (radix_rows_kernel<256, SimRowsFwd>).
// Every pass loads its whole lines into shared memory before it stores the same lines, so an op may store into the buffer
// it loads from (pnp_fft2c with dst == src; the simulator keeps T in x0).
//
// An op derives from LineOp and hides the members it replaces:
//   float2 load(const LineElem& e)                         input element e of the pass
//   void   store(const LineElem& e, float2 v, Pre pre)     v: the transformed element; pre: what preload(e) fetched
//   Pre    preload(const LineElem& e)                      loads the radix row pass issues KB elements ahead of the stores
//   bool   skip()                                          true: the launch does nothing (device flag, read first)
//   bool   image_active(int b)                             false: image b's stores are left out
//   bool   load_rows<N>(rows, b, row0, lane)               radix rows: fill the warp's rows itself and return true
//   kRowCtas<N>                                            radix rows: resident CTAs per SM asked of ptxas (0: its choice)
//   kMiddle, Mid middle_begin(int b), float2 middle(const Mid&, const LineElem&, float2 Z)
//                                                          column passes: Z -> the second transform's input
//   dense passes also: kRows (a line is an image row), bool inverse() (direction of the first transform), float scale(N)
#pragma once
#include <type_traits>
#include "common.cuh"
#include "fft_core.cuh"

namespace pnp {

// Element (i, j) of image b; o = i*W + j inside the image, g = b*H*W + o in the batch.
struct LineElem {
  int b, i, j;
  size_t o, g;
};

struct LineOp {
  static constexpr bool kMiddle = false;
  struct Pre {};
  __device__ bool skip() const { return false; }
  __device__ bool image_active(int) const { return true; }
  __device__ Pre preload(const LineElem&) const { return {}; }
  template <int N> __device__ bool load_rows(float2*, int, int, int) const { return false; }
  template <int N> static constexpr int kRowCtas = 0;
};

// s = (-1)^((H+W)/2): the centred transforms of even sizes are s.D.FFT2(D.w)/sqrt(HW), D[i,j] = (-1)^(i+j) (fftprox.cu)
inline float centre_sign(int H, int W) { return (((H + W) / 2) & 1) ? -1.f : 1.f; }

// Runs `kernel` on B images in slices of at most 65535 (the grid.y limit); image b0 + blockIdx.y is the CTA's.
template <class Op>
static int launch_lines(void (*kernel)(Op, int, int, int), const Op& op, int H, int W, int B, int nx, int threads,
                        size_t smem, cudaStream_t st) {
  for (int b0 = 0; b0 < B; b0 += 65535)
    kernel<<<dim3(nx, (B - b0 < 65535) ? (B - b0) : 65535), threads, smem, st>>>(op, H, W, b0);
  return int(cudaGetLastError());
}

// f(std::integral_constant<int, N>()) for the power of two n in 32..512
template <class F> static auto with_pow2(int n, F&& f) {
  switch (n) {
    case 32: return f(std::integral_constant<int, 32>());
    case 64: return f(std::integral_constant<int, 64>());
    case 128: return f(std::integral_constant<int, 128>());
    case 256: return f(std::integral_constant<int, 256>());
    default: return f(std::integral_constant<int, 512>());
  }
}

// ---------------------------------------------------------------- radix passes
// Element offsets use the batch row index b*H + i as an int (2^31 rows of at least 32 c64 are 512 GB, more than the
// device holds): a 64-bit image offset held across the transforms costs registers.

// Op::kRowCtas<N> for __launch_bounds__, where nvcc does not take the member template itself
template <int N, class Op> constexpr int row_ctas() { return Op::template kRowCtas<N>; }

// Row pass: N = W, a warp owns G rows, 8 warps a CTA.
template <int N, class Op>
__global__ void __launch_bounds__(256, row_ctas<N, Op>()) radix_rows_kernel(const Op op, int H, int W, int b0) {
  constexpr int G = FftPlan<N>::G;
  constexpr int P = fft_pitch(N);
  if (op.skip()) return;
  __shared__ float2 tw[kTwTotal];
  extern __shared__ float2 rows_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  fft_load_twiddles(tw, g_tw512);
  __syncthreads();
  const int b = b0 + blockIdx.y;
  const int row0 = (blockIdx.x * 8 + warp) * G;
  if (row0 >= H) return;
  float2* mine = rows_smem + warp * G * P;
  if (!op.template load_rows<N>(mine, b, row0, lane)) {
#pragma unroll 1
    for (int g = 0; g < G; ++g) {
      const int i = row0 + g;
      const size_t o = size_t(i) * N, base = size_t(b * H + i) * N;
      for (int j = lane; j < N; j += 32) mine[g * P + fpad(j)] = op.load(LineElem{b, i, j, o + j, base + j});
    }
  }
  __syncwarp();
  fft_warp_rows<N>(mine, P, tw, lane);
  if (!op.image_active(b)) return;
  // preload() is for plain loads that stay behind the preceding stores (the prox epilogue's u may alias u_out), so the
  // loads of KB elements are issued ahead of their stores by hand (load -> store -> load chains cost 25 % in the row-only
  // kernels)
  constexpr int KB = std::is_empty<typename Op::Pre>::value ? 1 : (N / 32 < 4) ? N / 32 : 4;
#pragma unroll 1
  for (int g = 0; g < G; ++g) {
    const int i = row0 + g;
    const size_t o = size_t(i) * N, base = size_t(b * H + i) * N;
    for (int j0 = lane; j0 < N; j0 += 32 * KB) {
      typename Op::Pre pre[KB];
#pragma unroll
      for (int q = 0; q < KB; ++q) {
        const int j = j0 + 32 * q;
        pre[q] = op.preload(LineElem{b, i, j, o + j, base + j});
      }
#pragma unroll
      for (int q = 0; q < KB; ++q) {
        const int j = j0 + 32 * q;
        op.store(LineElem{b, i, j, o + j, base + j}, mine[g * P + fpad(j)], pre[q]);
      }
    }
  }
}

// Column pass: N = H, a CTA owns NCOL = 8*G adjacent columns of one image, so loads and stores walk NCOL contiguous
// elements of a row.
template <int N> __host__ __device__ constexpr int radix_cols_pitch() {
  return fft_pitch(N) + ((fft_pitch(N) % 16 == 0) ? 4 : 0);   // de-conflict the transposed fill
}

template <int N, class Op>
__global__ void __launch_bounds__(256) radix_cols_kernel(const Op op, int H, int W, int b0) {
  constexpr int G = FftPlan<N>::G;
  constexpr int NCOL = 8 * G;
  constexpr int P = radix_cols_pitch<N>();
  if (op.skip()) return;
  __shared__ float2 tw[kTwTotal];
  extern __shared__ float2 cols_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  fft_load_twiddles(tw, g_tw512);
  const int b = b0 + blockIdx.y;
  const int c0 = blockIdx.x * NCOL;
  for (int e = threadIdx.x; e < N * NCOL; e += blockDim.x) {
    const int c = e % NCOL, i = e / NCOL, j = c0 + c;
    const LineElem el{b, i, j, size_t(i) * W + j, size_t(b * N + i) * W + j};
    cols_smem[c * P + fpad(i)] = (j < W) ? op.load(el) : make_float2(0.f, 0.f);
  }
  __syncthreads();
  float2* mine = cols_smem + warp * G * P;
  fft_warp_rows<N>(mine, P, tw, lane);
  if constexpr (Op::kMiddle) {
    __syncthreads();
    const auto m = op.middle_begin(b);
    for (int e = threadIdx.x; e < N * NCOL; e += blockDim.x) {
      const int c = e % NCOL, i = e / NCOL, j = c0 + c;
      if (j >= W) continue;
      const LineElem el{b, i, j, size_t(i) * W + j, size_t(b * N + i) * W + j};
      cols_smem[c * P + fpad(i)] = op.middle(m, el, cols_smem[c * P + fpad(i)]);
    }
    __syncthreads();
    fft_warp_rows<N>(mine, P, tw, lane);
  }
  __syncthreads();
  for (int e = threadIdx.x; e < N * NCOL; e += blockDim.x) {
    const int c = e % NCOL, i = e / NCOL, j = c0 + c;
    if (j >= W) continue;
    const LineElem el{b, i, j, size_t(i) * W + j, size_t(b * N + i) * W + j};
    op.store(el, cols_smem[c * P + fpad(i)], op.preload(el));
  }
}

template <class Op> static int radix_rows(const Op& op, int H, int W, int B, cudaStream_t st) {
  return with_pow2(W, [&](auto n) {
    constexpr int N = decltype(n)::value, G = FftPlan<N>::G;
    return launch_lines(radix_rows_kernel<N, Op>, op, H, W, B, (H + 8 * G - 1) / (8 * G), 256,
                        size_t(8) * G * fft_pitch(N) * sizeof(float2), st);
  });
}
template <class Op> static int radix_cols(const Op& op, int H, int W, int B, cudaStream_t st) {
  return with_pow2(H, [&](auto n) {
    constexpr int N = decltype(n)::value, G = FftPlan<N>::G;
    return launch_lines(radix_cols_kernel<N, Op>, op, H, W, B, (W + 8 * G - 1) / (8 * G), 256,
                        size_t(8) * G * radix_cols_pitch<N>() * sizeof(float2), st);
  });
}

// ---------------------------------------------------------------- dense pass (any length N in 2..1024)
// The centred 1-D transform as a dense sum (algebra in fftprox_any.cuh).  A CTA owns kAnyLines lines (adjacent columns
// are read as 64-byte row segments); both operand buffers are padded to an odd pitch so that the eight lines of a warp hit
// distinct banks.
constexpr int kAnyMaxN = 1024;
constexpr int kAnyLines = 8;
constexpr int kAnyThreads = 256;

__host__ __device__ inline int any_pitch(int N) { return N | 1; }
inline size_t any_smem_bytes(int N) { return (size_t(N) + 2 * size_t(kAnyLines) * any_pitch(N)) * sizeof(float2); }

// out[l][k] = scale * sum_m in[l][m] * tw[((m - h)(k - h)) mod N]  (tw holds the conjugates for the inverse direction)
__device__ __forceinline__ void any_dft_lines(const float2* __restrict__ in, float2* __restrict__ out,
                                              const float2* __restrict__ tw, int N, int P, int nl, float scale) {
  const int h = N / 2;
  for (int e = threadIdx.x; e < kAnyLines * N; e += kAnyThreads) {
    const int l = e % kAnyLines, k = e / kAnyLines;
    if (l >= nl) continue;
    const int step = (k >= h) ? (k - h) : (k - h + N);                       // (k - h) mod N
    int ex = int((long long)(N - h) % N * step % N);                          // (0 - h)(k - h) mod N
    const float2* a = in + l * P;
    float2 acc0 = make_float2(0.f, 0.f), acc1 = make_float2(0.f, 0.f);
    int m = 0;
    for (; m + 1 < N; m += 2) {
      const float2 w0 = tw[ex];
      ex += step; if (ex >= N) ex -= N;
      const float2 w1 = tw[ex];
      ex += step; if (ex >= N) ex -= N;
      const float2 v0 = a[m], v1 = a[m + 1];
      acc0.x = fmaf(v0.x, w0.x, acc0.x); acc0.x = fmaf(-v0.y, w0.y, acc0.x);
      acc0.y = fmaf(v0.x, w0.y, acc0.y); acc0.y = fmaf(v0.y, w0.x, acc0.y);
      acc1.x = fmaf(v1.x, w1.x, acc1.x); acc1.x = fmaf(-v1.y, w1.y, acc1.x);
      acc1.y = fmaf(v1.x, w1.y, acc1.y); acc1.y = fmaf(v1.y, w1.x, acc1.y);
    }
    if (m < N) {
      const float2 w0 = tw[ex];
      const float2 v0 = a[m];
      acc0.x = fmaf(v0.x, w0.x, acc0.x); acc0.x = fmaf(-v0.y, w0.y, acc0.x);
      acc0.y = fmaf(v0.x, w0.y, acc0.y); acc0.y = fmaf(v0.y, w0.x, acc0.y);
    }
    out[l * P + k] = make_float2((acc0.x + acc1.x) * scale, (acc0.y + acc1.y) * scale);
  }
}

// Lines are rows (Op::kRows: the transform runs over the column index) or columns; with a middle step the second
// transform runs in the opposite direction with the same scale (conjugated table).
template <class Op>
__global__ void __launch_bounds__(kAnyThreads) dense_lines_kernel(const Op op, int H, int W, int b0) {
  extern __shared__ float2 any_sm[];
  constexpr bool kRows = Op::kRows;
  const int N = kRows ? W : H;                         // transform length
  const int nlines = kRows ? H : W;
  const int P = any_pitch(N);
  float2* tw = any_sm;                                 // forward table exp(-2 pi i k / N)
  float2* bufa = tw + N;
  float2* bufc = bufa + kAnyLines * P;
  const int b = b0 + blockIdx.y, l0 = blockIdx.x * kAnyLines;
  const int nl = min(kAnyLines, nlines - l0);
  const size_t img = size_t(b) * H * W;
  const bool inv1 = op.inverse();
  for (int k = threadIdx.x; k < N; k += kAnyThreads) {
    float s, c;
    sincospif(2.0f * float(k) / float(N), &s, &c);
    tw[k] = make_float2(c, inv1 ? s : -s);
  }
  // ---- load: consecutive threads walk memory-contiguous elements; (l, m) = (line, position along it) ----
  for (int e = threadIdx.x; e < kAnyLines * N; e += kAnyThreads) {
    const int l = kRows ? e / N : e % kAnyLines, m = kRows ? e % N : e / kAnyLines;
    if (l >= nl) continue;
    const int i = kRows ? l0 + l : m, j = kRows ? m : l0 + l;
    const size_t o = size_t(i) * W + j;
    bufa[l * P + m] = op.load(LineElem{b, i, j, o, img + o});
  }
  __syncthreads();
  any_dft_lines(bufa, bufc, tw, N, P, nl, op.scale(N));
  __syncthreads();
  const float2* res = bufc;
  if constexpr (Op::kMiddle) {                         // lines are columns: element (l, k) is (row k, column l0 + l)
    static_assert(!kRows, "a middle step runs on column passes");
    const auto mid = op.middle_begin(b);
    for (int e = threadIdx.x; e < kAnyLines * N; e += kAnyThreads) {
      const int l = e % kAnyLines, k = e / kAnyLines;
      if (l >= nl) continue;
      const size_t o = size_t(k) * W + l0 + l;
      bufc[l * P + k] = op.middle(mid, LineElem{b, k, l0 + l, o, img + o}, bufc[l * P + k]);
    }
    for (int k = threadIdx.x; k < N; k += kAnyThreads) tw[k].y = -tw[k].y;   // own entries only: no barrier needed before
    __syncthreads();
    any_dft_lines(bufc, bufa, tw, N, P, nl, op.scale(N));
    __syncthreads();
    res = bufa;
  }
  // ---- store ----
  if (!op.image_active(b)) return;
  for (int e = threadIdx.x; e < kAnyLines * N; e += kAnyThreads) {
    const int l = kRows ? e / N : e % kAnyLines, m = kRows ? e % N : e / kAnyLines;
    if (l >= nl) continue;
    const int i = kRows ? l0 + l : m, j = kRows ? m : l0 + l;
    const LineElem el{b, i, j, size_t(i) * W + j, img + size_t(i) * W + j};
    op.store(el, res[l * P + m], op.preload(el));
  }
}

inline bool any_shape_supported(int H, int W) { return H >= 2 && W >= 2 && H <= kAnyMaxN && W <= kAnyMaxN; }

template <class Op> static int dense_lines(const Op& op, int H, int W, int B, cudaStream_t st) {
  static bool attr_done = false;                       // one flag per kernel instantiation
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(dense_lines_kernel<Op>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         int(any_smem_bytes(kAnyMaxN)));
    if (e != cudaSuccess) return int(e);
    attr_done = true;
  }
  const int N = Op::kRows ? W : H, nlines = Op::kRows ? H : W;
  return launch_lines(dense_lines_kernel<Op>, op, H, W, B, (nlines + kAnyLines - 1) / kAnyLines, kAnyThreads,
                      any_smem_bytes(N), st);
}

}  // namespace pnp
