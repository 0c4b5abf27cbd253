// FFT-prox + dual update for arbitrary sampling masks at 128x128 (the reference's native shape, evaluation/env.py:64):
// the cluster kernel of fftprox_cl.cuh re-dimensioned - 4-CTA clusters x 32 rows, 256 threads, two CTAs per SM, of which
// 71-74 clusters are resident (tools/cluster_occ.cu: 4-CTA clusters pack 96-100 % of the SMs).
//
// 128 = 16 x 8: a quarter-warp (8 lanes) owns a row, lane j holds x[j + 8 r], r < 16.
//   pass A  16-point DFT over r in registers, twiddle w128^(j q)
//   exchange through the row's own shared-memory slot (16-byte chunks, XOR-swizzled)
//   pass B  two 8-point DFTs over j (q = j'' and q = j'' + 8) -> X[j'' + 8 m], m < 16: the layout pass A consumes, so the
//           blend and the inverse transform chain register to register exactly as in the 256-point kernels.
// Columns: thread (c, jc), jc < 8, owns the 16 elements jc + 8 r of column c and transforms them in place (slot swap
// inside the received buffer, lanes along c: conflict free).  Staging (cp.async.bulk), exchanges (st.async + mbarrier tx
// counts), tensor memory for w = x + u and the algebra (y0R, packed rotated mask) are those of fftprox_cl.cuh.
#pragma once
#include "fftprox_cl.cuh"

namespace pnp {

constexpr int kC128N = 128, kC128CL = 4, kC128R = 32, kC128Threads = 256;
constexpr int kC128Buf = kC128R * kC128N;             // float2 elements per buffer (32 KB)
constexpr int kC128Blk = kC128R * kC128R;             // float2 elements per exchange block (8 KB)
constexpr size_t kC128Smem = size_t(3) * kC128Buf * 8 + size_t(kC128R) * kC128N * 4 + 96 * 8 + 64;

template <bool INV> __device__ __forceinline__ void dft8t(float2 (&v)[8]) {
  float2 e[4] = {v[0], v[2], v[4], v[6]};
  float2 o[4] = {v[1], v[3], v[5], v[7]};
  dft4t<INV>(e);
  dft4t<INV>(o);
  const float h = 0.70710678118654752440f;
  float2 o1, o2, o3;
  if constexpr (!INV) {
    o1 = make_float2(h * (o[1].x + o[1].y), h * (o[1].y - o[1].x));       // * (1 - i) / sqrt 2
    o2 = make_float2(o[2].y, -o[2].x);                                    // * (-i)
    o3 = make_float2(h * (o[3].y - o[3].x), -h * (o[3].x + o[3].y));      // * (-1 - i) / sqrt 2
  } else {
    o1 = make_float2(h * (o[1].x - o[1].y), h * (o[1].y + o[1].x));       // * (1 + i) / sqrt 2
    o2 = make_float2(-o[2].y, o[2].x);                                    // * (+i)
    o3 = make_float2(-h * (o[3].x + o[3].y), h * (o[3].x - o[3].y));      // * (-1 + i) / sqrt 2
  }
  v[0] = cadd(e[0], o[0]); v[4] = csub(e[0], o[0]);
  v[1] = cadd(e[1], o1);   v[5] = csub(e[1], o1);
  v[2] = cadd(e[2], o2);   v[6] = csub(e[2], o2);
  v[3] = cadd(e[3], o3);   v[7] = csub(e[3], o3);
}

// second pass of the 128-point transform: v[0..7] = V_j[q0], v[8..15] = V_j[q0 + 8] (j = 0..7) -> v[m] = X[q0 + 8 m]
template <bool INV> __device__ __forceinline__ void dft8x2_interleave(float2 (&v)[16]) {
  float2 a[8], b[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) { a[k] = v[k]; b[k] = v[8 + k]; }
  dft8t<INV>(a);
  dft8t<INV>(b);
#pragma unroll
  for (int k = 0; k < 8; ++k) { v[2 * k] = a[k]; v[2 * k + 1] = b[k]; }
}

// float2 index of position pos (0..127) of a local row inside a buffer blocked as [4][32 rows][32 columns]; `rowp` already
// points at buffer + rho * 32
__device__ __forceinline__ int c128_pos(int pos) { return (pos >> 5) * kC128Blk + (pos & 31); }

// 128-point DFT of one image row held by a quarter-warp: in v[r] = x[j + 8 r], out v[m] = X[j + 8 m].
// wtab[t][j] = exp(-2 pi i j m_t / 128), m_t in {1,2,3,4,8,12} (rows of 16 entries, j < 8 used).
template <bool INV>
__device__ __forceinline__ void fft128_row_blocked(float2 (&v)[16], float2* rowp, const float2* wtab, int j, int rho) {
  dft16t<INV>(v);
  twiddle16<INV>(v, wtab, j);                            // V_j[q] *= w128^(-+ j q)
  const int sw = (j & 7) ^ ((rho & 1) << 2);             // odd rows use the other half of the bank window
  {
    float4* dst = reinterpret_cast<float4*>(rowp + c128_pos(16 * j));   // logical 16 j + q -> chunk (q >> 1) ^ sw
#pragma unroll
    for (int m = 0; m < 8; ++m) dst[m ^ sw] = make_float4(v[2 * m].x, v[2 * m].y, v[2 * m + 1].x, v[2 * m + 1].y);
  }
  __syncwarp();
  // lane j'' = j reads V_jj[q] for q in {j, j + 8} from every writer jj
  const int qa = j, qb = j + 8;
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    const int swj = jj ^ ((rho & 1) << 2);
    v[jj] = rowp[c128_pos(16 * jj) + 2 * ((qa >> 1) ^ swj) + (qa & 1)];
    v[8 + jj] = rowp[c128_pos(16 * jj) + 2 * ((qb >> 1) ^ swj) + (qb & 1)];
  }
  __syncwarp();
  dft8x2_interleave<INV>(v);
}

__global__ void __launch_bounds__(kC128Threads, 2) fftprox_cl128_kernel(const ClParams p) {
  constexpr int N = kC128N, R = kC128R, BUF = kC128Buf, BLK = kC128Blk, CL = kC128CL;
  extern __shared__ __align__(128) uint8_t c128_smem[];
  float2* bufU = reinterpret_cast<float2*>(c128_smem);   // bulk-load target: R rows of u
  float2* bufA = bufU + BUF;                             // row domain: receives exchange 2; scratch of the row transforms
  float2* bufQ = bufA + BUF;                             // column domain: receives exchange 1, transformed in place
  float* X = reinterpret_cast<float*>(bufQ + BUF);       // bulk-load target: R rows of x
  float2* wf = reinterpret_cast<float2*>(X + R * N);
  uint64_t* bars = reinterpret_cast<uint64_t*>(wf + 96);
  uint64_t* tmafull = bars;
  uint64_t* bfull = bars + 1;
  uint64_t* afull = bars + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3);

  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t rank = cl_cluster_rank();
  const int cluster_id = blockIdx.x / CL, n_clusters = gridDim.x / CL;
  const int row0 = int(rank) * R;
  if (tid < 96) {
    const int t = tid >> 4, jj = tid & 15;
    const int m = (t < 4) ? t + 1 : (t == 4 ? 8 : 12);
    wf[tid] = g_tw512[(4 * jj * m) & 511];               // exp(-2 pi i jj m / 128); jj < 8 is used
  }
  if (tid == 0) {
    mbar_init(tmafull, 1);
    mbar_init(bfull, 1);
    mbar_init(afull, 1);
    fence_mbar_init();
  }
  grid_dep_wait();                                       // programmatic stream serialization: see fftprox_cl.cuh
  grid_dep_launch();
  if (p.skip_flag && *p.skip_flag != 0) return;
  constexpr uint32_t kRowBytesU = uint32_t(R) * N * 8, kRowBytesX = uint32_t(R) * N * 4;
  if (tid == 0 && cluster_id < p.B) {
    const size_t g = size_t(cluster_id) * N * N + size_t(row0) * N;
    mbar_arrive_expect_tx(tmafull, kRowBytesU + kRowBytesX);
    bulk_load_1d(bufU, p.u_in + g, kRowBytesU, tmafull);
    bulk_load_1d(X, p.x + g, kRowBytesX, tmafull);
    mbar_arrive_expect_tx(bfull, uint32_t(BUF) * 8);
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 64);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_w = *tmem_slot + (uint32_t(32 * (warp & 3)) << 16) + uint32_t(32 * (warp >> 2));
  cl_cluster_arrive_relaxed();                           // barrier inits are published by fence.mbarrier_init (see fftprox_cl.cuh)
  cl_cluster_wait();

  const int qw = tid >> 3, j = tid & 7;                  // row phases: quarter-warp qw owns local row qw, lane j
  const int cc = tid & 31, jc = tid >> 5;                // column phase: thread (column cc, residue jc < 8)
  const float inv2 = 1.0f / float(N * N);
  const uint32_t bfull_a = smem_u32(bfull), afull_a = smem_u32(afull);

  int it = 0;
  for (int b = cluster_id; b < p.B; b += n_clusters, ++it) {
    const uint32_t par = it & 1;
    const size_t img = size_t(b) * N * N;
    const bool has_next = b + n_clusters < p.B;
    const float mu = __ldg(p.mu + size_t(b) * p.mu_stride);

    // ================= rows forward =================
    if (tid == 0) mbar_arrive_expect_tx(afull, uint32_t(BUF) * 8);
    mbar_wait(tmafull, par);
    {
      const float2* Ur = bufU + qw * N;
      const float* Xr = X + qw * N;
      float2 v[16];
#pragma unroll
      for (int r = 0; r < 16; ++r) {
        const float2 uu = Ur[j + 8 * r];
        v[r] = make_float2(Xr[j + 8 * r] + uu.x, uu.y);
      }
      {
        uint32_t wr[32];
#pragma unroll
        for (int r = 0; r < 16; ++r) { wr[2 * r] = __float_as_uint(v[r].x); wr[2 * r + 1] = __float_as_uint(v[r].y); }
        tmem_st_32x32(tmem_w, wr);
      }
      fft128_row_blocked<false>(v, bufA + qw * R, wf, j, qw);       // v[m] = H[row][j + 8 m]
      // exchange 1: element (row, col = j + 8 m) -> CTA col / 32, slot [rank][row][col % 32] of its Q
      const uint32_t dst0 = smem_u32(bufQ + rank * BLK + qw * R + j);
#pragma unroll
      for (int m = 0; m < 16; ++m)
        cl_st_async(cl_mapa(dst0 + uint32_t((8 * m) % R) * 8u, (8 * m) / R), v[m], cl_mapa(bfull_a, (8 * m) / R));
    }
    const uint32_t mbits = __ldg(p.mpack + size_t(b) * p.mpack_bstride + jc * N + row0 + cc);
    {                                                    // the blend reads y0R under the mask: pull those sectors into L2 now
      const float2* yp = p.y0R + img + size_t(jc) * N + row0 + cc;
#pragma unroll
      for (int m = 0; m < 16; ++m)
        if ((mbits >> m) & 1u) asm volatile("prefetch.global.L2 [%0];" ::"l"(yp + 8 * m * N));
    }
    mbar_wait(bfull, par);
    if (tid == 0) mbar_arrive_expect_tx(bfull, uint32_t(BUF) * 8);

    // ================= columns: forward, blend, inverse - in place in Q =================
    {
      float2* Bc = bufQ + cc;
      const int col = row0 + cc;                         // kappa_j
      const float bb = 1.f / (1.f + mu), aa = mu * bb;
      float2 v[16];
#pragma unroll
      for (int r = 0; r < 16; ++r) v[r] = Bc[cl_col_idx<R>(jc + 8 * r, 0)];
      dft16t<false>(v);
      twiddle16<false>(v, wf, jc);
#pragma unroll
      for (int q = 0; q < 16; ++q) Bc[cl_col_idx<R>(jc + 8 * q, 0)] = v[q];      // V_jc[q] -> own slot jc + 8 q
      __syncthreads();
      if (tid == 0 && has_next) {
        const size_t g = img + size_t(n_clusters) * N * N + size_t(row0) * N;
        mbar_arrive_expect_tx(tmafull, kRowBytesU + kRowBytesX);
        bulk_load_1d(bufU, p.u_in + g, kRowBytesU, tmafull);
        bulk_load_1d(X, p.x + g, kRowBytesX, tmafull);
      }
      float2 y[16];
      {
        const float2* yp = p.y0R + img + size_t(jc) * N + col;
#pragma unroll
        for (int m = 0; m < 16; ++m) y[m] = ((mbits >> m) & 1u) ? __ldg(yp + 8 * m * N) : make_float2(0.f, 0.f);
      }
      // thread (c, jc) now takes q in {jc, jc + 8}: V_j[q] sits in slot j + 8 q
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) {
        v[jj] = Bc[cl_col_idx<R>(jj + 8 * jc, 0)];
        v[8 + jj] = Bc[cl_col_idx<R>(jj + 8 * jc + 64, 0)];
      }
      dft8x2_interleave<false>(v);                       // v[m] = H[kappa_i = jc + 8 m][kappa_j = col]
#pragma unroll
      for (int m = 0; m < 16; ++m)
        if ((mbits >> m) & 1u) v[m] = make_float2(aa * v[m].x + bb * y[m].x, aa * v[m].y + bb * y[m].y);
      dft16t<true>(v);
      twiddle16<true>(v, wf, jc);
#pragma unroll
      for (int q = 0; q < 16; ++q)                       // V'_jc[q] -> the slots this thread read: q + 8 jc (+ 56 for q >= 8)
        Bc[cl_col_idx<R>((q & 7) + 8 * jc + 64 * (q >> 3), 0)] = v[q];
      __syncthreads();
#pragma unroll
      for (int r = 0; r < 16; ++r) v[r] = Bc[cl_col_idx<R>(jc + 8 * r, 0)];      // r < 8: V'_r[jc]; r >= 8: V'_(r-8)[jc + 8]
      dft8x2_interleave<true>(v);                        // v[m] = column-inverse at image row jc + 8 m
      // exchange 2: element (row i = jc + 8 m, col) -> CTA i / 32, slot [rank][i % 32][cc] of its A
      const uint32_t dst0 = smem_u32(bufA + rank * BLK + jc * R + cc);
#pragma unroll
      for (int m = 0; m < 16; ++m)
        cl_st_async(cl_mapa(dst0 + uint32_t(((8 * m) % R) * R) * 8u, (8 * m) / R), v[m], cl_mapa(afull_a, (8 * m) / R));
    }
    mbar_wait(afull, par);

    // ================= rows inverse + epilogue =================
    {
      float2* rowp = bufA + qw * R;
      float2 v[16];
#pragma unroll
      for (int r = 0; r < 16; ++r) v[r] = rowp[c128_pos(j + 8 * r)];
      __syncwarp();
      fft128_row_blocked<true>(v, rowp, wf, j, qw);
      uint32_t wr[32];
      tmem_st_wait();
      tmem_ld_32x32(tmem_w, wr);
      tmem_ld_wait();
      const size_t g0 = img + size_t(row0 + qw) * N + j;
      if (!(p.active && p.active[b] == 0)) {
#pragma unroll
      for (int m = 0; m < 16; ++m) {
        const float2 zz = make_float2(v[m].x * inv2, v[m].y * inv2);
        const float2 un = make_float2(__uint_as_float(wr[2 * m]) - zz.x, __uint_as_float(wr[2 * m + 1]) - zz.y);
        p.z_out[g0 + 8 * m] = zz;
        p.u_out[g0 + 8 * m] = un;
        if (p.v_out) p.v_out[g0 + 8 * m] = zz.x - un.x;
      }
      }
    }
  }
  tc_fence_before();
  cl_cluster_arrive_relaxed();
  cl_cluster_wait();
  if (warp == 1) tmem_dealloc(*tmem_slot, 64);
}

// Trajectory constants at 128x128: y0R[ki][kj] = (-1)^(ki+kj) * 128 * y0[(ki+64)%128][(kj+64)%128]; packed rotated mask
// mpack[b][jj < 8][kj]: bit m = mask[(jj + 8 m + 64) % 128][(kj + 64) % 128].  grid (128, B), 128 threads.
__global__ void __launch_bounds__(128) prox_prepare_cl128_kernel(const float2* __restrict__ y0, const uint8_t* __restrict__ mask,
                                                                 long long mask_bstride, float2* __restrict__ y0R,
                                                                 uint16_t* __restrict__ mpack, int nb_mask,
                                                                 const int* skip_flag) {
  if (skip_flag && *skip_flag != 0) return;
  constexpr int N = kC128N;
  const int b = blockIdx.y, ki = blockIdx.x, kj = threadIdx.x;
  const size_t img = size_t(b) * N * N;
  const int si = (ki + N / 2) & (N - 1), sj = (kj + N / 2) & (N - 1);
  const float2 y = y0[img + size_t(si) * N + sj];
  const float s = ((ki + kj) & 1) ? -float(N) : float(N);
  y0R[img + size_t(ki) * N + kj] = make_float2(s * y.x, s * y.y);
  if (b < nb_mask && ki < 8) {
    const uint8_t* mk = mask + size_t(b) * mask_bstride + sj;
    uint32_t bits = 0;
#pragma unroll
    for (int m = 0; m < 16; ++m) bits |= (mk[size_t((ki + 8 * m + N / 2) & (N - 1)) * N] ? 1u : 0u) << m;
    mpack[size_t(b) * 8 * N + ki * N + kj] = uint16_t(bits);
  }
}

__global__ void __launch_bounds__(kC128Threads) cl128_occupancy_probe(int* p) {
  extern __shared__ int probe128_sm[];
  if (p) p[0] = probe128_sm[0];
}

static int launch_cl128(const ClParams& p, cudaStream_t st) {
  return launch_resident_clusters<fftprox_cl128_kernel, cl128_occupancy_probe>(p, kC128CL, kC128Threads, kC128Smem, st);
}

}  // namespace pnp
