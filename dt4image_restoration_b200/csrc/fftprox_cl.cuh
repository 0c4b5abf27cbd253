// FFT-prox + dual update for arbitrary sampling masks, 256x256: third-generation single-launch cluster kernel.
// Replaces reference evaluation/env.py:87-93 (fft -> masked k-space solve -> ifft -> dual update) with the centred
// transforms of evaluation/utils/transformations.py:6-19 folded into constants (see "Algebra" below).
//
// Design (what changed against round 1's fftprox_fused2 kernel, measured with tools/prox_phases.py - 40 % of its time was
// cluster barriers and register-staged transposes, x and u were read twice, every global load sat in front of an FFT;
// step-by-step numbers in profiles/r02_prox_cl_steps.txt).  One image per 16-CTA cluster, a CTA owns 16 image rows and 16
// k-space columns, 256 threads, two CTAs (of different images) per SM:
//   * all global READS of the image are 1-D bulk-async copies (cp.async.bulk, SASS UBLKCP): the 16 rows of u (32 KB) and
//     x (16 KB) of the NEXT image land in shared memory while the current image is transformed - no load instruction,
//     no register, no exposed DRAM latency.
//   * w = x + u is parked in TENSOR MEMORY (one tcgen05.st per thread, read back with tcgen05.ld in the epilogue:
//     u' = w - z, v' = Re(2 z - w)), so x and u cross L2 -> SM exactly once (DRAM traffic = the algorithmic 37 B/pixel)
//     and no shared-memory buffer stays occupied from the first phase to the last.
//   * the two cluster transposes are pushes through distributed shared memory straight from the registers the
//     transforms leave their results in (st.async.shared::cluster with mbarrier complete_tx: a warp writes 256 contiguous
//     bytes of one peer per instruction); the receiver waits on ONE mbarrier that counts the bytes of all 16 senders.
//     The column pass walks the received blocks with lanes along the column index (conflict free) and transforms IN
//     PLACE (thread (c, j) owns the 16 elements j + 16 r of column c; the radix-16 exchange is a strided slot swap inside
//     the buffer).  No register staging, no transposed copies of y0 / mask, no cluster barrier per image: a peer's
//     receive buffer is known to be free because its previous contribution has ARRIVED here (see the loop comments).
//   * measured limits (profiles/r02_prox_cl_steps.txt): distributed shared memory moves ~17 B/clk per SM, 16-CTA clusters
//     pack 14 at a time onto the chip, the kernel issues 2300 instructions per thread and image (832 packed FP32).
//
// Algebra.  With H = FFT2(w) (plain, unnormalised), h = N / 2 and k = (kappa + h) mod N:
//     fft_c(w)[k] = (-1)^kappa H[kappa] / N        (ifftshift = output modulation, fftshift = output rotation)
//     ifft_c(Z)[n] = IFFT2_plain(Y)[n] / N,  Y[kappa] = (-1)^kappa Z[k]
// so the reference step is   z = IFFT2_plain( m_R ? (mu H + y0R) / (1 + mu) : H ) / N^2   with the trajectory constants
//     y0R[kappa] = (-1)^(kappa_i + kappa_j) * N * y0[k],   m_R[kappa] = mask[k]
// prepared once (prox_prepare_cl_kernel): no sign flips, no shifts and no scaling inside the transforms.
#pragma once
#include "common.cuh"
#include "fft_core.cuh"
#include "fft256_reg.cuh"

namespace pnp {

struct ClParams {
  const float* x;
  const float2* u_in;
  const float2* y0R;          // 256x256: [B][kappa_j][kappa_i] (transposed: a half-warp owns a k-space column); 128x128: [B][kappa_i][kappa_j]
  const uint16_t* mpack;      // 256x256: [B or 1][256 kappa_j][16 jj]; 128x128: [B or 1][8 jj][128 kappa_j]; bit p = m_R[jj + 16 p (8 p)][kappa_j]
  long long mpack_bstride;    // in uint16 units: 16 * 256 (per-image masks) or 0 (one mask for the batch)
  const float* mu;
  int mu_stride;
  float2* z_out;
  float2* u_out;
  float* v_out;               // may be null
  int B;
  const int* skip_flag;       // optional: != 0 means the column-only-mask kernel (fftprox_sep.cuh) handles this batch
  const uint8_t* active;      // optional [B]: 0 = the image's z, u, v stay untouched (early exit of a trajectory, env.py:79-81)
};

constexpr int kClN = 256;

template <int CL> struct ClCfg {
  static constexpr int R = kClN / CL;                      // image rows (and k-space columns) per CTA
  static constexpr int THREADS = 16 * R;                   // a half-warp per row / 16 threads per column
  static constexpr int BUF = R * kClN;                     // float2 elements per buffer
  static constexpr int BLK = R * R;                        // float2 elements per exchange block
  static constexpr size_t SMEM = size_t(3) * BUF * 8 + size_t(R) * kClN * 4 + 96 * 8 + 64;   // + barriers, TMEM slot
};

// ---- directional radix-4 / radix-16 butterflies (INV: conjugated twiddles, i.e. the unnormalised inverse DFT) ----
template <bool INV> __device__ __forceinline__ void dft4t(float2 (&v)[4]) {
  const float2 a0 = cadd(v[0], v[2]), a1 = csub(v[0], v[2]);
  const float2 b0 = cadd(v[1], v[3]), b1 = csub(v[1], v[3]);
  v[0] = cadd(a0, b0);
  v[2] = csub(a0, b0);
  if constexpr (!INV) { v[1] = cadd_mi(a1, b1); v[3] = csub_mi(a1, b1); }
  else                { v[1] = csub_mi(a1, b1); v[3] = cadd_mi(a1, b1); }
}

template <bool INV> __device__ __forceinline__ void dft16t(float2 (&v)[16]) {
  const float c8 = 0.92387953251128675613f, s8 = 0.38268343236508977173f, h = 0.70710678118654752440f;
  constexpr float sg = INV ? 1.f : -1.f;              // sign of the imaginary part of w16^k
  float2 t[4][4];
#pragma unroll
  for (int b = 0; b < 4; ++b) {
    float2 a[4] = {v[b], v[b + 4], v[b + 8], v[b + 12]};
    dft4t<INV>(a);
#pragma unroll
    for (int q = 0; q < 4; ++q) t[b][q] = a[q];
  }
  t[1][1] = cmul(t[1][1], make_float2(c8, sg * s8));
  t[1][2] = cmul(t[1][2], make_float2(h, sg * h));
  t[1][3] = cmul(t[1][3], make_float2(s8, sg * c8));
  t[2][1] = cmul(t[2][1], make_float2(h, sg * h));
  t[2][2] = INV ? make_float2(-t[2][2].y, t[2][2].x) : make_float2(t[2][2].y, -t[2][2].x);   // * (+-i)
  t[2][3] = cmul(t[2][3], make_float2(-h, sg * h));
  t[3][1] = cmul(t[3][1], make_float2(s8, sg * c8));
  t[3][2] = cmul(t[3][2], make_float2(-h, sg * h));
  t[3][3] = cmul(t[3][3], make_float2(-c8, -sg * s8));
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float2 a[4] = {t[0][q], t[1][q], t[2][q], t[3][q]};
    dft4t<INV>(a);
#pragma unroll
    for (int p = 0; p < 4; ++p) v[q + 4 * p] = a[p];
  }
}

// v[r] *= w256^(-+j r) (INV: conjugates): wtab[t][j] = exp(-2 pi i j m_t / 256), m_t in {1,2,3,4,8,12}; six look-ups, nine products
template <bool INV>
__device__ __forceinline__ void twiddle16(float2 (&v)[16], const float2* wtab, int j) {
  float2 w1 = wtab[j], w2 = wtab[16 + j], w3 = wtab[32 + j];
  float2 w4 = wtab[48 + j], w8 = wtab[64 + j], w12 = wtab[80 + j];
  if constexpr (INV) { w1.y = -w1.y; w2.y = -w2.y; w3.y = -w3.y; w4.y = -w4.y; w8.y = -w8.y; w12.y = -w12.y; }
  v[1] = cmul(v[1], w1); v[2] = cmul(v[2], w2); v[3] = cmul(v[3], w3); v[4] = cmul(v[4], w4);
  v[5] = cmul(v[5], cmul(w4, w1)); v[6] = cmul(v[6], cmul(w4, w2)); v[7] = cmul(v[7], cmul(w4, w3));
  v[8] = cmul(v[8], w8);
  v[9] = cmul(v[9], cmul(w8, w1)); v[10] = cmul(v[10], cmul(w8, w2)); v[11] = cmul(v[11], cmul(w8, w3));
  v[12] = cmul(v[12], w12);
  v[13] = cmul(v[13], cmul(w12, w1)); v[14] = cmul(v[14], cmul(w12, w2)); v[15] = cmul(v[15], cmul(w12, w3));
}

// float2 index of element i (0..255) of local column c inside a buffer blocked as [256 / R][R][R] (i = sender * R + row)
template <int R> __device__ __forceinline__ int cl_col_idx(int i, int c) { return (i / R) * (R * R) + (i % R) * R + c; }

// 256-point DFT of one image row held by a half-warp: in v[r] = x[j + 16 r], out v[r] = X[16 r + j].  The radix-16
// exchange goes through the row's own storage `rowp` = buffer + rho * R (blocked layout, contents destroyed); chunks
// are XOR-swizzled so the 16-byte stores and the 8-byte loads are bank-conflict free.
template <int R, bool INV>
__device__ __forceinline__ void fft256_row_blocked(float2 (&v)[16], float2* rowp, const float2* wtab, int j) {
  dft16t<INV>(v);
  {
    // logical element 16 j + q -> position 16 j + 2 (m ^ (j & 7)) + (q & 1), m = q >> 1
    float4* dst = reinterpret_cast<float4*>(rowp + ((16 * j) / R) * (R * R) + ((16 * j) % R));
#pragma unroll
    for (int m = 0; m < 8; ++m) dst[m ^ (j & 7)] = make_float4(v[2 * m].x, v[2 * m].y, v[2 * m + 1].x, v[2 * m + 1].y);
  }
  __syncwarp();
#pragma unroll
  for (int r = 0; r < 16; ++r) v[r] = rowp[((16 * r) / R) * (R * R) + ((16 * r) % R) + (j ^ ((r & 7) << 1))];
  __syncwarp();
  twiddle16<INV>(v, wtab, j);
  dft16t<INV>(v);
}

// ---- exchange-buffer layouts of the 256x256 kernel (R = 16): XOR-swizzled so that a HALF-WARP can own a column (lanes along
// the row index) or a row (lanes along the column index) without bank conflicts and without a CTA barrier between passes ----
// Q (column domain): element (image row i, local column c).  The 16 lanes of a half-warp read i = l + 16 r (pass 1 / 3) or
// i = r + 16 l (pass 2): both vary (i & 15) ^ (i >> 4) over all 16 values, so the 16 float2 land in 16 different bank pairs.
__device__ __forceinline__ int cl_q_idx(int i, int c) { return 16 * i + (c ^ (i & 15) ^ (i >> 4)); }
// A (row domain): element (local row rho, column col = 16 s + cc) -> block s (sender), cc-major, rows swizzled by cc.
__device__ __forceinline__ int cl_a_idx(int rho, int s, int cc) { return 256 * s + 16 * cc + (rho ^ cc); }

// 256-point DFT of one image row held by a half-warp, radix-16 exchange through the row's own slots of the swizzled A
// buffer: lane j writes V_j[q] to slot (s = q, cc = j ^ q) and reads V_r[j] from slot (s = j, cc = r ^ j) - both touch 16
// different bank pairs.  in v[r] = x[j + 16 r], out v[r] = X[16 r + j] (contents of the row's slots destroyed).
template <bool INV>
__device__ __forceinline__ void fft256_row_swz(float2 (&v)[16], float2* A, const float2* wtab, int j, int rho) {
  dft16t<INV>(v);
#pragma unroll
  for (int q = 0; q < 16; ++q) A[cl_a_idx(rho, q, j ^ q)] = v[q];
  __syncwarp();
#pragma unroll
  for (int r = 0; r < 16; ++r) v[r] = A[cl_a_idx(rho, j, r ^ j)];
  __syncwarp();
  twiddle16<INV>(v, wtab, j);
  dft16t<INV>(v);
}

__device__ __forceinline__ uint32_t cl_mapa(uint32_t saddr, uint32_t rank) {
  uint32_t r;
#ifdef PNP_CL_LOCAL_ONLY   // timing experiment only (wrong results): every exchange targets the sender's own CTA - no SM-to-SM traffic
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
#endif
  asm("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cl_cluster_arrive() { asm volatile("barrier.cluster.arrive.release;" ::: "memory"); }
// Execution-only arrive (a released one is MEMBAR.ALL.GPU + ERRBAR: 9 % of the stall samples of the first version).  Used
// where nothing this thread WROTE has to be published: the accesses it orders are shared-memory reads whose values were
// already consumed by issued instructions (a warp issues in order), or an mbarrier wait that has returned.
__device__ __forceinline__ void cl_cluster_arrive_relaxed() { asm volatile("barrier.cluster.arrive.relaxed;" ::: "memory"); }
__device__ __forceinline__ void cl_cluster_wait() { asm volatile("barrier.cluster.wait.acquire;" ::: "memory"); }
__device__ __forceinline__ uint32_t cl_cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}

// register -> remote shared memory store (8 bytes) that completes 8 bytes on the mbarrier at cluster address `rbar`
__device__ __forceinline__ void cl_st_async(uint32_t raddr, float2 v, uint32_t rbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f32 [%0], {%1, %2}, [%3];" ::"r"(raddr),
               "f"(v.x), "f"(v.y), "r"(rbar)
               : "memory");
}

template <int CL>
__global__ void __launch_bounds__(ClCfg<CL>::THREADS, CL == 8 ? 1 : 2) fftprox_cl_kernel(const ClParams p) {
  using Cfg = ClCfg<CL>;
  constexpr int R = Cfg::R, BUF = Cfg::BUF, NT = Cfg::THREADS;
  static_assert(CL == 16 && R == 16, "the swizzled exchange layouts (cl_q_idx / cl_a_idx) assume 16 rows and 16 columns per CTA");
  constexpr uint32_t kTmemCols = NT / 4;               // 32 columns (16 float2) per thread: 4 lane quarters x NT/128 warps each
  constexpr uint32_t kTmemAlloc = 2 * kTmemCols;       // two images in flight (rows of image b+1 go out before image b is finished)
  extern __shared__ __align__(128) uint8_t cl_smem[];
  float2* bufU = reinterpret_cast<float2*>(cl_smem);     // bulk-load target: R rows of u; then scratch of the forward row transforms
  float2* bufA = bufU + BUF;                             // row domain: receives exchange 2; scratch of the inverse row transforms
  float2* bufQ = bufA + BUF;                             // column domain: receives exchange 1, transformed in place
  float* X = reinterpret_cast<float*>(bufQ + BUF);       // bulk-load target: R rows of x
  float2* wf = reinterpret_cast<float2*>(X + R * kClN);  // twiddle rows (forward; the inverse passes conjugate them)
  uint64_t* bars = reinterpret_cast<uint64_t*>(wf + 96);
  uint64_t* tmafull = bars;                              // bulk loads of u and x
  uint64_t* bfull = bars + 1;                            // exchange 1 received (R x 256 elements from the CL peers)
  uint64_t* afull = bars + 2;                            // exchange 2 received
  uint64_t* afree = bars + 3;                            // credits: every warp of every CTA of the cluster is done reading its A
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);

  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t rank = cl_cluster_rank();
  const int cluster_id = blockIdx.x / CL, n_clusters = gridDim.x / CL;
  const int row0 = int(rank) * R;
  if (tid < 96) {
    const int t = tid >> 4, jj = tid & 15;
    const int m = (t < 4) ? t + 1 : (t == 4 ? 8 : 12);
    wf[tid] = g_tw512[2 * jj * m];                       // exp(-2 pi i jj m / 256)
  }
  if (tid == 0) {
    mbar_init(tmafull, 1);
    mbar_init(bfull, 1);
    mbar_init(afull, 1);
    mbar_init(afree, uint32_t(CL) * (NT / 32));          // one arrival per warp of the cluster
    fence_mbar_init();
  }
  // Launched with programmatic stream serialization: everything above overlaps the tail of the previous kernel in the
  // stream; nothing it wrote (x, u, the prepared constants, the flag) is touched before this point.
  grid_dep_wait();
  grid_dep_launch();                                     // the next kernel in the stream may start its own prologue
  if (p.skip_flag && *p.skip_flag != 0) return;        // uniform over the whole grid, before any cluster operation
  constexpr uint32_t kRowBytesU = uint32_t(R) * kClN * 8, kRowBytesX = uint32_t(R) * kClN * 4;
  if (tid == 0 && cluster_id < p.B) {                    // first image: the loads fly while tensor memory is allocated
    const size_t g = size_t(cluster_id) * kClN * kClN + size_t(row0) * kClN;
    mbar_arrive_expect_tx(tmafull, kRowBytesU + kRowBytesX);
    bulk_load_1d(bufU, p.u_in + g, kRowBytesU, tmafull);
    bulk_load_1d(X, p.x + g, kRowBytesX, tmafull);
    mbar_arrive_expect_tx(bfull, uint32_t(BUF) * 8);     // armed before this CTA's cluster arrive: no peer can send earlier
  }
  if (warp == 1) {                                       // tensor memory keeps w = x + u of the images in flight
    tmem_alloc(tmem_slot, kTmemAlloc);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // this thread's 32 TMEM columns: lane quarter warp % 4 (the only one a warp can reach), column block warp / 4
  const uint32_t tmem_w = *tmem_slot + (uint32_t(32 * (warp & 3)) << 16) + uint32_t(32 * (warp >> 2));
  cl_cluster_arrive_relaxed();                           // every CTA's barriers are initialised (fence.mbarrier_init above) before anyone sends
  cl_cluster_wait();

  const int hw = tid >> 4, j = tid & 15;                 // row phases: half-warp hw owns local row hw, lane j
  const int cc = tid >> 4, jc = tid & 15;                // column phase: half-warp cc owns local column cc, lane jc = residue
  const float inv2 = 1.0f / 65536.0f;                    // 1 / (H W): both transforms are unnormalised
  const uint32_t bfull_a = smem_u32(bfull), afull_a = smem_u32(afull), afree_a = smem_u32(afree);

  // Software pipeline over the images of this cluster (image index it, batch index b = cluster_id + it * n_clusters):
  //     iteration it:   columns(it) -> rows forward(it + 1) -> rows inverse(it)
  // so that each exchange is in flight while independent work runs: the rows of image it+1 travel during the inverse
  // rows / epilogue of image it, the columns of image it during the forward rows of image it+1 (before: both waits were
  // exposed, 23 % of a CTA's time, profiles/r02_prox_phases_v6.txt).  What tells a sender that the target buffer is free:
  //   Q of every peer (exchange 1 of it+1): afull(it) has completed here, i.e. EVERY thread of the cluster has issued its
  //     column sends of image it, which follow its last read of Q;
  //   A of every peer (exchange 2 of it): explicit credits - each warp arrives on every peer's `afree` after its inverse-row
  //     reads of image it-1 (relaxed remote arrive: nothing it wrote has to be published, its reads have returned).
  const int n_img = (cluster_id < p.B) ? (p.B - cluster_id + n_clusters - 1) / n_clusters : 0;
  uint32_t mbits = 0;                                    // packed mask of the image whose rows were sent last
  F2_PHASE_BEGIN();
  for (int it = -1; it < n_img; ++it) {
    const int b = cluster_id + it * n_clusters;          // the image whose columns / inverse rows run in this iteration
    const size_t img = size_t(b) * kClN * kClN;
    const bool has_next = it + 1 < n_img;
    const uint32_t par = uint32_t(it) & 1u;

    if (it >= 0) {
      mbar_wait(bfull, par);
      if (tid == 0 && has_next) mbar_arrive_expect_tx(bfull, uint32_t(BUF) * 8);   // next image's exchange 1 (no peer sends it
      F2_PHASE(3);                                       //   before my columns of this image, sent below, have arrived there)
      // ================= columns: forward, blend, inverse - in place in Q; results -> peers' row buffers =================
      const float mu = __ldg(p.mu + size_t(b) * p.mu_stride);
      const int col = row0 + cc;                         // kappa_j
      const float bb = 1.f / (1.f + mu), aa = mu * bb;
      float2 v[16];
#pragma unroll
      for (int r = 0; r < 16; ++r) v[r] = bufQ[cl_q_idx(jc + 16 * r, cc)];
      dft16t<false>(v);
      twiddle16<false>(v, wf, jc);
#pragma unroll
      for (int q = 0; q < 16; ++q) bufQ[cl_q_idx(jc + 16 * q, cc)] = v[q];
      __syncwarp();                                      // the column's 16 threads are one half-warp: no CTA barrier
#pragma unroll
      for (int r = 0; r < 16; ++r) v[r] = bufQ[cl_q_idx(r + 16 * jc, cc)];
      dft16t<false>(v);                                  // v[q] = H[kappa_i = jc + 16 q][kappa_j = col]
      // the sampled k-space values (L2 hits after the prefetch in the row phase) are loaded where they are used: requesting them one
      // transform earlier kept 32 more registers live through it (measured: 759 vs 755 us; before the first pass: spills, 786 us)
      float2 y[16];
      {
        const float2* yp = p.y0R + img + size_t(col) * kClN + jc;        // y0R is stored [kappa_j][kappa_i]: lanes contiguous
#pragma unroll
        for (int q = 0; q < 16; ++q) y[q] = ((mbits >> q) & 1u) ? __ldg(yp + 16 * q) : make_float2(0.f, 0.f);
      }
#pragma unroll
      for (int q = 0; q < 16; ++q)
        if ((mbits >> q) & 1u) v[q] = make_float2(aa * v[q].x + bb * y[q].x, aa * v[q].y + bb * y[q].y);
      dft16t<true>(v);
      twiddle16<true>(v, wf, jc);
#pragma unroll
      for (int q = 0; q < 16; ++q) bufQ[cl_q_idx(q + 16 * jc, cc)] = v[q];
      __syncwarp();
#pragma unroll
      for (int r = 0; r < 16; ++r) v[r] = bufQ[cl_q_idx(jc + 16 * r, cc)];
      dft16t<true>(v);                                   // v[q] = column-inverse at image row jc + 16 q
      F2_PHASE(4);                                       // columns
      if (it > 0) mbar_wait(afree, (uint32_t(it) - 1u) & 1u);   // every peer is done with the previous image's A
      F2_PHASE(1);                                       // wait for the A credits
      // exchange 2: element (row i = jc + 16 q, col) -> CTA q, slot cl_a_idx(jc, rank, cc) of its A: the 16 lanes write one
      // (permuted) 128-byte segment, the two half-warps of a warp adjacent segments
      const uint32_t dst0 = smem_u32(bufA + cl_a_idx(jc, int(rank), cc));
#pragma unroll
      for (int q = 0; q < 16; ++q) cl_st_async(cl_mapa(dst0, q), v[q], cl_mapa(afull_a, q));
      F2_PHASE(5);                                       // column sends
    }

    if (has_next) {
      // ================= rows forward of the NEXT image: shared (bulk-loaded) -> registers -> peers' column buffers =========
      const int bn = b + n_clusters;
      const size_t imgn = size_t(bn) * kClN * kClN;
      mbar_wait(tmafull, par ^ 1u);
      F2_PHASE(0);                                       // wait for the bulk loads of u and x
      const float2* Ur = bufU + hw * kClN;
      const float* Xr = X + hw * kClN;
      float2 v[16];
#pragma unroll
      for (int r = 0; r < 16; ++r) {
        const float2 uu = Ur[j + 16 * r];
        v[r] = make_float2(Xr[j + 16 * r] + uu.x, uu.y);
      }
      {                                                  // w stays in tensor memory until the epilogue of that image
        uint32_t wr[32];
#pragma unroll
        for (int r = 0; r < 16; ++r) { wr[2 * r] = __float_as_uint(v[r].x); wr[2 * r + 1] = __float_as_uint(v[r].y); }
        tmem_st_32x32(tmem_w + (par ^ 1u) * kTmemCols, wr);
      }
      __syncwarp();                                      // the row's own storage in U becomes the transform's scratch
      fft256_row_blocked<kClN, false>(v, bufU + hw * kClN, wf, j);  // v[r] = H[row][16 r + j]
      // the blend of that image reads y0R under the mask: pull exactly those elements' sectors into L2 now
      mbits = __ldg(p.mpack + size_t(bn) * p.mpack_bstride + (row0 + cc) * 16 + jc);
      {
        const float2* yp = p.y0R + imgn + size_t(row0 + cc) * kClN + jc;
#pragma unroll
        for (int q = 0; q < 16; ++q)
          if ((mbits >> q) & 1u) asm volatile("prefetch.global.L2 [%0];" ::"l"(yp + 16 * q));
      }
      F2_PHASE(2);                                       // rows forward
      if (it >= 0) mbar_wait(afull, par);                // columns of image it have arrived: every peer's Q is free (see above)
      if (tid == 0) mbar_arrive_expect_tx(afull, uint32_t(BUF) * 8);   // exchange 2 of the next image cannot start before my rows left
      F2_PHASE(6);                                       // wait for the peers' columns
      // exchange 1: element (row, col = 16 r + j) -> CTA r, slot cl_q_idx(row0 + hw, j) of its Q: the 16 lanes write one
      // (permuted) 128-byte segment, the two half-warps of a warp adjacent rows
      const uint32_t dst0 = smem_u32(bufQ + cl_q_idx(row0 + hw, j));
#pragma unroll
      for (int r = 0; r < 16; ++r) cl_st_async(cl_mapa(dst0, r), v[r], cl_mapa(bfull_a, r));
      // (reporting "this warp is done with U, X" on a local mbarrier that only thread 0 waits for, instead of this CTA
      // barrier, was measured: 781 vs 759 us at B = 1024 - the barrier keeps the warps of the two co-resident CTAs in step)
      fence_proxy_async_smem();                          // my scratch writes to U are ordered before the bulk load that refills it
      __syncthreads();
      if (tid == 0 && it + 2 < n_img) {                  // every thread is past the row phase: u and x buffers are free
        const size_t g = imgn + size_t(n_clusters) * kClN * kClN + size_t(row0) * kClN;
        mbar_arrive_expect_tx(tmafull, kRowBytesU + kRowBytesX);
        bulk_load_1d(bufU, p.u_in + g, kRowBytesU, tmafull);
        bulk_load_1d(X, p.x + g, kRowBytesX, tmafull);
      }
      F2_PHASE(7);                                       // row sends
    } else {
      mbar_wait(afull, par);                             // last image (it >= 0 here: a cluster has at least one image)
      F2_PHASE(6);
    }

    if (it >= 0) {
      // ================= rows inverse: A -> registers -> epilogue -> global =================
      float2 v[16];
#pragma unroll
      for (int r = 0; r < 16; ++r) v[r] = bufA[cl_a_idx(hw, r, j)];    // element (row hw, col = j + 16 r)
      __syncwarp();
      fft256_row_swz<true>(v, bufA, wf, j, hw);
      if (has_next && (tid & 31) < CL)                   // credit: this warp no longer reads A (v depends on every value it loaded)
        asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cl_mapa(afree_a, uint32_t(tid & 31))),
                     "r"(__float_as_uint(v[0].x))
                     : "memory");
      uint32_t wr[32];
      tmem_st_wait();
      tmem_ld_32x32(tmem_w + par * kTmemCols, wr);
      tmem_ld_wait();
      const size_t g0 = img + size_t(row0 + hw) * kClN + j;
      if (!(p.active && p.active[b] == 0)) {
#pragma unroll
        for (int r = 0; r < 16; ++r) {
          const float2 zz = make_float2(v[r].x * inv2, v[r].y * inv2);
          const float2 un = make_float2(__uint_as_float(wr[2 * r]) - zz.x, __uint_as_float(wr[2 * r + 1]) - zz.y);   // u' = u + x - z
          p.z_out[g0 + 16 * r] = zz;
          p.u_out[g0 + 16 * r] = un;
          if (p.v_out) p.v_out[g0 + 16 * r] = zz.x - un.x;                // Re(z - u')
        }
      }
      F2_PHASE(8);                                       // rows inverse + epilogue
#ifdef PNP_PROX_PHASE_TIMING
      if (tid == 0) atomicAdd(&g_f2_phase[15], 1ull);
#endif
    }
  }
  tc_fence_before();
  cl_cluster_arrive_relaxed();                           // no CTA leaves while a peer may still write to its shared memory
  cl_cluster_wait();
  if (warp == 1) tmem_dealloc(*tmem_slot, kTmemAlloc);
}

// Trajectory constants of the cluster kernel (see "Algebra"): y0R and the packed rotated mask.  grid (256, B), 256 threads.
__global__ void __launch_bounds__(256) prox_prepare_cl_kernel(const float2* __restrict__ y0, const uint8_t* __restrict__ mask,
                                                              long long mask_bstride, float2* __restrict__ y0R,
                                                              uint16_t* __restrict__ mpack, int nb_mask,
                                                              const int* skip_flag) {
  if (skip_flag && *skip_flag != 0) return;            // column-only masks: the row-only kernel needs none of this
  const int b = blockIdx.y, ki = blockIdx.x, kj = threadIdx.x;
  const size_t img = size_t(b) * kClN * kClN;
  const int si = (ki + 128) & 255, sj = (kj + 128) & 255;
  const float2 y = y0[img + size_t(si) * kClN + sj];
  const float s = ((ki + kj) & 1) ? -256.f : 256.f;
  y0R[img + size_t(kj) * kClN + ki] = make_float2(s * y.x, s * y.y);      // stored [kappa_j][kappa_i] (see the column phase)
  if (b < nb_mask && ki < 16) {                          // entry (jj = ki, kappa_j = kj)
    const uint8_t* mk = mask + size_t(b) * mask_bstride + sj;
    uint32_t bits = 0;
#pragma unroll
    for (int q = 0; q < 16; ++q) bits |= (mk[size_t((ki + 16 * q + 128) & 255) * kClN] ? 1u : 0u) << q;
    mpack[size_t(b) * 16 * kClN + kj * 16 + ki] = uint16_t(bits);
  }
}

// cudaOccupancyMaxActiveClusters of the real kernel (128 registers x 256 threads x 2 CTAs = the whole register file) answers 7
// for 16-CTA clusters where the hardware runs 14 at once (measured: forcing 14 is 1.3x faster, 15 falls off a cliff); a probe
// with the same block size and shared memory but few registers gives the figure the hardware follows (tools/cluster_occ.cu).
template <int CL> __global__ void __launch_bounds__(ClCfg<CL>::THREADS) cl_occupancy_probe(int* p) {
  extern __shared__ int probe_sm[];
  if (p) p[0] = probe_sm[0];
}

// Launch of a persistent cluster kernel (one image per cluster at a time) with every cluster that can be resident, at
// most one per image.  `Probe` stands in for `Kernel` in the occupancy query (see cl_occupancy_probe).
template <void (*Kernel)(ClParams), void (*Probe)(int*)>
static int launch_resident_clusters(const ClParams& p, int cl, int threads, size_t smem, cudaStream_t st) {
  static bool attr_done = false;
  if (!attr_done) {
    for (const void* f : {reinterpret_cast<const void*>(Kernel), reinterpret_cast<const void*>(Probe)}) {
      cudaError_t e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
      if (e == cudaSuccess && cl > 8) e = cudaFuncSetAttribute(f, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
      if (e != cudaSuccess) return int(e);
    }
    attr_done = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(cl * 64);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cl;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  // (default cluster scheduling policy: load balancing reports a 15th 16-CTA cluster that never becomes resident with the
  // 256x256 kernel's register use, and the launch falls off a wave cliff - profiles/r02_prox_cl_steps.txt)
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;                                      // the occupancy query below does not take the PDL attribute
  static int max_clusters = 0;
  if (max_clusters == 0) {
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, Probe, &cfg) != cudaSuccess || n < 1) {
      (void)cudaGetLastError();
      n = 1;
    }
    max_clusters = n;
  }
  int clusters = max_clusters < p.B ? max_clusters : p.B;
  if (clusters < 1) clusters = 1;
  // all resident clusters are used even when the last round is partial (evening the rounds out - the smallest cluster count
  // with the same number of rounds - was right for the unpipelined kernel; now the clusters of a partial last round run with
  // less contention, all resident vs evened out: 256x256 B = 20: 21.6 vs 27.8 us, B = 100: 84.2 vs 89.9 us, B = 64: 59.0 vs
  // 59.8 us; 128x128 B = 100: 21.8 vs 28.7 us, B = 1024: 192.0 vs 197.3 us)
  cfg.gridDim = dim3(clusters * cl);
  cfg.numAttrs = 2;
  return int(cudaLaunchKernelEx(&cfg, Kernel, p));
}

static int launch_cl(const ClParams& p, cudaStream_t st) {
  return launch_resident_clusters<fftprox_cl_kernel<16>, cl_occupancy_probe<16>>(p, 16, ClCfg<16>::THREADS, ClCfg<16>::SMEM,
                                                                                  st);
}

}  // namespace pnp
