/* libpnp_b200 - C-ABI of the B200-native PnP-ADMM CS-MRI environment step.
 *
 * The reference (joesharratt1229/DT4Image_Restoration) is pure Python/PyTorch and has no FFI; these entry
 * points are what a binding for its hot path would bind.  Each one cites the reference code it replaces.
 * Conventions (SURVEY.md section 8b):
 *   - plain pointers and sizes only; every data pointer is a DEVICE pointer owned by the caller;
 *   - every call is asynchronous on the caller-supplied `stream` (a cudaStream_t passed as void*), performs
 *     no allocation and no synchronisation (pnp_init and plan creation excepted);
 *   - return value: 0 = ok, <0 = argument error, >0 = cudaError_t / 1000+CUresult; text via pnp_last_error();
 *   - complex64 tensors are interleaved (re, im) float pairs, i.e. torch.complex64 / float2;
 *   - images are [B, H, W] row-major (the reference's [B,1,H,W] with the singleton channel dropped).
 * Built for sm_100a only.  There is no CPU fallback.
 */
#ifndef PNP_B200_H_
#define PNP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pnp_unet_plan pnp_unet_plan;

/* One-time per-process setup: twiddle tables, kernel attributes, TMA driver entry point. */
int pnp_init(void);
/* Last error message of the calling thread ("" if none). */
const char* pnp_last_error(void);
int pnp_num_sms(void);
int pnp_abi_version(void);

/* Reward: replaces torch_psnr (evaluation/env.py:120-125) as called by PnPEnv.compute_reward (env.py:112-116):
 * out[b] = 10*log10(1 / mean((clamp(x[b],0,1) - gt[b])^2)).  gt_batch_stride = H*W, or 0 to share one gt. */
int pnp_psnr(const float* x, const float* gt, long long gt_batch_stride, float* out, int B, int HW, void* stream);

/* Reward + all-gather in ONE kernel over NVLink peer memory: the exchange a multi-GPU tree search needs for its global
 * selection (select_p_ucb / backprop over all candidates, evaluation/mcts.py:74-88,34-38; the reference is single-process).
 * Every rank owns one copy of a symmetric buffer of (2*world*slot_floats + 1) 4-byte words, zero-initialised before the
 * first call, and peer_base[p] (HOST array, `world` entries) is the address of rank p's copy as mapped into this process:
 *   floats [parity][rank][slot_floats] gathered rewards (double-buffered by call parity), word flag_word = arrival counter.
 * Call number n = 1, 2, ... (the same on all ranks): parity = n & 1, flag_target = world * n, count_target = total B
 * over all calls so far including this one (local_count: zero-initialised device word; err_flag: device int set to 1 if
 * a rank has not arrived after 10 s).  When the kernel completes, rank r's rewards of this call are in
 * floats [parity][r][0..B_r) of the local copy.  out_local (may be NULL) also receives the local rewards.  world <= 8. */
int pnp_psnr_allgather(const float* x, const float* gt, long long gt_batch_stride, float* out_local,
                       const unsigned long long* peer_base, int rank, int world, int slot_floats, int parity,
                       int flag_word, unsigned int* local_count, unsigned int count_target, unsigned int flag_target,
                       int* err_flag, int B, int HW, void* stream);

/* Image-quality metric next to the PSNR reward: SSIM per image.  The reference ships `calculate_ssim`
 * (evaluation/utils/transformations.py:61-95) but never calls it; this is the standard SSIM of Wang et al. (2004) in the
 * form of pytorch-msssim / BasicSR, and parity with that function is not claimed:
 *   X = clamp(x[b], 0, 1), Y = gt[b] (not clamped, as in pnp_psnr);  g[k] = exp(-(k-5)^2 / 4.5) / sum, k = 0..10, applied
 *   separably with VALID filtering ((H-10) x (W-10) map, no padding);  mu_x = g*X, mu_y = g*Y, s_xx = g*(X.X) - mu_x^2,
 *   s_yy = g*(Y.Y) - mu_y^2, s_xy = g*(X.Y) - mu_x mu_y (population moments);  C1 = 0.01^2, C2 = 0.03^2 (L = 1);
 *   out[b] = mean of ((2 mu_x mu_y + C1)(2 s_xy + C2)) / ((mu_x^2 + mu_y^2 + C1)(s_xx + s_yy + C2)).
 * gt_batch_stride = H*W, or 0 to share one gt.  out: fp32 [B].  H, W >= 11, no upper limit.  workspace:
 * pnp_ssim_workspace_bytes(B,H,W) bytes, 16-byte aligned.  The value of an image is bitwise the same on every call and at
 * any position of any batch (the summation order depends on H and W only). */
size_t pnp_ssim_workspace_bytes(int B, int H, int W);
int pnp_ssim(const float* x, const float* gt, long long gt_batch_stride, float* out, void* workspace, int B, int H, int W,
             void* stream);

/* Centred orthonormal 2-D FFT / inverse FFT: replaces fft / ifft (evaluation/utils/transformations.py:6-12,
 * 14-19).  H, W in 2..1024: radix kernels for powers of two in 32..512, a dense-DFT path for every other size (torch.fft
 * is mixed-radix, so the reference accepts them).  dst may alias src. */
int pnp_fft2c(const void* src_c64, void* dst_c64, int B, int H, int W, int inverse, void* stream);

/* Episode generation on the device: undersampled, noisy k-space measurements of fully-sampled images (what the reference
 * loads from precomputed .mat items, dataset/datasets.py:148-168; synth.make_item is the host-side NumPy version).
 * Per image b, with fft_c / ifft_c the centred orthonormal transforms (transformations.py:6-19), and every index (i, j) in
 * the centred k-space layout of y0:
 *   p = i*W + j
 *   (w0, w1, _, _) = philox4x32_10(counter = (p, 0, 0, 0), key = (lo32(seed[b]), hi32(seed[b])))
 *   u1 = (w0 + 0.5) * 2^-32,   u2 = (w1 + 0.5) * 2^-32
 *   n_r = sqrt(-2 ln u1) * cos(2 pi u2),   n_i = sqrt(-2 ln u1) * sin(2 pi u2)
 *   y0[b,i,j]   = mask[b,i,j] != 0 ? fft_c(gt[b])[i,j] + (sigma_n[b] / 255) * (n_r + i*n_i) : 0
 *   ATy0[b]     = ifft_c(y0[b])
 *   x0[b]       = (max(Re ATy0, 0), max(Im ATy0, 0))          # datasets.py:160,199 / synth.make_item
 * philox4x32_10 is the Random123 generator: 10 rounds of
 *   (c0, c1, c2, c3) -> (hi(M1*c2) ^ c1 ^ k0, lo(M1*c2), hi(M0*c0) ^ c3 ^ k1, lo(M0*c0)),  M0 = 0xD2511F53, M1 = 0xCD9E8D57,
 * with the key bumped by (0x9E3779B9, 0xBB67AE85) between rounds.  The noise depends only on (seed, H, W, i, j): not on the
 * mask, the batch position or the other images.  With sigma_n[b] == 0, y0 = mask . fft_c(gt).
 * gt: fp32 [B,H,W] with gt_batch_stride = H*W, or one [H,W] with stride 0; mask: uint8 likewise; sigma_n: device fp32,
 * sigma_n[b*sigma_stride] (0 = one value for the batch); seeds: device uint64 [B].  Outputs c64 [B,H,W]; aty0_out may be
 * NULL.  H, W in 2..1024 (radix kernels for powers of two in 32..512, dense DFT otherwise); no workspace; outputs must not
 * overlap each other, gt or mask.  Results are bitwise reproducible and independent of the batch position. */
int pnp_simulate_measurements(const float* gt, long long gt_batch_stride, const uint8_t* mask, long long mask_batch_stride,
                              const float* sigma_n, int sigma_stride, const unsigned long long* seeds,
                              void* y0_out_c64, void* x0_out_c64, void* aty0_out_c64, int B, int H, int W, void* stream);

/* Seeded Cartesian undersampling masks (the structure of synth.cartesian_mask, drawn with the generator above).  Per image b:
 *   n_keep = max(1, W / accel[b]) (integer division);  n_acs = min(n_keep, acs_cols);  c0 = W/2 - n_acs/2
 *   columns [c0, c0 + n_acs) are sampled (ACS band);
 *   key_j = philox4x32_10(counter = (j, 1, 0, 0), key = seed split as above).w0  for every column j;
 *   the n_keep - n_acs non-ACS columns with the smallest (key_j, j), compared lexicographically, are sampled;
 *   mask[b, i, j] = 1 for every row i of a sampled column, else 0.
 * accel: device int32, accel[b*accel_stride] (accel < 1 samples every column); seeds: device uint64 [B]; mask_out: uint8
 * [B,H,W].  H, W in 2..1024, acs_cols >= 1 (synth.cartesian_mask uses max(1, round(0.08 W))).  These masks depend on the
 * column index only, so pnp_prox_prepare routes them to the row-only prox kernel. */
int pnp_cartesian_masks(const int* accel, int accel_stride, const unsigned long long* seeds, int acs_cols, uint8_t* mask_out,
                        int B, int H, int W, void* stream);

/* Seeded golden-angle radial masks (synth.radial_mask's lines, rotated per image).  Per image b, in float64:
 *   cy = H / 2, cx = W / 2 (integer division);  R = 1 + the smallest integer r with 4 r^2 >= H^2 + W^2
 *   golden = 0x1.f10d6bc8e0e35p+0 (pi (sqrt 5 - 1) / 2 as NumPy computes it)
 *   phi = 0 if seeds == NULL, else double(philox4x32_10(counter = (0, 2, 0, 0), key = seed[b] split as above).w0)
 *         * 0x1.921fb54442d18p-31 (pi * 2^-32, so phi is in [0, pi))
 *   target = (frac[b*frac_stride] * H) * W;  count = 0, n = 0
 *   while count < target and n < 8 * max(H, W):
 *       ang = n * golden + phi                                    (two roundings, no FMA)
 *       for t in -R .. R:  y = rint(cy + t sin(ang)),  x = rint(cx + t cos(ang))   (each op rounded, no FMA; rint rounds
 *           half to even);  if 0 <= y < H and 0 <= x < W: mask[b, y, x] = 1
 *       count = number of sampled pixels of image b;  n += 1
 *   lines_out[b] = n
 * With seeds == NULL the mask is exactly synth.radial_mask(H, W, frac).  frac <= 0 or NaN draws no line; frac > 1 runs to the
 * 8 max(H, W) line cap.  Counter word 1 = 2 keeps this stream apart from the noise (word 1 = 0) and the Cartesian column
 * keys (word 1 = 1).  frac: device float64 (0 stride = one value for the batch); seeds: device uint64 [B] or NULL;
 * mask_out: uint8 [B,H,W]; lines_out: device int32 [B] or NULL.  H, W in 2..1024; the outputs must not overlap each other,
 * frac or seeds.  Results are bitwise reproducible and independent of the batch position. */
int pnp_radial_masks(const double* frac, int frac_stride, const unsigned long long* seeds, uint8_t* mask_out,
                     int* lines_out, int B, int H, int W, void* stream);

/* Seeded 2-D variable-density random masks (Lustig, Donoho and Pauly, 2007): dense near the k-space centre, sparser
 * towards the edge, with exactly max(n_keep, |ACS|) sampled pixels.  Per image b, for every index (i, j) in the centred
 * k-space layout, in float64 with every operation rounded on its own (no FMA):
 *   cy = H / 2,  cx = W / 2                                   (integer division; H, W >= 2 so both >= 1)
 *   ky = (i - cy) / cy,   kx = (j - cx) / cx                  (both in [-1, 1])
 *   r  = sqrt(0.5 * (ky*ky + kx*kx))                          (in [0, 1]; r = 1 only where |ky| = |kx| = 1)
 *   w  = 1; repeat `power` times: w = w * (1 - r)             (power 0: w = 1, uniform sampling)
 *   p  = i*W + j
 *   u  = (philox4x32_10(counter = (p, 3, 0, 0), key = (lo32(seed[b]), hi32(seed[b]))).w0 + 0.5) * 2^-32
 *   key[p] = float32(u / w)                                   (round to nearest; w = 0 or overflow gives +inf)
 *   n_keep = accel[b] >= 1 ? max(1, (H*W) / accel[b]) : H*W  (integer division; same rule as pnp_cartesian_masks)
 *   ACS    = rows [cy - acs_h/2, cy - acs_h/2 + acs_h) x columns [cx - acs_w/2, cx - acs_w/2 + acs_w)
 *   mask[b] = 1 on ACS, plus on the max(0, n_keep - |ACS|) pixels outside ACS with the smallest (key[p], p),
 *             compared lexicographically; 0 elsewhere
 * Selecting the smallest u/w is Bernoulli sampling of pixel p when u_p <= t w_p, with the threshold t that makes the count
 * exact: the density (1 - r)^power, scaled to the sample budget.  Counter word 1 = 3 keeps this stream apart from the
 * noise (0), the Cartesian column keys (1) and the radial rotation (2).  The key uses only + - * /, sqrt and the double ->
 * float rounding, so a NumPy restatement reproduces the masks bit for bit.  accel: device int32, accel[b*accel_stride]
 * (0 stride = one value for the batch); seeds: device uint64 [B]; mask_out: uint8 [B,H,W], must not overlap accel or
 * seeds.  H, W in 2..1024, 0 <= acs_h <= H, 0 <= acs_w <= W, 0 <= power <= 16.  Results are bitwise reproducible and
 * independent of the batch position.  These masks are general (not column-only, unless every pixel is sampled), so
 * pnp_prox_prepare routes them to the cluster prox kernel. */
int pnp_variable_density_masks(const int* accel, int accel_stride, const unsigned long long* seeds, int acs_h, int acs_w,
                               int power, uint8_t* mask_out, int B, int H, int W, void* stream);

/* v = Re(z - u): the denoiser input of PnPEnv.step (env.py:85-86). */
int pnp_residual_real(const void* z_c64, const void* u_c64, float* v, long long n, void* stream);

/* Data-fidelity prox + dual update: replaces env.py:87-93
 *     z = ifft(blend(fft(x + u))), blend(Z)[mask] = (mu*Z + y0)[mask] / (1 + mu);   u_out = u_in + x - z
 * and emits v_next = Re(z - u_out) (next step's env.py:85) when v_next != NULL.
 * mask: uint8 (0/1) [B,H,W] with mask_batch_stride = H*W, or one [H,W] mask with stride 0.
 * mu: device fp32, mu[b*mu_stride]; mu_stride = 0 reproduces the reference's scalar mu (env.py:88).
 * u_out may alias u_in.  workspace: pnp_prox_workspace_bytes(B,H,W) bytes, 16-byte aligned.  H, W in 2..1024 (as pnp_fft2c). */
size_t pnp_prox_workspace_bytes(int B, int H, int W);
int pnp_prox_dual(const float* x, const void* u_in_c64, const void* y0_c64, const uint8_t* mask,
                  long long mask_batch_stride, const float* mu, int mu_stride, void* z_out_c64, void* u_out_c64,
                  float* v_next, void* workspace, int B, int H, int W, void* stream);

/* Prepared variant (pnp_prox_prepared_supported: 256x256): y0 and the mask are constants of a trajectory (set in
 * PnPEnv.reset, env.py:64-66), so everything that depends only on them is computed ONCE by pnp_prox_prepare into two
 * caller-owned device buffers whose sizes pnp_prox_prepared_bytes returns:
 *   y0p   : y0 transposed and sign-folded (c64 [B,W,H]) for the general single-launch cluster kernel, followed by
 *           Yt = Fc^-1(s*D.y0) (c64 [B,H,W]) for the row-only kernel;
 *   maskp : the transposed mask (uint8 [B or 1,W,H]), the packed row mask and a device flag saying whether every mask of
 *           the batch depends on the column index only (Cartesian undersampling, fully sampled columns).
 * pnp_prox_dual_prepared then runs, per iteration, the row-only kernel (half the FFT work, no transposes; csrc/
 * fftprox_sep.cuh) when the flag is set and the general cluster kernel otherwise - both are launched, the one whose case
 * it is not exits immediately, so nothing synchronises with the host.  Results equal pnp_prox_dual's to rounding. */
int pnp_prox_prepared_supported(int H, int W);
int pnp_prox_prepared_bytes(int B, int H, int W, size_t* y0p_bytes, size_t* maskp_bytes);
int pnp_prox_prepare(const void* y0_c64, const uint8_t* mask, long long mask_batch_stride, void* y0T_c64, uint8_t* maskT,
                     int B, int H, int W, void* stream);
int pnp_prox_dual_prepared(const float* x, const void* u_in_c64, const void* y0T_c64, const uint8_t* maskT,
                           long long mask_batch_stride, const float* mu, int mu_stride, void* z_out_c64,
                           void* u_out_c64, float* v_next, int B, int H, int W, void* stream);

/* Host-side copy of the mask-structure flag (1 = every mask of the batch depends on the column index only, 0 = general):
 * enqueues an asynchronous 4-byte device-to-host copy into *kind_host (pinned host memory; valid once the work enqueued on
 * `stream` so far has completed - record an event, do not synchronise).  Passing the value as `kind` to the _kind variants
 * launches only the kernel whose case it is (kind = -1: both are launched and the device flag decides, as in
 * pnp_prox_dual_prepared).  The flag is a constant of a trajectory (set by pnp_prox_prepare from env.py:64's mask). */
int pnp_prox_prepared_kind_async(const uint8_t* maskT, long long mask_batch_stride, int B, int H, int W, int* kind_host,
                                 void* stream);
int pnp_prox_dual_prepared_kind(const float* x, const void* u_in_c64, const void* y0T_c64, const uint8_t* maskT,
                                long long mask_batch_stride, const float* mu, int mu_stride, void* z_out_c64,
                                void* u_out_c64, float* v_next, int B, int H, int W, int kind, void* stream);

/* U-Net denoiser: replaces UNetDenoiser2D.forward (evaluation/noise.py:155-164) and UNet.forward
 * (noise.py:119-133).  Weights arrive as the reference state_dict (noise.py:147-148) flattened to one fp32
 * device vector in module-registration order (pnp_unet_num_params() floats: for inc, down1-4, up1-4:
 * conv-0/1/2 weight then bias; then outc weight, bias) and are repacked once to bf16 tensor-core tiles. */
size_t pnp_unet_num_params(void);
size_t pnp_unet_packed_bytes(void);
int pnp_unet_pack_weights(const float* flat_params, void* packed, void* stream);
/* The denoiser runs in micro-batches that share one workspace, so this is bounded (<= 8 GiB, or one image's worth) for any B. */
size_t pnp_unet_workspace_bytes(int B, int H, int W);
/* packed and workspace must be 1024-byte aligned and outlive the plan. */
int pnp_unet_plan_create(pnp_unet_plan** plan, const void* packed, void* workspace, size_t workspace_bytes, int B,
                         int H, int W);
void pnp_unet_plan_destroy(pnp_unet_plan* plan);
/* x_out[b] = clamp(v[b] + residual, 0, 1); preclamp (optional) receives v + residual. sigma: [B] device fp32. */
int pnp_unet_forward(pnp_unet_plan* plan, const float* v, const float* sigma, float* x_out, float* preclamp,
                     void* stream);
/* Profiling pass (SYNCHRONISES the stream): one forward with a CUDA-event pair around every launch.  On return
 * ms[i], kinds[i] (0 first conv, 1 tcgen05 conv, 3 upsample) and ids[i] (conv: layer 0..26 in state_dict order;
 * upsample: 200+level) describe launch i; *n_inout = capacity in, count out. */
int pnp_unet_profile(pnp_unet_plan* plan, const float* v, const float* sigma, float* x_out, void* stream, float* ms,
                     int* kinds, int* ids, int* n_inout);
/* Kernel launches one pnp_unet_forward issues for this plan (all micro-batches). */
int pnp_unet_num_launches(const pnp_unet_plan* plan);
/* Images per micro-batch of this plan (== B when the whole batch fits the workspace cap). */
int pnp_unet_micro_batch(const pnp_unet_plan* plan);
/* Process-wide activation-workspace budget of plans created from now on (default 8 GiB); returns the previous value
 * (bytes = 0 only queries).  pnp_unet_workspace_bytes follows it. */
size_t pnp_unet_set_workspace_cap(size_t bytes);
/* Kernel choice of the convs of plans / single convs created from now on: -1 (default) the split-K cluster kernel serves
 * launches with few output tiles (batch 1-4 at the deep levels), 0 never, 1 every eligible conv (parity tests).  Any other
 * value only queries.  Returns the previous mode. */
int pnp_unet_set_splitk(int mode);
/* Locate a named NHWC bf16 activation inside the workspace (layer-wise parity tests), e.g. "down2.conv-1".  Fails (-1) for
 * micro-batched plans, whose workspace holds one micro-batch at a time. */
int pnp_unet_plan_tensor(const pnp_unet_plan* plan, const char* name, size_t* byte_offset, int* C, int* H, int* W);
/* Per-launch window into a plan, for tests that check each launch alone.  Both fail (-1) for micro-batched plans.
 * pnp_unet_forward_ops runs launches [first_op, end_op) of pnp_unet_forward (0 <= first_op <= end_op <=
 * pnp_unet_num_launches); the launches read their inputs from the workspace as the earlier launches left it.
 * pnp_unet_op_describe writes PNP_UNET_OP_DESC_LEN values describing launch i to desc[]:
 *   [0] kind (0 first conv, 1 tcgen05 conv, 3 upsample)   [1] id, as pnp_unet_profile reports it
 *   [2] H, [3] W of the launch's output level
 *   [4] [5]  in0 workspace byte offset, channels      [6] [7]  in1 (second concat segment)
 *   [8] [9]  out                                      [10] [11] pool_out (fused MaxPool2d(2), H/2 x W/2)
 *            (offset and channels -1 where the launch has none or the tensor is not in the workspace: the first conv
 *             reads v and sigma, the FINAL conv writes x_out and preclamp)
 *   [12] kernel: 0 first conv, 1 conv3x3_umma, 2 conv3x3_umma FINAL epilogue, 3 kw-stacked, 4 CTA pair, 5 split-K
 *        cluster, 6 fast upsample (exact doubling), 7 general upsample (zero pad)
 *   [13] KC, or the cluster size S of the split-K kernel     [14] BN (output channels per tile)
 *   [15] rev (1: tiles walked in descending order)          [16] wres (1: weights resident in shared memory)
 *   [17] [18] output tile width, height in pixels          [19] work tiles (pair kernel: tile pairs)   [20] grid (CTAs)
 *   (fields 13, 14, 16 .. 20 are 0 for launches that are not tcgen05 convs) */
#define PNP_UNET_OP_DESC_LEN 21
int pnp_unet_forward_ops(pnp_unet_plan* plan, const float* v, const float* sigma, float* x_out, float* preclamp,
                         int first_op, int end_op, void* stream);
int pnp_unet_op_describe(const pnp_unet_plan* plan, int i, long long* desc);

/* One 3x3 conv + bias + LeakyReLU(0.2) on the tensor cores (reference ConvLayer, noise.py:75-89) on NHWC bf16
 * tensors; the input is the channel concat of in0 (C0 ch) and in1 (C1 ch, may be NULL/0) as in `up`
 * (noise.py:59).  weights fp32 [Cout][C0+C1][3][3].  scratch: pnp_conv3x3_packed_bytes() bytes, 1024-aligned. */
size_t pnp_conv3x3_packed_bytes(int Cin, int Cout);
int pnp_conv3x3_bf16(const void* in0, int C0, const void* in1, int C1, const float* weights, const float* bias,
                     void* out, void* scratch, int B, int H, int W, int Cout, void* stream);

/* The policy that produces the actions (SURVEY 8f row 1; reference transformer/decision_transformer.py:212-275 as driven by
 * evaluation/eval.py:147-186): ONE kernel per rollout iteration computes the action head at the newest observation token and,
 * with that action written into the context, the return head at the new action token (the reference runs two forwards).
 * packed: pnp_policy_packed_floats(n_time, n_task) fp32 words laid out as csrc/policy.cu:PolicyOffsets (GEMM weights
 * transposed to [in][out]); context window of K <= 6 entries: rtg [B,K,1], emb [B,K,128] (state-encoder outputs),
 * act [B,K,3] (in/out: entry *pos receives the new action), timesteps / task int64 [B,K], pos device int64 (newest entry).
 * act_out [B,3] = scaled actions in head order, rtg_out [B]. */
size_t pnp_policy_packed_floats(int n_time, int n_task);
int pnp_policy_step(const float* packed, const float* rtg, const float* emb, float* act, const long long* timesteps,
                    const long long* task, const long long* pos, float* act_out, float* rtg_out, float scale0, float scale1,
                    float scale2, int B, int K, int n_time, int n_task, void* stream);

/* Observation side of the same iteration (reference evaluation/eval.py:204-217 + transformer/decision_transformer.py:128-132,
 * 215) as ONE kernel: x [B,H,W] (H = W = 128 f) -> f x f area mean -> state encoder (3 convs + Linear 2304->128 + Tanh) ->
 * appended to each trajectory's context window (a full window first moves one entry to the left): the new entry gets
 * next_rtg [B], the encoding, an empty action and time step (*t_dev + 1) % n_time.  *pos / *t_dev are READ (newest entry and its
 * time step before the call); the caller advances them.  enc_packed: pnp_policy_encoder_packed_floats() fp32 words =
 * conv1 [ky][kx][co] | b | conv2 [ci][ky][kx][co] | b | conv3 [ci][ky][kx][co] | b | Linear [k][o] | b. */
size_t pnp_policy_encoder_packed_floats(void);
int pnp_policy_observe(const float* enc_packed, const float* x, int H, int W, const float* next_rtg, float* rtg, float* emb,
                       float* act, long long* timesteps, const long long* pos, const long long* t_dev, int B, int K,
                       int n_time, void* stream);

/* One whole PnPEnv.step body (env.py:85-93) for a batch: x = denoise(v, sigma); z,u = prox/dual; v_next. */
int pnp_step(pnp_unet_plan* plan, const float* v, const float* sigma, const void* u_in_c64, const void* y0_c64,
             const uint8_t* mask, long long mask_batch_stride, const float* mu, int mu_stride, float* x_out,
             void* z_out_c64, void* u_out_c64, float* v_next, void* prox_workspace, void* stream);

/* pnp_step with prepared y0T / maskT (see pnp_prox_prepare). */
int pnp_step_prepared(pnp_unet_plan* plan, const float* v, const float* sigma, const void* u_in_c64,
                      const void* y0T_c64, const uint8_t* maskT, long long mask_batch_stride, const float* mu,
                      int mu_stride, float* x_out, void* z_out_c64, void* u_out_c64, float* v_next, void* stream);

/* pnp_step_prepared with the host-side mask-structure hint (see pnp_prox_prepared_kind_async). */
int pnp_step_prepared_kind(pnp_unet_plan* plan, const float* v, const float* sigma, const void* u_in_c64,
                           const void* y0T_c64, const uint8_t* maskT, long long mask_batch_stride, const float* mu,
                           int mu_stride, float* x_out, void* z_out_c64, void* u_out_c64, float* v_next, int kind,
                           void* stream);

/* pnp_step_prepared_kind with a per-image predicate: active[b] == 0 leaves x_out, z_out, u_out, v_next of image b untouched
 * (the batched form of the reference's early exit `if T > 0.5: return states, True`, env.py:79-81).  The predicate is
 * applied in the epilogues of the last conv and of the prox kernels: no copies, no extra pass.  active: device uint8 [B]
 * or NULL (all active).  Outputs must alias the state to be kept (x_out = x, z_out = z, u_out = u_in, v_next = v). */
int pnp_step_prepared_active(pnp_unet_plan* plan, const float* v, const float* sigma, const void* u_in_c64,
                             const void* y0T_c64, const uint8_t* maskT, long long mask_batch_stride, const float* mu,
                             int mu_stride, float* x_out, void* z_out_c64, void* u_out_c64, float* v_next, int kind,
                             const uint8_t* active, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PNP_B200_H_ */
