// extern "C" entry points of libpnp_b200.so (declared in include/pnp_b200.h).
#include <mutex>
#include <string>
#include "../../include/pnp_b200.h"
#include "common.cuh"
#include "pnp_internal.h"

namespace pnp {
static thread_local std::string t_err;
void set_error(const std::string& msg) { t_err = msg; }
static std::once_flag g_once;
static int g_init_rc = -100;

static int fail_cuda(int rc, const char* where) {
  if (rc > 0 && rc < 1000) set_error(std::string(where) + ": " + cudaGetErrorString(cudaError_t(rc)));
  return rc;
}

__global__ void residual_real_kernel(const float2* __restrict__ z, const float2* __restrict__ u, float* __restrict__ v,
                                     long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    v[i] = z[i].x - u[i].x;
}
}  // namespace pnp

using namespace pnp;

// A plan runs the denoiser in micro-batches of at most `mb` images (impl) plus one remainder batch (tail), all on the SAME
// workspace, so the activation workspace is bounded for any B (BASELINE config 5 sweeps to B = 4096: one 32-channel
// full-resolution bf16 tensor alone would be 16 GiB at 256x256, SURVEY 7.3-5).
struct pnp_unet_plan {
  UnetPlan* impl;            // micro-batch of `mb` images (== B when the whole batch fits the cap)
  UnetPlan* tail;            // B % mb images, or null
  int B, H, W, mb;
};

namespace pnp {
static size_t kUnetWorkspaceCap = size_t(8) << 30;          // bytes; pnp_unet_set_workspace_cap
// largest micro-batch whose workspace stays under the cap, rounded down to a multiple of 8 images (>= 1)
static int unet_micro_batch(int B, int H, int W) {
  if (unet_workspace_bytes(B, H, W) <= kUnetWorkspaceCap) return B;
  const size_t per8 = unet_workspace_bytes(8, H, W);
  long long m = (long long)(kUnetWorkspaceCap / per8) * 8;
  if (m < 1) m = 1;                                          // a single image over the cap: still runs, one by one
  while (m > 1 && unet_workspace_bytes(int(m), H, W) > kUnetWorkspaceCap) m -= (m > 8 ? 8 : 1);
  return int(m < B ? m : B);
}
}  // namespace pnp

extern "C" {

int pnp_abi_version(void) { return 1; }

int pnp_init(void) {
  std::call_once(g_once, [] {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) { g_init_rc = int(e); set_error("no CUDA device"); return; }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, dev);
    if (prop.major != 10) {
      set_error("libpnp_b200 requires an sm_100a (B200) device; found sm_" + std::to_string(prop.major) +
                std::to_string(prop.minor));
      g_init_rc = -10;
      return;
    }
    init_fft_tables();
    int rc = unet_global_init();
    if (rc == 0) rc = int(cudaGetLastError());
    g_init_rc = rc;
  });
  return g_init_rc;
}

const char* pnp_last_error(void) { return t_err.c_str(); }
int pnp_num_sms(void) { return num_sms(); }

#define REQUIRE_INIT()                                          \
  if (g_init_rc != 0) {                                         \
    set_error("pnp_init() has not succeeded");                  \
    return -3;                                                  \
  }

int pnp_psnr(const float* x, const float* gt, long long gt_batch_stride, float* out, int B, int HW, void* stream) {
  REQUIRE_INIT();
  if (!x || !gt || !out) { set_error("pnp_psnr: null pointer"); return -1; }
  return fail_cuda(psnr_launch(x, gt, gt_batch_stride, out, B, HW, cudaStream_t(stream)), "pnp_psnr");
}

int pnp_psnr_allgather(const float* x, const float* gt, long long gt_batch_stride, float* out_local,
                       const unsigned long long* peer_base, int rank, int world, int slot_floats, int parity,
                       int flag_word, unsigned int* local_count, unsigned int count_target, unsigned int flag_target,
                       int* err_flag, int B, int HW, void* stream) {
  REQUIRE_INIT();
  if (!x || !gt || !peer_base || !local_count || !err_flag) { set_error("pnp_psnr_allgather: null pointer"); return -1; }
  if (world < 1 || world > 8 || rank < 0 || rank >= world || B > slot_floats) {
    set_error("pnp_psnr_allgather: need 1 <= world <= 8, 0 <= rank < world, B <= slot_floats");
    return -1;
  }
  return fail_cuda(psnr_allgather_launch(x, gt, gt_batch_stride, out_local, peer_base, rank, world, slot_floats, parity,
                                         flag_word, local_count, count_target, flag_target, err_flag, B, HW,
                                         cudaStream_t(stream)), "pnp_psnr_allgather");
}

size_t pnp_ssim_workspace_bytes(int B, int H, int W) { return ssim_workspace_bytes(B, H, W); }

int pnp_ssim(const float* x, const float* gt, long long gt_batch_stride, float* out, void* workspace, int B, int H, int W,
             void* stream) {
  REQUIRE_INIT();
  if (!x || !gt || !out || !workspace) { set_error("pnp_ssim: null pointer"); return -1; }
  if (B <= 0) { set_error("pnp_ssim: need B > 0"); return -1; }
  if (H < 11 || W < 11) { set_error("pnp_ssim: H and W must be at least 11 (11x11 window, valid filtering)"); return -2; }
  if (reinterpret_cast<uintptr_t>(workspace) & 15) { set_error("pnp_ssim: workspace must be 16-byte aligned"); return -1; }
  return fail_cuda(ssim_launch(x, gt, gt_batch_stride, out, workspace, B, H, W, cudaStream_t(stream)), "pnp_ssim");
}

int pnp_fft2c(const void* src, void* dst, int B, int H, int W, int inverse, void* stream) {
  REQUIRE_INIT();
  if (!src || !dst || B <= 0) { set_error("pnp_fft2c: bad argument"); return -1; }
  if (!fft_any_shape_supported(H, W)) { set_error("pnp_fft2c: H and W must be in [2, 1024]"); return -2; }
  return fail_cuda(fft2c_general(static_cast<const float2*>(src), static_cast<float2*>(dst), B, H, W, inverse,
                                 cudaStream_t(stream)), "pnp_fft2c");
}

// Byte ranges [lo, hi) of the buffers of pnp_simulate_measurements and the mask calls, for the overlap test.
static bool ranges_overlap(const void* a, size_t na, const void* b, size_t nb) {
  const uintptr_t pa = reinterpret_cast<uintptr_t>(a), pb = reinterpret_cast<uintptr_t>(b);
  return a && b && pa < pb + nb && pb < pa + na;
}

// The argument checks of the simulator and mask entry points come before REQUIRE_INIT, so a bad call is refused with its own
// message whether or not pnp_init has run.
int pnp_simulate_measurements(const float* gt, long long gt_batch_stride, const uint8_t* mask, long long mask_batch_stride,
                              const float* sigma_n, int sigma_stride, const unsigned long long* seeds, void* y0_out,
                              void* x0_out, void* aty0_out, int B, int H, int W, void* stream) {
  if (!gt || !mask || !sigma_n || !seeds || !y0_out || !x0_out) {
    set_error("pnp_simulate_measurements: null pointer");
    return -1;
  }
  if (B <= 0 || gt_batch_stride < 0 || mask_batch_stride < 0 || sigma_stride < 0) {
    set_error("pnp_simulate_measurements: need B > 0 and non-negative strides");
    return -1;
  }
  if (!fft_any_shape_supported(H, W)) { set_error("pnp_simulate_measurements: H and W must be in [2, 1024]"); return -2; }
  const size_t hw = size_t(H) * W, nout = size_t(B) * hw * sizeof(float2);
  const size_t ngt = (size_t(B - 1) * gt_batch_stride + hw) * sizeof(float);
  const size_t nmask = size_t(B - 1) * mask_batch_stride + hw;
  const void* outs[3] = {y0_out, x0_out, aty0_out};
  for (int k = 0; k < 3; ++k) {
    bool bad = ranges_overlap(outs[k], nout, gt, ngt) || ranges_overlap(outs[k], nout, mask, nmask);
    for (int q = k + 1; q < 3; ++q) bad |= ranges_overlap(outs[k], nout, outs[q], nout);
    if (bad) { set_error("pnp_simulate_measurements: outputs overlap each other, gt or mask"); return -1; }
  }
  REQUIRE_INIT();
  return fail_cuda(simulate_measurements(gt, gt_batch_stride, mask, mask_batch_stride, sigma_n, sigma_stride, seeds,
                                         static_cast<float2*>(y0_out), static_cast<float2*>(x0_out),
                                         static_cast<float2*>(aty0_out), B, H, W, cudaStream_t(stream)),
                   "pnp_simulate_measurements");
}

int pnp_cartesian_masks(const int* accel, int accel_stride, const unsigned long long* seeds, int acs_cols, uint8_t* mask_out,
                        int B, int H, int W, void* stream) {
  if (!accel || !seeds || !mask_out) { set_error("pnp_cartesian_masks: null pointer"); return -1; }
  if (B <= 0 || accel_stride < 0 || acs_cols < 1) {
    set_error("pnp_cartesian_masks: need B > 0, accel_stride >= 0 and acs_cols >= 1");
    return -1;
  }
  if (!fft_any_shape_supported(H, W)) { set_error("pnp_cartesian_masks: H and W must be in [2, 1024]"); return -2; }
  REQUIRE_INIT();
  return fail_cuda(cartesian_masks(accel, accel_stride, seeds, acs_cols, mask_out, B, H, W, cudaStream_t(stream)),
                   "pnp_cartesian_masks");
}

int pnp_radial_masks(const double* frac, int frac_stride, const unsigned long long* seeds, uint8_t* mask_out,
                     int* lines_out, int B, int H, int W, void* stream) {
  if (!frac || !mask_out) { set_error("pnp_radial_masks: null pointer"); return -1; }
  if (B <= 0 || frac_stride < 0) { set_error("pnp_radial_masks: need B > 0 and frac_stride >= 0"); return -1; }
  if (!fft_any_shape_supported(H, W)) { set_error("pnp_radial_masks: H and W must be in [2, 1024]"); return -2; }
  const size_t nmask = size_t(B) * H * W, nlines = size_t(B) * sizeof(int);
  const size_t nfrac = (size_t(B - 1) * frac_stride + 1) * sizeof(double), nseeds = size_t(B) * sizeof(unsigned long long);
  const bool bad = ranges_overlap(lines_out, nlines, mask_out, nmask) || ranges_overlap(mask_out, nmask, frac, nfrac) ||
                   ranges_overlap(mask_out, nmask, seeds, nseeds) || ranges_overlap(lines_out, nlines, frac, nfrac) ||
                   ranges_overlap(lines_out, nlines, seeds, nseeds);
  if (bad) { set_error("pnp_radial_masks: outputs overlap each other, frac or seeds"); return -1; }
  REQUIRE_INIT();
  return fail_cuda(radial_masks(frac, frac_stride, seeds, mask_out, lines_out, B, H, W, cudaStream_t(stream)),
                   "pnp_radial_masks");
}

int pnp_variable_density_masks(const int* accel, int accel_stride, const unsigned long long* seeds, int acs_h, int acs_w,
                               int power, uint8_t* mask_out, int B, int H, int W, void* stream) {
  if (!accel || !seeds || !mask_out) { set_error("pnp_variable_density_masks: null pointer"); return -1; }
  if (B <= 0 || accel_stride < 0) { set_error("pnp_variable_density_masks: need B > 0 and accel_stride >= 0"); return -1; }
  if (!fft_any_shape_supported(H, W)) { set_error("pnp_variable_density_masks: H and W must be in [2, 1024]"); return -2; }
  if (acs_h < 0 || acs_h > H || acs_w < 0 || acs_w > W || power < 0 || power > 16) {
    set_error("pnp_variable_density_masks: need 0 <= acs_h <= H, 0 <= acs_w <= W and 0 <= power <= 16");
    return -1;
  }
  const size_t nmask = size_t(B) * H * W, nseeds = size_t(B) * sizeof(unsigned long long);
  const size_t naccel = (size_t(B - 1) * accel_stride + 1) * sizeof(int);
  if (ranges_overlap(mask_out, nmask, accel, naccel) || ranges_overlap(mask_out, nmask, seeds, nseeds)) {
    set_error("pnp_variable_density_masks: mask_out overlaps accel or seeds");
    return -1;
  }
  REQUIRE_INIT();
  return fail_cuda(variable_density_masks(accel, accel_stride, seeds, acs_h, acs_w, power, mask_out, B, H, W,
                                          cudaStream_t(stream)), "pnp_variable_density_masks");
}

int pnp_residual_real(const void* z, const void* u, float* v, long long n, void* stream) {
  REQUIRE_INIT();
  long long g = (n + 255) / 256;
  if (g > 148 * 16) g = 148 * 16;
  if (g < 1) g = 1;
  residual_real_kernel<<<int(g), 256, 0, cudaStream_t(stream)>>>(static_cast<const float2*>(z),
                                                                 static_cast<const float2*>(u), v, n);
  return fail_cuda(int(cudaGetLastError()), "pnp_residual_real");
}

size_t pnp_prox_workspace_bytes(int B, int H, int W) { return size_t(B) * H * W * (sizeof(float2) + 1); }

int pnp_prox_prepared_supported(int H, int W) { return fft_shape_supported(H, W); }

int pnp_prox_prepared_bytes(int B, int H, int W, size_t* y0p_bytes, size_t* maskp_bytes) {
  if (!y0p_bytes || !maskp_bytes || B <= 0) { set_error("pnp_prox_prepared_bytes: bad argument"); return -1; }
  if (!pnp_prox_prepared_supported(H, W)) { set_error("pnp_prox_prepared_bytes: H and W must be powers of two in 32..512"); return -2; }
  prox_prepared_bytes(B, H, W, y0p_bytes, maskp_bytes);
  return 0;
}

int pnp_prox_prepare(const void* y0, const uint8_t* mask, long long mask_batch_stride, void* y0T, uint8_t* maskT, int B,
                     int H, int W, void* stream) {
  REQUIRE_INIT();
  if (!y0 || !mask || !y0T || !maskT) { set_error("pnp_prox_prepare: null pointer"); return -1; }
  if (!pnp_prox_prepared_supported(H, W)) { set_error("pnp_prox_prepare: H and W must be powers of two in 32..512"); return -2; }
  return fail_cuda(prox_prepare(static_cast<const float2*>(y0), mask, mask_batch_stride, static_cast<float2*>(y0T), maskT,
                                B, H, W, cudaStream_t(stream)), "pnp_prox_prepare");
}

int pnp_prox_prepared_kind_async(const uint8_t* maskT, long long mask_batch_stride, int B, int H, int W, int* kind_host,
                                 void* stream) {
  REQUIRE_INIT();
  if (!maskT || !kind_host) { set_error("pnp_prox_prepared_kind_async: null pointer"); return -1; }
  if (!pnp_prox_prepared_supported(H, W)) { set_error("pnp_prox_prepared_kind_async: unsupported shape"); return -2; }
  return fail_cuda(int(cudaMemcpyAsync(kind_host, prox_prepared_flag(maskT, mask_batch_stride, B, H, W), sizeof(int),
                                       cudaMemcpyDeviceToHost, cudaStream_t(stream))), "pnp_prox_prepared_kind_async");
}

int pnp_prox_dual_prepared(const float* x, const void* u_in, const void* y0T, const uint8_t* maskT,
                           long long mask_batch_stride, const float* mu, int mu_stride, void* z_out, void* u_out,
                           float* v_next, int B, int H, int W, void* stream) {
  return pnp_prox_dual_prepared_kind(x, u_in, y0T, maskT, mask_batch_stride, mu, mu_stride, z_out, u_out, v_next, B, H, W,
                                     -1, stream);
}

int pnp_prox_dual_prepared_kind(const float* x, const void* u_in, const void* y0T, const uint8_t* maskT,
                                long long mask_batch_stride, const float* mu, int mu_stride, void* z_out, void* u_out,
                                float* v_next, int B, int H, int W, int kind, void* stream) {
  REQUIRE_INIT();
  if (kind < -1 || kind > 1) { set_error("pnp_prox_dual_prepared_kind: kind must be -1, 0 or 1"); return -1; }
  if (!x || !u_in || !y0T || !maskT || !mu || !z_out || !u_out) { set_error("pnp_prox_dual_prepared: null pointer"); return -1; }
  if (!pnp_prox_prepared_supported(H, W)) { set_error("pnp_prox_dual_prepared: H and W must be powers of two in 32..512"); return -2; }
  return fail_cuda(prox_dual_prepared(x, static_cast<const float2*>(u_in), static_cast<const float2*>(y0T), maskT,
                                      mask_batch_stride, mu, mu_stride, static_cast<float2*>(z_out),
                                      static_cast<float2*>(u_out), v_next, B, H, W, kind, cudaStream_t(stream)),
                   "pnp_prox_dual_prepared");
}

int pnp_prox_dual(const float* x, const void* u_in, const void* y0, const uint8_t* mask, long long mask_batch_stride,
                  const float* mu, int mu_stride, void* z_out, void* u_out, float* v_next, void* workspace, int B,
                  int H, int W, void* stream) {
  REQUIRE_INIT();
  if (!x || !u_in || !y0 || !mask || !mu || !z_out || !u_out || !workspace) {
    set_error("pnp_prox_dual: null pointer");
    return -1;
  }
  if (!fft_any_shape_supported(H, W)) {
    set_error("pnp_prox_dual: H and W must be in [2, 1024]");
    return -2;
  }
  return fail_cuda(prox_dual_general(x, static_cast<const float2*>(u_in), static_cast<const float2*>(y0), mask,
                                     mask_batch_stride, mu, mu_stride, static_cast<float2*>(z_out),
                                     static_cast<float2*>(u_out), v_next, static_cast<float2*>(workspace), B, H, W,
                                     cudaStream_t(stream)), "pnp_prox_dual");
}

size_t pnp_unet_num_params(void) { return unet_num_params(); }
size_t pnp_unet_packed_bytes(void) { return unet_packed_bytes(); }
size_t pnp_unet_workspace_bytes(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  return unet_workspace_bytes(unet_micro_batch(B, H, W), H, W);
}

int pnp_unet_pack_weights(const float* flat_params, void* packed, void* stream) {
  REQUIRE_INIT();
  return fail_cuda(unet_pack(flat_params, static_cast<uint8_t*>(packed), cudaStream_t(stream)), "pnp_unet_pack_weights");
}

int pnp_unet_plan_create(pnp_unet_plan** plan, const void* packed, void* workspace, size_t workspace_bytes, int B,
                         int H, int W) {
  REQUIRE_INIT();
  if (B <= 0) { set_error("pnp_unet_plan_create: B must be positive"); return -1; }
  const int mb = unet_micro_batch(B, H, W);
  UnetPlan *impl = nullptr, *tail = nullptr;
  int rc = unet_plan_create(&impl, static_cast<const uint8_t*>(packed), static_cast<uint8_t*>(workspace),
                            workspace_bytes, mb, H, W);
  if (rc) return rc;
  if (B % mb) {
    rc = unet_plan_create(&tail, static_cast<const uint8_t*>(packed), static_cast<uint8_t*>(workspace), workspace_bytes,
                          B % mb, H, W);
    if (rc) { unet_plan_destroy(impl); return rc; }
  }
  *plan = new pnp_unet_plan{impl, tail, B, H, W, mb};
  return 0;
}

void pnp_unet_plan_destroy(pnp_unet_plan* plan) {
  if (!plan) return;
  unet_plan_destroy(plan->impl);
  if (plan->tail) unet_plan_destroy(plan->tail);
  delete plan;
}

int pnp_unet_forward(pnp_unet_plan* plan, const float* v, const float* sigma, float* x_out, float* preclamp,
                     void* stream) {
  REQUIRE_INIT();
  if (!plan || !v || !sigma || !x_out) { set_error("pnp_unet_forward: null pointer"); return -1; }
  const size_t hw = size_t(plan->H) * plan->W;
  for (int i0 = 0; i0 < plan->B; i0 += plan->mb) {
    UnetPlan* p = (plan->B - i0 >= plan->mb) ? plan->impl : plan->tail;
    int rc = unet_forward(p, v + i0 * hw, sigma + i0, x_out + i0 * hw, preclamp ? preclamp + i0 * hw : nullptr,
                          cudaStream_t(stream));
    if (rc) return fail_cuda(rc, "pnp_unet_forward");
  }
  return 0;
}

int pnp_unet_profile(pnp_unet_plan* plan, const float* v, const float* sigma, float* x_out, void* stream, float* ms,
                     int* kinds, int* ids, int* n_inout) {
  REQUIRE_INIT();
  if (!plan || !v || !sigma || !x_out || !ms || !kinds || !ids || !n_inout) {
    set_error("pnp_unet_profile: null pointer");
    return -1;
  }
  // per-launch timing of every micro-batch, appended (callers sum by id)
  const size_t hw = size_t(plan->H) * plan->W;
  const int cap = *n_inout;
  int used = 0;
  for (int i0 = 0; i0 < plan->B; i0 += plan->mb) {
    UnetPlan* p = (plan->B - i0 >= plan->mb) ? plan->impl : plan->tail;
    int n = cap - used;
    int rc = unet_profile(p, v + i0 * hw, sigma + i0, x_out + i0 * hw, cudaStream_t(stream), ms + used, kinds + used,
                          ids + used, &n);
    if (rc) return fail_cuda(rc, "pnp_unet_profile");
    used += n;
  }
  *n_inout = used;
  return 0;
}

int pnp_unet_num_launches(const pnp_unet_plan* plan) {
  if (!plan) return -1;
  return (plan->B / plan->mb) * unet_num_launches(plan->impl) + (plan->tail ? unet_num_launches(plan->tail) : 0);
}

int pnp_unet_micro_batch(const pnp_unet_plan* plan) { return plan ? plan->mb : -1; }

size_t pnp_unet_set_workspace_cap(size_t bytes) {
  const size_t old = kUnetWorkspaceCap;
  if (bytes) kUnetWorkspaceCap = bytes;
  return old;
}

int pnp_unet_set_splitk(int mode) { return unet_set_splitk(mode); }

int pnp_unet_plan_tensor(const pnp_unet_plan* plan, const char* name, size_t* byte_offset, int* C, int* H, int* W) {
  if (!plan || !name) return -1;
  if (plan->mb != plan->B) return -1;        // micro-batched plans reuse the workspace: no whole-batch intermediates
  return unet_plan_tensor(plan->impl, name, byte_offset, C, H, W);
}

size_t pnp_policy_packed_floats(int n_time, int n_task) { return policy_packed_floats(n_time, n_task); }

int pnp_policy_step(const float* packed, const float* rtg, const float* emb, float* act, const long long* timesteps,
                    const long long* task, const long long* pos, float* act_out, float* rtg_out, float scale0, float scale1,
                    float scale2, int B, int K, int n_time, int n_task, void* stream) {
  REQUIRE_INIT();
  if (!packed || !rtg || !emb || !act || !timesteps || !task || !pos || !act_out || !rtg_out) {
    set_error("pnp_policy_step: null pointer");
    return -1;
  }
  if (K < 1 || K > 6 || B < 1) { set_error("pnp_policy_step: need 1 <= K <= 6 context entries and B >= 1"); return -1; }
  return fail_cuda(policy_step_launch(packed, rtg, emb, act, timesteps, task, pos, act_out, rtg_out, scale0, scale1, scale2,
                                      B, K, n_time, n_task, cudaStream_t(stream)), "pnp_policy_step");
}

size_t pnp_policy_encoder_packed_floats(void) { return policy_encoder_packed_floats(); }

int pnp_policy_observe(const float* enc_packed, const float* x, int H, int W, const float* next_rtg, float* rtg, float* emb,
                       float* act, long long* timesteps, const long long* pos, const long long* t_dev, int B, int K,
                       int n_time, void* stream) {
  if (!enc_packed || !x || !next_rtg || !rtg || !emb || !act || !timesteps || !pos || !t_dev) {
    set_error("pnp_policy_observe: null pointer");
    return -1;
  }
  if (K < 1 || K > 6 || B < 1 || H != W || H < 128 || H % 128 != 0 || n_time < 1) {
    set_error("pnp_policy_observe: need square images whose edge is a multiple of 128, 1 <= K <= 6 and B >= 1");
    return -1;
  }
  return fail_cuda(policy_observe_launch(enc_packed, x, H, W, next_rtg, rtg, emb, act, timesteps, pos, t_dev, B, K, n_time,
                                         cudaStream_t(stream)), "pnp_policy_observe");
}

size_t pnp_conv3x3_packed_bytes(int Cin, int Cout) { return (conv_packed_bytes(Cin, Cout) + 1023) / 1024 * 1024; }

int pnp_conv3x3_bf16(const void* in0, int C0, const void* in1, int C1, const float* weights, const float* bias,
                     void* out, void* scratch, int B, int H, int W, int Cout, void* stream) {
  REQUIRE_INIT();
  return fail_cuda(conv3x3_single(static_cast<const __nv_bfloat16*>(in0), C0, static_cast<const __nv_bfloat16*>(in1),
                                  C1, weights, bias, static_cast<__nv_bfloat16*>(out), static_cast<uint8_t*>(scratch),
                                  B, H, W, Cout, cudaStream_t(stream)), "pnp_conv3x3_bf16");
}

int pnp_step_prepared(pnp_unet_plan* plan, const float* v, const float* sigma, const void* u_in, const void* y0T,
                      const uint8_t* maskT, long long mask_batch_stride, const float* mu, int mu_stride, float* x_out,
                      void* z_out, void* u_out, float* v_next, void* stream) {
  return pnp_step_prepared_kind(plan, v, sigma, u_in, y0T, maskT, mask_batch_stride, mu, mu_stride, x_out, z_out, u_out,
                                v_next, -1, stream);
}

int pnp_step_prepared_kind(pnp_unet_plan* plan, const float* v, const float* sigma, const void* u_in, const void* y0T,
                           const uint8_t* maskT, long long mask_batch_stride, const float* mu, int mu_stride, float* x_out,
                           void* z_out, void* u_out, float* v_next, int kind, void* stream) {
  int rc = pnp_unet_forward(plan, v, sigma, x_out, nullptr, stream);
  if (rc) return rc;
  return pnp_prox_dual_prepared_kind(x_out, u_in, y0T, maskT, mask_batch_stride, mu, mu_stride, z_out, u_out, v_next,
                                     plan->B, plan->H, plan->W, kind, stream);
}

int pnp_step_prepared_active(pnp_unet_plan* plan, const float* v, const float* sigma, const void* u_in, const void* y0T,
                             const uint8_t* maskT, long long mask_batch_stride, const float* mu, int mu_stride,
                             float* x_out, void* z_out, void* u_out, float* v_next, int kind, const uint8_t* active,
                             void* stream) {
  REQUIRE_INIT();
  if (!plan || !v || !sigma || !u_in || !y0T || !maskT || !mu || !x_out || !z_out || !u_out) {
    set_error("pnp_step_prepared_active: null pointer");
    return -1;
  }
  if (kind < -1 || kind > 1) { set_error("pnp_step_prepared_active: kind must be -1, 0 or 1"); return -1; }
  const size_t hw = size_t(plan->H) * plan->W;
  for (int i0 = 0; i0 < plan->B; i0 += plan->mb) {
    UnetPlan* p = (plan->B - i0 >= plan->mb) ? plan->impl : plan->tail;
    int rc = unet_forward(p, v + i0 * hw, sigma + i0, x_out + i0 * hw, nullptr, cudaStream_t(stream),
                          active ? active + i0 : nullptr);
    if (rc) return fail_cuda(rc, "pnp_step_prepared_active");
  }
  return fail_cuda(prox_dual_prepared(x_out, static_cast<const float2*>(u_in), static_cast<const float2*>(y0T), maskT,
                                      mask_batch_stride, mu, mu_stride, static_cast<float2*>(z_out),
                                      static_cast<float2*>(u_out), v_next, plan->B, plan->H, plan->W, kind,
                                      cudaStream_t(stream), active), "pnp_step_prepared_active");
}

int pnp_step(pnp_unet_plan* plan, const float* v, const float* sigma, const void* u_in, const void* y0,
             const uint8_t* mask, long long mask_batch_stride, const float* mu, int mu_stride, float* x_out,
             void* z_out, void* u_out, float* v_next, void* prox_workspace, void* stream) {
  int rc = pnp_unet_forward(plan, v, sigma, x_out, nullptr, stream);
  if (rc) return rc;
  return pnp_prox_dual(x_out, u_in, y0, mask, mask_batch_stride, mu, mu_stride, z_out, u_out, v_next, prox_workspace,
                       plan->B, plan->H, plan->W, stream);
}

}  // extern "C"
