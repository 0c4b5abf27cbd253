// Internal (C++) interfaces between the translation units of libpnp_b200.so. Not part of the C-ABI.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stddef.h>
#include <stdint.h>
#include <string>

namespace pnp {

void set_error(const std::string& msg);

// psnr.cu
int psnr_launch(const float* x, const float* gt, long long gt_bstride, float* out, int B, int HW, cudaStream_t st);
int psnr_allgather_launch(const float* x, const float* gt, long long gt_bstride, float* out_local,
                          const unsigned long long* peer_base, int rank, int world, int slot, int parity, int flag_word,
                          unsigned int* local_count, unsigned int count_target, unsigned int flag_target, int* err,
                          int B, int HW, cudaStream_t st);

// ssim.cu
size_t ssim_workspace_bytes(int B, int H, int W);
int ssim_launch(const float* x, const float* gt, long long gt_bstride, float* out, void* workspace, int B, int H, int W,
                cudaStream_t st);

// fftprox.cu
void init_fft_tables();
int fft_shape_supported(int H, int W);       // radix kernels + prepared path: powers of two in 32..512
int fft_any_shape_supported(int H, int W);   // any kernel: 2..1024 (dense-DFT path for the rest)
int prox_dual_general(const float* x, const float2* u_in, const float2* y0, const uint8_t* mask,
                      long long mask_bstride, const float* mu, int mu_stride, float2* z_out, float2* u_out,
                      float* v_out, float2* work, int B, int H, int W, cudaStream_t st);
void prox_prepared_bytes(int B, int H, int W, size_t* y0p_bytes, size_t* maskp_bytes);
int prox_prepare(const float2* y0, const uint8_t* mask, long long mask_bstride, float2* y0T, uint8_t* maskT, int B, int H,
                 int W, cudaStream_t st);
int prox_dual_prepared(const float* x, const float2* u_in, const float2* y0T, const uint8_t* maskT,
                       long long mask_bstride, const float* mu, int mu_stride, float2* z_out, float2* u_out,
                       float* v_out, int B, int H, int W, int kind, cudaStream_t st, const uint8_t* active = nullptr);
const int* prox_prepared_flag(const uint8_t* maskp, long long mask_bstride, int B, int H, int W);
int fft2c_general(const float2* src, float2* dst, int B, int H, int W, int inverse, cudaStream_t st);
// measure.cuh (compiled into fftprox.cu)
int simulate_measurements(const float* gt, long long gt_bstride, const uint8_t* mask, long long mask_bstride,
                          const float* sigma, int sigma_stride, const unsigned long long* seeds, float2* y0, float2* x0,
                          float2* aty0, int B, int H, int W, cudaStream_t st);
int cartesian_masks(const int* accel, int accel_stride, const unsigned long long* seeds, int acs_cols, uint8_t* mask,
                    int B, int H, int W, cudaStream_t st);
int radial_masks(const double* frac, int frac_stride, const unsigned long long* seeds, uint8_t* mask, int* lines_out,
                 int B, int H, int W, cudaStream_t st);
int variable_density_masks(const int* accel, int accel_stride, const unsigned long long* seeds, int acs_h, int acs_w,
                           int power, uint8_t* mask, int B, int H, int W, cudaStream_t st);

// policy.cu
size_t policy_packed_floats(int n_time, int n_task);
int policy_step_launch(const float* w, const float* rtg, const float* emb, float* act, const long long* ts,
                       const long long* task, const long long* pos, float* act_out, float* rtg_out, float s0, float s1,
                       float s2, int B, int K, int n_time, int n_task, cudaStream_t st);
// policy_observe.cu
size_t policy_encoder_packed_floats();
int policy_observe_launch(const float* w, const float* x, int H, int W, const float* nxt_rtg, float* w_rtg, float* w_emb,
                          float* w_act, long long* w_ts, const long long* pos, const long long* t_dev, int B, int K,
                          int n_time, cudaStream_t st);

// unet.cu
struct UnetPlan;
int unet_global_init();
int num_sms();
size_t unet_num_params();
size_t unet_packed_bytes();
size_t unet_workspace_bytes(int B, int H, int W);
int unet_pack(const float* flat_fp32, uint8_t* packed, cudaStream_t st);
int unet_plan_create(UnetPlan** out, const uint8_t* packed, uint8_t* workspace, size_t workspace_bytes, int B, int H,
                     int W);
void unet_plan_destroy(UnetPlan* p);
int unet_plan_tensor(const UnetPlan* p, const char* name, size_t* off, int* C, int* H, int* W);
int unet_forward(UnetPlan* p, const float* v, const float* sigma, float* x_out, float* preclamp, cudaStream_t st,
                 const uint8_t* active = nullptr);
int unet_profile(UnetPlan* p, const float* v, const float* sigma, float* x_out, cudaStream_t st, float* ms, int* kinds,
                 int* ids, int* n_inout);
int unet_num_launches(const UnetPlan* p);
int unet_forward_ops(UnetPlan* p, const float* v, const float* sigma, float* x_out, float* preclamp, int first, int end,
                     cudaStream_t st);
constexpr int kUnetOpDescLen = 21;      // PNP_UNET_OP_DESC_LEN
int unet_op_describe(const UnetPlan* p, int i, long long* desc);
int unet_set_splitk(int mode);
size_t conv_packed_bytes(int Cin, int Cout);
int conv3x3_single(const __nv_bfloat16* in0, int C0, const __nv_bfloat16* in1, int C1, const float* w_fp32,
                   const float* bias, __nv_bfloat16* out, uint8_t* wpk_scratch, int B, int H, int W, int Cout,
                   cudaStream_t st);

}  // namespace pnp
