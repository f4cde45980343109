// Internal launcher interface between the C-ABI entry points (bbb_api.cu) and the kernel files.
#pragma once
#include "bbb_common.cuh"

namespace bbb {

// Arguments of the weight-sampling layer kernels (forward and backward share one struct).
struct LinArgs {
  // forward operands
  const float *x;
  int64_t x_sstride;
  const float *w_mu, *w_rho, *b_mu, *b_rho, *eps_w, *eps_b;
  RngDev rng;
  PriorDev prior;
  int S;
  int64_t B, in, out;
  int flags;
  float *y;
  double *logp, *logq;
  // backward operands
  const float *dy, *mask;
  float gp, gq;
  const float *gp_dev, *gq_dev;
  int64_t g_dev_stride;
  const float *out_scale_dev;
  float *dx, *g_w_mu, *g_w_rho, *g_b_mu, *g_b_rho;
  // derived
  bool vec_in;   // in % 4 == 0 and every [*, in] base pointer 16-byte aligned
  bool vec_out;  // out % 4 == 0 and every [*, out] base pointer 16-byte aligned
};

// Arguments of the local-reparameterisation layer kernels.
struct LrArgs {
  const float *x;
  int64_t x_sstride;
  const float *w_mu, *w_rho, *b_mu, *b_rho, *eps_a, *eps_b;
  RngDev rng;
  float sigma_p;
  int S;
  int64_t B, in, out;
  int flags;
  float *y, *delta;
  double *kl;
  const float *dy, *mask, *delta_in;
  float g_kl;
  const float *g_kl_dev, *out_scale_dev;
  float *dx, *g_w_mu, *g_w_rho, *g_b_mu, *g_b_rho;
  bool vec_in, vec_out;
};

int launch_linear_fwd_fma(const LinArgs &a, cudaStream_t st);
int launch_linear_bwd_fma(const LinArgs &a, cudaStream_t st);
int launch_lr_fwd_fma(const LrArgs &a, cudaStream_t st);
int launch_lr_bwd_fma(const LrArgs &a, cudaStream_t st);

// local reparameterisation on tcgen05 kind::tf32, batch <= 128 (bbb_lr_tc.cu)
bool lr_tc_supported(const LrArgs &a);
int launch_lr_fwd_tc(const LrArgs &a, cudaStream_t st);
bool lr_bwd_tc_supported(const LrArgs &a);
int launch_lr_bwd_tc(const LrArgs &a, cudaStream_t st);   // overwrites the forward's delta with dV

// tcgen05 kind::tf32 path (bbb_linear_tc.cu); returns BBB_EUNSUPPORTED when the shape does not fit.
bool linear_tc_supported(const LinArgs &a);
int launch_linear_fwd_tc(const LinArgs &a, cudaStream_t st);
int launch_linear_bwd_tc(const LinArgs &a, cudaStream_t st);

// tcgen05 kind::tf32 forward / dgrad for large batches (bbb_wide.cu): the batch is the MMA's N dimension, a CTA's
// accumulator [128 weight rows x 512 batch rows] fills TMEM, activation tiles arrive by TMA and every sampled weight
// tile is shared by the CTAs of a cluster.  Support conditions and wgrad in bbb_linear_big.cu.
bool linear_big_fwd_supported(const LinArgs &a);
bool linear_big_dgrad_supported(const LinArgs &a);
int launch_linear_fwd_wide(const LinArgs &a, cudaStream_t st);
int launch_linear_dgrad_wide(const LinArgs &a, cudaStream_t st);
bool linear_big_wgrad_supported(const LinArgs &a);
int launch_linear_wgrad_big(const LinArgs &a, cudaStream_t st);   // plain MN-major GEMM over the batch + sampling epilogue

// tcgen05 kind::tf32 forward for batches of at most 128 rows (bbb_linear_sk.cu): stream-K, two co-resident CTAs per SM.
bool linear_sk_supported(const LinArgs &a);
int launch_linear_fwd_sk(const LinArgs &a, cudaStream_t st);

// narrow-output layers (out <= 16: classification / regression heads), exact fp32, both modes (bbb_linear_narrow.cu)
bool linear_narrow_supported(const LinArgs &a);
int launch_linear_fwd_narrow(const LinArgs &a, cudaStream_t st);
int launch_linear_bwd_narrow(const LinArgs &a, cudaStream_t st);
bool lr_narrow_supported(const LrArgs &a);
int launch_lr_fwd_narrow(const LrArgs &a, cudaStream_t st);
int launch_lr_bwd_narrow(const LrArgs &a, cudaStream_t st);

// the network's head (out <= 16), exact fp32, cluster split-K forward (+ likelihood + ELBO assembly through
// bbb_head_fwd) and column-owned backward (bbb_head.cu)
bool head_supported(const LinArgs &a);
int launch_linear_fwd_head(const LinArgs &a, cudaStream_t st);
int launch_linear_bwd_head(const LinArgs &a, cudaStream_t st);
bool lr_head_bwd_supported(const LrArgs &a);
int launch_lr_bwd_head(const LrArgs &a, cudaStream_t st);   // LR head backward, exact fp32, same organisation

// fused backward (wgrad + analytic epilogue + dgrad, one eps regeneration) for batches of at most 128 rows
// (bbb_linear_bwd_fused.cu)
bool linear_bwd_fused_supported(const LinArgs &a);
int launch_linear_bwd_fused(const LinArgs &a, cudaStream_t st);

}  // namespace bbb
