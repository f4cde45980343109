// C-ABI entry points of the layer kernels (include/bbb.h): argument validation, host-side folding
// of the prior / RNG descriptors, and dispatch between the exact-fp32 FMA kernels and the tcgen05
// kind::tf32 kernels.  No allocation, no synchronisation, no global state.
#include "bbb_common.cuh"
#include "bbb_kernels.h"

using namespace bbb;

namespace {
inline bool al16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline bool all16(std::initializer_list<const void *> ps) {
  for (const void *p : ps)
    if (p && !al16(p)) return false;
  return true;
}
}  // namespace

extern "C" int bbb_linear_fwd(const float *x, int64_t x_sample_stride, const float *w_mu, const float *w_rho,
                              const float *b_mu, const float *b_rho, const float *eps_w, const float *eps_b,
                              const bbb_rng *rng, const bbb_prior *prior, int64_t S, int64_t B, int64_t in,
                              int64_t out, int32_t flags, float *y, double *logp, double *logq, void *stream) {
  BBB_CHECK_ARG(S >= 0 && B >= 0 && in >= 0 && out >= 0 && S <= 65535, "bad shape");
  BBB_CHECK_ARG(w_mu && b_mu && ((x && y) || S * B == 0), "null pointer");  // empty batches carry null activations
  BBB_CHECK_ARG(x_sample_stride == 0 || x_sample_stride == B * in, "x_sample_stride must be 0 or B*in");
  const bool sample = flags & BBB_F_SAMPLE, lpq = flags & BBB_F_LOGPROB;
  BBB_CHECK_ARG(!(sample || lpq) || (w_rho && b_rho), "rho pointers required");
  BBB_CHECK_ARG(!lpq || (prior && logp && logq), "log-prob outputs and prior required with BBB_F_LOGPROB");
  BBB_CHECK_ARG(!sample || (eps_w && eps_b) || (!eps_w && !eps_b && rng), "give both eps pointers or an rng");
  BBB_CHECK_ARG(!prior || prior->kind == BBB_PRIOR_GAUSSIAN || prior->kind == BBB_PRIOR_MIXTURE, "bad prior kind");
  if (S == 0 || B == 0 || out == 0) return BBB_OK;
  LinArgs a{};
  a.x = x; a.x_sstride = x_sample_stride;
  a.w_mu = w_mu; a.w_rho = w_rho; a.b_mu = b_mu; a.b_rho = b_rho; a.eps_w = eps_w; a.eps_b = eps_b;
  a.rng = make_rng_dev(rng);
  if (prior) a.prior = make_prior_dev(prior);
  a.S = (int)S; a.B = B; a.in = in; a.out = out; a.flags = flags;
  a.y = y; a.logp = logp; a.logq = logq;
  a.vec_in = (in % 4 == 0) && all16({x, w_mu, w_rho, eps_w});
  a.vec_out = (out % 4 == 0) && all16({y});
  cudaStream_t st = (cudaStream_t)stream;
  const bool big = (flags & BBB_F_TF32) && !head_supported(a) && !linear_sk_supported(a) && linear_big_fwd_supported(a);
  if ((flags & BBB_F_RELU_OUT) && !big)
    return fail(BBB_EUNSUPPORTED, "BBB_F_RELU_OUT: only the large-batch tensor kernels store post-activations "
                                  "(bbb_linear_fwd_relu_out_supported)");
  if (head_supported(a)) return launch_linear_fwd_head(a, st);                // out <= 16, both modes, exact fp32
  if ((flags & BBB_F_TF32) && linear_sk_supported(a)) return launch_linear_fwd_sk(a, st);
  if (big) return launch_linear_fwd_wide(a, st);   // batch >= 384: TMA-fed, weight tiles shared in a cluster
  if ((flags & BBB_F_TF32) && linear_tc_supported(a)) return launch_linear_fwd_tc(a, st);
  if (linear_narrow_supported(a)) return launch_linear_fwd_narrow(a, st);   // exact-fp32 mode, out <= 16
  return launch_linear_fwd_fma(a, st);
}

extern "C" int bbb_linear_fwd_relu_out_supported(int64_t B, int64_t in, int64_t out, int32_t flags) {
  if (B <= 0 || in <= 0 || out <= 0) return 0;
  LinArgs a{};
  a.S = 1; a.B = B; a.in = in; a.out = out; a.flags = flags;
  a.vec_in = in % 4 == 0;
  a.vec_out = out % 4 == 0;
  return ((flags & BBB_F_TF32) && !head_supported(a) && !linear_sk_supported(a) && linear_big_fwd_supported(a)) ? 1 : 0;
}

extern "C" int bbb_linear_bwd(const float *dy, const float *dy_mask_src, const float *x, int64_t x_sample_stride,
                              const float *w_mu, const float *w_rho, const float *b_mu, const float *b_rho,
                              const float *eps_w, const float *eps_b, const bbb_rng *rng, const bbb_prior *prior,
                              int64_t S, int64_t B, int64_t in, int64_t out, int32_t flags, float gp, float gq,
                              const float *gp_dev, const float *gq_dev, int64_t g_dev_stride,
                              const float *out_scale_dev, float *dx, float *grad_w_mu, float *grad_w_rho,
                              float *grad_b_mu, float *grad_b_rho, void *stream) {
  BBB_CHECK_ARG(w_mu && w_rho && b_mu && b_rho && ((dy && x) || S * B == 0), "null pointer");
  BBB_CHECK_ARG((flags & BBB_F_NO_WGRAD) || (grad_w_mu && grad_w_rho && grad_b_mu && grad_b_rho),
                "null gradient pointer");
  BBB_CHECK_ARG((flags & BBB_F_NO_DX) || dx || S * B == 0, "dx required unless BBB_F_NO_DX");
  BBB_CHECK_ARG(S >= 0 && B >= 0 && in >= 0 && out >= 0 && S <= 65535, "bad shape");
  BBB_CHECK_ARG(x_sample_stride == 0 || x_sample_stride == B * in, "x_sample_stride must be 0 or B*in");
  const bool sample = flags & BBB_F_SAMPLE;
  BBB_CHECK_ARG(!sample || (eps_w && eps_b) || (!eps_w && !eps_b && rng), "give both eps pointers or an rng");
  BBB_CHECK_ARG(((gp == 0.0f) && !gp_dev) || prior, "prior required when gp != 0");
  BBB_CHECK_ARG(!prior || prior->kind == BBB_PRIOR_GAUSSIAN || prior->kind == BBB_PRIOR_MIXTURE, "bad prior kind");
  if (out == 0 || in == 0) return BBB_OK;
  LinArgs a{};
  a.x = x; a.x_sstride = x_sample_stride;
  a.w_mu = w_mu; a.w_rho = w_rho; a.b_mu = b_mu; a.b_rho = b_rho; a.eps_w = eps_w; a.eps_b = eps_b;
  a.rng = make_rng_dev(rng);
  if (prior) a.prior = make_prior_dev(prior);
  a.S = (int)S; a.B = B; a.in = in; a.out = out; a.flags = flags;
  BBB_CHECK_ARG(g_dev_stride == 0 || g_dev_stride == 1, "g_dev_stride must be 0 or 1");
  a.dy = dy; a.mask = dy_mask_src; a.gp = gp; a.gq = gq; a.gp_dev = gp_dev; a.gq_dev = gq_dev;
  a.g_dev_stride = g_dev_stride; a.out_scale_dev = out_scale_dev;
  a.dx = dx; a.g_w_mu = grad_w_mu; a.g_w_rho = grad_w_rho; a.g_b_mu = grad_b_mu; a.g_b_rho = grad_b_rho;
  a.vec_in = (in % 4 == 0) && all16({x, w_mu, w_rho, eps_w, dx});
  a.vec_out = (out % 4 == 0) && all16({dy, dy_mask_src});
  if (S == 0 || B == 0) a.S = (B == 0) ? a.S : 0;  // degenerate: gradients reduce to the prior/posterior terms
  cudaStream_t st = (cudaStream_t)stream;
  if (a.S > 0 && head_supported(a)) return launch_linear_bwd_head(a, st);   // out <= 16, both modes, exact fp32
  if ((flags & BBB_F_TF32) && a.S > 0 && linear_bwd_fused_supported(a)) return launch_linear_bwd_fused(a, st);
  if ((flags & BBB_F_TF32) && linear_tc_supported(a)) {
    // batch >= 384: batch-resident dgrad (bbb_wide.cu) and the MN-major wgrad (bbb_linear_big.cu); anything they do
    // not cover goes to the batch-tiled kernels
    LinArgs rest = a;
    if (a.S > 0 && !(flags & BBB_F_NO_DX) && linear_big_dgrad_supported(a)) {
      if (int r = launch_linear_dgrad_wide(a, st)) return r;
      rest.flags |= BBB_F_NO_DX;
    }
    if (a.S > 0 && !(flags & BBB_F_NO_WGRAD) && linear_big_wgrad_supported(a)) {
      if (int r = launch_linear_wgrad_big(a, st)) return r;
      rest.flags |= BBB_F_NO_WGRAD;
    }
    if ((rest.flags & BBB_F_NO_DX) && (rest.flags & BBB_F_NO_WGRAD)) return BBB_OK;
    return launch_linear_bwd_tc(rest, st);
  }
  if (a.S > 0 && linear_narrow_supported(a)) return launch_linear_bwd_narrow(a, st);   // exact-fp32 mode, out <= 16
  return launch_linear_bwd_fma(a, st);
}

extern "C" int bbb_lr_linear_fwd(const float *x, int64_t x_sample_stride, const float *w_mu, const float *w_rho,
                                 const float *b_mu, const float *b_rho, const float *eps_a, const float *eps_b,
                                 const bbb_rng *rng, float sigma_p, int64_t S, int64_t B, int64_t in, int64_t out,
                                 int32_t flags, float *y, float *delta, double *kl, void *stream) {
  BBB_CHECK_ARG(x && w_mu && b_mu && y, "null pointer");
  BBB_CHECK_ARG(S >= 0 && B >= 0 && in >= 0 && out >= 0 && S <= 65535, "bad shape");
  BBB_CHECK_ARG(x_sample_stride == 0 || x_sample_stride == B * in, "x_sample_stride must be 0 or B*in");
  const bool sample = flags & BBB_F_SAMPLE, lpq = flags & BBB_F_LOGPROB;
  BBB_CHECK_ARG(!(sample || lpq) || (w_rho && b_rho), "rho pointers required");
  BBB_CHECK_ARG(!lpq || (kl && sigma_p > 0), "kl output and sigma_p > 0 required with BBB_F_LOGPROB");
  BBB_CHECK_ARG(!sample || (eps_a && eps_b) || (!eps_a && !eps_b && rng), "give both eps pointers or an rng");
  if (S == 0 || B == 0 || out == 0) return BBB_OK;
  LrArgs a{};
  a.x = x; a.x_sstride = x_sample_stride;
  a.w_mu = w_mu; a.w_rho = w_rho; a.b_mu = b_mu; a.b_rho = b_rho; a.eps_a = eps_a; a.eps_b = eps_b;
  a.rng = make_rng_dev(rng);
  a.sigma_p = sigma_p > 0 ? sigma_p : 1.0f;
  a.S = (int)S; a.B = B; a.in = in; a.out = out; a.flags = flags;
  a.y = y; a.delta = delta; a.kl = kl;
  a.vec_in = (in % 4 == 0) && all16({x});
  a.vec_out = (out % 4 == 0) && all16({w_mu, w_rho, eps_a, y, delta});
  if ((flags & BBB_F_TF32) && lr_tc_supported(a)) return launch_lr_fwd_tc(a, (cudaStream_t)stream);
  if (lr_narrow_supported(a)) return launch_lr_fwd_narrow(a, (cudaStream_t)stream);   // heads: out <= 16, exact fp32
  return launch_lr_fwd_fma(a, (cudaStream_t)stream);
}

extern "C" int bbb_lr_linear_bwd(const float *dy, const float *dy_mask_src, const float *x, int64_t x_sample_stride,
                                 const float *w_mu, const float *w_rho, const float *b_mu, const float *b_rho,
                                 const float *eps_a, const float *eps_b, const bbb_rng *rng, const float *delta,
                                 float sigma_p, int64_t S, int64_t B, int64_t in, int64_t out, int32_t flags,
                                 float g_kl, const float *g_kl_dev, const float *out_scale_dev, float *dx,
                                 float *grad_w_mu, float *grad_w_rho, float *grad_b_mu, float *grad_b_rho,
                                 void *stream) {
  // empty batches carry null activations, as in bbb_linear_bwd
  BBB_CHECK_ARG(w_mu && w_rho && b_mu && b_rho && ((dy && x) || S * B == 0), "null pointer");
  BBB_CHECK_ARG((flags & BBB_F_NO_WGRAD) || (grad_w_mu && grad_w_rho && grad_b_mu && grad_b_rho),
                "null gradient pointer");
  BBB_CHECK_ARG((flags & BBB_F_NO_DX) || dx || S * B == 0, "dx required unless BBB_F_NO_DX");
  BBB_CHECK_ARG(S >= 0 && B >= 0 && in >= 0 && out >= 0 && S <= 65535 && sigma_p > 0, "bad shape or sigma_p");
  BBB_CHECK_ARG(x_sample_stride == 0 || x_sample_stride == B * in, "x_sample_stride must be 0 or B*in");
  const bool sample = flags & BBB_F_SAMPLE;
  BBB_CHECK_ARG(!sample || delta || S * B == 0, "delta (saved by the forward) required when sampling");
  BBB_CHECK_ARG(!sample || (eps_a && eps_b) || (!eps_a && !eps_b && rng), "give both eps pointers or an rng");
  if (out == 0 || in == 0) return BBB_OK;
  LrArgs a{};
  a.x = x; a.x_sstride = x_sample_stride;
  a.w_mu = w_mu; a.w_rho = w_rho; a.b_mu = b_mu; a.b_rho = b_rho; a.eps_a = eps_a; a.eps_b = eps_b;
  a.rng = make_rng_dev(rng);
  a.sigma_p = sigma_p;
  a.S = (int)S; a.B = B; a.in = in; a.out = out; a.flags = flags;
  a.dy = dy; a.mask = dy_mask_src; a.delta_in = delta; a.g_kl = g_kl;
  a.g_kl_dev = g_kl_dev; a.out_scale_dev = out_scale_dev;
  a.dx = dx; a.g_w_mu = grad_w_mu; a.g_w_rho = grad_w_rho; a.g_b_mu = grad_b_mu; a.g_b_rho = grad_b_rho;
  a.vec_in = (in % 4 == 0) && all16({x});
  a.vec_out = (out % 4 == 0) && all16({w_mu, w_rho, eps_a, dy, dy_mask_src, delta});
  if ((flags & BBB_F_TF32) && lr_bwd_tc_supported(a)) return launch_lr_bwd_tc(a, (cudaStream_t)stream);
  if (a.S > 0 && a.B > 0 && lr_head_bwd_supported(a)) return launch_lr_bwd_head(a, (cudaStream_t)stream);   // out <= 16
  if (a.S > 0 && a.B > 0 && lr_narrow_supported(a)) return launch_lr_bwd_narrow(a, (cudaStream_t)stream);
  return launch_lr_bwd_fma(a, (cudaStream_t)stream);
}
