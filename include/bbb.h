/*
 * bbb.h -- C ABI of libbbb.so, the sm_100a Bayes-by-Backprop hot path.
 *
 * The reference (tennisonliu/bayesian-neural-network) has no FFI: its hot path is the
 * Python module networks.py.  Each entry point below replaces the chain of eager ATen
 * ops behind one reference function; the citation after "replaces" is the reference
 * file:line.  The Python host (top-level networks.py + bayesian-neural-network_b200/)
 * binds these with ctypes; INTEGRATION.md shows the stub a reference maintainer adds.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer unless said otherwise;
 *    tensors are fp32, row-major, contiguous; sizes are int64_t; `stream` is a cudaStream_t.
 *  - every function returns 0 on success, a negative BBB_E* code otherwise, never throws,
 *    never synchronises; launch errors are read with cudaGetLastError right after the launch.
 *    bbb_last_error_string() returns a thread-local message for the last failure.
 *  - the library owns no device memory and keeps no state between calls.
 *  - "S" is the number of Monte-Carlo samples handled by one call (one launch covers all).
 *  - eps pointers are nullable.  Non-NULL: parity mode, eps is read from memory in the
 *    reference's draw layout.  NULL: eps is generated in registers by Philox4x32-10 keyed by
 *    (seed; element/4, sample_base + s, tensor id, step) and is never stored; the backward
 *    call regenerates it from the same coordinates.
 *  - double* accumulators are ADDED to (callers zero them once per step).
 */
#ifndef BBB_H_
#define BBB_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BBB_VERSION 101

/* error codes */
#define BBB_OK 0
#define BBB_EINVAL (-1)   /* bad argument (null pointer, negative size, unsupported flag)   */
#define BBB_ECUDA (-2)    /* CUDA runtime / launch error, see bbb_last_error_string()        */
#define BBB_EUNSUPPORTED (-3) /* shape not supported by the requested kernel family          */

/* prior kinds: networks.py:61-68 */
#define BBB_PRIOR_GAUSSIAN 0 /* Normal(0, sigma1); pi, sigma2 ignored                         */
#define BBB_PRIOR_MIXTURE 1  /* pi N(0,sigma1) + (1-pi) N(0,sigma2)                           */

/* flags */
#define BBB_F_SAMPLE 1     /* w = mu + softplus(rho) eps; otherwise w = mu (networks.py:74-79) */
#define BBB_F_LOGPROB 2    /* accumulate log prior / log posterior (or KL) (networks.py:81-83) */
#define BBB_F_RELU_IN 4    /* the input x is a pre-activation: apply max(x,0) while loading    */
#define BBB_F_ACCUM 8      /* backward: add into the grad buffers instead of overwriting       */
#define BBB_F_TF32 16      /* allow the tcgen05 kind::tf32 tensor path when the shape supports it */
#define BBB_F_NO_DX 32     /* backward: do not compute dx                                      */
#define BBB_F_SCALE_DX 64  /* backward: out_scale_dev also multiplies dx                       */
#define BBB_F_NO_WGRAD 128 /* backward: do not compute parameter gradients (dx only)           */
#define BBB_F_DX_PREACT 512 /* backward: dx is multiplied by (x > 0) (x the stored input: a pre-activation with
                               BBB_F_RELU_IN, the post-activation itself without it), i.e. it is the gradient
                              w.r.t. the PRE-activation input; the layer below then needs no dy_mask_src      */
#define BBB_F_RELU_OUT 1024 /* forward: store max(y, 0) instead of y.  The consumers of such an output are then called
                               WITHOUT BBB_F_RELU_IN (BBB_F_DX_PREACT still masks by (x > 0), which is the same mask), so
                               no kernel spends shared-memory bandwidth on a ReLU pass over TMA-landed tiles.  Implemented
                               by the large-batch tensor kernels only: ask bbb_linear_fwd_relu_out_supported first; a
                               call that sets it on any other path returns BBB_EUNSUPPORTED. */
#define BBB_F_OUT_ZEROED 256 /* y (forward) / dx (backward) is already zero-filled by the caller: kernels that
                               combine split-K partial sums with red.add skip their own memset              */

/* Philox tensor ids: weight tensor of layer l -> 2l, bias -> 2l+1, LR activation noise -> 2l */
typedef struct bbb_rng {
  uint64_t seed;        /* Philox key                                                          */
  uint32_t step;        /* counter word 3: training step / call index                          */
  uint32_t sample_base; /* counter word 1 = sample_base + s : global MC-sample index           */
  uint32_t layer;       /* counter word 2 = 2*layer (+1 for the bias)                          */
  const uint32_t *step_dev; /* optional DEVICE counter added to `step` when the kernel starts, so a
                               CUDA graph that replays the launch still advances the eps stream    */
} bbb_rng;

typedef struct bbb_prior {
  int32_t kind;
  float pi, sigma1, sigma2;
} bbb_prior;

int bbb_version(void);
const char *bbb_last_error_string(void);
/* number of kernels this library has launched in this process (diagnostic; bench.py's gpu_launches) */
uint64_t bbb_launch_count(void);

/* ---- weight-sampling layer ------------------------------------------------------------
 * replaces BayesianLinear.forward (networks.py:73-88) = GaussianNode.sample (41-43) for W and b,
 * ScaleMixtureGaussian.log_prob (24-27) / Normal.log_prob (67-68,82), GaussianNode.log_prob (45-46)
 * and F.linear (88), for S samples at once.
 *   x      [Sx,B,in]   x_sample_stride = B*in, or 0 when all samples share one input
 *   w_mu,w_rho [out,in]; b_mu,b_rho [out]; eps_w [S,out,in] / eps_b [S,out] or NULL
 *   y      [S,B,out]   written
 *   logp, logq [S]     += sum log prior / sum log posterior over W and b (BBB_F_LOGPROB)
 * S, B or out == 0: nothing is launched and no output is touched (logp / logq included).
 */
int bbb_linear_fwd(const float *x, int64_t x_sample_stride, const float *w_mu, const float *w_rho,
                   const float *b_mu, const float *b_rho, const float *eps_w, const float *eps_b,
                   const bbb_rng *rng, const bbb_prior *prior, int64_t S, int64_t B, int64_t in,
                   int64_t out, int32_t flags, float *y, double *logp, double *logq, void *stream);
/* 1 when bbb_linear_fwd honours BBB_F_RELU_OUT for this shape and `flags` (16-byte aligned pointers assumed) */
int bbb_linear_fwd_relu_out_supported(int64_t B, int64_t in, int64_t out, int32_t flags);

/* replaces the autograd backward of the above (triggered at reg_task.py:72, class_task.py:78,
 * bandits.py:49).  With t = dy^T x - gp w R(w):  grad_mu = sum_s t,  grad_rho = sum_s
 * sigmoid(rho) (t eps - gq / sigma)  (SURVEY App. A-2; gp, gq = d loss / d logp_s, d logq_s).
 *   dy        [S,B,out]  gradient w.r.t. y;  if dy_mask_src != NULL the effective gradient is
 *                        dy * (dy_mask_src > 0)  (ReLU of this layer's output fused here)
 *   gp, gq    host scalars;  gp_dev/gq_dev optional device multipliers read as gp_dev[s*g_dev_stride]
 *             (stride 0: one value for all samples, 1: per sample) -- autograd hands these over as
 *             device tensors and reading them on the device avoids a host synchronisation
 *   out_scale_dev optional device scalar multiplying every parameter gradient written (d loss upstream)
 *   dx        [S,B,in] written unless BBB_F_NO_DX (gradient w.r.t. the post-ReLU input); with BBB_F_NO_DX a
 *             non-NULL dx is left untouched
 *   grad_*    same shapes as the parameters; overwritten, or added to with BBB_F_ACCUM; with BBB_F_NO_WGRAD
 *             non-NULL gradient buffers are left untouched
 *   B == 0 (or S == 0): no dx; the gradients reduce to the prior / posterior terms of the S samples
 */
int bbb_linear_bwd(const float *dy, const float *dy_mask_src, const float *x, int64_t x_sample_stride,
                   const float *w_mu, const float *w_rho, const float *b_mu, const float *b_rho,
                   const float *eps_w, const float *eps_b, const bbb_rng *rng, const bbb_prior *prior,
                   int64_t S, int64_t B, int64_t in, int64_t out, int32_t flags, float gp, float gq,
                   const float *gp_dev, const float *gq_dev, int64_t g_dev_stride,
                   const float *out_scale_dev, float *dx, float *grad_w_mu, float *grad_w_rho,
                   float *grad_b_mu, float *grad_b_rho, void *stream);

/* ---- local-reparameterisation layer ----------------------------------------------------
 * replaces BayesianLinearLR.forward (networks.py:116-138) and compute_kl_cost (109-114).
 *   w_mu,w_rho [in,out] (the reference's LR layout, networks.py:95-96)
 *   eps_a [S,B,out] / eps_b [S,out] or NULL (Philox)
 *   y [S,B,out] written;  delta [S,B,out] = sqrt(x^2 sigma^2) written when non-NULL (backward needs it);
 *     with BBB_F_OUT_ZEROED both y and delta must arrive zero-filled (the tcgen05 path adds partial sums into both)
 *   kl  += closed-form KL(q || N(0,sigma_p)) of W and b, ONCE per call (it is sample-independent)
 */
int bbb_lr_linear_fwd(const float *x, int64_t x_sample_stride, const float *w_mu, const float *w_rho,
                      const float *b_mu, const float *b_rho, const float *eps_a, const float *eps_b,
                      const bbb_rng *rng, float sigma_p, int64_t S, int64_t B, int64_t in, int64_t out,
                      int32_t flags, float *y, float *delta, double *kl, void *stream);

/* backward of the above (SURVEY App. A-3).  g_kl = d loss / d kl (host scalar), times
 * g_kl_dev[0] when non-NULL, applied with BBB_F_LOGPROB only; out_scale_dev, BBB_F_NO_DX, BBB_F_NO_WGRAD,
 * BBB_F_ACCUM and BBB_F_DX_PREACT as in bbb_linear_bwd.  B == 0 (or S == 0): dy, x, delta and dx may be NULL; no dx, and
 * the gradients reduce to the KL terms.
 * With BBB_F_TF32 (tcgen05 path: B <= 128, in and out multiples of 4, no dy_mask_src) the call OVERWRITES `delta`
 * with dV = dz eps_a / (2 delta), which the two contractions of the backward consume; delta has no other use in
 * the backward, but a caller must not run the backward twice on the same forward buffers in that mode. */
int bbb_lr_linear_bwd(const float *dy, const float *dy_mask_src, const float *x, int64_t x_sample_stride,
                      const float *w_mu, const float *w_rho, const float *b_mu, const float *b_rho,
                      const float *eps_a, const float *eps_b, const bbb_rng *rng, const float *delta,
                      float sigma_p, int64_t S, int64_t B, int64_t in, int64_t out, int32_t flags,
                      float g_kl, const float *g_kl_dev, const float *out_scale_dev, float *dx,
                      float *grad_w_mu, float *grad_w_rho, float *grad_b_mu, float *grad_b_rho,
                      void *stream);

/* ---- stand-alone single-pass reductions -------------------------------------------------
 * bbb_logprob_reduce: one pass over (mu, rho[, eps]) -> optional w = mu + sigma eps, sum log p(w),
 * sum log q(w)  (networks.py:24-27, 41-46, 82-83).  tensor_id is the full Philox counter word 2.
 * bbb_kl_gauss: closed-form KL(q || N(0, sigma_p)) (networks.py:109-114).
 * bbb_philox_fill_normal: the eps stream itself, for the statistical tests.
 */
int bbb_logprob_reduce(const float *mu, const float *rho, const float *eps, uint64_t seed, uint32_t step,
                       uint32_t sample, uint32_t tensor_id, const bbb_prior *prior, int64_t n,
                       int32_t flags, float *w_out, double *logp, double *logq, void *stream);
int bbb_kl_gauss(const float *mu, const float *rho, float sigma_p, int64_t n, double *kl, void *stream);
int bbb_philox_fill_normal(float *out, int64_t n, uint64_t seed, uint32_t step, uint32_t sample,
                           uint32_t tensor_id, void *stream);

/* ---- per-weight Gaussian priors p(w_i) = N(m_i, sp_i^2), sp_i = softplus(r_i) -----------------------------------------
 * The prior is stored in the posterior's own parametrisation, so a trained posterior becomes the next task's prior by a
 * copy of (mu, rho) (variational continual learning, Nguyen et al. 2018).  The layer kernels do not read it: a caller
 * runs them WITHOUT BBB_F_LOGPROB (weight sampling: gp = gq = 0 and no gp_dev / gq_dev in the backward) and adds the
 * prior terms with the calls below, one launch for all tensors of a network (at most BBB_GAUSS_PRIOR_MAX_TENSORS).
 * One tensor of the table: */
#define BBB_GAUSS_PRIOR_MAX_TENSORS 64
typedef struct bbb_gauss_prior_tensor {
  const float *mu, *rho;             /* q: a layer's weight or bias parameters, n elements                               */
  const float *prior_mu, *prior_rho; /* p = N(prior_mu, softplus(prior_rho)^2), n elements                              */
  const float *eps;                  /* [S, n] injected eps (parity mode) or NULL: Philox                               */
  float *grad_mu, *grad_rho;         /* backward only: ADDED to                                                         */
  int64_t n;
  uint32_t tensor_id;                /* Philox counter word 2: 2l for a weight, 2l+1 for its bias                       */
} bbb_gauss_prior_tensor;
/* weight sampling (Monte Carlo, as sample_elbo): w_s = mu + softplus(rho) eps_s, eps_s regenerated at
 * (element/4, rng->sample_base + s, tensor_id, rng->step [+ *rng->step_dev]), i.e. the SAME eps the layer kernels drew
 * (rng->layer is ignored: every tensor carries its own id).
 *   logp[s] += sum log N(w_s; m, sp^2),  logq[s] += sum log N(w_s; mu, sigma^2)          (logp, logq: [S] fp64)   */
int bbb_gauss_prior_logprob(const bbb_gauss_prior_tensor *t, int32_t n_tensors, int64_t S, const bbb_rng *rng,
                            double *logp, double *logq, void *stream);
/* its gradient, gp_s / gq_s / out_scale exactly as bbb_linear_bwd defines them (gp_s = gp * gp_dev[s * g_dev_stride]
 * when gp_dev is given, likewise gq_s; c = out_scale_dev ? *out_scale_dev : 1):
 *   grad_mu  += c sum_s gp_s (-(w_s - m) / sp^2)
 *   grad_rho += c sigmoid(rho) sum_s [ gp_s (-(w_s - m) / sp^2) eps_s - gq_s / sigma ]                                */
int bbb_gauss_prior_logprob_bwd(const bbb_gauss_prior_tensor *t, int32_t n_tensors, int64_t S, const bbb_rng *rng,
                                float gp, float gq, const float *gp_dev, const float *gq_dev, int64_t g_dev_stride,
                                const float *out_scale_dev, void *stream);
/* local reparameterisation: closed-form KL(q || p) = sum [ log(sp/sigma) + (sigma^2 + (mu - m)^2) / (2 sp^2) - 1/2 ]
 * (networks.py:109-114 with p_mu = m), *kl += it; exactly 0 per element when (mu, rho) == (m, r).
 * bwd: grad_mu += c (mu - m)/sp^2,  grad_rho += c sigmoid(rho) (sigma/sp^2 - 1/sigma),
 *   c = g_kl * (g_kl_dev ? *g_kl_dev : 1) * (out_scale_dev ? *out_scale_dev : 1)
 * All four: any n (n % 4 tails, pointers without 16-byte alignment), n == 0 is a no-op for that tensor; launched with
 * programmatic dependent launch.  BBB_EINVAL before any device work for n_tensors outside [0, 64], a null table with
 * n_tensors > 0, n < 0, a null mu / rho / prior_mu / prior_rho (grad_mu / grad_rho in a backward) of a non-empty
 * tensor, a null logp / logq / rng / kl, or S <= 0 on the log-prob calls. */
int bbb_gauss_prior_kl(const bbb_gauss_prior_tensor *t, int32_t n_tensors, double *kl, void *stream);
int bbb_gauss_prior_kl_bwd(const bbb_gauss_prior_tensor *t, int32_t n_tensors, float g_kl, const float *g_kl_dev,
                           const float *out_scale_dev, void *stream);

/* ---- consumers of the (mu, rho) stream: SNR pruning (weight_pruning.py:81-115) -------------------------------------------
 * bbb_snr:       snr_out[i] = 10 log10(|mu_i| / softplus(rho_i))   (compute_snr, weight_pruning.py:81-83; decibels)
 * bbb_snr_prune: mu_i, rho_i *= (snr_i > threshold_db), in place (prune_weights, weight_pruning.py:85-115: the same mask
 *                multiplies mu AND rho, so a pruned weight keeps sigma = softplus(0)); *kept (nullable device counter) +=
 *                number of parameters that survive.  One pass over (mu, rho), any n.
 * bbb_softmax_mean: probs[b][c] = mean_s softmax(logits[s][b][:])[c]   (BNN_Classification.predict, class_task.py:81-87) */
int bbb_snr(const float *mu, const float *rho, int64_t n, float *snr_out, void *stream);
int bbb_snr_prune(float *mu, float *rho, int64_t n, float threshold_db, unsigned long long *kept, void *stream);
int bbb_softmax_mean(const float *logits, int64_t S, int64_t B, int64_t C, float *probs, void *stream);

/* ---- posterior predictive: uncertainty and calibration of sampled outputs (one pass over [S,B,C]) ---------------------
 * replaces the host-side analysis after the prediction loops of class_task.py:81-87 / reg_task.py:76-83 (mean +- std
 * of reg_task.evaluate) and the ECE of the reference's compute_ece.py.  One warp per row, the row's S samples read once.
 *   out     [S,B,C] sampled outputs (logits, or regression outputs with C = D);  1 <= C <= 1024, S >= 1
 *   target  nullable: int64 [B] labels (BBB_NLL_CE) or float [B,D] (BBB_NLL_GAUSS; [B] when D = 1), row for row
 *   kind    BBB_NLL_CE: p_s = softmax(out[s,b,:]).
 *             mean [B,C] = pbar = (1/S) sum_s p_s;  pred [B] (nullable) = argmax pbar (lowest index on ties);
 *             row_stats [B,5] = { confidence pbar[pred], entropy H[pbar] (0 log 0 = 0),
 *               expected entropy (1/S) sum_s H[p_s] (aleatoric), mutual information max(H[pbar] - E H[p_s], 0)
 *               (epistemic), log pbar[y] formed as LSE_s(log p_s[y]) - log S (NaN without a valid target) }
 *           BBB_NLL_GAUSS: likelihood N(y; f_s, sigma^2).
 *             mean [B,D] = mu = (1/S) sum_s f_s;  row_stats [B,D+1] = { epistemic variance (1/S) sum_s (f_s - mu)^2 per
 *               output (total = that + sigma^2), log predictive density LSE_s(sum_d log N(y_d; f_s,d, sigma^2)) - log S }
 *           BBB_NLL_GAUSS_HET: heteroscedastic likelihood N(y; f_s, sigma_s^2), C = 2D even, each row [f (D) | r (D)],
 *             sigma_s = sigma + softplus(r_s) (`sigma` is sigma_min here, see bbb_nll_gauss_het); the predictive is the
 *             mixture (1/S) sum_s N(f_s, sigma_s^2).  mean [B,D] = mu = (1/S) sum_s f_s;  row_stats [B,2D+1] = { epistemic
 *             variance (1/S) sum_s (f_s - mu)^2 [D], aleatoric variance (1/S) sum_s sigma_s^2 [D] (total = their sum, the
 *             law of total variance), log predictive density LSE_s(sum_d log N(y_d; f_s,d, sigma_s,d^2)) - log S }
 *   n_bins  BBB_NLL_CE: 1..1024 confidence bins; bin m holds confidences in (m/M, (m+1)/M], i.e.
 *           m = clamp(ceil(conf M) - 1, 0, M - 1)
 *   acc     fp64 aggregates, ADDED to (required with a target, ignored without):
 *             [0] rows counted n  [1] rows whose label is outside [0, C) (not read out of bounds, not counted in n or
 *             the bins: the host reports them)  [2] sum -log pbar[y] / sum -lpd
 *             BBB_NLL_CE:    [3] sum correct  [4] sum Brier sum_c (pbar_c - [c = y])^2
 *                            [5 + 3m ..] bin m: count, sum confidence, sum correct      (5 + 3 n_bins doubles)
 *             BBB_NLL_GAUSS, BBB_NLL_GAUSS_HET: [3] sum_d (mu_d - y_d)^2                 (4 doubles)
 *           ECE = (1/n) sum_m |sum correct_m - sum confidence_m|.  Counts are integers, exact in fp64.
 * B == 0 is a no-op.  Bad kind or shape (an odd C with BBB_NLL_GAUSS_HET), n_bins out of range, sigma <= 0, a null
 * required pointer: BBB_EINVAL. */
int bbb_predictive_stats(const float *out, const void *target, int64_t S, int64_t B, int64_t C, int32_t kind,
                         float sigma, int32_t n_bins, float *mean, float *row_stats, int64_t *pred, double *acc,
                         void *stream);

/* ---- likelihood terms (BayesianNetwork.get_nll, networks.py:183-190) --------------------
 * nll += sum over (s, b) of the negative log likelihood; dout (nullable) = grad_scale * d nll / d out.
 * bbb_nll_ce:    logits [S,B,C], target int64 [B]       (CrossEntropyLoss(reduction='sum'))
 * bbb_nll_gauss: out [S,B,D], target [B,D]              (-Normal(out, sigma).log_prob(target).sum())
 */
int bbb_nll_ce(const float *logits, const int64_t *target, int64_t S, int64_t B, int64_t C,
               float grad_scale, double *nll, float *dlogits, void *stream);
int bbb_nll_gauss(const float *out, const float *target, float sigma, int64_t S, int64_t B, int64_t D,
                  float grad_scale, double *nll, float *dout, void *stream);
/* heteroscedastic regression (a learned per-input noise, Kendall & Gal 2017): the net has 2D outputs per row,
 * out [S,B,2D] = [f | r]: mean f = columns [0, D), raw scale r = columns [D, 2D), target [B,D];
 *   sigma = sigma_min + softplus(r),  softplus(r) = max(r, 0) + log1p(exp(-|r|)),  sigma_min > 0
 *   nll  += sum over (s, b, d) of (y - f)^2 / (2 sigma^2) + log sigma + log(2 pi) / 2
 *   dout (nullable) [S,B,2D], written in full:  d/df = g (f - y) / sigma^2,
 *                                               d/dr = g sigmoid(r) (1/sigma - (y - f)^2 / sigma^3),  g = grad_scale
 * Finite for r in [-40, 40] and large residuals (formed from (y - f) / sigma, never from sigma^3).  Launched with
 * programmatic dependent launch like its siblings.  Null out / target / nll, a negative size, D == 0 with S B > 0 or
 * sigma_min <= 0: BBB_EINVAL.  No network-level call (bbb_head_fwd, bbb_mlp_fwd) implements this likelihood. */
#define BBB_NLL_GAUSS_HET 3
int bbb_nll_gauss_het(const float *out, const float *target, float sigma_min, int64_t S, int64_t B, int64_t D,
                      float grad_scale, double *nll, float *dout, void *stream);

/* ---- the network's head in one launch --------------------------------------------------------
 * bbb_head_fwd = bbb_linear_fwd of a narrow layer (out <= 16: the classification / regression head, networks.py:164)
 * + bbb_nll_ce / bbb_nll_gauss on its outputs + bbb_elbo_finalize, i.e. the tail of sample_elbo (networks.py:199-209)
 * from the last layer's forward to the four returned scalars.  Exact fp32, deterministic.
 *   nll_kind  BBB_NLL_NONE: plain layer forward (target, nll, dy, out4 ignored);  BBB_NLL_CE: target = int64 [B];
 *             BBB_NLL_GAUSS: target = float [B,out], sigma = likelihood std;  any other kind (BBB_NLL_GAUSS_HET
 *             included): BBB_EINVAL
 *   y  [S,B,out] written;  dy (nullable) [S,B,out] = grad_scale * d nll / d y;  nll += sum over (s, b)
 *   logp, logq [S] += this layer's terms (BBB_F_LOGPROB); they must already hold the other layers' sums when out4 is
 *             requested, because the CTA that finishes last assembles out4 exactly as bbb_elbo_finalize does
 *   done_counter  zeroed device word used to find that CTA (required with out4; left zero again)
 * Needs in % 4 == 0, in <= 8192 and 16-byte aligned x / w rows; returns BBB_EUNSUPPORTED otherwise. */
#define BBB_NLL_NONE 0
#define BBB_NLL_CE 1
#define BBB_NLL_GAUSS 2
int bbb_head_fwd(const float *x, int64_t x_sample_stride, const float *w_mu, const float *w_rho,
                 const float *b_mu, const float *b_rho, const float *eps_w, const float *eps_b,
                 const bbb_rng *rng, const bbb_prior *prior, int64_t S, int64_t B, int64_t in, int64_t out,
                 int32_t flags, int32_t nll_kind, const void *target, float sigma, float grad_scale,
                 float *y, float *dy, double *logp, double *logq, double *nll, float beta,
                 const float *beta_dev, float *out4, uint32_t *done_counter, void *stream);

/* ---- the whole network in one call (batches of at most 128 rows, tcgen05 kind::tf32) ---------------------------------
 * bbb_mlp_fwd = the body of BayesianNetwork.sample_elbo (networks.py:192-209): BayesianNetwork.forward (166-172) for
 * all S samples -- every hidden BayesianLinear.forward (73-88); the ReLU between layers is applied by the CONSUMER, in
 * shared memory, to the tile its TMA has loaded -- then the head as bbb_head_fwd does it (last layer + get_nll (183-190)
 * and its gradient + the four returned scalars).  Replaces n_layers calls of bbb_linear_fwd / bbb_head_fwd: one host call
 * per network pass.
 *   layers[l]  w_mu, w_rho [out,in]; b_mu, b_rho [out]; eps_w [S,out,in] / eps_b [S,out] or NULL (Philox, tensor ids
 *              2l / 2l+1: rng->layer is ignored);  in of layer l+1 == out of layer l
 *              y [S,B,out]: the layer's PRE-activation output x W_s^T + b_s.  Hidden layers: must be ZERO-FILLED (the
 *              split-K partial tiles are added into it with TMA reduce-add); last layer: written
 *              dz, g_*: backward only (bbb_mlp_bwd)
 *   x [B,in0] is shared by all samples;  nll_kind / target / sigma / grad_scale / d_out / nll / beta / beta_dev / out4 /
 *   done_counter exactly as in bbb_head_fwd (d_out [S,B,out_last] = grad_scale * d nll / d outputs).
 * bbb_mlp_supported: 1 when bbb_mlp_fwd / bbb_mlp_bwd cover this network (dims[0..n_layers], BBB_F_TF32 in flags, B <= 128,
 * hidden widths multiples of 4, last layer a head of <= 16 outputs), else 0; otherwise the calls return
 * BBB_EUNSUPPORTED without launching anything and the per-layer entry points apply. */
typedef struct bbb_mlp_layer {
  const float *w_mu, *w_rho, *b_mu, *b_rho, *eps_w, *eps_b;
  int64_t in, out;
  float *y;                                       /* [S,B,out] pre-activation output (hidden layers: zero-filled)          */
  float *dz;                                      /* [S,B,out]: hidden layers zero-filled, accumulated by the layer above */
  float *g_w_mu, *g_w_rho, *g_b_mu, *g_b_rho;     /* parameter gradients, overwritten                                     */
} bbb_mlp_layer;
int bbb_mlp_supported(const int64_t *dims, int32_t n_layers, int64_t S, int64_t B, int32_t flags);
int bbb_mlp_fwd(const bbb_mlp_layer *layers, int32_t n_layers, const float *x, int64_t S, int64_t B,
                const bbb_rng *rng, const bbb_prior *prior, int32_t flags, int32_t nll_kind, const void *target,
                float sigma, float grad_scale, float *d_out, double *logp, double *logq, double *nll, float beta,
                const float *beta_dev, float *out4, uint32_t *done_counter, void *stream);
/* bbb_mlp_bwd = the autograd backward of the above (triggered at reg_task.py:72, class_task.py:78, bandits.py:49), all
 * layers in one call; replaces n_layers calls of bbb_linear_bwd (same gp / gq / gp_dev / gq_dev / g_dev_stride /
 * out_scale_dev meaning, eps regenerated from the same Philox coordinates).  Reads layers[l].y (the pre-activations the
 * forward stored) and layers[n-1].dz (= d_out of bbb_mlp_fwd); layers[l].dz of the hidden layers must be zero-filled:
 * the layer above adds (dz W_s) (y > 0) into it.  Writes g_w_mu / g_w_rho / g_b_mu / g_b_rho of every layer
 * (added to with BBB_F_ACCUM). */
int bbb_mlp_bwd(const bbb_mlp_layer *layers, int32_t n_layers, const float *x, int64_t S, int64_t B,
                const bbb_rng *rng, const bbb_prior *prior, int32_t flags, float gp, float gq, const float *gp_dev,
                const float *gq_dev, int64_t g_dev_stride, const float *out_scale_dev, void *stream);

/* ELBO assembly (networks.py:205-209 / 221-225):
 * out4 = { beta mean(logq) - beta mean(logp) + nll/S, mean(logp), mean(logq), nll/S }   (kl == NULL)
 * out4 = { beta kl + nll/S, kl, nll/S, 0 }                                              (kl != NULL)
 */
int bbb_elbo_finalize(const double *logp, const double *logq, const double *kl, const double *nll,
                      int64_t S, float beta, const float *beta_dev, float *out4, void *stream);
/* beta_dev (nullable): device scalar multiplied into `beta`, so a captured CUDA graph can follow the
 * reference's per-minibatch beta schedule (reg_task.py:63) without re-capture. */

/* ---- optimiser (SURVEY 8f-1): torch.optim.Adam.step() over all parameter tensors in ONE launch ----
 * replaces torch.optim.Adam at reg_task.py:53,73 / class_task.py:60,79 / bandits.py:36,50 (same update rule:
 * m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2; p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps)).
 * params/grads/exp_avg/exp_avg_sq/sizes are HOST arrays of n_tensors (<= 32) device pointers / element counts.
 * t = step + (step_dev ? *step_dev : 0) is the 1-based Adam step; lr is multiplied by *lr_scale_dev if given.
 * The hyper-parameters are doubles because torch forms 1-beta, the bias corrections and the step size in double. */
int bbb_adam_step(int32_t n_tensors, float *const *params, const float *const *grads, float *const *exp_avg,
                  float *const *exp_avg_sq, const int64_t *sizes, double lr, double beta1, double beta2, double eps,
                  uint32_t step, const uint32_t *step_dev, const float *lr_scale_dev, void *stream);

/* ---- multi-GPU optimiser step over NVLink peer memory (SURVEY 8e: the gradient exchange) -----------------------
 * Gradient reduce-scatter + Adam + parameter all-gather in ONE kernel: rank r sums the W ranks' flat gradient
 * buckets over its slice [r n/W, (r+1) n/W) with peer loads, applies torch.optim.Adam's update with its local
 * exp_avg / exp_avg_sq (only that slice is ever touched), and stores the new parameters into every rank's flat
 * parameter buffer with peer stores.  Replaces ncclAllReduce + optimiser.step() of a data-parallel step.  The
 * gradient is the MEAN over the ranks (each rank holds the gradient of its own Monte-Carlo samples).
 *   grads / params / flags   pointers to every rank's buffers AS MAPPED IN THIS PROCESS (cudaIpcOpenMemHandle, or the
 *                            same process for several devices); flags: 2*world zero-initialised uint32 per rank
 *   epoch, done_blocks       zero-initialised device words of THIS rank: epoch[0] = call count; done_blocks[0] = block
 *                            counter, done_blocks[1] = error word, set to 1 when a peer did not show up within the
 *                            kernel's bounded wait (seconds): the results of that call are then undefined
 * Every rank must make the call once per step, on any stream; the kernel completes only when all ranks have
 * finished with this rank's buffers.  world == 1 degenerates to a flat single-tensor Adam. */
#define BBB_MAX_PEERS 8
typedef struct bbb_peer_comm {
  int32_t world, rank;
  const float *grads[BBB_MAX_PEERS];
  float *params[BBB_MAX_PEERS];
  uint32_t *flags[BBB_MAX_PEERS];
  uint32_t *epoch;
  uint32_t *done_blocks;
  const float *mc_grads;   /* optional NVLS multicast mappings of the SAME gradient / parameter buffers (every rank's copy  */
  float *mc_params;        /* bound to one multicast object, e.g. torch symmetric memory's multicast_ptr).  With mc_grads
                              the kernel reads its slice of the gradient SUM with one multimem.ld_reduce per 16 bytes
                              (the NVSwitch adds the W copies: inbound traffic n/W instead of (W-1) n/W); with mc_params it
                              writes the new parameters to every rank with one multimem.st (outbound n/W likewise).
                              NULL: peer loads / stores through grads[] / params[] */
} bbb_peer_comm;
/* let kernels of the CURRENT device load / store memory of `peer_device` (cudaDeviceEnablePeerAccess; idempotent) */
int bbb_enable_peer_access(int32_t peer_device);
/* map an allocation another process of this node exported with cudaIpcGetMemHandle (64-byte handle, HOST pointer)
 * into this process for the CURRENT device; *out_ptr = mapped base + offset_bytes.  Open a handle once per process. */
int bbb_ipc_open(const void *handle, int64_t offset_bytes, void **out_ptr);
int bbb_adam_step_peer(const bbb_peer_comm *comm, float *exp_avg, float *exp_avg_sq, int64_t n, double lr,
                       double beta1, double beta2, double eps, uint32_t step, const uint32_t *step_dev,
                       const float *lr_scale_dev, void *stream);

/* ---- diagnostic: device time of every kernel the network-level calls launch ------------------------------------------
 * bbb_timing_enable(1) clears the records and starts bracketing each kernel of bbb_mlp_fwd / bbb_mlp_bwd with CUDA events
 * on the launching stream (do not enable while a CUDA graph is being captured); bbb_timing_report synchronises the
 * device and writes a JSON object {"kernel[inxout]": [total ms, launches], ...} into buf (HOST pointer). */
int bbb_timing_enable(int32_t on);
/* debug aid: when buf != NULL every CTA of the network-level kernels launched afterwards writes 16 %globaltimer stamps
 * (phase boundaries, ns) at buf[2560 * launch + 16 * cta ..] (launch = 0..7, in launch order; buf holds 8 * 2560 words);
 * tools/kernel_timeline.py prints the phase durations.  NULL switches it off. */
int bbb_debug_set_timeline(unsigned long long *buf);
/* Debug / test aid: the large-batch wgrad splits the sample groups of a tile over two CTAs (partial gradients in a
 * stream-ordered workspace, added in by a second kernel) when that fills the SMs better.  mode 0: decide by shape
 * (default), 1: split whenever there are two sample groups, -1: never. */
int bbb_debug_wgrad_split(int mode);
int bbb_timing_report(char *buf, int64_t buf_bytes);

/* *counter += inc  (advances a bbb_rng.step_dev between steps; one tiny launch, graph-capturable) */
int bbb_counter_add(uint32_t *counter, uint32_t inc, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* BBB_H_ */
