// Bandwidth-bound single-pass kernels: ELBO reductions over (mu, rho[, eps]), closed-form KL,
// the Philox eps stream, likelihood terms and ELBO assembly.
//
// Roofline: HBM.  bbb_logprob_reduce reads 8 B/weight (mu, rho; +4 with injected eps, +4 when W is
// written) and does ~60 flops + Philox per weight; bbb_kl_gauss reads 8 B/weight.  Loads are 16-byte
// vectors, four independent vectors in flight per thread, grid = a multiple of the 148 SMs.
// bbb_gauss_prior_logprob / bbb_gauss_prior_kl (per-weight priors) read 16 B/parameter (mu, rho, prior mu, prior rho;
// +4 S with injected eps), the log-prob call once per group of 8 samples (one group for S <= 8); their backward calls
// read the same 16 B and read-modify-write both gradients: 32 B/parameter (+4 S injected).
#include <stdarg.h>

#include <atomic>

#include "bbb_common.cuh"

namespace bbb {

// ---- error plumbing ------------------------------------------------------------------
char *last_error_buf() {
  static thread_local char buf[512] = "ok";
  return buf;
}
int fail(int code, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(last_error_buf(), 512, fmt, ap);
  va_end(ap);
  return code;
}

static std::atomic<uint64_t> g_launches{0};
void note_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

namespace {

constexpr int RT = 256;  // threads per CTA of the reduction kernels

template <bool kInjected, bool kWriteW>
__global__ void __launch_bounds__(RT) logprob_reduce_kernel(const float *__restrict__ mu,
                                                            const float *__restrict__ rho,
                                                            const float *__restrict__ eps, RngDev rng,
                                                            uint32_t tensor, uint32_t sample, PriorDev prior,
                                                            int64_t n, int sample_flag, float *__restrict__ w_out,
                                                            double *logp, double *logq) {
  __shared__ float red[64];
  rng_resolve(rng);
  float lp = 0.0f, lq = 0.0f;
  const int64_t nq = n >> 2;  // whole quads
  const int64_t stride = (int64_t)gridDim.x * RT;
  for (int64_t q = (int64_t)blockIdx.x * RT + threadIdx.x; q < nq; q += stride) {
    const float4 m4 = __ldg(reinterpret_cast<const float4 *>(mu) + q);
    const float4 r4 = __ldg(reinterpret_cast<const float4 *>(rho) + q);
    const float m[4] = {m4.x, m4.y, m4.z, m4.w}, r[4] = {r4.x, r4.y, r4.z, r4.w};
    float e[4] = {0.f, 0.f, 0.f, 0.f}, w[4];
    if (sample_flag) {
      if (kInjected) {
        const float4 e4 = __ldg(reinterpret_cast<const float4 *>(eps) + q);
        e[0] = e4.x; e[1] = e4.y; e[2] = e4.z; e[3] = e4.w;
      } else {
        philox_normal4(rng, tensor, sample, (uint32_t)q, e);
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float sg = softplus_f(r[j]);
      w[j] = __fadd_rn(m[j], __fmul_rn(sg, e[j]));
      lp += logp_elem(prior, w[j]);
      lq += logq_elem(sg, e[j]);
    }
    if (kWriteW) reinterpret_cast<float4 *>(w_out)[q] = make_float4(w[0], w[1], w[2], w[3]);
  }
  // tail (n % 4 elements) handled by the first threads of block 0
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const int64_t i = (nq << 2) + threadIdx.x;
    const float sg = softplus_f(rho[i]);
    float e = 0.0f;
    if (sample_flag) e = kInjected ? eps[i] : philox_normal1(rng, tensor, sample, (uint64_t)i);
    const float w = __fadd_rn(mu[i], __fmul_rn(sg, e));
    lp += logp_elem(prior, w);
    lq += logq_elem(sg, e);
    if (kWriteW) w_out[i] = w;
  }
  block_sum2_atomic(lp, lq, red, logp, logq);
}

__global__ void __launch_bounds__(RT) kl_gauss_kernel(const float *__restrict__ mu, const float *__restrict__ rho,
                                                      float log_sp, float inv_sp2, int64_t n, double *kl) {
  __shared__ float red[64];
  float acc = 0.0f;
  const int64_t nq = n >> 2, stride = (int64_t)gridDim.x * RT;
  for (int64_t q = (int64_t)blockIdx.x * RT + threadIdx.x; q < nq; q += stride) {
    const float4 m4 = __ldg(reinterpret_cast<const float4 *>(mu) + q);
    const float4 r4 = __ldg(reinterpret_cast<const float4 *>(rho) + q);
    const float m[4] = {m4.x, m4.y, m4.z, m4.w}, r[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float sg = softplus_f(r[j]);
      acc += 2.0f * (log_sp - logf(sg)) - 1.0f + (sg * sg + m[j] * m[j]) * inv_sp2;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const int64_t i = (nq << 2) + threadIdx.x;
    const float sg = softplus_f(rho[i]);
    acc += 2.0f * (log_sp - logf(sg)) - 1.0f + (sg * sg + mu[i] * mu[i]) * inv_sp2;
  }
  block_sum2_atomic(0.5f * acc, 0.0f, red, kl, nullptr);
}

__global__ void __launch_bounds__(RT) philox_fill_kernel(float *__restrict__ out, int64_t n, RngDev rng,
                                                         uint32_t tensor, uint32_t sample) {
  const int64_t nq = (n + 3) >> 2, stride = (int64_t)gridDim.x * RT;
  for (int64_t q = (int64_t)blockIdx.x * RT + threadIdx.x; q < nq; q += stride) {
    float z[4];
    philox_normal4(rng, tensor, sample, (uint32_t)q, z);
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if ((q << 2) + j < n) out[(q << 2) + j] = z[j];
  }
}

// one warp per (s, b) row of logits
__global__ void __launch_bounds__(128) nll_ce_kernel(const float *__restrict__ logits,
                                                     const int64_t *__restrict__ target, int64_t rows, int64_t B,
                                                     int64_t C, float grad_scale, double *nll,
                                                     float *__restrict__ dlogits) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float red[64];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float local = 0.0f;
  for (int64_t row = (int64_t)blockIdx.x * 4 + warp; row < rows; row += (int64_t)gridDim.x * 4) {
    const float *z = logits + row * C;
    const int64_t t = target[row % B];
    float mx = -INFINITY;
    for (int64_t c = lane; c < C; c += 32) mx = fmaxf(mx, z[c]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float se = 0.0f;
    for (int64_t c = lane; c < C; c += 32) se += expf(z[c] - mx);
    se = warp_sum(se);
    const float lse = mx + logf(se);
    if (lane == 0) local += lse - z[t];
    if (dlogits) {
      float *g = dlogits + row * C;
      for (int64_t c = lane; c < C; c += 32) g[c] = grad_scale * (expf(z[c] - lse) - (c == t ? 1.0f : 0.0f));
    }
  }
  block_sum2_atomic(local, 0.0f, red, nll, nullptr);
}

__global__ void __launch_bounds__(RT) nll_gauss_kernel(const float *__restrict__ out, const float *__restrict__ target,
                                                       float inv_2var, float inv_var, float cst, int64_t n,
                                                       int64_t per_sample, float grad_scale, double *nll,
                                                       float *__restrict__ dout) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float red[64];
  float acc = 0.0f;
  for (int64_t i = (int64_t)blockIdx.x * RT + threadIdx.x; i < n; i += (int64_t)gridDim.x * RT) {
    const float d = out[i] - target[i % per_sample];
    acc += fmaf(d * d, inv_2var, cst);
    if (dout) dout[i] = grad_scale * d * inv_var;
  }
  block_sum2_atomic(acc, 0.0f, red, nll, nullptr);
}

// Heteroscedastic Gaussian: row (s, b) of `out` is [f (D) | r (D)], sigma = sigma_min + softplus(r).  One thread per
// (s, b, d).  With a = (y - f) / sigma every term is formed from a and 1 / sigma, never from sigma^2 or sigma^3, so the
// value and both gradients stay finite for r in [-40, 40] and residuals of 1e3 down to sigma_min ~ 1e-6.
__global__ void __launch_bounds__(RT) nll_gauss_het_kernel(const float *__restrict__ out,
                                                           const float *__restrict__ target, float sigma_min,
                                                           float cst, int64_t n, int64_t B, int64_t D,
                                                           float grad_scale, double *nll, float *__restrict__ dout) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float red[64];
  float acc = 0.0f;
  for (int64_t i = (int64_t)blockIdx.x * RT + threadIdx.x; i < n; i += (int64_t)gridDim.x * RT) {
    const int64_t row = i / D, d = i - row * D;
    const int64_t o = row * 2 * D + d;
    const float f = out[o], r = out[o + D];
    const float e = expf(-fabsf(r));
    const float sg = fmaxf(r, 0.0f) + log1pf(e);                  // softplus(r), stable for either sign
    const float sig = r >= 0.0f ? 1.0f / (1.0f + e) : e / (1.0f + e);   // sigmoid(r) = d softplus / dr
    const float sigma = sigma_min + sg, inv_s = 1.0f / sigma;
    const float a = (target[(row % B) * D + d] - f) * inv_s;
    acc += fmaf(0.5f * a, a, logf(sigma) + cst);
    if (dout) {
      dout[o] = -grad_scale * a * inv_s;                             // g (f - y) / sigma^2
      dout[o + D] = grad_scale * sig * inv_s * fmaf(-a, a, 1.0f);    // g sigmoid(r) (1/sigma - (y - f)^2 / sigma^3)
    }
  }
  block_sum2_atomic(acc, 0.0f, red, nll, nullptr);
}

__global__ void elbo_finalize_kernel(const double *logp, const double *logq, const double *kl, const double *nll,
                                     int S, float beta, const float *beta_dev, float *out4) {
  pdl_launch_dependents();
  pdl_wait();
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (beta_dev) beta *= *beta_dev;
  const float nll_m = (float)(nll[0] / S);
  if (kl) {
    const float k = (float)kl[0];
    out4[0] = beta * k + nll_m; out4[1] = k; out4[2] = nll_m; out4[3] = 0.0f;
  } else {
    double lp = 0.0, lq = 0.0;
    for (int s = 0; s < S; ++s) { lp += (double)(float)logp[s]; lq += (double)(float)logq[s]; }
    const float lpm = (float)(lp / S), lqm = (float)(lq / S);
    out4[0] = beta * lqm - beta * lpm + nll_m; out4[1] = lpm; out4[2] = lqm; out4[3] = nll_m;
  }
}

// signal-to-noise ratio in decibels of every Gaussian parameter, 10 log10(|mu| / softplus(rho)) (weight_pruning.py:81-83),
// and/or the pruning pass of weight_pruning.py:85-115: mu, rho *= (snr > threshold), in place.  One pass over (mu, rho).
__global__ void __launch_bounds__(RT) snr_kernel(float *__restrict__ mu, float *__restrict__ rho, int64_t n,
                                                 float *__restrict__ snr_out, int prune, float threshold,
                                                 unsigned long long *kept) {
  const int64_t stride = (int64_t)gridDim.x * RT;
  unsigned long long mine = 0;
  for (int64_t i = (int64_t)blockIdx.x * RT + threadIdx.x; i < n; i += stride) {
    const float m = mu[i], r = rho[i];
    const float snr = 10.0f * log10f(fabsf(m) / softplus_f(r));
    if (snr_out) snr_out[i] = snr;
    if (prune) {
      const bool keep = snr > threshold;        // (NaN and -inf, i.e. mu == 0, are dropped, as `snrs > threshold` does)
      if (!keep) { mu[i] = m * 0.0f; rho[i] = r * 0.0f; }
      mine += keep ? 1ull : 0ull;
    }
  }
  if (prune && kept) {
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(kept, mine);
  }
}

// BNN_Classification.predict (class_task.py:81-87): softmax of every sampled forward, averaged over the samples.
// One warp per batch row; logits [S,B,C], probs [B,C].
__global__ void __launch_bounds__(128) softmax_mean_kernel(const float *__restrict__ logits, int64_t S, int64_t B, int64_t C,
                                                           float *__restrict__ probs) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t b = (int64_t)blockIdx.x * 4 + warp; b < B; b += (int64_t)gridDim.x * 4) {
    for (int64_t c0 = 0; c0 < C; c0 += 32) {        // (C <= 32: one pass; wider heads accumulate chunk by chunk)
      const int64_t c = c0 + lane;
      float acc = 0.0f;
      for (int64_t s = 0; s < S; ++s) {
        const float *z = logits + (s * B + b) * C;
        float mx = -INFINITY;
        for (int64_t j = lane; j < C; j += 32) mx = fmaxf(mx, z[j]);
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        float sum = 0.0f;
        for (int64_t j = lane; j < C; j += 32) sum += expf(z[j] - mx);
        sum = warp_sum(sum);
        if (c < C) acc += expf(z[c] - mx) / sum;
      }
      if (c < C) probs[b * C + c] = acc / (float)S;
    }
  }
}

// ---- per-weight Gaussian priors p = N(m, sp^2), sp = softplus(r) (bbb_gauss_prior_*) ------------------------------------
// One launch streams every tensor of a network: the table travels by value in the kernel parameters (4.4 KB, the
// large-parameter launch of CUDA 12.1+), each thread takes quads (4 consecutive elements) of each tensor in turn with
// a grid stride.  A tensor whose pointers are 16-byte aligned (and, with injected eps, whose n is a multiple of 4, so
// every eps row is) uses float4 loads; otherwise, and for the n % 4 tail, scalar loads of the valid elements.
// Every term is formed from (w - m)/sp, (mu - m)/sp and sigma/sp, so sigma, sp ~ 1e-5 stay finite.
constexpr int kGpMax = BBB_GAUSS_PRIOR_MAX_TENSORS;
constexpr int kGpS = 8;   // samples per CTA row of the log-prob kernel: their partial sums live in registers
struct GpTable {
  const float *mu[kGpMax], *rho[kGpMax], *pm[kGpMax], *pr[kGpMax], *eps[kGpMax];
  float *gm[kGpMax], *gr[kGpMax];
  int64_t n[kGpMax];
  uint32_t id[kGpMax];
  bool vec[kGpMax];
  int nt;
};

__device__ __forceinline__ void ld4_rw(const float *p, int64_t i, int valid, bool vec, float v[4]) {
  if (vec && valid == 4) {
    const float4 t = *reinterpret_cast<const float4 *>(p + i);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = j < valid ? p[i + j] : 0.0f;
  }
}
__device__ __forceinline__ void st4(float *p, int64_t i, int valid, bool vec, const float v[4]) {
  if (vec && valid == 4) {
    *reinterpret_cast<float4 *>(p + i) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (j < valid) p[i + j] = v[j];
  }
}
// the eps of the 4 elements of quad q, sample `smp` (index s of the call): injected row s, or Philox exactly as the
// layer kernels draw it (the linear-index quad mapping of logprob_reduce_kernel)
__device__ __forceinline__ void gp_eps(const GpTable &t, int k, const RngDev &rng, int64_t s, int64_t q, int valid,
                                       float e[4]) {
  if (t.eps[k]) ld4(t.eps[k] + s * t.n[k], q << 2, valid, t.vec[k], e);
  else philox_normal4(rng, t.id[k], rng.sample_base + (uint32_t)s, (uint32_t)q, e);
}

// logp[s] += sum log N(w_s; m, sp^2), logq[s] += sum log N(w_s; mu, sigma^2) for the kGpS samples of blockIdx.y
__global__ void __launch_bounds__(RT, 2) gauss_prior_logprob_kernel(const GpTable t, int64_t S, RngDev rng, double *logp,
                                                                 double *logq) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float red[64];
  rng_resolve(rng);
  const int64_t s0 = (int64_t)blockIdx.y * kGpS;
  const int ns = (int)(S - s0 < kGpS ? S - s0 : kGpS);
  float lp[kGpS], lq[kGpS];
#pragma unroll
  for (int j = 0; j < kGpS; ++j) lp[j] = lq[j] = 0.0f;
  const int64_t stride = (int64_t)gridDim.x * RT;
  for (int k = 0; k < t.nt; ++k) {
    const int64_t n = t.n[k], nq = (n + 3) >> 2;
    for (int64_t q = (int64_t)blockIdx.x * RT + threadIdx.x; q < nq; q += stride) {
      const int valid = (int)(n - (q << 2) < 4 ? n - (q << 2) : 4);
      float m[4], r[4], pm[4], pr[4];
      ld4(t.mu[k], q << 2, valid, t.vec[k], m);
      ld4(t.rho[k], q << 2, valid, t.vec[k], r);
      ld4(t.pm[k], q << 2, valid, t.vec[k], pm);
      ld4(t.pr[k], q << 2, valid, t.vec[k], pr);
      // cp, cq: the sample-independent parts of the quad's log p and log q, -sum (log sp + log(2 pi)/2) and
      // -sum (log sigma + log(2 pi)/2)
      float sg[4], isp[4], cp = 0.0f, cq = 0.0f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        sg[j] = softplus_f(r[j]);
        const float sp = softplus_f(pr[j]);
        isp[j] = 1.0f / sp;
        if (j < valid) {
          cp -= kHalfLog2Pi + logf(sp);
          cq -= kHalfLog2Pi + logf(sg[j]);
        }
      }
#pragma unroll
      for (int js = 0; js < kGpS; ++js) {
        if (js < ns) {
          float e[4];
          gp_eps(t, k, rng, s0 + js, q, valid, e);
          float ap = 0.0f, aq = 0.0f;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (j < valid) {
              const float w = __fadd_rn(m[j], __fmul_rn(sg[j], e[j]));
              const float a = (w - pm[j]) * isp[j];
              ap = fmaf(a, a, ap);
              aq = fmaf(e[j], e[j], aq);
            }
          }
          lp[js] += fmaf(-0.5f, ap, cp);
          lq[js] += fmaf(-0.5f, aq, cq);
        }
      }
    }
  }
#pragma unroll
  for (int js = 0; js < kGpS; ++js)
    if (js < ns) block_sum2_atomic(lp[js], lq[js], red, logp + s0 + js, logq + s0 + js);
}

// grad_mu += c sum_s gp_s (-(w_s - m)/sp^2),  grad_rho += c sigmoid(rho) sum_s [gp_s (-(w_s - m)/sp^2) eps_s - gq_s/sigma]
__global__ void __launch_bounds__(RT) gauss_prior_logprob_bwd_kernel(const GpTable t, int64_t S, RngDev rng, float gp,
                                                                     float gq, const float *gp_dev,
                                                                     const float *gq_dev, int64_t gstride,
                                                                     const float *out_scale_dev) {
  pdl_launch_dependents();
  pdl_wait();
  rng_resolve(rng);
  const float c = out_scale_dev ? __ldg(out_scale_dev) : 1.0f;
  const int64_t stride = (int64_t)gridDim.x * RT;
  for (int k = 0; k < t.nt; ++k) {
    const int64_t n = t.n[k], nq = (n + 3) >> 2;
    for (int64_t q = (int64_t)blockIdx.x * RT + threadIdx.x; q < nq; q += stride) {
      const int64_t i = q << 2;
      const int valid = (int)(n - i < 4 ? n - i : 4);
      float m[4], r[4], pm[4], pr[4];
      ld4(t.mu[k], i, valid, t.vec[k], m);
      ld4(t.rho[k], i, valid, t.vec[k], r);
      ld4(t.pm[k], i, valid, t.vec[k], pm);
      ld4(t.pr[k], i, valid, t.vec[k], pr);
      float sg[4], isp[4], gm[4], gr[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        sg[j] = softplus_f(r[j]);
        isp[j] = 1.0f / softplus_f(pr[j]);
        gm[j] = gr[j] = 0.0f;
      }
      float gq_sum = 0.0f;
      for (int64_t s = 0; s < S; ++s) {
        const float gps = gp_dev ? gp * __ldg(gp_dev + s * gstride) : gp;
        gq_sum += gq_dev ? gq * __ldg(gq_dev + s * gstride) : gq;
        float e[4];
        gp_eps(t, k, rng, s, q, valid, e);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float w = __fadd_rn(m[j], __fmul_rn(sg[j], e[j]));
          const float tt = -gps * ((w - pm[j]) * isp[j]) * isp[j];
          gm[j] += tt;
          gr[j] = fmaf(tt, e[j], gr[j]);
        }
      }
      float om[4], orh[4];
      ld4_rw(t.gm[k], i, valid, t.vec[k], om);
      ld4_rw(t.gr[k], i, valid, t.vec[k], orh);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        om[j] = fmaf(c, gm[j], om[j]);
        orh[j] = fmaf(c * sigmoid_f(r[j]), gr[j] - gq_sum / sg[j], orh[j]);
      }
      st4(t.gm[k], i, valid, t.vec[k], om);
      st4(t.gr[k], i, valid, t.vec[k], orh);
    }
  }
}

// The scale part of one element's KL, (u^2 - 1)/2 - log u with u = sigma/sp and v = u - 1 = (sigma - sp)/sp (formed
// from the difference, exact near u = 1).  For |v| < 0.1 the closed form cancels; there it is the series
// v^2 - v^3/3 + v^4/4 - ... to v^9 (truncation < 1e-8 relative), exactly 0 at v = 0.
__device__ __forceinline__ float kl_scale_term(float u, float v) {
  if (fabsf(v) >= 0.1f) return fmaf(0.5f * u, u, -0.5f) - logf(u);
  float p = -1.0f / 9.0f;
  p = fmaf(p, v, 1.0f / 8.0f);
  p = fmaf(p, v, -1.0f / 7.0f);
  p = fmaf(p, v, 1.0f / 6.0f);
  p = fmaf(p, v, -1.0f / 5.0f);
  p = fmaf(p, v, 1.0f / 4.0f);
  p = fmaf(p, v, -1.0f / 3.0f);
  p = fmaf(p, v, 1.0f);
  return p * v * v;
}

// bwd == false: *kl += sum [f(v) + d^2/2], v = (sigma - sp)/sp, d = (mu - m)/sp  (= log(sp/sigma) + (sigma^2 +
// (mu - m)^2)/(2 sp^2) - 1/2);  bwd == true: grad_mu += c d/sp, grad_rho += c sigmoid(rho) v (1/sp + 1/sigma)
// (= c sigmoid(rho) (sigma/sp^2 - 1/sigma)).  q == p gives v = d = 0: exactly zero terms and gradients.
template <bool kBwd>
__global__ void __launch_bounds__(RT) gauss_prior_kl_kernel(const GpTable t, double *kl, float g_kl,
                                                            const float *g_kl_dev, const float *out_scale_dev) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float red[64];
  float c = 0.0f;
  if (kBwd) c = g_kl * (g_kl_dev ? __ldg(g_kl_dev) : 1.0f) * (out_scale_dev ? __ldg(out_scale_dev) : 1.0f);
  float acc = 0.0f;
  const int64_t stride = (int64_t)gridDim.x * RT;
  for (int k = 0; k < t.nt; ++k) {
    const int64_t n = t.n[k], nq = (n + 3) >> 2;
    for (int64_t q = (int64_t)blockIdx.x * RT + threadIdx.x; q < nq; q += stride) {
      const int64_t i = q << 2;
      const int valid = (int)(n - i < 4 ? n - i : 4);
      float m[4], r[4], pm[4], pr[4];
      ld4(t.mu[k], i, valid, t.vec[k], m);
      ld4(t.rho[k], i, valid, t.vec[k], r);
      ld4(t.pm[k], i, valid, t.vec[k], pm);
      ld4(t.pr[k], i, valid, t.vec[k], pr);
      float om[4], orh[4];
      if (kBwd) {
        ld4_rw(t.gm[k], i, valid, t.vec[k], om);
        ld4_rw(t.gr[k], i, valid, t.vec[k], orh);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float sg = softplus_f(r[j]), sp = softplus_f(pr[j]);
        const float v = __fdiv_rn(sg - sp, sp), d = __fdiv_rn(m[j] - pm[j], sp);
        if (kBwd) {
          om[j] = fmaf(c, __fdiv_rn(d, sp), om[j]);
          orh[j] = fmaf(c * sigmoid_f(r[j]), v * (__fdiv_rn(1.0f, sp) + __fdiv_rn(1.0f, sg)), orh[j]);
        } else if (j < valid) {
          acc += fmaf(0.5f * d, d, kl_scale_term(__fdiv_rn(sg, sp), v));
        }
      }
      if (kBwd) {
        st4(t.gm[k], i, valid, t.vec[k], om);
        st4(t.gr[k], i, valid, t.vec[k], orh);
      }
    }
  }
  if (!kBwd) block_sum2_atomic(acc, 0.0f, red, kl, nullptr);
}

inline int grid_for(int64_t work_items, int per_cta) {

  int64_t need = (work_items + per_cta - 1) / per_cta;
  int64_t cap = (int64_t)sm_count() * 8;  // 8 resident CTAs of 256 threads per SM
  if (need < 1) need = 1;
  return (int)(need < cap ? need : cap);
}
inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace
}  // namespace bbb

using namespace bbb;

extern "C" int bbb_logprob_reduce(const float *mu, const float *rho, const float *eps, uint64_t seed, uint32_t step,
                                  uint32_t sample, uint32_t tensor_id, const bbb_prior *prior, int64_t n,
                                  int32_t flags, float *w_out, double *logp, double *logq, void *stream) {
  BBB_CHECK_ARG(mu && rho && prior && logp && logq, "null pointer");
  BBB_CHECK_ARG(n >= 0, "negative size");
  BBB_CHECK_ARG(aligned16(mu) && aligned16(rho) && (!eps || aligned16(eps)) && (!w_out || aligned16(w_out)),
                "pointers must be 16-byte aligned");
  if (n == 0) return BBB_OK;
  bbb_rng r{seed, step, 0, 0, nullptr};
  RngDev rng = make_rng_dev(&r);
  PriorDev pd = make_prior_dev(prior);
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = grid_for(n >> 2, RT * 4);
  const int sf = (flags & BBB_F_SAMPLE) ? 1 : 0;
#define LAUNCH(INJ, WR) \
  logprob_reduce_kernel<INJ, WR><<<grid, RT, 0, st>>>(mu, rho, eps, rng, tensor_id, sample, pd, n, sf, w_out, logp, logq)
  if (eps && w_out) LAUNCH(true, true);
  else if (eps) LAUNCH(true, false);
  else if (w_out) LAUNCH(false, true);
  else LAUNCH(false, false);
#undef LAUNCH
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

extern "C" int bbb_kl_gauss(const float *mu, const float *rho, float sigma_p, int64_t n, double *kl, void *stream) {
  BBB_CHECK_ARG(mu && rho && kl, "null pointer");
  BBB_CHECK_ARG(n >= 0 && sigma_p > 0, "bad size or sigma_p");
  BBB_CHECK_ARG(aligned16(mu) && aligned16(rho), "pointers must be 16-byte aligned");
  if (n == 0) return BBB_OK;
  kl_gauss_kernel<<<grid_for(n >> 2, RT * 4), RT, 0, (cudaStream_t)stream>>>(
      mu, rho, logf(sigma_p), 1.0f / (sigma_p * sigma_p), n, kl);
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

namespace bbb { namespace {
// the by-value kernel table of a bbb_gauss_prior_* call, and the quads it covers (0: nothing to launch); BBB_EINVAL
// for a bad table (see bbb.h)
int gp_table(const bbb_gauss_prior_tensor *t, int32_t n_tensors, bool bwd, GpTable &g, int64_t &quads) {
  BBB_CHECK_ARG(n_tensors >= 0 && n_tensors <= kGpMax, "n_tensors outside [0, 64]");
  BBB_CHECK_ARG(t || n_tensors == 0, "null tensor table");
  g.nt = 0;
  quads = 0;
  for (int32_t k = 0; k < n_tensors; ++k) {
    const bbb_gauss_prior_tensor &x = t[k];
    BBB_CHECK_ARG(x.n >= 0, "negative size");
    if (x.n == 0) continue;
    BBB_CHECK_ARG(x.mu && x.rho && x.prior_mu && x.prior_rho, "null mu / rho / prior_mu / prior_rho");
    BBB_CHECK_ARG(!bwd || (x.grad_mu && x.grad_rho), "null grad_mu / grad_rho");
    const int i = g.nt++;
    g.mu[i] = x.mu; g.rho[i] = x.rho; g.pm[i] = x.prior_mu; g.pr[i] = x.prior_rho; g.eps[i] = x.eps;
    g.gm[i] = bwd ? x.grad_mu : nullptr; g.gr[i] = bwd ? x.grad_rho : nullptr;
    g.n[i] = x.n;
    g.id[i] = x.tensor_id;
    g.vec[i] = aligned16(x.mu) && aligned16(x.rho) && aligned16(x.prior_mu) && aligned16(x.prior_rho) &&
               (!x.eps || (aligned16(x.eps) && x.n % 4 == 0)) && (!bwd || (aligned16(x.grad_mu) && aligned16(x.grad_rho)));
    quads += (x.n + 3) >> 2;
  }
  return BBB_OK;
}
} }

extern "C" int bbb_gauss_prior_logprob(const bbb_gauss_prior_tensor *t, int32_t n_tensors, int64_t S,
                                       const bbb_rng *rng, double *logp, double *logq, void *stream) {
  BBB_CHECK_ARG(S > 0, "S <= 0");
  BBB_CHECK_ARG(rng && logp && logq, "null rng / logp / logq");
  GpTable g;
  int64_t quads;
  if (int st = gp_table(t, n_tensors, false, g, quads)) return st;
  if (quads == 0) return BBB_OK;
  BBB_CHECK_CUDA(launch_pdl(gauss_prior_logprob_kernel, dim3(grid_for(quads, RT), (unsigned)((S + kGpS - 1) / kGpS)),
                            dim3(RT), 0, (cudaStream_t)stream, g, S, make_rng_dev(rng), logp, logq));
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

extern "C" int bbb_gauss_prior_logprob_bwd(const bbb_gauss_prior_tensor *t, int32_t n_tensors, int64_t S,
                                           const bbb_rng *rng, float gp, float gq, const float *gp_dev,
                                           const float *gq_dev, int64_t g_dev_stride, const float *out_scale_dev,
                                           void *stream) {
  BBB_CHECK_ARG(S > 0, "S <= 0");
  BBB_CHECK_ARG(rng, "null rng");
  BBB_CHECK_ARG(g_dev_stride >= 0, "negative g_dev_stride");
  GpTable g;
  int64_t quads;
  if (int st = gp_table(t, n_tensors, true, g, quads)) return st;
  if (quads == 0) return BBB_OK;
  BBB_CHECK_CUDA(launch_pdl(gauss_prior_logprob_bwd_kernel, dim3(grid_for(quads, RT)), dim3(RT), 0,
                            (cudaStream_t)stream, g, S, make_rng_dev(rng), gp, gq, gp_dev, gq_dev, g_dev_stride,
                            out_scale_dev));
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

extern "C" int bbb_gauss_prior_kl(const bbb_gauss_prior_tensor *t, int32_t n_tensors, double *kl, void *stream) {
  BBB_CHECK_ARG(kl, "null kl");
  GpTable g;
  int64_t quads;
  if (int st = gp_table(t, n_tensors, false, g, quads)) return st;
  if (quads == 0) return BBB_OK;
  BBB_CHECK_CUDA(launch_pdl(gauss_prior_kl_kernel<false>, dim3(grid_for(quads, RT)), dim3(RT), 0, (cudaStream_t)stream,
                            g, kl, 0.0f, (const float *)nullptr, (const float *)nullptr));
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

extern "C" int bbb_gauss_prior_kl_bwd(const bbb_gauss_prior_tensor *t, int32_t n_tensors, float g_kl,
                                      const float *g_kl_dev, const float *out_scale_dev, void *stream) {
  GpTable g;
  int64_t quads;
  if (int st = gp_table(t, n_tensors, true, g, quads)) return st;
  if (quads == 0) return BBB_OK;
  BBB_CHECK_CUDA(launch_pdl(gauss_prior_kl_kernel<true>, dim3(grid_for(quads, RT)), dim3(RT), 0, (cudaStream_t)stream,
                            g, (double *)nullptr, g_kl, g_kl_dev, out_scale_dev));
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

extern "C" int bbb_philox_fill_normal(float *out, int64_t n, uint64_t seed, uint32_t step, uint32_t sample,
                                      uint32_t tensor_id, void *stream) {
  BBB_CHECK_ARG(out && n >= 0, "null pointer or negative size");
  if (n == 0) return BBB_OK;
  bbb_rng r{seed, step, 0, 0, nullptr};
  philox_fill_kernel<<<grid_for((n + 3) >> 2, RT * 4), RT, 0, (cudaStream_t)stream>>>(out, n, make_rng_dev(&r),
                                                                                    tensor_id, sample);
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

extern "C" int bbb_nll_ce(const float *logits, const int64_t *target, int64_t S, int64_t B, int64_t C,
                          float grad_scale, double *nll, float *dlogits, void *stream) {
  BBB_CHECK_ARG(logits && target && nll, "null pointer");
  BBB_CHECK_ARG(S >= 0 && B >= 0 && C > 0, "bad shape");
  const int64_t rows = S * B;
  if (rows == 0) return BBB_OK;
  BBB_CHECK_CUDA(launch_pdl(nll_ce_kernel, dim3(grid_for(rows, 4)), dim3(128), 0, (cudaStream_t)stream, logits, target, rows, B,
                            C, grad_scale, nll, dlogits));
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

extern "C" int bbb_nll_gauss(const float *out, const float *target, float sigma, int64_t S, int64_t B, int64_t D,
                             float grad_scale, double *nll, float *dout, void *stream) {
  BBB_CHECK_ARG(out && target && nll, "null pointer");
  BBB_CHECK_ARG(S >= 0 && B >= 0 && D >= 0 && sigma > 0, "bad shape or sigma");
  const int64_t n = S * B * D;
  if (n == 0) return BBB_OK;
  const double var = (double)sigma * sigma;
  BBB_CHECK_CUDA(launch_pdl(nll_gauss_kernel, dim3(grid_for(n, RT)), dim3(RT), 0, (cudaStream_t)stream, out, target,
                            (float)(0.5 / var), (float)(1.0 / var),
                            (float)(log((double)sigma) + 0.918938533204672741780329736406), n, B * D, grad_scale, nll, dout));
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

extern "C" int bbb_nll_gauss_het(const float *out, const float *target, float sigma_min, int64_t S, int64_t B,
                                 int64_t D, float grad_scale, double *nll, float *dout, void *stream) {
  BBB_CHECK_ARG(out && target && nll, "null pointer");
  BBB_CHECK_ARG(S >= 0 && B >= 0 && D >= 0, "negative size");
  BBB_CHECK_ARG(D > 0 || S * B == 0, "D == 0 with S * B > 0");
  BBB_CHECK_ARG(sigma_min > 0.0f, "sigma_min must be > 0");
  const int64_t n = S * B * D;
  if (n == 0) return BBB_OK;
  BBB_CHECK_CUDA(launch_pdl(nll_gauss_het_kernel, dim3(grid_for(n, RT)), dim3(RT), 0, (cudaStream_t)stream, out, target,
                            sigma_min, (float)0.918938533204672741780329736406, n, B, D, grad_scale, nll, dout));
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

extern "C" int bbb_elbo_finalize(const double *logp, const double *logq, const double *kl, const double *nll,
                                 int64_t S, float beta, const float *beta_dev, float *out4, void *stream) {
  BBB_CHECK_ARG(nll && out4 && S > 0, "null pointer or S <= 0");
  BBB_CHECK_ARG(kl || (logp && logq), "need kl or logp+logq");
  BBB_CHECK_CUDA(launch_pdl(elbo_finalize_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, logp, logq, kl, nll, (int)S, beta,
                            beta_dev, out4));
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

namespace bbb { namespace {
__global__ void counter_add_kernel(uint32_t *c, uint32_t inc) {
  pdl_launch_dependents();
  pdl_wait();
  if (threadIdx.x == 0 && blockIdx.x == 0) *c += inc;
}
} }
extern "C" int bbb_counter_add(uint32_t *counter, uint32_t inc, void *stream) {
  BBB_CHECK_ARG(counter, "null pointer");
  BBB_CHECK_CUDA(launch_pdl(counter_add_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, counter, inc));
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

extern "C" uint64_t bbb_launch_count(void) { return bbb::g_launches.load(std::memory_order_relaxed); }
extern "C" int bbb_version(void) { return BBB_VERSION; }
extern "C" const char *bbb_last_error_string(void) { return last_error_buf(); }

// ---- consumers of the (mu, rho) stream and of the sampled outputs (SURVEY 8 f2 / f3) ---------------------------------
extern "C" int bbb_snr(const float *mu, const float *rho, int64_t n, float *snr_out, void *stream) {
  BBB_CHECK_ARG(n >= 0 && ((mu && rho && snr_out) || n == 0), "null pointer or negative size");
  if (n == 0) return BBB_OK;
  snr_kernel<<<grid_for(n, RT * 4), RT, 0, (cudaStream_t)stream>>>(const_cast<float *>(mu), const_cast<float *>(rho), n,
                                                                    snr_out, 0, 0.0f, nullptr);
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

extern "C" int bbb_snr_prune(float *mu, float *rho, int64_t n, float threshold_db, unsigned long long *kept, void *stream) {
  BBB_CHECK_ARG(n >= 0 && ((mu && rho) || n == 0), "null pointer or negative size");
  if (n == 0) return BBB_OK;
  snr_kernel<<<grid_for(n, RT * 4), RT, 0, (cudaStream_t)stream>>>(mu, rho, n, nullptr, 1, threshold_db, kept);
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

extern "C" int bbb_softmax_mean(const float *logits, int64_t S, int64_t B, int64_t C, float *probs, void *stream) {
  BBB_CHECK_ARG(S >= 1 && B >= 0 && C >= 1 && ((logits && probs) || B == 0), "null pointer or bad shape");
  if (B == 0) return BBB_OK;
  softmax_mean_kernel<<<grid_for(B, 4), 128, 0, (cudaStream_t)stream>>>(logits, S, B, C, probs);
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}
