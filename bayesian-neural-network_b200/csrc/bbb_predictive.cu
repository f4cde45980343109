// Posterior-predictive summaries of sampled network outputs, one pass over [S,B,C] (include/bbb.h:
// bbb_predictive_stats).  Replaces the host-side analysis the reference's callers do after their predict loops
// (class_task.py:81-87, reg_task.py:76-83) and the ECE of its compute_ece.py.
//
// One warp per batch row; a lane holds the classes (outputs) c = lane + 32 j, j < NPL, in registers, so every
// quantity of a row is formed in registers while its S samples stream through once (the next sample's loads are
// issued before the current one is reduced).  Per-row outputs are written by lane 0; the aggregates are summed per
// block (warp registers -> shared memory) and added to the fp64 accumulators with one atomic per block and quantity.
// Bound: one read of 4 S B C bytes plus the writes of [B,C] and [B,K]; launch- and latency-bound at the sizes of a test
// set (MNIST: 10 000 rows x 10 samples x 10 classes = 4 MB).
#include "bbb_common.cuh"

namespace bbb {
namespace {

constexpr int PT = 256;          // threads per CTA: 8 rows in flight
constexpr int kWarps = PT / 32;
constexpr int kMaxBins = 1024;   // shared-memory bin table: kMaxBins x (2 counters + 1 double)

// header of the accumulator vector, both kinds (documented in bbb.h)
constexpr int A_N = 0, A_ERR = 1, A_NLL = 2, A_CORRECT = 3, A_BRIER = 4, A_SQERR = 3, A_BINS = 5;

template <int NPL>
__device__ __forceinline__ void load_row(const float *__restrict__ z, int64_t C, int lane, float v[NPL]) {
#pragma unroll
  for (int j = 0; j < NPL; ++j) {
    const int64_t c = lane + 32 * j;
    v[j] = c < C ? __ldg(z + c) : 0.0f;
  }
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// block-wide sum of one float per warp (lane 0's value), added to *dst by one thread; all threads call
__device__ __forceinline__ void block_add(float v, float *red, double *dst) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) red[warp] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) s += (double)red[w];
    if (s != 0.0) atomicAdd(dst, s);
  }
  __syncthreads();
}

// ---- classification: p_s = softmax(z_s) ------------------------------------------------------------------------------
template <int NPL>
__global__ void __launch_bounds__(PT) predictive_cls_kernel(const float *__restrict__ out,
                                                             const int64_t *__restrict__ target, int64_t S,
                                                             int64_t B, int64_t C, int n_bins,
                                                             float *__restrict__ mean, float *__restrict__ row_stats,
                                                             int64_t *__restrict__ pred, double *acc) {
  extern __shared__ unsigned char smem[];
  unsigned *bin_cnt = reinterpret_cast<unsigned *>(smem);
  unsigned *bin_cor = bin_cnt + n_bins;
  double *bin_conf = reinterpret_cast<double *>(smem + ((8u * (unsigned)n_bins + 15u) & ~15u));
  __shared__ float red[kWarps];
  const bool agg = target != nullptr && acc != nullptr;
  if (agg)
    for (int m = threadIdx.x; m < n_bins; m += PT) { bin_cnt[m] = 0u; bin_cor[m] = 0u; bin_conf[m] = 0.0; }
  __syncthreads();

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float inv_s = 1.0f / (float)S, log_s = logf((float)S);
  float w_n = 0.0f, w_err = 0.0f, w_nll = 0.0f, w_cor = 0.0f, w_brier = 0.0f;   // this warp's rows (lane 0)

  for (int64_t b = (int64_t)blockIdx.x * kWarps + warp; b < B; b += (int64_t)gridDim.x * kWarps) {
    int64_t y = -1;
    bool bad = false;
    if (target) {
      y = __ldg(target + b);
      bad = y < 0 || y >= C;
    }
    const int y_lane = (int)(y & 31), y_j = (int)(y >> 5);
    float pbar[NPL], zc[NPL], zn[NPL];
#pragma unroll
    for (int j = 0; j < NPL; ++j) pbar[j] = 0.0f;
    float ent_sum = 0.0f;                       // sum_s H[p_s]
    float lp_max = -INFINITY, lp_sum = 0.0f;    // online LSE over s of log p_s[y]
    load_row<NPL>(out + b * C, C, lane, zc);
    for (int64_t s = 0; s < S; ++s) {
      if (s + 1 < S) load_row<NPL>(out + ((s + 1) * B + b) * C, C, lane, zn);
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < NPL; ++j)
        if (lane + 32 * j < C) mx = fmaxf(mx, zc[j]);
      mx = warp_max(mx);
      float e[NPL], se = 0.0f;
#pragma unroll
      for (int j = 0; j < NPL; ++j) {
        zc[j] -= mx;                            // shifted logits z' <= 0
        e[j] = lane + 32 * j < C ? expf(zc[j]) : 0.0f;
        se += e[j];
      }
      se = warp_sum(se);
      const float lse = logf(se), inv_se = 1.0f / se;   // LSE of the shifted logits, in [0, log C]
      // H[p_s] = LSE(z) - sum_c p_c z_c, summed as sum_c p_c (LSE(z') - z'_c): non-negative terms, no cancellation
      float h = 0.0f;
#pragma unroll
      for (int j = 0; j < NPL; ++j) {
        const float p = e[j] * inv_se;
        pbar[j] += p;
        h += lane + 32 * j < C ? p * (lse - zc[j]) : 0.0f;
      }
      ent_sum += warp_sum(h);
      if (target && !bad) {
        float zy = 0.0f;
#pragma unroll
        for (int j = 0; j < NPL; ++j)
          if (j == y_j) zy = zc[j];
        const float l = __shfl_sync(0xffffffffu, zy, y_lane) - lse;     // log p_s[y]
        const float m = fmaxf(lp_max, l);
        lp_sum = lp_sum * expf(lp_max - m) + expf(l - m);
        lp_max = m;
      }
#pragma unroll
      for (int j = 0; j < NPL; ++j) zc[j] = zn[j];
    }
    // mean over the samples; argmax (lowest index on ties), entropy of the mean, Brier score
    float best = -1.0f, ent = 0.0f, brier = 0.0f;
    int64_t arg = 0;
#pragma unroll
    for (int j = 0; j < NPL; ++j) {
      const int64_t c = lane + 32 * j;
      if (c < C) {
        const float p = pbar[j] * inv_s;
        pbar[j] = p;
        mean[b * C + c] = p;
        if (p > best) { best = p; arg = c; }
        if (p > 0.0f) ent -= p * logf(p);
        const float d = p - (c == y ? 1.0f : 0.0f);
        brier += d * d;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int64_t oa = __shfl_xor_sync(0xffffffffu, arg, o);
      if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
    }
    ent = warp_sum(ent);
    brier = warp_sum(brier);
    if (lane == 0) {
      const float ee = ent_sum * inv_s;
      const float log_pred = (target && !bad) ? lp_max + logf(lp_sum) - log_s : __int_as_float(0x7fc00000);
      float *rs = row_stats + b * 5;
      rs[0] = best; rs[1] = ent; rs[2] = ee; rs[3] = fmaxf(ent - ee, 0.0f); rs[4] = log_pred;
      if (pred) pred[b] = arg;
      if (agg) {
        if (bad) {
          w_err += 1.0f;
        } else {
          const bool ok = arg == y;
          w_n += 1.0f;
          w_cor += ok ? 1.0f : 0.0f;
          w_nll -= log_pred;
          w_brier += brier;
          // bin m holds confidences in (m/M, (m+1)/M]
          int m = (int)ceilf(best * (float)n_bins) - 1;
          m = m < 0 ? 0 : (m >= n_bins ? n_bins - 1 : m);
          atomicAdd(bin_cnt + m, 1u);
          if (ok) atomicAdd(bin_cor + m, 1u);
          atomicAdd(bin_conf + m, (double)best);
        }
      }
    }
  }
  if (!agg) return;
  // per-warp sums of at most ceil(B / #warps) rows: integers stay exact in fp32 below 2^24 rows
  block_add(w_n, red, acc + A_N);
  block_add(w_err, red, acc + A_ERR);
  block_add(w_nll, red, acc + A_NLL);
  block_add(w_cor, red, acc + A_CORRECT);
  block_add(w_brier, red, acc + A_BRIER);
  for (int m = threadIdx.x; m < n_bins; m += PT) {
    if (bin_cnt[m] == 0u) continue;
    double *a = acc + A_BINS + 3 * m;
    atomicAdd(a + 0, (double)bin_cnt[m]);
    atomicAdd(a + 1, bin_conf[m]);
    if (bin_cor[m]) atomicAdd(a + 2, (double)bin_cor[m]);
  }
}

// ---- Gaussian likelihood N(y; f_s, sigma^2) ---------------------------------------------------------------------------
template <int NPL>
__global__ void __launch_bounds__(PT) predictive_gauss_kernel(const float *__restrict__ out,
                                                               const float *__restrict__ target, int64_t S, int64_t B,
                                                               int64_t D, float inv_2var, float log_norm,
                                                               float *__restrict__ mean,
                                                               float *__restrict__ row_stats, double *acc) {
  __shared__ float red[kWarps];
  const bool agg = target != nullptr && acc != nullptr;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float log_s = logf((float)S);
  float w_n = 0.0f, w_nll = 0.0f, w_sq = 0.0f;
  for (int64_t b = (int64_t)blockIdx.x * kWarps + warp; b < B; b += (int64_t)gridDim.x * kWarps) {
    float yv[NPL], mu[NPL], m2[NPL], fc[NPL], fn[NPL];
    if (target) load_row<NPL>(target + b * D, D, lane, yv);
#pragma unroll
    for (int j = 0; j < NPL; ++j) { mu[j] = 0.0f; m2[j] = 0.0f; }
    float lp_max = -INFINITY, lp_sum = 0.0f;
    load_row<NPL>(out + b * D, D, lane, fc);
    for (int64_t s = 0; s < S; ++s) {
      if (s + 1 < S) load_row<NPL>(out + ((s + 1) * B + b) * D, D, lane, fn);
      const float inv_n = 1.0f / (float)(s + 1);
      float sq = 0.0f;
#pragma unroll
      for (int j = 0; j < NPL; ++j) {
        const float d = fc[j] - mu[j];          // Welford: mean and sum of squared deviations
        mu[j] += d * inv_n;
        m2[j] += d * (fc[j] - mu[j]);
        if (target) { const float r = yv[j] - fc[j]; sq += r * r; }
      }
      if (target) {
        const float l = -warp_sum(sq) * inv_2var - log_norm;   // sum_d log N(y_d; f_s,d, sigma^2)
        const float m = fmaxf(lp_max, l);
        lp_sum = lp_sum * expf(lp_max - m) + expf(l - m);
        lp_max = m;
      }
#pragma unroll
      for (int j = 0; j < NPL; ++j) fc[j] = fn[j];
    }
    const float inv_s = 1.0f / (float)S;
    float sqerr = 0.0f;
    float *rs = row_stats + b * (D + 1);
#pragma unroll
    for (int j = 0; j < NPL; ++j) {
      const int64_t d = lane + 32 * j;
      if (d < D) {
        mean[b * D + d] = mu[j];
        rs[d] = m2[j] * inv_s;
        if (target) { const float r = mu[j] - yv[j]; sqerr += r * r; }
      }
    }
    sqerr = warp_sum(sqerr);
    if (lane == 0) {
      const float log_pred = target ? lp_max + logf(lp_sum) - log_s : __int_as_float(0x7fc00000);
      rs[D] = log_pred;
      w_n += 1.0f;
      w_nll -= log_pred;
      w_sq += sqerr;
    }
  }
  if (!agg) return;
  block_add(w_n, red, acc + A_N);
  block_add(w_nll, red, acc + A_NLL);
  block_add(w_sq, red, acc + A_SQERR);
}

// ---- heteroscedastic Gaussian: the mixture (1/S) sum_s N(f_s, sigma_s^2), row = [f (D) | r (D)] -------------------------
// sigma_s = sigma_min + softplus(r_s).  Welford over f (epistemic), a running sum of sigma_s^2 (aleatoric), online LSE of
// sum_d log N(y_d; f_s,d, sigma_s,d^2) (log predictive density).  The explicit minimum of one block per SM keeps ptxas
// from capping the NPL = 4 instance at 64 registers, where it spilled.
template <int NPL>
__global__ void __launch_bounds__(PT, 1) predictive_gauss_het_kernel(const float *__restrict__ out,
                                                                   const float *__restrict__ target, int64_t S,
                                                                   int64_t B, int64_t D, float sigma_min,
                                                                   float *__restrict__ mean,
                                                                   float *__restrict__ row_stats, double *acc) {
  __shared__ float red[kWarps];
  const bool agg = target != nullptr && acc != nullptr;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float log_s = logf((float)S), half_log_2pi = 0.918938533204672741780329736406f;
  float w_n = 0.0f, w_nll = 0.0f, w_sq = 0.0f;
  for (int64_t b = (int64_t)blockIdx.x * kWarps + warp; b < B; b += (int64_t)gridDim.x * kWarps) {
    float yv[NPL], mu[NPL], m2[NPL], var[NPL], fc[NPL], rc[NPL], fn[NPL], rn[NPL];
    if (target) load_row<NPL>(target + b * D, D, lane, yv);
#pragma unroll
    for (int j = 0; j < NPL; ++j) { mu[j] = 0.0f; m2[j] = 0.0f; var[j] = 0.0f; }
    float lp_max = -INFINITY, lp_sum = 0.0f;
    load_row<NPL>(out + b * 2 * D, D, lane, fc);
    load_row<NPL>(out + b * 2 * D + D, D, lane, rc);
    for (int64_t s = 0; s < S; ++s) {
      if (s + 1 < S) {
        const float *z = out + ((s + 1) * B + b) * 2 * D;
        load_row<NPL>(z, D, lane, fn);
        load_row<NPL>(z + D, D, lane, rn);
      }
      const float inv_n = 1.0f / (float)(s + 1);
      float ll = 0.0f;
#pragma unroll
      for (int j = 0; j < NPL; ++j) {
        const float d = fc[j] - mu[j];
        mu[j] += d * inv_n;
        m2[j] += d * (fc[j] - mu[j]);
        const float sigma = sigma_min + fmaxf(rc[j], 0.0f) + log1pf(expf(-fabsf(rc[j])));
        var[j] += sigma * sigma;
        if (target && lane + 32 * j < D) {
          const float a = (yv[j] - fc[j]) / sigma;
          ll -= fmaf(0.5f * a, a, logf(sigma) + half_log_2pi);
        }
      }
      if (target) {
        const float l = warp_sum(ll);
        const float m = fmaxf(lp_max, l);
        lp_sum = lp_sum * expf(lp_max - m) + expf(l - m);
        lp_max = m;
      }
#pragma unroll
      for (int j = 0; j < NPL; ++j) { fc[j] = fn[j]; rc[j] = rn[j]; }
    }
    const float inv_s = 1.0f / (float)S;
    float sqerr = 0.0f;
    float *rs = row_stats + b * (2 * D + 1);
#pragma unroll
    for (int j = 0; j < NPL; ++j) {
      const int64_t d = lane + 32 * j;
      if (d < D) {
        mean[b * D + d] = mu[j];
        rs[d] = m2[j] * inv_s;
        rs[D + d] = var[j] * inv_s;
        if (target) { const float r = mu[j] - yv[j]; sqerr += r * r; }
      }
    }
    sqerr = warp_sum(sqerr);
    if (lane == 0) {
      const float log_pred = target ? lp_max + logf(lp_sum) - log_s : __int_as_float(0x7fc00000);
      rs[2 * D] = log_pred;
      w_n += 1.0f;
      w_nll -= log_pred;
      w_sq += sqerr;
    }
  }
  if (!agg) return;
  block_add(w_n, red, acc + A_N);
  block_add(w_nll, red, acc + A_NLL);
  block_add(w_sq, red, acc + A_SQERR);
}

template <int NPL>
cudaError_t launch_het(const float *out, const float *target, int64_t S, int64_t B, int64_t D, float sigma_min,
                       float *mean, float *row_stats, double *acc, cudaStream_t st) {
  const int64_t blocks = (B + kWarps - 1) / kWarps;
  const int64_t cap = (int64_t)sm_count() * (2048 / PT);   // one resident wave
  predictive_gauss_het_kernel<NPL><<<(int)(blocks < cap ? blocks : cap), PT, 0, st>>>(out, target, S, B, D, sigma_min,
                                                                                      mean, row_stats, acc);
  return cudaGetLastError();
}

template <int NPL>
cudaError_t launch_stats(const float *out, const void *target, int64_t S, int64_t B, int64_t C, int32_t kind,
                         float sigma, int n_bins, float *mean, float *row_stats, int64_t *pred, double *acc,
                         cudaStream_t st) {
  int64_t blocks = (B + kWarps - 1) / kWarps;
  const int64_t cap = (int64_t)sm_count() * (2048 / PT);   // one resident wave
  const int grid = (int)(blocks < cap ? blocks : cap);
  if (kind == BBB_NLL_CE) {
    // bin table (<= 16 KB at kMaxBins): the two counters, then the confidence sums 16-byte aligned
    const size_t smem = target && acc ? ((8u * (size_t)n_bins + 15u) & ~(size_t)15u) + 8u * (size_t)n_bins : 0;
    predictive_cls_kernel<NPL><<<grid, PT, smem, st>>>(out, static_cast<const int64_t *>(target), S, B, C, n_bins,
                                                       mean, row_stats, pred, acc);
  } else {
    const double var = (double)sigma * sigma;
    const float log_norm = (float)((double)C * (log((double)sigma) + 0.918938533204672741780329736406));
    predictive_gauss_kernel<NPL><<<grid, PT, 0, st>>>(out, static_cast<const float *>(target), S, B, C,
                                                      (float)(0.5 / var), log_norm, mean, row_stats, acc);
  }
  return cudaGetLastError();
}

}  // namespace
}  // namespace bbb

using namespace bbb;

// kind BBB_NLL_GAUSS_HET of bbb_predictive_stats: C = 2D outputs per row, sigma = sigma_min
static int predictive_stats_het(const float *out, const float *target, int64_t S, int64_t B, int64_t C,
                                float sigma_min, float *mean, float *row_stats, double *acc, cudaStream_t st) {
  BBB_CHECK_ARG(S >= 1 && B >= 0 && C >= 2 && C % 2 == 0, "bad shape (need S >= 1, B >= 0, C = 2D >= 2)");
  BBB_CHECK_ARG(C <= 32 * 32, "more than 1024 outputs per row");
  BBB_CHECK_ARG(sigma_min > 0.0f, "sigma_min must be > 0");
  BBB_CHECK_ARG(!target || acc, "aggregates (acc) required with a target");
  BBB_CHECK_ARG(B == 0 || (out && mean && row_stats), "null pointer");
  if (B == 0) return BBB_OK;
  const int64_t D = C / 2;
  cudaError_t e;
  if (D <= 32) e = launch_het<1>(out, target, S, B, D, sigma_min, mean, row_stats, acc, st);
  else if (D <= 64) e = launch_het<2>(out, target, S, B, D, sigma_min, mean, row_stats, acc, st);
  else if (D <= 128) e = launch_het<4>(out, target, S, B, D, sigma_min, mean, row_stats, acc, st);
  else if (D <= 256) e = launch_het<8>(out, target, S, B, D, sigma_min, mean, row_stats, acc, st);
  else e = launch_het<16>(out, target, S, B, D, sigma_min, mean, row_stats, acc, st);
  BBB_CHECK_CUDA(e);
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

extern "C" int bbb_predictive_stats(const float *out, const void *target, int64_t S, int64_t B, int64_t C,
                                    int32_t kind, float sigma, int32_t n_bins, float *mean, float *row_stats,
                                    int64_t *pred, double *acc, void *stream) {
  if (kind == BBB_NLL_GAUSS_HET)
    return predictive_stats_het(out, static_cast<const float *>(target), S, B, C, sigma, mean, row_stats, acc,
                                (cudaStream_t)stream);
  BBB_CHECK_ARG(kind == BBB_NLL_CE || kind == BBB_NLL_GAUSS, "kind must be BBB_NLL_CE or BBB_NLL_GAUSS");
  BBB_CHECK_ARG(S >= 1 && B >= 0 && C >= 1, "bad shape (need S >= 1, B >= 0, C >= 1)");
  BBB_CHECK_ARG(C <= 32 * 32, "more than 1024 classes / outputs per row");
  BBB_CHECK_ARG(kind == BBB_NLL_GAUSS || (n_bins >= 1 && n_bins <= kMaxBins), "n_bins must be in [1, 1024]");
  BBB_CHECK_ARG(kind == BBB_NLL_CE || sigma > 0.0f, "sigma must be > 0");
  BBB_CHECK_ARG(!target || acc, "aggregates (acc) required with a target");
  BBB_CHECK_ARG(B == 0 || (out && mean && row_stats), "null pointer");
  if (B == 0) return BBB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e;
  if (C <= 32) e = launch_stats<1>(out, target, S, B, C, kind, sigma, n_bins, mean, row_stats, pred, acc, st);
  else if (C <= 64) e = launch_stats<2>(out, target, S, B, C, kind, sigma, n_bins, mean, row_stats, pred, acc, st);
  else if (C <= 128) e = launch_stats<4>(out, target, S, B, C, kind, sigma, n_bins, mean, row_stats, pred, acc, st);
  else if (C <= 256) e = launch_stats<8>(out, target, S, B, C, kind, sigma, n_bins, mean, row_stats, pred, acc, st);
  else if (C <= 512) e = launch_stats<16>(out, target, S, B, C, kind, sigma, n_bins, mean, row_stats, pred, acc, st);
  else e = launch_stats<32>(out, target, S, B, C, kind, sigma, n_bins, mean, row_stats, pred, acc, st);
  BBB_CHECK_CUDA(e);
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}
