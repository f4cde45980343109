// Local-reparameterisation Bayesian linear layer, exact-fp32 path (CUDA-core FMA).
//
// The reference (networks.py:116-138) runs two GEMMs per layer, x mu and x^2 sigma^2, plus ~10
// elementwise passes.  Here both contractions share one staged x tile (x^2 is formed in the FMA
// loop), sigma^2 is formed from rho while the weight tile is staged, and the pre-activation noise
// delta * eps_a + (mu_b + sigma_b eps_b) is applied in the epilogue with eps from Philox or memory.
// The closed-form KL (networks.py:109-114) is accumulated once per call by the CTAs that stage
// each weight for sample 0.  Weights are laid out [in, out] as in the reference (networks.py:95-96).
#include "bbb_common.cuh"
#include "bbb_kernels.h"

namespace bbb {
namespace {

constexpr int TM = 64, TN = 64, TK = 16, NT = 256, PAD = 4;
typedef float Tile[TK][TM + PAD];

template <class F>
__device__ __forceinline__ void for_kcontig(int tid, F f) {  // f(row, kq) -- 4 consecutive k per thread
  f(tid >> 2, (tid & 3) << 2);
}
template <class F>
__device__ __forceinline__ void for_mncontig(int tid, F f) {  // f(k, q) -- 4 consecutive m/n per thread
  f(tid >> 4, (tid & 15) << 2);
}
__device__ __forceinline__ void put_k(Tile &t, int r, int kq, const float v[4]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) t[kq + j][r] = v[j];
}
__device__ __forceinline__ void put_mn(Tile &t, int k, int q, const float v[4]) {
  *reinterpret_cast<float4 *>(&t[k][q]) = make_float4(v[0], v[1], v[2], v[3]);
}

// activation noise eps_a for elements (s, b, o..o+3)
__device__ __forceinline__ void eps_a4(const LrArgs &a, int s, int64_t b, int64_t o, int valid, float e[4]) {
  const int64_t idx = b * a.out + o;
  if (a.eps_a) {
    ld4(a.eps_a + (int64_t)s * a.B * a.out, idx, valid, a.vec_out, e);
  } else if (a.vec_out) {
    philox_normal4(a.rng, a.rng.tensor_w, a.rng.sample_base + s, (uint32_t)(idx >> 2), e);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      e[j] = j < valid ? philox_normal1(a.rng, a.rng.tensor_w, a.rng.sample_base + s, (uint64_t)(idx + j)) : 0.0f;
  }
}
__device__ __forceinline__ float eps_b1(const LrArgs &a, int s, int64_t o) {
  return a.eps_b ? __ldg(a.eps_b + (int64_t)s * a.out + o)
                 : philox_normal1(a.rng, a.rng.tensor_b, a.rng.sample_base + s, (uint64_t)o);
}

// masked upstream gradient dz and dV = dz eps_a / (2 delta) for (s, b, o..o+3); zero where delta == 0
// (the reference divides by zero there, SURVEY App. B-7).
__device__ __forceinline__ void dz_dv4(const LrArgs &a, int s, int64_t b, int64_t o, int valid, bool sample,
                                       float dz[4], float dv[4]) {
  const int64_t base = (int64_t)s * a.B * a.out, idx = b * a.out + o;
  ld4(a.dy + base, idx, valid, a.vec_out, dz);
  if (a.mask) {
    float m[4];
    ld4(a.mask + base, idx, valid, a.vec_out, m);
#pragma unroll
    for (int j = 0; j < 4; ++j) dz[j] = m[j] > 0.0f ? dz[j] : 0.0f;
  }
  if (sample) {
    float e[4], d[4];
    eps_a4(a, s, b, o, valid, e);
    ld4(a.delta_in + base, idx, valid, a.vec_out, d);
#pragma unroll
    for (int j = 0; j < 4; ++j) dv[j] = (j < valid && d[j] > 0.0f) ? dz[j] * e[j] / (2.0f * d[j]) : 0.0f;
  } else {
    dv[0] = dv[1] = dv[2] = dv[3] = 0.0f;
  }
}

__device__ __forceinline__ float kl_elem(float mu, float sg, float log_sp, float inv_sp2) {
  return 0.5f * (2.0f * (log_sp - logf(sg)) - 1.0f + (sg * sg + mu * mu) * inv_sp2);
}

// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT) lr_fwd_kernel(const LrArgs a_in) {
  LrArgs a = a_in;
  rng_resolve(a.rng);
  __shared__ __align__(16) Tile As, Bm, Bv;
  __shared__ float bias_s[TN];
  __shared__ float red[64];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int s = blockIdx.z;
  const int64_t b0 = (int64_t)blockIdx.y * TM, o0 = (int64_t)blockIdx.x * TN;
  const float *xs = a.x + (int64_t)s * a.x_sstride;
  const bool relu = a.flags & BBB_F_RELU_IN, sample = a.flags & BBB_F_SAMPLE;
  const bool klcta = (a.flags & BBB_F_LOGPROB) && blockIdx.y == 0 && s == 0;
  const float log_sp = logf(a.sigma_p), inv_sp2 = 1.0f / (a.sigma_p * a.sigma_p);
  float acc1[4][4] = {}, acc2[4][4] = {};
  float kl = 0.0f;

  if (tid < TN) {
    const int64_t o = o0 + tid;
    float bv = 0.0f;
    if (o < a.out) {
      const float mu = __ldg(a.b_mu + o);
      bv = mu;
      if (sample || klcta) {
        const float sg = softplus_f(__ldg(a.b_rho + o));
        if (sample) bv = fmaf(sg, eps_b1(a, s, o), mu);
        if (klcta) kl += kl_elem(mu, sg, log_sp, inv_sp2);
      }
    }
    bias_s[tid] = bv;
  }

  for (int64_t k0 = 0; k0 < a.in; k0 += TK) {
    for_kcontig(tid, [&](int r, int kq) {
      const int64_t b = b0 + r, k = k0 + kq;
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      if (b < a.B && k < a.in) {
        ld4(xs, b * a.in + k, (int)min((int64_t)4, a.in - k), a.vec_in, v);
        if (relu) {
#pragma unroll
          for (int j = 0; j < 4; ++j) v[j] = fmaxf(v[j], 0.0f);
        }
      }
      put_k(As, r, kq, v);
    });
    for_mncontig(tid, [&](int kr, int nq) {
      const int64_t i = k0 + kr, o = o0 + nq;
      float m[4] = {0.f, 0.f, 0.f, 0.f}, v[4] = {0.f, 0.f, 0.f, 0.f};
      if (i < a.in && o < a.out) {
        const int valid = (int)min((int64_t)4, a.out - o);
        ld4(a.w_mu, i * a.out + o, valid, a.vec_out, m);
        if (sample || klcta) {
          float r[4];
          ld4(a.w_rho, i * a.out + o, valid, a.vec_out, r);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (j < valid) {
              const float sg = softplus_f(r[j]);
              v[j] = sg * sg;
              if (klcta) kl += kl_elem(m[j], sg, log_sp, inv_sp2);
            }
          }
        }
      }
      put_mn(Bm, kr, nq, m);
      put_mn(Bv, kr, nq, v);
    });
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < TK; ++kk) {
      const float4 av = *reinterpret_cast<const float4 *>(&As[kk][ty * 4]);
      const float4 mv = *reinterpret_cast<const float4 *>(&Bm[kk][tx * 4]);
      const float4 vv = *reinterpret_cast<const float4 *>(&Bv[kk][tx * 4]);
      const float a_[4] = {av.x, av.y, av.z, av.w}, m_[4] = {mv.x, mv.y, mv.z, mv.w}, v_[4] = {vv.x, vv.y, vv.z, vv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float a2 = a_[i] * a_[i];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          acc1[i][j] = fmaf(a_[i], m_[j], acc1[i][j]);
          acc2[i][j] = fmaf(a2, v_[j], acc2[i][j]);
        }
      }
    }
    __syncthreads();
  }
  __syncthreads();

  const int64_t base = (int64_t)s * a.B * a.out;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t b = b0 + ty * 4 + i, o = o0 + tx * 4;
    if (b >= a.B || o >= a.out) continue;
    const int valid = (int)min((int64_t)4, a.out - o);
    float e[4] = {0.f, 0.f, 0.f, 0.f}, yv[4], dl[4];
    if (sample) eps_a4(a, s, b, o, valid, e);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      dl[j] = sample ? sqrtf(acc2[i][j]) : 0.0f;
      yv[j] = acc1[i][j] + dl[j] * e[j] + bias_s[tx * 4 + j];
    }
    if (a.vec_out && valid == 4) {
      *reinterpret_cast<float4 *>(a.y + base + b * a.out + o) = make_float4(yv[0], yv[1], yv[2], yv[3]);
      if (a.delta) *reinterpret_cast<float4 *>(a.delta + base + b * a.out + o) = make_float4(dl[0], dl[1], dl[2], dl[3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (j < valid) {
          a.y[base + b * a.out + o + j] = yv[j];
          if (a.delta) a.delta[base + b * a.out + o + j] = dl[j];
        }
    }
  }
  if (klcta) block_sum2_atomic(kl, 0.0f, red, a.kl, nullptr);
}

// dx[s][b][i] = sum_o dz mu[i][o] + 2 x[b][i] sum_o dV sigma^2[i][o]
__global__ void __launch_bounds__(NT) lr_dgrad_kernel(const LrArgs a_in) {
  LrArgs a = a_in;
  rng_resolve(a.rng);
  __shared__ __align__(16) Tile A1, A2, Bm, Bv;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int s = blockIdx.z;
  const int64_t b0 = (int64_t)blockIdx.y * TM, i0 = (int64_t)blockIdx.x * TN;
  const bool relu = a.flags & BBB_F_RELU_IN, sample = a.flags & BBB_F_SAMPLE;
  float acc1[4][4] = {}, acc2[4][4] = {};

  for (int64_t k0 = 0; k0 < a.out; k0 += TK) {
    for_kcontig(tid, [&](int r, int kq) {
      const int64_t b = b0 + r, o = k0 + kq;
      float dz[4] = {0.f, 0.f, 0.f, 0.f}, dv[4] = {0.f, 0.f, 0.f, 0.f};
      if (b < a.B && o < a.out) dz_dv4(a, s, b, o, (int)min((int64_t)4, a.out - o), sample, dz, dv);
      put_k(A1, r, kq, dz);
      put_k(A2, r, kq, dv);
    });
    for_kcontig(tid, [&](int r, int kq) {
      const int64_t i = i0 + r, o = k0 + kq;
      float m[4] = {0.f, 0.f, 0.f, 0.f}, v[4] = {0.f, 0.f, 0.f, 0.f};
      if (i < a.in && o < a.out) {
        const int valid = (int)min((int64_t)4, a.out - o);
        ld4(a.w_mu, i * a.out + o, valid, a.vec_out, m);
        if (sample) {
          float rr[4];
          ld4(a.w_rho, i * a.out + o, valid, a.vec_out, rr);
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (j < valid) { const float sg = softplus_f(rr[j]); v[j] = sg * sg; }
        }
      }
      put_k(Bm, r, kq, m);
      put_k(Bv, r, kq, v);
    });
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < TK; ++kk) {
      const float4 a1 = *reinterpret_cast<const float4 *>(&A1[kk][ty * 4]);
      const float4 a2 = *reinterpret_cast<const float4 *>(&A2[kk][ty * 4]);
      const float4 mv = *reinterpret_cast<const float4 *>(&Bm[kk][tx * 4]);
      const float4 vv = *reinterpret_cast<const float4 *>(&Bv[kk][tx * 4]);
      const float p[4] = {a1.x, a1.y, a1.z, a1.w}, q[4] = {a2.x, a2.y, a2.z, a2.w};
      const float m_[4] = {mv.x, mv.y, mv.z, mv.w}, v_[4] = {vv.x, vv.y, vv.z, vv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          acc1[i][j] = fmaf(p[i], m_[j], acc1[i][j]);
          acc2[i][j] = fmaf(q[i], v_[j], acc2[i][j]);
        }
    }
    __syncthreads();
  }

  const float *xs = a.x + (int64_t)s * a.x_sstride;
  float *dxs = a.dx + (int64_t)s * a.B * a.in;
  const float dsc = ((a.flags & BBB_F_SCALE_DX) && a.out_scale_dev) ? __ldg(a.out_scale_dev) : 1.0f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t b = b0 + ty * 4 + i, c = i0 + tx * 4;
    if (b >= a.B) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (c + j < a.in) {
        float xv = xs[b * a.in + c + j];
        if (relu) xv = fmaxf(xv, 0.0f);
        float d = dsc * fmaf(2.0f * xv, acc2[i][j], acc1[i][j]);
        if ((a.flags & BBB_F_DX_PREACT) && !(xv > 0.0f)) d = 0.0f;   // gradient w.r.t. the pre-activation input
        dxs[b * a.in + c + j] = d;
      }
    }
  }
}

// grad_mu[i][o] = sum_s x^T dz + g_kl mu / sp^2 ; grad_rho = sigmoid(rho)(2 sigma sum_s (x^2)^T dV + g_kl(-1/sigma + sigma/sp^2))
__global__ void __launch_bounds__(NT) lr_wgrad_kernel(const LrArgs a_in) {
  LrArgs a = a_in;
  rng_resolve(a.rng);
  __shared__ __align__(16) Tile As, B1, B2;  // As[b][i], B1[b][o] = dz, B2[b][o] = dV
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t o0 = (int64_t)blockIdx.x * TN, i0 = (int64_t)blockIdx.y * TM;
  const bool relu = a.flags & BBB_F_RELU_IN, sample = a.flags & BBB_F_SAMPLE;
  const bool bias_cta = blockIdx.y == 0;
  const float inv_sp2 = 1.0f / (a.sigma_p * a.sigma_p);
  float acc1[4][4] = {}, acc2[4][4] = {};
  float gbmu = 0.0f, gbrho = 0.0f;

  for (int s = 0; s < a.S; ++s) {
    const float *xs = a.x + (int64_t)s * a.x_sstride;
    float colsum = 0.0f;
    for (int64_t k0 = 0; k0 < a.B; k0 += TK) {
      for_mncontig(tid, [&](int kr, int mq) {
        const int64_t b = k0 + kr, i = i0 + mq;
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        if (b < a.B && i < a.in) {
          ld4(xs, b * a.in + i, (int)min((int64_t)4, a.in - i), a.vec_in, v);
          if (relu) {
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = fmaxf(v[j], 0.0f);
          }
        }
        put_mn(As, kr, mq, v);
      });
      for_mncontig(tid, [&](int kr, int nq) {
        const int64_t b = k0 + kr, o = o0 + nq;
        float dz[4] = {0.f, 0.f, 0.f, 0.f}, dv[4] = {0.f, 0.f, 0.f, 0.f};
        if (b < a.B && o < a.out) dz_dv4(a, s, b, o, (int)min((int64_t)4, a.out - o), sample, dz, dv);
        put_mn(B1, kr, nq, dz);
        put_mn(B2, kr, nq, dv);
      });
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < TK; ++kk) {
        const float4 av = *reinterpret_cast<const float4 *>(&As[kk][ty * 4]);
        const float4 p = *reinterpret_cast<const float4 *>(&B1[kk][tx * 4]);
        const float4 q = *reinterpret_cast<const float4 *>(&B2[kk][tx * 4]);
        const float a_[4] = {av.x, av.y, av.z, av.w}, p_[4] = {p.x, p.y, p.z, p.w}, q_[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float a2 = a_[i] * a_[i];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            acc1[i][j] = fmaf(a_[i], p_[j], acc1[i][j]);
            acc2[i][j] = fmaf(a2, q_[j], acc2[i][j]);
          }
        }
      }
      if (bias_cta && tid < TN) {
#pragma unroll
        for (int kk = 0; kk < TK; ++kk) colsum += B1[kk][tid];
      }
      __syncthreads();
    }
    if (bias_cta && tid < TN && o0 + tid < a.out) {
      gbmu += colsum;
      if (sample) gbrho += colsum * eps_b1(a, s, o0 + tid);
    }
  }

  const bool accum = a.flags & BBB_F_ACCUM;
  const float osc = a.out_scale_dev ? __ldg(a.out_scale_dev) : 1.0f;
  const float gk = (a.flags & BBB_F_LOGPROB) ? a.g_kl * (a.g_kl_dev ? __ldg(a.g_kl_dev) : 1.0f) : 0.0f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t r = i0 + ty * 4 + i, c = o0 + tx * 4;
    if (r >= a.in) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (c + j < a.out) {
        const int64_t e = r * a.out + c + j;
        const float mu = a.w_mu[e], sg = softplus_f(a.w_rho[e]);
        const float gm = fmaf(gk * mu, inv_sp2, acc1[i][j]);
        const float gr = -expm1f(-sg) * (2.0f * sg * acc2[i][j] + gk * (sg * inv_sp2 - 1.0f / sg));
        a.g_w_mu[e] = accum ? fmaf(osc, gm, a.g_w_mu[e]) : osc * gm;
        a.g_w_rho[e] = accum ? fmaf(osc, gr, a.g_w_rho[e]) : osc * gr;
      }
    }
  }
  if (bias_cta && tid < TN) {
    const int64_t o = o0 + tid;
    if (o < a.out) {
      const float mu = a.b_mu[o], sg = softplus_f(a.b_rho[o]);
      const float gm = fmaf(gk * mu, inv_sp2, gbmu);
      const float gr = -expm1f(-sg) * (gbrho + gk * (sg * inv_sp2 - 1.0f / sg));
      a.g_b_mu[o] = accum ? fmaf(osc, gm, a.g_b_mu[o]) : osc * gm;
      a.g_b_rho[o] = accum ? fmaf(osc, gr, a.g_b_rho[o]) : osc * gr;
    }
  }
}

inline unsigned cdiv(int64_t a, int64_t b) { return (unsigned)((a + b - 1) / b); }

}  // namespace

int launch_lr_fwd_fma(const LrArgs &a, cudaStream_t st) {
  dim3 grid(cdiv(a.out, TN), cdiv(a.B, TM), (unsigned)a.S);
  lr_fwd_kernel<<<grid, NT, 0, st>>>(a);
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

int launch_lr_bwd_fma(const LrArgs &a, cudaStream_t st) {
  if (!(a.flags & BBB_F_NO_DX) && a.S > 0 && a.B > 0) {   // an empty batch has no dx (and a zero grid is no launch)
    dim3 grid(cdiv(a.in, TN), cdiv(a.B, TM), (unsigned)a.S);
    lr_dgrad_kernel<<<grid, NT, 0, st>>>(a);
    BBB_CHECK_LAUNCH();
  }
  if (a.flags & BBB_F_NO_WGRAD) return BBB_OK;
  dim3 grid(cdiv(a.out, TN), cdiv(a.in, TM));
  lr_wgrad_kernel<<<grid, NT, 0, st>>>(a);
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

}  // namespace bbb
