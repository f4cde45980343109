// Shared device math for the BBB kernels: Philox4x32-10 eps stream, softplus, prior/posterior
// log-densities and their derivatives, block reductions, error plumbing.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/bbb.h"

namespace bbb {

// ---------------------------------------------------------------------------------------
// error plumbing (thread-local message, integer status; never throws)
// ---------------------------------------------------------------------------------------
char *last_error_buf();
int fail(int code, const char *fmt, ...);
void note_launch(int n = 1);  // diagnostic launch counter (bbb_launch_count)
#define BBB_CHECK_ARG(cond, msg)                                         \
  do {                                                                   \
    if (!(cond)) return ::bbb::fail(BBB_EINVAL, "%s: %s", __func__, msg); \
  } while (0)
#define BBB_CHECK_LAUNCH()                                                                        \
  do {                                                                                            \
    cudaError_t e__ = cudaGetLastError();                                                         \
    if (e__ != cudaSuccess) return ::bbb::fail(BBB_ECUDA, "%s: %s", __func__, cudaGetErrorString(e__)); \
    ::bbb::note_launch();                                                                         \
  } while (0)
#define BBB_CHECK_CUDA(expr)                                                                      \
  do {                                                                                            \
    cudaError_t e__ = (expr);                                                                     \
    if (e__ != cudaSuccess) return ::bbb::fail(BBB_ECUDA, "%s: %s", __func__, cudaGetErrorString(e__)); \
  } while (0)

// ---------------------------------------------------------------------------------------
// Programmatic dependent launch.  The kernels of a train step form one dependent chain; launched with the
// programmatic-serialisation attribute, kernel N+1 becomes resident while kernel N drains and runs its prologue
// (shared-memory carve-up, TMEM allocation, barrier init) until pdl_wait(), which returns when every prerequisite
// grid has completed and its memory is visible.  Every kernel launched through launch_pdl() calls pdl_wait() before
// it touches global memory, and pdl_launch_dependents() first thing (all grids here fit in one wave, so letting
// the successor in early cannot starve the running grid).  Without the attribute both are no-ops.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---------------------------------------------------------------------------------------
// constants
// ---------------------------------------------------------------------------------------
constexpr float kHalfLog2Pi = 0.918938533204672741780329736406f;
// SM count of the CURRENT device (148 on B200), queried once per device: grids are sized from it
inline int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  int n = cached[dev];
  if (n == 0) {
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;   // benign race: every thread writes the same value
  }
  return n;
}

// Prior descriptor with the per-call constants folded on the host.
struct PriorDev {
  int kind;
  float c1, k1, inv_var1;  // component 1: log(pi) - log(s1) - .5log2pi ; 1/(2 s1^2) ; 1/s1^2
  float c2, k2, inv_var2;  // component 2 (mixture only)
  float c1l, k1l, c2l, k2l;  // c and k times log2(e): the density terms in the base the SFU works in
  float dkl, dcl;            // k1l - k2l, c2l - c1l: log2 of the component ratio p2/p1 is dkl w^2 + dcl
};

inline PriorDev make_prior_dev(const bbb_prior *p) {
  PriorDev d{};
  d.kind = p->kind;
  if (p->kind == BBB_PRIOR_MIXTURE) {
    double s1 = p->sigma1, s2 = p->sigma2, pi = p->pi;
    d.c1 = (float)(log(pi) - log(s1) - 0.918938533204672741780329736406);
    d.c2 = (float)(log1p(-pi) - log(s2) - 0.918938533204672741780329736406);
    d.k1 = (float)(1.0 / (2.0 * s1 * s1));
    d.k2 = (float)(1.0 / (2.0 * s2 * s2));
    d.inv_var1 = (float)(1.0 / (s1 * s1));
    d.inv_var2 = (float)(1.0 / (s2 * s2));
  } else {
    double s1 = p->sigma1;
    d.c1 = (float)(-log(s1) - 0.918938533204672741780329736406);
    d.k1 = (float)(1.0 / (2.0 * s1 * s1));
    d.inv_var1 = (float)(1.0 / (s1 * s1));
  }
  const double l2e = 1.4426950408889634074;
  d.c1l = (float)(d.c1 * l2e); d.k1l = (float)(d.k1 * l2e);
  d.c2l = (float)(d.c2 * l2e); d.k2l = (float)(d.k2 * l2e);
  d.dkl = (float)(((double)d.k1 - (double)d.k2) * l2e); d.dcl = (float)(((double)d.c2 - (double)d.c1) * l2e);
  return d;
}

struct RngDev {
  uint32_t key0, key1;  // seed
  // the ten Philox round keys (key + r * Weyl constant), formed on the host: as kernel parameters they are constant-bank
  // operands of the round's xor and cost neither a register nor the two additions per round
  uint32_t rk0[10], rk1[10];
  uint32_t step;
  uint32_t sample_base;
  uint32_t tensor_w, tensor_b;
  const uint32_t *step_dev;
};

inline RngDev make_rng_dev(const bbb_rng *r) {
  RngDev d{};
  if (r) {
    d.key0 = (uint32_t)(r->seed & 0xffffffffu);
    d.key1 = (uint32_t)(r->seed >> 32);
    uint32_t k0 = d.key0, k1 = d.key1;
    for (int i = 0; i < 10; ++i) { d.rk0[i] = k0; d.rk1[i] = k1; k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    d.step = r->step;
    d.sample_base = r->sample_base;
    d.tensor_w = 2u * r->layer;
    d.tensor_b = 2u * r->layer + 1u;
    d.step_dev = r->step_dev;
  }
  return d;
}

// ---------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011) -> 4 standard normals by Box-Muller.
// counter = (quad index, global sample, tensor id, step); key = seed.  The mapping depends only
// on the element's linear index, never on the tiling, so forward and backward regenerate
// bit-identical eps.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const RngDev &rng) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {   // 2 IMAD.WIDE + 2 LOP3 per round
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ rng.rk0[r], n2 = (uint32_t)(p0 >> 32) ^ c3 ^ rng.rk1[r];
    c1 = (uint32_t)p1; c3 = (uint32_t)p0; c0 = n0; c2 = n2;
  }
  return make_uint4(c0, c1, c2, c3);
}

// low 23 bits of a Philox word -> float in [1, 2): (x & 0x7fffff) | 0x3f800000 as ONE lop3 (the 1.0f pattern is handed
// over in a register so that the expression is not split into two immediates)
__device__ __forceinline__ float bits_to_12(uint32_t x) {
  uint32_t one, r;
  asm("mov.b32 %0, 0x3f800000;" : "=r"(one));
  asm("lop3.b32 %0, %1, 0x007fffff, %2, 0xEA;" : "=r"(r) : "r"(x), "r"(one));
  return __uint_as_float(r);
}

// Box-Muller on the SFU: lg2 / sqrt / sin / cos approximations (abs error ~2^-21, far below the sampling noise;
// moments and KS are checked in tests/test_gpu_parity.py).  The uniforms carry 23 bits: u' = 2 - u in (0, 1] for the
// radius (|z| <= 5.65), and sin / cos take 2 pi v with v in [1, 2) as it is (they are periodic).
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float &z0, float &z1) {
  const float u = bits_to_12(a), v = bits_to_12(b);
  float lg, r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(2.0f - u));
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-1.3862943611198906f * lg));   // sqrt(-2 ln u')
  float s, c;
  __sincosf(6.283185307179586f * v, &s, &c);
  z0 = r * s;
  z1 = r * c;
}

// fold the optional device-side step counter into the by-value descriptor (call once per thread)
__device__ __forceinline__ void rng_resolve(RngDev &rng) {
  if (rng.step_dev) rng.step += __ldg(rng.step_dev);
}

// 4 normals for elements 4q..4q+3 of tensor `tensor`, global sample `sample`.
__device__ __forceinline__ void philox_normal4(const RngDev &rng, uint32_t tensor, uint32_t sample,
                                               uint32_t quad, float z[4]) {
  uint4 r = philox4x32_10(quad, sample, tensor, rng.step, rng);
  box_muller(r.x, r.y, z[0], z[1]);
  box_muller(r.z, r.w, z[2], z[3]);
}

// one normal for linear element index e (slow path for rows that are not 16-byte aligned)
__device__ __forceinline__ float philox_normal1(const RngDev &rng, uint32_t tensor, uint32_t sample,
                                                uint64_t e) {
  uint4 r = philox4x32_10((uint32_t)(e >> 2), sample, tensor, rng.step, rng);
  uint32_t lane = (uint32_t)(e & 3u);
  float z0, z1;
  if (lane < 2) box_muller(r.x, r.y, z0, z1);
  else box_muller(r.z, r.w, z0, z1);
  return (lane & 1u) ? z1 : z0;
}

// ---------------------------------------------------------------------------------------
// posterior / prior math
// ---------------------------------------------------------------------------------------
// sigma = log(1 + e^rho)  (networks.py:39).  Above rho = 15 the algebraically identical
// rho + log1p(e^-rho) is used, which stays finite where the reference overflows (SURVEY B-6).
__device__ __forceinline__ float softplus_f(float rho) {
  return rho > 15.0f ? rho + log1pf(expf(-rho)) : log1pf(expf(rho));
}
__device__ __forceinline__ float sigmoid_f(float rho) { return 1.0f / (1.0f + expf(-rho)); }

// log q contribution of one element: -0.5 log 2pi - log sigma - eps^2 / 2   (networks.py:46)
__device__ __forceinline__ float logq_elem(float sigma, float eps) {
  return -kHalfLog2Pi - logf(sigma) - 0.5f * eps * eps;
}

// log p(w) of one element (stable log-sum-exp form of networks.py:24-27, or networks.py:67-68)
__device__ __forceinline__ float logp_elem(const PriorDev &p, float w) {
  float w2 = w * w;
  float a = fmaf(-p.k1, w2, p.c1);
  if (p.kind == BBB_PRIOR_GAUSSIAN) return a;
  float b = fmaf(-p.k2, w2, p.c2);
  float m = fmaxf(a, b);
  return m + logf(expf(a - m) + expf(b - m));
}

// R(w) with d log p / d w = -w R(w): responsibilities-weighted inverse variance (SURVEY App. A-2)
__device__ __forceinline__ float prior_R(const PriorDev &p, float w) {
  if (p.kind == BBB_PRIOR_GAUSSIAN) return p.inv_var1;
  float w2 = w * w;
  float a = fmaf(-p.k1, w2, p.c1), b = fmaf(-p.k2, w2, p.c2);
  float m = fmaxf(a, b);
  float ea = expf(a - m), eb = expf(b - m);
  float inv = 1.0f / (ea + eb);
  return (ea * p.inv_var1 + eb * p.inv_var2) * inv;
}

// SFU-based variants used by the tensor-core (TF32) kernels, where the stated bound is 5e-3 on GEMM outputs
// and 1e-5 on the log-prob sums: ex2.approx / lg2.approx carry ~1e-7 absolute error per element here.
__device__ __forceinline__ float logp_elem_fast(const PriorDev &p, float w) {
  const float w2 = w * w;
  const float a = fmaf(-p.k1, w2, p.c1);
  if (p.kind == BBB_PRIOR_GAUSSIAN) return a;
  const float b = fmaf(-p.k2, w2, p.c2);
  const float m = fmaxf(a, b), d = fminf(a, b) - m;   // exp(max - m) = 1
  return m + __logf(1.0f + __expf(d));
}
__device__ __forceinline__ float rcp_approx_f(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// R(w) = (1/s1^2 + t/s2^2) / (1 + t) with t = p2(w)/p1(w) = 2^(dkl w^2 + dcl): one exponential, one reciprocal, no
// selects.  (t is bounded by its value at w = 0 when s2 < s1; the clamp covers priors given the other way round.)
__device__ __forceinline__ float prior_R_fast(const PriorDev &p, float w) {
  if (p.kind == BBB_PRIOR_GAUSSIAN) return p.inv_var1;
  float t;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fminf(fmaf(p.dkl, w * w, p.dcl), 100.0f)));
  return fmaf(t, p.inv_var2, p.inv_var1) * rcp_approx_f(1.0f + t);
}

// ---------------------------------------------------------------------------------------
// SFU math for the tensor-core (TF32) kernels.  Stated bounds for that mode: 5e-3 on anything downstream of a
// contraction, 1e-5 on the log-prob sums; every function below is accurate to ~1e-6 relative or better.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// sigma = log1p(t), t = e^rho, plus sigmoid(rho) = t / (1 + t) from the same exponential.
// t < 1/8: alternating series to t^6 (truncation 5e-7 relative); else log(1 + t) on the SFU; rho > 15: sigma = rho.
__device__ __forceinline__ void softplus_sigmoid_fast(float rho, float &sigma, float &sigmoid) {
  const float t = ex2_approx(rho * 1.4426950408889634f);
  const float u = 1.0f + t;
  float ser = fmaf(t, -0.16666667f, 0.2f);
  ser = fmaf(t, ser, -0.25f);
  ser = fmaf(t, ser, 0.33333334f);
  ser = fmaf(t, ser, -0.5f);
  ser = fmaf(t, ser, 1.0f);
  ser *= t;
  const float lg = 0.6931471805599453f * lg2_approx(u);
  sigma = rho > 15.0f ? rho : (t < 0.125f ? ser : lg);
  sigmoid = rho > 15.0f ? 1.0f : t * rcp_approx_f(u);
}
__device__ __forceinline__ float softplus_fast(float rho) {
  float sg, sm;
  softplus_sigmoid_fast(rho, sg, sm);
  return sg;
}
// sum of log p(w_j) over the 4 weights of a quad.  Mixture: p = 2^a + 2^b in the base-2 domain, one lg2 per PAIR of
// weights (the product of two densities cannot underflow for |w| < 9 sigma1); same exp -> mix -> log order as
// networks.py:24-27.
__device__ __forceinline__ float logp_quad_fast(const PriorDev &p, const float w[4]) {
  const float s2 = fmaf(w[0], w[0], fmaf(w[1], w[1], fmaf(w[2], w[2], w[3] * w[3])));
  if (p.kind == BBB_PRIOR_GAUSSIAN) return fmaf(-p.k1, s2, 4.0f * p.c1);
  // log2 p(w) = (c1l - k1l w^2) + log2(1 + t),  t = p2/p1 = 2^(dkl w^2 + dcl): ONE exponential per weight and one
  // logarithm per pair (1 <= 1 + t <= 1 + 2^dcl, so the product of two cannot overflow)
  float u[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) u[j] = 1.0f + ex2_approx(fminf(fmaf(p.dkl, w[j] * w[j], p.dcl), 60.0f));
  const float lg = lg2_approx(u[0] * u[1]) + lg2_approx(u[2] * u[3]);
  return 0.6931471805599453f * (fmaf(-p.k1l, s2, 4.0f * p.c1l) + lg);
}
// sum of log sigma_j over a quad: one lg2 per pair (sigma > 1e-19 keeps the product normal)
__device__ __forceinline__ float logsigma_quad_fast(const float sg[4]) {
  return 0.6931471805599453f * (lg2_approx(sg[0] * sg[1]) + lg2_approx(sg[2] * sg[3]));
}

// ---------------------------------------------------------------------------------------
// Adam (torch.optim.Adam, no amsgrad, no weight decay): the update rule of the multi-tensor kernels (bbb_adam.cu).
// ---------------------------------------------------------------------------------------
struct AdamConst {
  float b1, b2, omb1, omb2, step_size, bc2_sqrt, eps;
};
// 1-beta, the bias corrections and the step size are formed in double, as torch does on the host
__device__ __forceinline__ AdamConst adam_consts(double lr, double b1, double b2, float eps, uint32_t step,
                                                 const uint32_t *step_dev, const float *lr_scale_dev) {
  const uint32_t t = step + (step_dev ? *step_dev : 0u);
  const double bc1 = 1.0 - pow(b1, (double)t), bc2 = 1.0 - pow(b2, (double)t);
  const double lr_t = lr * (lr_scale_dev ? (double)*lr_scale_dev : 1.0);
  AdamConst c;
  c.b1 = (float)b1; c.b2 = (float)b2;
  c.omb1 = (float)(1.0 - b1); c.omb2 = (float)(1.0 - b2);
  c.step_size = (float)(lr_t / bc1); c.bc2_sqrt = (float)sqrt(bc2); c.eps = eps;
  return c;
}
// lerp_(g, 1-b1);  mul_(b2).addcmul_(g, g, 1-b2);  denom = sqrt(v)/sqrt(bc2) + eps;  addcdiv_(m, denom, -step_size)
__device__ __forceinline__ void adam1(float &p, float g, float &m, float &v, const AdamConst &c) {
  m = fmaf(c.omb1, g - m, m);
  v = fmaf(c.omb2 * g, g, c.b2 * v);
  const float denom = sqrtf(v) / c.bc2_sqrt + c.eps;
  p = fmaf(-c.step_size, m / denom, p);
}

// the same update with the SFU's sqrt and reciprocal (1 ulp-level approximations) for the kernels that apply the
// optimiser inside a compute-bound epilogue: ~10 instructions instead of ~30
__device__ __forceinline__ void adam1_fast(float &p, float g, float &m, float &v, const AdamConst &c, float inv_bc2_sqrt) {
  m = fmaf(c.omb1, g - m, m);
  v = fmaf(c.omb2 * g, g, c.b2 * v);
  float sq;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq) : "f"(v));
  float inv;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(fmaf(sq, inv_bc2_sqrt, c.eps)));
  p = fmaf(-c.step_size * m, inv, p);
}

// ---------------------------------------------------------------------------------------
// reductions
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum of two floats, result added to two double accumulators by one thread.
// `red` is a __shared__ float[2*32] scratch.  All threads of the block must call.
__device__ __forceinline__ void block_sum2_atomic(float a, float b, float *red, double *dst_a,
                                                  double *dst_b) {
  a = warp_sum(a);
  b = warp_sum(b);
  int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
  if (lane == 0) { red[warp] = a; red[32 + warp] = b; }
  __syncthreads();
  if (warp == 0) {
    double da = lane < nwarp ? (double)red[lane] : 0.0;
    double db = lane < nwarp ? (double)red[32 + lane] : 0.0;
    da = warp_sum_d(da);
    db = warp_sum_d(db);
    if (lane == 0) {
      if (dst_a) atomicAdd(dst_a, da);
      if (dst_b) atomicAdd(dst_b, db);
    }
  }
  __syncthreads();
}

// 4 consecutive floats starting at base[idx], zero-filled past `valid` elements.
__device__ __forceinline__ void ld4(const float *__restrict__ base, int64_t idx, int valid, bool vec,
                                    float v[4]) {
  if (vec && valid >= 4) {
    float4 t = __ldg(reinterpret_cast<const float4 *>(base + idx));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = j < valid ? __ldg(base + idx + j) : 0.0f;
  }
}

}  // namespace bbb
