// Internal interface of the network-level step for batches of at most 128 rows (bbb_mlp_fwd / bbb_mlp_bwd, include/bbb.h):
// per-layer descriptors and the launchers of the TMA-fed tcgen05 kernels (bbb_mlp_fwd.cu, bbb_mlp_bwd.cu).
#pragma once
#include "bbb_common.cuh"

namespace bbb {

// one weight-sampling layer inside a network-level call
struct MlpLayerDesc {
  const float *x;            // forward input [S,B,in]: the PRE-activation output of the layer below (ReLU is applied to the
  bool x_shared;             // loaded tiles in shared memory), or [B,in] when x_shared (the network's input, no ReLU)
  const float *w_mu, *w_rho, *b_mu, *b_rho, *eps_w, *eps_b;
  int64_t in, out;
  float *y;                  // [S,B,out] zero-filled: the pre-activation output, split-K partial tiles are reduce-added into it
  // backward
  const float *dz;           // [S,B,out] gradient w.r.t. the layer's pre-activation output
  float *dx;                 // [S,B,in] zero-filled: gradient w.r.t. the pre-activation input (masked by x > 0), or NULL
  float *g_w_mu, *g_w_rho, *g_b_mu, *g_b_rho;
};

struct MlpFwdArgs {
  const float *b_mu, *b_rho, *eps_w, *eps_b;
  double *logp, *logq;
  RngDev rng;
  PriorDev prior;
  int S, B, in, out, in4;
  int n_ot, T_o, nkb;        // output-row tiles of T_o rows; 32-wide k blocks
  int base, rem;             // CTA -> (pair, part): the first `rem` pairs get base + 1 CTAs, the others base
  int flags, x_shared;
  unsigned long long *timeline;   // debug (bbb_debug_set_timeline): 16 globaltimer stamps per CTA, or NULL
};

struct MlpBwdArgs {
  const float *w_mu, *w_rho, *b_mu, *b_rho, *eps_w, *eps_b;
  const float *dz;           // (plain loads: bias column sums)
  const float *x;            // (plain loads: the (x > 0) mask of dgrad)
  float *dx, *g_w_mu, *g_w_rho, *g_b_mu, *g_b_rho;
  RngDev rng;
  PriorDev prior;
  int S, B, in, out;
  int n_ot, T_o;             // output-row tiles
  int n_c;                   // column ranges per row tile (grid = n_c x n_ot)
  int flags, x_shared;
  float gp, gq;              // d loss / d logp_s, d loss / d logq_s (host factors) ...
  const float *gp_dev, *gq_dev, *out_scale_dev;   // ... times optional device scalars (bbb_linear_bwd semantics)
  int g_dev_stride;
  unsigned long long *timeline;   // debug: 16 globaltimer stamps per CTA, or NULL
};

// debug: phase time stamps of the network-level kernels (tools/kernel_timeline.py)
unsigned long long *debug_timeline();
// the peer-exchange kernel's six stamps: slot 8 of the same buffer (words 20480..20485), or NULL
unsigned long long *peer_timeline();
__device__ __forceinline__ void stamp(unsigned long long *tl, int slot) {
  if (tl) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    tl[(size_t)(blockIdx.y * gridDim.x + blockIdx.x) * 16 + slot] = t;
  }
}

bool mlp_fwd_layer_supported(const MlpLayerDesc &l, int64_t S, int64_t B);
int launch_mlp_fwd_layer(const MlpLayerDesc &l, int64_t S, int64_t B, const RngDev &rng, const PriorDev &prior, int flags,
                         double *logp, double *logq, cudaStream_t st);
bool mlp_bwd_layer_supported(const MlpLayerDesc &l, int64_t S, int64_t B);
int launch_mlp_bwd_layer(const MlpLayerDesc &l, int64_t S, int64_t B, const RngDev &rng, const PriorDev &prior, int flags,
                         float gp, float gq, const float *gp_dev, const float *gq_dev, int g_dev_stride,
                         const float *out_scale_dev, cudaStream_t st);

}  // namespace bbb
