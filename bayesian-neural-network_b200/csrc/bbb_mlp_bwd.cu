// Weight-sampling Bayesian linear layer, fused backward, for batches of at most 128 rows -- round-2 organisation.
//
// One kernel per layer: wgrad, the analytic mu/rho-gradient epilogue and dgrad with ONE eps regeneration, like
// csrc/bbb_linear_bwd_fused.cu, but no thread ever stages an operand tile and nothing is transposed by hand:
//
//   * warp 0 (one lane) is the TMA producer.  A row-major [batch][features] matrix IS an MN-major tcgen05 operand when
//     it lands in the SWIZZLE_128B_ATOM_32B layout (bbb_tma.cuh), so for  G_s[o][i] = sum_b dz_s[b][o] x_s[b][i]  the
//     dz and x tiles are streamed as 32-batch-row chunks through a 4-deep ring straight from where the forward / the layer
//     above left them (x_s is the post-ReLU activation the forward stored);  for  dX_s[b][i] = sum_o dz_s[b][o] W_s[o][i]
//     the same dz tile is loaded K-major (SWIZZLE_128B).  mu and rho of the CTA's block are TMA-loaded INTO the two
//     weight-tile slots: the sampler that owns a quad reads (mu, rho) from them and overwrites them in place with
//     (W_0, W_1), the MN-major B operands of dgrad -- the block's parameters cost no global-load instruction and no
//     extra shared memory.
//   * warp 1 (one lane) issues the MMAs: accumulators G_0, G_1, dX_0, dX_1 in TMEM (4 x 96 columns).
//   * warps 2..17 (512 threads): a thread owns weight ROW o = its TMEM lane, so it reads its G quads straight from TMEM
//     (no shared-memory round trip), regenerates eps (Philox), forms w, t = G - gp w R(w), and sums grad_mu / grad_rho
//     over the samples of the group in 8 registers per quad.  Gradients and dX leave through a small swizzled staging
//     tile that turns the row-per-lane ownership into coalesced 16-byte global accesses.
//
// A CTA owns rows [o_t0, o_t0 + rows) of one output-row tile x a 4-aligned column range of at most 32 XWR columns;
// sample groups of 2 are processed one after the other (gradients of later groups are added by the same CTA).
#include "bbb_tc_tiles.cuh"
#include "bbb_tma.cuh"
#include "bbb_mlp.h"

namespace bbb {
namespace {

using namespace tc;

constexpr int kEpiWarps = 16;
constexpr int kEpi = kEpiWarps * 32;              // 512
constexpr int kThreadsB = 64 + kEpi;
constexpr int REG = 128 * 128;                    // bytes of one [128 rows][128 B] region
constexpr int CH_ROWS = 32;                       // batch rows per MMA1 chunk
constexpr int CH_REG = CH_ROWS * 128;             // bytes of one [32 rows][128 B] chunk region
constexpr int NRING = 4;

template <int XWR>
struct BwdCfg {
  static constexpr int kW = XWR * REG;                            // one weight-tile slot
  static constexpr int kChunk = (4 + XWR) * CH_REG;               // dz (4 o groups) | x (XWR i groups)
  static constexpr int kRing = NRING * kChunk;                    // later reused: dz K-major (4 REG) | staging (2 REG)
  static constexpr int kArea = kRing > 6 * REG ? kRing : 6 * REG;
  static constexpr int kDyn = 2 * kW + kArea + 1024;
  static constexpr int kN = 32 * XWR;                             // MMA N
};

struct BwdCtl {
  uint64_t murho_full, ring_full[NRING], ring_fixed[NRING], ring_empty[NRING], g_full, dzk_full, w_full, dx_full[2], tail_done;
  uint32_t tmem_base;
};

__device__ __forceinline__ void bar_epi() { asm volatile("bar.sync 1, 512;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_l(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
// staging tile [128 rows][32 fp32]: 16-byte chunk index XOR (row & 7): conflict-free for a lane-per-row writer and for a
// quarter-warp-per-row reader
__device__ __forceinline__ uint32_t stg_off(int row, int c16) { return (uint32_t)((row << 7) + ((c16 ^ (row & 7)) << 4)); }

// MODE 0: eps from Philox, 1: eps injected from memory, 2: w = mu
template <int XWR, int MODE, bool kDx>
__global__ void __launch_bounds__(kThreadsB, 1)
ws_bwd_kernel(const __grid_constant__ CUtensorMap tm_mu, const __grid_constant__ CUtensorMap tm_rho,
              const __grid_constant__ CUtensorMap tm_dz, const __grid_constant__ CUtensorMap tm_x,
              const __grid_constant__ CUtensorMap tm_dzk, const MlpBwdArgs a) {
  using Cfg = BwdCfg<XWR>;
  constexpr int N = Cfg::kN;
  extern __shared__ uint8_t dsm[];
  __shared__ BwdCtl ctl;
  __shared__ float csum[2][128];
  const uint32_t base = (smem_u32(dsm) + 1023u) & ~1023u;
  const uint32_t w_s[2] = {base, base + Cfg::kW};        // weight-tile slots (mu / rho land here)
  const uint32_t area = base + 2 * Cfg::kW;              // MMA1 ring, later dz K-major (4 REG) + staging (2 REG)
  const uint32_t dzk = area, stg = area + 4 * REG;
  const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
  unsigned long long *tl = tid == 64 ? a.timeline : nullptr;     // the first epilogue thread stamps the phases (group 0)
  stamp(tl, 0);

  // ---- this CTA's block ----------------------------------------------------------------------------------------------
  const int ot = blockIdx.y;
  const int o_t0 = ot * a.T_o, rows = min(a.T_o, a.out - o_t0);
  const int nq_i = a.in >> 2;
  const int q_lo = (int)((int64_t)blockIdx.x * nq_i / gridDim.x), q_hi = (int)((int64_t)(blockIdx.x + 1) * nq_i / gridDim.x);
  const int tq = q_hi - q_lo, i_lo = q_lo * 4;
  const int groups = (a.S + 1) >> 1;
  const bool bias_cta = blockIdx.x == 0;

  if (wid == 1) tmem_alloc(smem_u32(&ctl.tmem_base), 512);
  if (tid == 0) {
    mbar_init(smem_u32(&ctl.murho_full), 1);
    for (int i = 0; i < NRING; ++i) {
      mbar_init(smem_u32(&ctl.ring_full[i]), 1); mbar_init(smem_u32(&ctl.ring_empty[i]), 1);
      mbar_init(smem_u32(&ctl.ring_fixed[i]), kEpiWarps);
    }
    mbar_init(smem_u32(&ctl.g_full), 1);
    mbar_init(smem_u32(&ctl.dzk_full), 1);
    mbar_init(smem_u32(&ctl.w_full), kEpiWarps);
    mbar_init(smem_u32(&ctl.dx_full[0]), 1);
    mbar_init(smem_u32(&ctl.dx_full[1]), 1);
    mbar_init(smem_u32(&ctl.tail_done), kEpiWarps);
    mbar_fence_init();
    tma::prefetch_map(&tm_mu); tma::prefetch_map(&tm_rho); tma::prefetch_map(&tm_dz); tma::prefetch_map(&tm_x);
    if (kDx) tma::prefetch_map(&tm_dzk);
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = ctl.tmem_base;
  const uint32_t tm_g[2] = {tmem, tmem + 96}, tm_dx[2] = {tmem + 192, tmem + 288};
  stamp(tl, 1);
  const bool relu_in = a.flags & BBB_F_RELU_IN;      // x is the pre-activation of the layer below: max(., 0) in shared memory
  // (mu / rho are written by the optimiser only: the producer requests the block's tiles before the dependency wait)
  if (wid != 0) pdl_wait();
  stamp(tl, 2);

  if (wid == 0) {
    // ================================ TMA producer ====================================================================
    if (lane == 0) {
      int rit = 0;                                        // ring iteration counter over all groups
      for (int g = 0; g < groups; ++g) {
        const int s0 = 2 * g, ns = min(2, a.S - s0);
        const uint32_t gph = (uint32_t)(g & 1);
        if (g > 0) mbar_wait(smem_u32(&ctl.tail_done), gph ^ 1u);   // the previous group is out of every buffer
        // the block's mu -> slot 0, rho -> slot 1 (MN-major layout: rows = o, 128 B = 32 consecutive i)
        tma::arrive_expect_tx(smem_u32(&ctl.murho_full), (uint32_t)(2 * XWR * REG));
#pragma unroll
        for (int r = 0; r < XWR; ++r) {
          tma::load_2d(w_s[0] + r * REG, &tm_mu, smem_u32(&ctl.murho_full), i_lo + 32 * r, o_t0);
          tma::load_2d(w_s[1] + r * REG, &tm_rho, smem_u32(&ctl.murho_full), i_lo + 32 * r, o_t0);
        }
        if (g == 0) pdl_wait();
        // MMA1 operands: per sample 4 chunks of 32 batch rows, dz [4 o groups] + x [XWR i groups]
        for (int s = 0; s < ns; ++s) {
          for (int ch = 0; ch < 4; ++ch, ++rit) {
            const int slot = rit % NRING;
            // (a new group's first chunks also waited on tail_done above: the ring aliases the dgrad buffers)
            if (rit >= NRING) mbar_wait(smem_u32(&ctl.ring_empty[slot]), (uint32_t)(((rit / NRING) - 1) & 1));
            const uint32_t cb = area + slot * Cfg::kChunk, bar = smem_u32(&ctl.ring_full[slot]);
            tma::arrive_expect_tx(bar, (uint32_t)Cfg::kChunk);
#pragma unroll
            for (int og = 0; og < 4; ++og) tma::load_3d(cb + og * CH_REG, &tm_dz, bar, o_t0 + 32 * og, CH_ROWS * ch, s0 + s);
#pragma unroll
            for (int r = 0; r < XWR; ++r)
              tma::load_3d(cb + (4 + r) * CH_REG, &tm_x, bar, i_lo + 32 * r, CH_ROWS * ch, a.x_shared ? 0 : s0 + s);
          }
        }
        if (kDx) {
          // dgrad's A operand: dz_s K-major, once MMA1 of the whole group has left the ring, then once MMA2(0) is done
          for (int s = 0; s < ns; ++s) {
            if (s == 0) mbar_wait(smem_u32(&ctl.g_full), gph);
            else mbar_wait(smem_u32(&ctl.dx_full[0]), gph);
            tma::arrive_expect_tx(smem_u32(&ctl.dzk_full), (uint32_t)(4 * REG));
#pragma unroll
            for (int og = 0; og < 4; ++og) tma::load_3d(dzk + og * REG, &tm_dzk, smem_u32(&ctl.dzk_full), o_t0 + 32 * og, 0, s0 + s);
          }
        }
      }
    } else {
      pdl_wait();
    }
    __syncwarp();
    pdl_launch_dependents();
  } else if (wid == 1) {
    // ================================ MMA issuer ======================================================================
    if (lane == 0) {
      constexpr uint32_t idesc1 = idesc_tf32_major(128, N, 1, 1);   // G  = dz^T x : A, B MN-major
      constexpr uint32_t idesc2 = idesc_tf32_major(128, N, 0, 1);   // dX = dz W  : A K-major, B MN-major
      int rit = 0, dzk_it = 0, wph = 0;
      for (int g = 0; g < groups; ++g) {
        const int s0 = 2 * g, ns = min(2, a.S - s0);
        for (int s = 0; s < ns; ++s) {
          for (int ch = 0; ch < 4; ++ch, ++rit) {
            const int slot = rit % NRING;
            mbar_wait_parked(smem_u32(&ctl.ring_full[slot]), (uint32_t)((rit / NRING) & 1));
            if (relu_in) mbar_wait_parked(smem_u32(&ctl.ring_fixed[slot]), (uint32_t)((rit / NRING) & 1));
            tc_fence_after_sync();
            const uint32_t cb = area + slot * Cfg::kChunk;
#pragma unroll
            for (int k8 = 0; k8 < 4; ++k8)
              mma_tf32(tm_g[s], smem_desc_mn32(cb + k8 * 1024, CH_REG), smem_desc_mn32(cb + 4 * CH_REG + k8 * 1024, CH_REG),
                       idesc1, (ch | k8) ? 1u : 0u);
            mma_commit(smem_u32(&ctl.ring_empty[slot]));
          }
        }
        mma_commit(smem_u32(&ctl.g_full));
        if (kDx) {
          // dgrad.  Sample 0 region by region (N = 32) as the epilogue completes each 32-column region of the weight
          // tiles -- only the last region's MMAs are left when the epilogue ends --; sample 1 in one piece once its
          // K-major dz tile has replaced sample 0's.
          constexpr uint32_t idesc2r = idesc_tf32_major(128, 32, 0, 1);
          const int nk = (rows + 7) >> 3;
          mbar_wait_parked(smem_u32(&ctl.dzk_full), (uint32_t)(dzk_it & 1));
          ++dzk_it;
          for (int r = 0; r < XWR; ++r, ++wph) {
            mbar_wait_parked(smem_u32(&ctl.w_full), (uint32_t)(wph & 1));
            tc_fence_after_sync();
            for (int k8 = 0; k8 < nk; ++k8)
              mma_tf32(tm_dx[0] + 32 * r, smem_desc_sw128(dzk + (k8 >> 2) * REG + (k8 & 3) * 32),
                       smem_desc_mn32(w_s[0] + r * REG + k8 * 1024, REG), idesc2r, k8 ? 1u : 0u);
          }
          mma_commit(smem_u32(&ctl.dx_full[0]));
          if (ns > 1) {
            mbar_wait_parked(smem_u32(&ctl.dzk_full), (uint32_t)(dzk_it & 1));
            ++dzk_it;
            tc_fence_after_sync();
            for (int k8 = 0; k8 < nk; ++k8)
              mma_tf32(tm_dx[1], smem_desc_sw128(dzk + (k8 >> 2) * REG + (k8 & 3) * 32),
                       smem_desc_mn32(w_s[1] + k8 * 1024, REG), idesc2, k8 ? 1u : 0u);
            mma_commit(smem_u32(&ctl.dx_full[1]));
          }
        }
      }
    }
    __syncwarp();
    pdl_launch_dependents();
  } else {
    // ================================ samplers / epilogue =============================================================
    RngDev rng = a.rng;
    rng_resolve(rng);
    const int et = tid - 64;
    const int q = wid & 3, cgp = (wid - 2) >> 2;          // TMEM lane quarter, column sub-group (2 quads per region)
    const int row = q * 32 + lane;                        // weight row o (wgrad) / batch row b (dgrad) of this thread
    const bool row_ok = row < rows;
    const float osc = a.out_scale_dev ? __ldg(a.out_scale_dev) : 1.0f;
    const bool accum_flag = a.flags & BBB_F_ACCUM;
    const int c_row = et >> 3, c_chk = et & 7;            // coalesced mapping: rows c_row + 64 h, 16-byte chunk c_chk
    int erit = 0;                                          // MMA1 chunk counter (the ring's iteration index)
    for (int g = 0; g < groups; ++g) {
      const int s0 = 2 * g, ns = min(2, a.S - s0);
      const uint32_t gph = (uint32_t)(g & 1);
      float gps[2], gqs[2];
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const int si = min(s0 + s, a.S - 1);
        gps[s] = a.gp * (a.gp_dev ? __ldg(a.gp_dev + si * a.g_dev_stride) : 1.0f);
        gqs[s] = a.gq * (a.gq_dev ? __ldg(a.gq_dev + si * a.g_dev_stride) : 1.0f);
      }
      if (relu_in) {
        // the x part of every MMA1 chunk holds PRE-activations: max(., 0) in place, chunk by chunk as they land
        // (XWR regions of [32 rows][128 B]: 256 16-byte quads each; elementwise, so the swizzle does not matter)
        for (int c8 = 0; c8 < 4 * ns; ++c8, ++erit) {
          const int slot = erit % NRING;
          mbar_wait_parked(smem_u32(&ctl.ring_full[slot]), (uint32_t)((erit / NRING) & 1));
          const uint32_t xb = area + slot * Cfg::kChunk + 4 * CH_REG;
          for (int i = et; i < XWR * 256; i += kEpi) {
            const float4 v = lds128(xb + i * 16);
            sts128(xb + i * 16, fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f));
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive_l(smem_u32(&ctl.ring_fixed[slot]));
        }
      }
      // ---- bias gradients (the CTAs of column range 0): column sums of dz over the batch, then the analytic terms ----
      if (bias_cta && et < 256) {
        const int o_l = et & 127, s = et >> 7;
        float acc = 0.0f;
        if (s < ns && o_l < rows) {
          const float *zp = a.dz + ((int64_t)(s0 + s) * a.B) * a.out + o_t0 + o_l;
          for (int b = 0; b < a.B; ++b) acc += __ldg(zp + (int64_t)b * a.out);
        }
        csum[s][o_l] = acc;
      }
      mbar_wait_parked(smem_u32(&ctl.murho_full), gph);     // (parked: a spinning warp would take issue slots from the
      if (g == 0) stamp(tl, 3);
      mbar_wait_parked(smem_u32(&ctl.g_full), gph);         //  TMA and MMA warps, which have the lowest priority)
      tc_fence_after_sync();
      if (g == 0) stamp(tl, 4);
      if (bias_cta) {
        bar_epi();
        if (et < rows) {
          const int o = o_t0 + et;
          const float bmu = __ldg(a.b_mu + o), brho = __ldg(a.b_rho + o);
          const float bsg = softplus_f(brho);
          float gbm = 0.0f, gbr = 0.0f;
          for (int s = 0; s < ns; ++s) {
            float ep = 0.0f;
            if (MODE == 0) ep = philox_normal1(rng, rng.tensor_b, rng.sample_base + (uint32_t)(s0 + s), (uint64_t)o);
            if (MODE == 1) ep = __ldg(a.eps_b + (int64_t)(s0 + s) * a.out + o);
            const float bv = MODE == 2 ? bmu : __fadd_rn(bmu, __fmul_rn(bsg, ep));
            float t = csum[s][et];
            if (gps[s] != 0.0f) t = fmaf(-gps[s] * bv, prior_R(a.prior, bv), t);
            gbm += t;
            gbr += -expm1f(-bsg) * (t * ep - gqs[s] / bsg);
          }
          const bool acc_b = accum_flag || g > 0;
          a.g_b_mu[o] = acc_b ? fmaf(osc, gbm, a.g_b_mu[o]) : osc * gbm;
          a.g_b_rho[o] = acc_b ? fmaf(osc, gbr, a.g_b_rho[o]) : osc * gbr;
        }
      }
      // ---- the block's weights, region by region (32 columns): two adjacent quads per thread ----------------------------
#pragma unroll 1
      for (int r = 0; r < XWR; ++r) {
        float G[2][8];
#pragma unroll
        for (int s = 0; s < 2; ++s)
          if (s < ns) tmem_ld8(tm_g[s] + ((uint32_t)(q * 32) << 16) + (uint32_t)(32 * r + 8 * cgp), G[s]);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int c16 = 2 * cgp + h, qd = 8 * r + c16;                 // quad index inside the window
          const uint32_t off = (uint32_t)(r * REG) + mn32_off(row, c16);
          float gm[4] = {0.f, 0.f, 0.f, 0.f}, gr[4] = {0.f, 0.f, 0.f, 0.f};
          if (row_ok && qd < tq) {
            const float4 m4 = lds128(w_s[0] + off), r4 = lds128(w_s[1] + off);
            const float mu[4] = {m4.x, m4.y, m4.z, m4.w}, rho[4] = {r4.x, r4.y, r4.z, r4.w};
            float sg[4], sgm[4], isg[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              softplus_sigmoid_fast(rho[e], sg[e], sgm[e]);
              isg[e] = rcp_approx_f(sg[e]);
            }
            const uint32_t quad = (uint32_t)(o_t0 + row) * (uint32_t)nq_i + (uint32_t)(q_lo + qd);
#pragma unroll
            for (int s = 0; s < 2; ++s) {
              if (s >= ns) break;
              float ep[4] = {0.f, 0.f, 0.f, 0.f}, w[4];
              if (MODE == 0) philox_normal4(rng, rng.tensor_w, rng.sample_base + (uint32_t)(s0 + s), quad, ep);
              if (MODE == 1) {
                const float4 e4 = __ldg(reinterpret_cast<const float4 *>(a.eps_w + (int64_t)(s0 + s) * a.out * a.in) + quad);
                ep[0] = e4.x; ep[1] = e4.y; ep[2] = e4.z; ep[3] = e4.w;
              }
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                w[e] = MODE == 2 ? mu[e] : fmaf(sg[e], ep[e], mu[e]);
                float t = G[s][4 * h + e];
                if (gps[s] != 0.0f) t = fmaf(-gps[s] * w[e], prior_R_fast(a.prior, w[e]), t);
                gm[e] += t;
                gr[e] += sgm[e] * fmaf(t, ep[e], -gqs[s] * isg[e]);
              }
              if (kDx) sts128(w_s[s] + off, to_tf32(w[0]), to_tf32(w[1]), to_tf32(w[2]), to_tf32(w[3]));
            }
          } else if (kDx && !row_ok) {
            // rows of the next tile inside the MMA's last K step must not contribute to dX
            sts128(w_s[0] + off, 0.f, 0.f, 0.f, 0.f);
            sts128(w_s[1] + off, 0.f, 0.f, 0.f, 0.f);
          }
          // stage the gradient quads: [row][c16] of the mu tile and of the rho tile
          sts128(stg + stg_off(row, c16), osc * gm[0], osc * gm[1], osc * gm[2], osc * gm[3]);
          sts128(stg + REG + stg_off(row, c16), osc * gr[0], osc * gr[1], osc * gr[2], osc * gr[3]);
        }
        if (kDx) {      // this warp's part of the region's weight tiles is complete: dgrad of the region may start
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive_l(smem_u32(&ctl.w_full));
        }
        // coalesced write-back of the region: a quarter warp per row
        bar_epi();
        {
          const int qd = 8 * r + c_chk;
          if (qd < tq) {
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              const int rr = c_row + 64 * hh;
              if (rr < rows) {
                const int64_t e = (int64_t)(o_t0 + rr) * a.in + i_lo + 4 * qd;
                float4 vm = lds128(stg + stg_off(rr, c_chk)), vr = lds128(stg + REG + stg_off(rr, c_chk));
                float4 *pm = reinterpret_cast<float4 *>(a.g_w_mu + e), *pr = reinterpret_cast<float4 *>(a.g_w_rho + e);
                if (accum_flag || g > 0) {
                  const float4 om = *pm, orr = *pr;
                  vm.x += om.x; vm.y += om.y; vm.z += om.z; vm.w += om.w;
                  vr.x += orr.x; vr.y += orr.y; vr.z += orr.z; vr.w += orr.w;
                }
                *pm = vm;
                *pr = vr;
              }
            }
          }
        }
        bar_epi();      // the staging tiles are rewritten by the next region
        if (g == 0 && r < 3) stamp(tl, 5 + r);
      }
      if (kDx) {
        // ---- dgrad: dX_s [lane = b][column = i] -> mask -> red.add ----------------------------------------------------------
        if (g == 0) stamp(tl, 8);
        for (int s = 0; s < ns; ++s) {
          // the activations this layer consumed (the (x > 0) mask), in the coalesced mapping: requested before the wait
          float4 xm[XWR][2];
#pragma unroll
          for (int r = 0; r < XWR; ++r)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              const int b = c_row + 64 * hh, qd = 8 * r + c_chk;
              xm[r][hh] = make_float4(0.f, 0.f, 0.f, 0.f);
              if (qd < tq && b < a.B)
                xm[r][hh] = __ldg(reinterpret_cast<const float4 *>(a.x + ((int64_t)(s0 + s) * a.B + b) * a.in + i_lo + 4 * qd));
            }
          mbar_wait_parked(smem_u32(&ctl.dx_full[s]), gph);
          tc_fence_after_sync();
          if (g == 0) stamp(tl, 9 + 2 * s);
#pragma unroll
          for (int r = 0; r < XWR; ++r) {
            float v[8];
            tmem_ld8(tm_dx[s] + ((uint32_t)(q * 32) << 16) + (uint32_t)(32 * r + 8 * cgp), v);
            // two staging tiles, used alternately: one barrier per region instead of two
            const uint32_t sg_t = stg + (uint32_t)((r & 1) * REG);
            sts128(sg_t + stg_off(row, 2 * cgp), v[0], v[1], v[2], v[3]);
            sts128(sg_t + stg_off(row, 2 * cgp + 1), v[4], v[5], v[6], v[7]);
            bar_epi();
            const int qd = 8 * r + c_chk;
            if (qd < tq) {
#pragma unroll
              for (int hh = 0; hh < 2; ++hh) {
                const int b = c_row + 64 * hh;
                if (b < a.B) {
                  const int64_t e = ((int64_t)(s0 + s) * a.B + b) * a.in + i_lo + 4 * qd;
                  const float4 d = tcx::mask4(lds128(sg_t + stg_off(b, c_chk)), xm[r][hh]);
                  tcx::red_add_v4(a.dx + e, d);
                }
              }
            }
          }
          bar_epi();      // (the staging tiles are rewritten by the next sample)
          if (g == 0) stamp(tl, 10 + 2 * s);
        }
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive_l(smem_u32(&ctl.tail_done));
    }
    pdl_launch_dependents();
  }
  stamp(tl, 15);
  tc_fence_before_sync();
  __syncthreads();
  if (wid == 1) tmem_dealloc(tmem, 512);
}

inline int cdiv_i(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }
inline bool al16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

template <int XWR, int MODE, bool kDx>
int launch_one(const CUtensorMap *tm, const MlpBwdArgs &a, dim3 grid, cudaStream_t st) {
  auto kernel = ws_bwd_kernel<XWR, MODE, kDx>;
  BBB_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BwdCfg<XWR>::kDyn));
  BBB_CHECK_CUDA(launch_pdl(kernel, grid, dim3(kThreadsB), (size_t)BwdCfg<XWR>::kDyn, st, tm[0], tm[1], tm[2], tm[3], tm[4], a));
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}
template <int XWR>
int launch_x(const CUtensorMap *tm, const MlpBwdArgs &a, dim3 grid, int mode, bool dx, cudaStream_t st) {
  if (mode == 0) return dx ? launch_one<XWR, 0, true>(tm, a, grid, st) : launch_one<XWR, 0, false>(tm, a, grid, st);
  if (mode == 1) return dx ? launch_one<XWR, 1, true>(tm, a, grid, st) : launch_one<XWR, 1, false>(tm, a, grid, st);
  return dx ? launch_one<XWR, 2, true>(tm, a, grid, st) : launch_one<XWR, 2, false>(tm, a, grid, st);
}

}  // namespace

bool mlp_bwd_layer_supported(const MlpLayerDesc &l, int64_t S, int64_t B) {
  if (!(B >= 1 && B <= 128 && S >= 1 && l.in >= 4 && l.in % 4 == 0 && l.out >= 4 && l.out % 4 == 0)) return false;
  return al16(l.x) && al16(l.w_mu) && al16(l.w_rho) && al16(l.eps_w) && al16(l.dz) && al16(l.dx) && al16(l.g_w_mu) &&
         al16(l.g_w_rho) && l.in * l.out / 4 < (int64_t)1 << 32;     // (NULL gradient pointers count as aligned)
}

// One layer's backward: dz [S,B,out], x [Sx,B,in] (post-ReLU activations, or the network input when x_shared) ->
// parameter gradients (overwritten, or added to with BBB_F_ACCUM) and, when dx != NULL, dx [S,B,in] += (dz W_s) (x > 0)
// (zero-filled by the caller: the CTAs of different row tiles add their partial sums).
int launch_mlp_bwd_layer(const MlpLayerDesc &l, int64_t S, int64_t B, const RngDev &rng, const PriorDev &prior, int flags,
                         float gp, float gq, const float *gp_dev, const float *gq_dev, int g_dev_stride,
                         const float *out_scale_dev, cudaStream_t st) {
  const bool sample = flags & BBB_F_SAMPLE;
  const int mode = !sample ? 2 : (l.eps_w ? 1 : 0);
  MlpBwdArgs a{};
  a.w_mu = l.w_mu; a.w_rho = l.w_rho; a.b_mu = l.b_mu; a.b_rho = l.b_rho; a.eps_w = l.eps_w; a.eps_b = l.eps_b;
  a.dz = l.dz; a.x = l.x; a.dx = l.dx;
  a.g_w_mu = l.g_w_mu; a.g_w_rho = l.g_w_rho; a.g_b_mu = l.g_b_mu; a.g_b_rho = l.g_b_rho;
  a.rng = rng; a.prior = prior;
  a.S = (int)S; a.B = (int)B; a.in = (int)l.in; a.out = (int)l.out;
  a.n_ot = cdiv_i(l.out, 128);
  a.T_o = ((cdiv_i(l.out, a.n_ot) + 3) / 4) * 4;
  a.n_ot = cdiv_i(l.out, a.T_o);
  a.flags = flags; a.x_shared = l.x_shared ? 1 : 0;
  a.timeline = debug_timeline();
  a.gp = gp; a.gq = gq; a.gp_dev = gp_dev; a.gq_dev = gq_dev; a.g_dev_stride = g_dev_stride; a.out_scale_dev = out_scale_dev;
  const int nq_i = (int)(l.in / 4);
  int n_c = sm_count() / a.n_ot;                                   // about one CTA per SM
  const int need = cdiv_i(nq_i, 24);                               // a column range is at most 96 wide
  if (n_c < need) n_c = need;
  if (n_c > nq_i) n_c = nq_i;
  if (n_c < 1) n_c = 1;
  a.n_c = n_c;
  const int width = cdiv_i(nq_i, n_c) * 4;
  const int xwr = width <= 32 ? 1 : width <= 64 ? 2 : 3;
  CUtensorMap tm[5];
  if (int r = tma::make_map(&tm[0], l.w_mu, l.in, l.out, 0, 32, 128, tma::kSw128Atom32)) return r;
  if (int r = tma::make_map(&tm[1], l.w_rho, l.in, l.out, 0, 32, 128, tma::kSw128Atom32)) return r;
  if (int r = tma::make_map(&tm[2], l.dz, l.out, B, S, 32, CH_ROWS, tma::kSw128Atom32)) return r;
  if (int r = tma::make_map(&tm[3], l.x, l.in, B, l.x_shared ? 1 : S, 32, CH_ROWS, tma::kSw128Atom32)) return r;
  tm[4] = tm[2];
  if (l.dx)
    if (int r = tma::make_map(&tm[4], l.dz, l.out, B, S, 32, 128, tma::kSw128)) return r;
  dim3 grid(n_c, a.n_ot);
  const bool dx = l.dx != nullptr;
  if (xwr == 1) return launch_x<1>(tm, a, grid, mode, dx, st);
  if (xwr == 2) return launch_x<2>(tm, a, grid, mode, dx, st);
  return launch_x<3>(tm, a, grid, mode, dx, st);
}

}  // namespace bbb
