// Weight-sampling Bayesian linear layer on tcgen05 kind::tf32 for LARGE batches (BASELINE.json config 5: 4096-wide
// layers, batch 4096): the weight gradient, and the support conditions of the large-batch path.  The forward and dgrad
// of these shapes run in bbb_wide.cu (wide_kernel), behind the same conditions.
//
// wgrad is a dense contraction over the batch, G_s[o][i] = sum_b dz_s[b][o] x_s[b][i], followed by an epilogue that
// regenerates eps from the forward's Philox coordinates and folds in the prior and posterior terms; W never leaves the
// SM.  Warp-specialised: 16 worker warps, one MMA-issuing warp and (TMA variant) one TMA warp; 1 CTA per SM (512 TMEM
// columns).
#include "bbb_tc_tiles.cuh"
#include "bbb_tma.cuh"
#include <cmath>
#include <cstring>

namespace bbb {
namespace {

using namespace tc;
using namespace tcx;

constexpr int PW = 16;                    // producer warps
constexpr int PT = PW * 32;               // producer threads
constexpr int BT = PT + 32;               // + the MMA-issuing warp

__device__ __forceinline__ void mbar_arrive1(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// ==================================================================================================
// wgrad for large batches:  G_s[o][i] = sum_b dz_s[b][o] x_s[b][i]  (M = 128 o, N = 256 i, K = the batch), then
//   t = G - gp w R(w);  grad_mu += t;  grad_rho += sigmoid(rho) (t eps - gq / sigma)      (eps regenerated)
// Both operands are MN-major: a [32 batch rows][128 B] slab of the row-major dz / x matrices IS an operand region
// (SWIZZLE_128B_BASE32B, bbb_tc.cuh), so the main loop is a plain copy global -> shared with no transposes, 4 stages
// of 32 batch rows deep, and runs at the tensor pipe's pace.  TMEM holds the accumulators of TWO samples
// (2 x 256 columns): their K loops run back to back and the epilogue then finishes both with mu / rho / sigma loaded
// once.  The epilogue reads TMEM directly: a thread owns one weight row o and 64 consecutive columns i.
// ==================================================================================================
constexpr int WN = 256;                    // i columns per CTA tile
constexpr int WKB = 32;                    // batch rows per stage
constexpr int WSTG = 4;
constexpr int WREG = WKB * 128;            // one [32 rows][128 B] region
constexpr int WA_BYTES = (BM / 32) * WREG; // dz slab: 4 regions (128 o)
constexpr int WB_BYTES = (WN / 32) * WREG; // x slab : 8 regions (256 i)
constexpr int WSTAGE = WA_BYTES + WB_BYTES;
constexpr int kWgradDyn = WSTG * WSTAGE + 1024;

struct WCtl {
  uint64_t full[WSTG], fixed[WSTG], empty[WSTG], acc;
  uint32_t tmem_base;
};
// gridDim.z = 2 splits the sample groups of every tile over two CTAs (the 512 tiles of a 4096 x 4096 layer fill 3.46
// waves of 148 SMs, 1024 half-jobs fill 6.92): z = 0 writes the gradient tensors, z = 1 these partial tensors, which
// wgrad_combine_kernel adds in afterwards (two addends: the sum does not depend on any order)
struct WgradPart {
  float *w_mu, *w_rho, *b_mu, *b_rho;
};

// kTma: the slabs are loaded by TMA (one extra warp; grouped 4-D maps, bbb_tma.cuh: one box = the 4 dz regions, one =
// the 8 x regions of a stage, already in the MN-major layout), which streams them from L2 several times faster than
// per-thread copies can (tools/wide_probe.cu); the 16 worker warps only touch a stage when it needs the ReLU or feeds
// the bias column sums.  Needs in % 32 == 0 and out % 32 == 0; the cp.async variant covers every other shape.
template <bool kTma>
__global__ void __launch_bounds__(kTma ? BT + 32 : BT, 1)
big_wgrad_kernel(const __grid_constant__ CUtensorMap tm_dz, const __grid_constant__ CUtensorMap tm_x, const LinArgs a_in,
                 const WgradPart part) {
  extern __shared__ uint8_t dsm[];
  __shared__ WCtl ctl;
  __shared__ float colsum_s[2][BM];     // sum_b dz[b][o] of the two samples in flight (bias gradients)
  LinArgs a = a_in;
  uint8_t *tiles = align1024(dsm);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool sample = a.flags & BBB_F_SAMPLE, relu = a.flags & BBB_F_RELU_IN;
  bool accum_flag = a.flags & BBB_F_ACCUM;
  const int64_t o0 = (int64_t)blockIdx.x * BM, i0 = (int64_t)blockIdx.y * WN;
  const bool bias_cta = blockIdx.y == 0;
  const int nkb = (int)((a.B + WKB - 1) / WKB);
  // this CTA's share of the sample groups: groups [g_lo, g_hi) = samples [s_base, s_base + S_loc)
  const int ngroups_all = (a.S + 1) / 2;
  const int g_lo = ngroups_all * (int)blockIdx.z / (int)gridDim.z, g_hi = ngroups_all * ((int)blockIdx.z + 1) / (int)gridDim.z;
  const int s_base = 2 * g_lo, S_loc = min(a.S, 2 * g_hi) - s_base, ngroups = g_hi - g_lo;
  if (blockIdx.z > 0) {
    a.g_w_mu = part.w_mu; a.g_w_rho = part.w_rho; a.g_b_mu = part.b_mu; a.g_b_rho = part.b_rho;
    accum_flag = false;
  }
  const bool need_fix = relu || bias_cta;      // (kTma) the worker warps pass over every stage before the MMAs read it

  if (warp == PW) tmem_alloc(smem_u32(&ctl.tmem_base), 512);
  if (tid == 0) {
#pragma unroll
    for (int st = 0; st < WSTG; ++st) {
      mbar_init(smem_u32(&ctl.full[st]), kTma ? 1 : PW);
      mbar_init(smem_u32(&ctl.fixed[st]), PW);
      mbar_init(smem_u32(&ctl.empty[st]), 1);
    }
    mbar_init(smem_u32(&ctl.acc), 1);
    mbar_fence_init();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = ctl.tmem_base;
  pdl_wait();
  rng_resolve(a.rng);
  const float osc = a.out_scale_dev ? __ldg(a.out_scale_dev) : 1.0f;

  if (warp == PW) {
    // ---- MMA warp: the stage counter runs on across samples and groups ------------------------------
    constexpr uint32_t idesc = idesc_tf32_major(BM, WN, 1, 1);
    int it = 0;
    for (int g = 0; g < ngroups; ++g) {
      const int ns = min(2, S_loc - 2 * g);
      if (lane == 0) {
        for (int sl = 0; sl < ns; ++sl) {
          for (int kb = 0; kb < nkb; ++kb, ++it) {
            const int st = it % WSTG;
            mbar_wait_parked(smem_u32((kTma && need_fix) ? &ctl.fixed[st] : &ctl.full[st]), (uint32_t)((it / WSTG) & 1));
            tc_fence_after_sync();
            const uint32_t As = smem_u32(tiles + st * WSTAGE), Bs = As + WA_BYTES;
#pragma unroll
            for (int k8 = 0; k8 < WKB / 8; ++k8)
              mma_tf32(tmem + sl * WN, smem_desc_mn32(As + k8 * 1024, WREG), smem_desc_mn32(Bs + k8 * 1024, WREG), idesc,
                       (kb == 0 && k8 == 0) ? 0u : 1u);
            mma_commit(smem_u32(&ctl.empty[st]));
          }
        }
        mma_commit(smem_u32(&ctl.acc));
      }
      __syncwarp();
      // the accumulators are overwritten by the next group: the whole warp waits until the epilogue has read them
      if (g + 1 < ngroups) {
        asm volatile("bar.sync 2, %0;" ::"n"(BT) : "memory");
        tc_fence_after_sync();
      }
    }
  } else if (kTma && warp == PW + 1) {
    // ---- TMA warp: two boxes per stage, running ahead of the MMAs by up to WSTG stages (across samples and groups) ----
    if (lane == 0) {
      tma::prefetch_map(&tm_dz);
      tma::prefetch_map(&tm_x);
      int it = 0;
      for (int s = s_base; s < s_base + S_loc; ++s) {
        const int sx = a.x_sstride ? s : 0;
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int st = it % WSTG;
          if (it >= WSTG) mbar_wait(smem_u32(&ctl.empty[st]), (uint32_t)(((it / WSTG) - 1) & 1));
          const uint32_t base = smem_u32(tiles + st * WSTAGE), bar = smem_u32(&ctl.full[st]);
          tma::arrive_expect_tx(bar, (uint32_t)WSTAGE);
          tma::load_4d(base, &tm_dz, bar, 0, kb * WKB, (int)(o0 >> 5), s);
          tma::load_4d(base + WA_BYTES, &tm_x, bar, 0, kb * WKB, (int)(i0 >> 5), sx);
        }
      }
    }
    __syncwarp();
  } else {
    // ---- producers: slab copies.  dz: thread t -> batch rows t/32 + 16 h (h < 2), 16-byte chunk t%32 (4 o columns);
    //                              x : thread t -> batch rows t/64 + 8 h (h < 4),  16-byte chunk t%64 (4 i columns)
    const int ar = tid >> 5, ac = tid & 31, br = tid >> 6, bc = tid & 63;
    const uint32_t a_off = (uint32_t)(ac >> 3) * WREG, b_off = (uint32_t)(bc >> 3) * WREG;
    const int64_t ao = o0 + ac * 4, bi = i0 + bc * 4;
    const bool ao_ok = ao < a.out, bi_ok = bi < a.in;
    int it = 0;
    for (int g = 0; g < ngroups; ++g) {
      const int s0 = s_base + 2 * g, ns = min(2, S_loc - 2 * g);
      if (bias_cta && tid < 2 * BM) colsum_s[tid >> 7][tid & (BM - 1)] = 0.0f;
      for (int sl = 0; sl < ns; ++sl) {
        const float *dzs = a.dy + (int64_t)(s0 + sl) * a.B * a.out + (ao_ok ? ao : 0);
        const float *xs = a.x + (int64_t)(s0 + sl) * a.x_sstride + (bi_ok ? bi : 0);
        float4 bsum = make_float4(0.f, 0.f, 0.f, 0.f);
        // Slab copies with cp.async (global -> shared, 16 bytes, L2 only, zero fill outside the matrices), kAhead
        // batch blocks in flight per thread: no registers are staged, so the latency of streaming dz and x (together
        // as large as the L2: every wave of tiles reads them from HBM again) hides behind three slabs of copies.
        // ReLU and the bias column sums are applied to the thread's own chunks once they have landed.
        constexpr int kAhead = WSTG - 1;
        // per-thread constants of the copy: the six shared-memory offsets inside a stage and the six global row
        // pointers of batch block 0 (columns outside the matrix: pointer clamped, zero bytes copied); a block
        // advances every pointer by 32 rows, so the loop carries no index arithmetic
        uint32_t zoff[2], xoff[4];
        const float *zp[2], *xp[4];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          zoff[h] = a_off + mn32_off(ar + 16 * h, ac & 7);
          zp[h] = dzs + (int64_t)(ar + 16 * h) * a.out;
        }
#pragma unroll
        for (int h = 0; h < 4; ++h) {
          xoff[h] = WA_BYTES + b_off + mn32_off(br + 8 * h, bc & 7);
          xp[h] = xs + (int64_t)(br + 8 * h) * a.in;
        }
        if constexpr (kTma) {
          // the slabs arrive by TMA; this thread owns the same chunks of a stage as in the copying variant
          if (need_fix) {
            for (int kb = 0; kb < nkb; ++kb, ++it) {
              const int st = it % WSTG;
              mbar_wait(smem_u32(&ctl.full[st]), (uint32_t)((it / WSTG) & 1));
              uint8_t *stage = tiles + st * WSTAGE;
              if (bias_cta) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                  const float4 z = *reinterpret_cast<const float4 *>(stage + zoff[h]);
                  bsum.x += z.x; bsum.y += z.y; bsum.z += z.z; bsum.w += z.w;
                }
              }
              if (relu) {
#pragma unroll
                for (int h = 0; h < 4; ++h) {
                  float4 *px = reinterpret_cast<float4 *>(stage + xoff[h]);
                  *px = relu4(*px);
                }
                fence_proxy_async_smem();
              }
              __syncwarp();
              if (lane == 0) mbar_arrive1(smem_u32(&ctl.fixed[st]));
            }
          } else {
            it += nkb;
          }
        } else {
        const int64_t zstep = (int64_t)WKB * a.out, xstep = (int64_t)WKB * a.in;
        const uint32_t ring = smem_u32(tiles);
        auto issue_slab = [&](int kb, int j) {      // j: running stage index of that slab; called for kb = 0, 1, 2, ...
          const int st = j % WSTG;
          if (j >= WSTG) mbar_wait(smem_u32(&ctl.empty[st]), (uint32_t)(((j / WSTG) - 1) & 1));
          const uint32_t base = ring + st * WSTAGE;
          if ((int64_t)(kb + 1) * WKB <= a.B) {     // whole block inside the batch: the common case
#pragma unroll
            for (int h = 0; h < 2; ++h)
              asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(base + zoff[h]), "l"(zp[h]), "r"(ao_ok ? 16 : 0) : "memory");
#pragma unroll
            for (int h = 0; h < 4; ++h)
              asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(base + xoff[h]), "l"(xp[h]), "r"(bi_ok ? 16 : 0) : "memory");
          } else {                                   // last, partial block: rows past the batch are zero-filled
            const int64_t b0 = (int64_t)kb * WKB;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const bool ok = ao_ok && b0 + ar + 16 * h < a.B;
              asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(base + zoff[h]), "l"(ok ? zp[h] : dzs), "r"(ok ? 16 : 0) : "memory");
            }
#pragma unroll
            for (int h = 0; h < 4; ++h) {
              const bool ok = bi_ok && b0 + br + 8 * h < a.B;
              asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(base + xoff[h]), "l"(ok ? xp[h] : xs), "r"(ok ? 16 : 0) : "memory");
            }
          }
#pragma unroll
          for (int h = 0; h < 2; ++h) zp[h] += zstep;
#pragma unroll
          for (int h = 0; h < 4; ++h) xp[h] += xstep;
        };
        for (int p = 0; p < kAhead; ++p) {
          if (p < nkb) issue_slab(p, it + p);
          asm volatile("cp.async.commit_group;" ::: "memory");
        }
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          if (kb + kAhead < nkb) issue_slab(kb + kAhead, it + kAhead);
          asm volatile("cp.async.commit_group;" ::: "memory");      // (an empty group keeps the count uniform)
          asm volatile("cp.async.wait_group %0;" ::"n"(kAhead) : "memory");   // this thread's copies of block kb landed
          const int st = it % WSTG;
          uint8_t *stage = tiles + st * WSTAGE;
          if (bias_cta) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const float4 z = *reinterpret_cast<const float4 *>(stage + zoff[h]);
              bsum.x += z.x; bsum.y += z.y; bsum.z += z.z; bsum.w += z.w;
            }
          }
          if (relu) {
#pragma unroll
            for (int h = 0; h < 4; ++h) {
              float4 *px = reinterpret_cast<float4 *>(stage + xoff[h]);
              *px = relu4(*px);
            }
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive1(smem_u32(&ctl.full[st]));
        }
        }   // !kTma
        if (bias_cta) {
          atomicAdd(&colsum_s[sl][ac * 4 + 0], bsum.x); atomicAdd(&colsum_s[sl][ac * 4 + 1], bsum.y);
          atomicAdd(&colsum_s[sl][ac * 4 + 2], bsum.z); atomicAdd(&colsum_s[sl][ac * 4 + 3], bsum.w);
        }
      }
      // ---- epilogue of the group: thread = weight row o (TMEM lane), 64 consecutive columns i ------------------
      mbar_wait_parked(smem_u32(&ctl.acc), (uint32_t)(g & 1));
      tc_fence_after_sync();
      asm volatile("bar.sync 1, %0;" ::"n"(PT) : "memory");   // colsum_s complete
      const bool accum = accum_flag || g > 0;
      float gps[2], gqs[2];
#pragma unroll
      for (int sl = 0; sl < 2; ++sl) {
        gps[sl] = sl < ns ? a.gp * (a.gp_dev ? __ldg(a.gp_dev + (s0 + sl) * a.g_dev_stride) : 1.0f) : 0.0f;
        gqs[sl] = sl < ns ? a.gq * (a.gq_dev ? __ldg(a.gq_dev + (s0 + sl) * a.g_dev_stride) : 1.0f) : 0.0f;
      }
      const int q4 = warp & 3, cq = warp >> 2;
      const int64_t o = o0 + q4 * 32 + lane;
#pragma unroll 1
      for (int c0 = 0; c0 < 64; c0 += 8) {
        const int col = cq * 64 + c0;
        if (i0 + col >= a.in) break;                       // warp-uniform
        // two quads at a time, every load of the pair (mu, rho, the running gradient sums) issued before the accumulators
        // are read and before the first store: interleaved with the stores they would go out one L2 round trip at a
        // time (possible aliasing).  (tcgen05.ld is warp-collective: rows past `out` take part with their loads clamped.)
        const bool o_ok = o < a.out;
        float4 m4[2], r4[2], om[2], orr[2];
        bool ok[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int64_t i = i0 + col + 4 * u;
          ok[u] = o_ok && i < a.in;
          const int64_t e = ok[u] ? o * a.in + i : 0;
          m4[u] = __ldg(reinterpret_cast<const float4 *>(a.w_mu + e));
          r4[u] = __ldg(reinterpret_cast<const float4 *>(a.w_rho + e));
          om[u] = orr[u] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (accum && ok[u]) {
            om[u] = *reinterpret_cast<const float4 *>(a.g_w_mu + e);
            orr[u] = *reinterpret_cast<const float4 *>(a.g_w_rho + e);
          }
        }
        float G[2][8];
        tmem_ld8(tmem + ((uint32_t)(q4 * 32) << 16) + (uint32_t)col, G[0]);
        if (ns > 1) tmem_ld8(tmem + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(WN + col), G[1]);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          if (!ok[u]) continue;
          const int64_t e = o * a.in + i0 + col + 4 * u;
          Quad q;
          q.mu[0] = m4[u].x; q.mu[1] = m4[u].y; q.mu[2] = m4[u].z; q.mu[3] = m4[u].w;
          q.rho[0] = r4[u].x; q.rho[1] = r4[u].y; q.rho[2] = r4[u].z; q.rho[3] = r4[u].w;
#pragma unroll
          for (int c = 0; c < 4; ++c) q.sg[c] = softplus_fast(q.rho[c]);
          float gm[4] = {0.f, 0.f, 0.f, 0.f}, gr[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int sl = 0; sl < 2; ++sl) {
            if (sl < ns) {
              float ep[4], w[4];
              sample_quad(a, s0 + sl, e, q, sample, ep, w);
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                float t = G[sl][4 * u + c];
                if (gps[sl] != 0.0f) t = fmaf(-gps[sl] * w[c], prior_R_fast(a.prior, w[c]), t);
                gm[c] += t;
                gr[c] += t * ep[c] - gqs[sl] * __fdividef(1.0f, q.sg[c]);
              }
            }
          }
#pragma unroll
          for (int c = 0; c < 4; ++c) gr[c] *= sigmoid_fast(q.rho[c]);
          *reinterpret_cast<float4 *>(a.g_w_mu + e) = make_float4(fmaf(osc, gm[0], om[u].x), fmaf(osc, gm[1], om[u].y),
                                                                  fmaf(osc, gm[2], om[u].z), fmaf(osc, gm[3], om[u].w));
          *reinterpret_cast<float4 *>(a.g_w_rho + e) = make_float4(fmaf(osc, gr[0], orr[u].x), fmaf(osc, gr[1], orr[u].y),
                                                                   fmaf(osc, gr[2], orr[u].z), fmaf(osc, gr[3], orr[u].w));
        }
      }
      // bias gradients: column sums of dz, by the CTAs of the first i tile
      if (bias_cta && tid < BM) {
        const int64_t ob = o0 + tid;
        if (ob < a.out) {
          float gbm = 0.0f, gbr = 0.0f;
          for (int sl = 0; sl < ns; ++sl) {
            float bv, sg, ep;
            bias_elem(a, s0 + sl, ob, sample, true, bv, sg, ep);
            float t = colsum_s[sl][tid];
            if (gps[sl] != 0.0f) t = fmaf(-gps[sl] * bv, prior_R(a.prior, bv), t);
            gbm += t;
            gbr += -expm1f(-sg) * (t * ep - gqs[sl] / sg);
          }
          a.g_b_mu[ob] = accum ? fmaf(osc, gbm, a.g_b_mu[ob]) : osc * gbm;
          a.g_b_rho[ob] = accum ? fmaf(osc, gbr, a.g_b_rho[ob]) : osc * gbr;
        }
      }
      tc_fence_before_sync();
      if (g + 1 < ngroups) asm volatile("bar.sync 2, %0;" ::"n"(BT) : "memory");   // accumulators and colsum_s are free
    }
  }
  pdl_launch_dependents();
  tc_fence_before_sync();
  __syncthreads();
  if (warp == PW) tmem_dealloc(tmem, 512);
}

inline int cdiv_i(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

}  // namespace

// Batches of at least 384 rows (3/4 of one 512-row tile) with 16-byte aligned rows; the weight matrix must be wide
// enough for full tiles to matter (narrow heads go to bbb_head.cu); no dy mask (the network path fuses the ReLU
// mask into the producer of dy: BBB_F_DX_PREACT)
bool linear_big_fwd_supported(const LinArgs &a) {
  return a.vec_in && a.B >= 384 && a.out >= 32 && a.in >= 32 && a.S >= 1;
}
bool linear_big_dgrad_supported(const LinArgs &a) {
  return a.vec_in && a.vec_out && a.B >= 384 && a.out >= 32 && a.in >= 32 && a.S >= 1 && !a.mask;
}

// wgrad: rows of dz and x must be 16-byte multiples (slab copies), no dy mask
bool linear_big_wgrad_supported(const LinArgs &a) {
  return a.vec_in && a.vec_out && a.B >= 384 && a.out >= 32 && a.in >= 32 && a.S >= 1 && !a.mask;
}
namespace {
// g += p for the four gradient tensors (float4 where the weight matrices allow it: in % 4 == 0 on this path)
__global__ void __launch_bounds__(256) wgrad_combine_kernel(float *g_w_mu, float *g_w_rho, float *g_b_mu, float *g_b_rho,
                                                            const WgradPart p, int64_t n_w4, int64_t n_b) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_w4; i += stride) {
    float4 a = reinterpret_cast<float4 *>(g_w_mu)[i], b = reinterpret_cast<const float4 *>(p.w_mu)[i];
    reinterpret_cast<float4 *>(g_w_mu)[i] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
    a = reinterpret_cast<float4 *>(g_w_rho)[i]; b = reinterpret_cast<const float4 *>(p.w_rho)[i];
    reinterpret_cast<float4 *>(g_w_rho)[i] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
  }
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_b; i += stride) {
    g_b_mu[i] += p.b_mu[i];
    g_b_rho[i] += p.b_rho[i];
  }
}
}  // namespace

static int g_wgrad_split_mode = 0;
extern "C" int bbb_debug_wgrad_split(int mode) {
  g_wgrad_split_mode = mode;
  return BBB_OK;
}

int launch_linear_wgrad_big(const LinArgs &a, cudaStream_t st) {
  dim3 grid(cdiv_i(a.out, BM), cdiv_i(a.in, WN));
  // Split the sample groups of every tile over two CTAs when that fills the SMs better (see WgradPart)
  const int ngroups = (a.S + 1) / 2;
  const double waves = (double)grid.x * grid.y / sm_count();
  const double eff1 = waves / ceil(waves), eff2 = 2 * waves / ceil(2 * waves);
  const int mode = g_wgrad_split_mode;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  BBB_CHECK_CUDA(cudaStreamIsCapturing(st, &cap));      // (no workspace allocation inside a graph capture)
  const bool split = ngroups >= 2 && mode >= 0 && (mode > 0 || eff2 > eff1 + 0.03) && cap == cudaStreamCaptureStatusNone;
  WgradPart part{};
  float *wsp = nullptr;
  const int64_t n_w = a.in * a.out, n_b4 = (a.out + 3) / 4 * 4;
  if (split) {
    grid.z = 2;
    // stream-ordered workspace from the device's default pool; the pool keeps what it is given back (without a release
    // threshold it would return the memory to the driver at every synchronisation and re-map it on the next call)
    static bool pool_set[64] = {false};
    int dev = 0;
    BBB_CHECK_CUDA(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && !pool_set[dev]) {
      cudaMemPool_t pool;
      BBB_CHECK_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
      uint64_t keep = UINT64_MAX;
      BBB_CHECK_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
      pool_set[dev] = true;
    }
    BBB_CHECK_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&wsp), (size_t)(2 * n_w + 2 * n_b4) * sizeof(float), st));
    part.w_mu = wsp; part.w_rho = wsp + n_w; part.b_mu = wsp + 2 * n_w; part.b_rho = wsp + 2 * n_w + n_b4;
  }
  CUtensorMap tm_dz, tm_x;
  if (a.in % 32 == 0 && a.out % 32 == 0) {
    if (int r = tma::make_map_grouped(&tm_dz, a.dy, a.out, a.B, a.S, WKB, BM / 32, tma::kSw128Atom32)) return r;
    if (int r = tma::make_map_grouped(&tm_x, a.x, a.in, a.B, a.x_sstride ? a.S : 1, WKB, WN / 32, tma::kSw128Atom32)) return r;
    BBB_CHECK_CUDA(cudaFuncSetAttribute(big_wgrad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgradDyn));
    BBB_CHECK_CUDA(launch_pdl(big_wgrad_kernel<true>, grid, dim3(BT + 32), kWgradDyn, st, tm_dz, tm_x, a, part));
  } else {
    memset(&tm_dz, 0, sizeof(tm_dz));
    memset(&tm_x, 0, sizeof(tm_x));
    BBB_CHECK_CUDA(cudaFuncSetAttribute(big_wgrad_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgradDyn));
    BBB_CHECK_CUDA(launch_pdl(big_wgrad_kernel<false>, grid, dim3(BT), kWgradDyn, st, tm_dz, tm_x, a, part));
  }
  BBB_CHECK_LAUNCH();
  if (split) {
    wgrad_combine_kernel<<<sm_count() * 4, 256, 0, st>>>(a.g_w_mu, a.g_w_rho, a.g_b_mu, a.g_b_rho, part, n_w / 4, a.out);
    BBB_CHECK_LAUNCH();
    BBB_CHECK_CUDA(cudaFreeAsync(wsp, st));
  }
  return BBB_OK;
}

}  // namespace bbb
