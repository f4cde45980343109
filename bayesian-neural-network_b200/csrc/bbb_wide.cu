// Weight-sampling Bayesian linear layer on tcgen05 kind::tf32 for LARGE batches, second generation (BASELINE.json
// config 5: 4096-wide layers, batch 4096): forward and dgrad with
//   * the activation tile streamed by TMA (one warp; [256 batch rows][32 k] half-tiles, SWIZZLE_128B = the K-major UMMA
//     operand as it lands; tools/wide_probe.cu: 90 B/clk per SM from L2 where per-thread copies reached 15), and
//   * every sampled weight tile SHARED by the CTAs of a thread-block cluster laid along the batch: a CTA samples 1 / CL
//     of the [128 weight rows][32 k] tile of a stage into its own shared memory and pushes that piece into the same
//     place of its CL - 1 peers with one bulk shared::cta -> shared::cluster copy each (completing on the peer's
//     mbarrier); a stage is recycled when the MMAs of ALL CTAs of the cluster have read it (tcgen05.commit multicast).
// With CL = 4 a weight is sampled once per 2048 batch rows (twice for the whole batch of config 5) instead of once per
// 512, which takes the CUDA-core work (Philox + Box-Muller + softplus [+ log-densities], ~65 instructions per weight)
// off the critical path: what remains is the tensor pipe.  W still never leaves the SMs.
//
//   D^T[m][b] (+)= A[m][k] * Bop[b][k]     M = 128 weight rows, N = 512 batch rows (two N = 256 MMAs), K = 32 / stage
//     forward:  A = W_s[o][k]   K-major SWIZZLE_128B                       Bop = x_s[b][k]   (ReLU applied in place)
//     dgrad:    A = W_s^T[i][o] MN-major SWIZZLE_128B_BASE32B (4 regions)   Bop = dz_s[b][o]
//
// Warps: 16 samplers (they also apply the ReLU to landed activation tiles and drain TMEM), one MMA issuer, one TMA
// issuer.  Shared memory: a ring of 5 activation half-tiles (160 KB) + a ring of 4 weight tiles (64 KB).
// Grid (weight-row tiles, batch tiles of 512, samples), clusters (1, CL, 1); the first cluster along the batch also
// accumulates the log-prob terms of the pieces it samples.
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "bbb_tc_tiles.cuh"
#include "bbb_tma.cuh"

namespace bbb {
namespace {

using namespace tc;
using namespace tcx;

constexpr int SW = 16;                    // sampler warps
constexpr int STH = SW * 32;              // sampler threads
constexpr int WT = STH + 64;              // + MMA warp + TMA warp
constexpr int NBT = 512;                  // batch rows per CTA tile = TMEM columns
constexpr int XH = 256;                   // batch rows per activation half-tile (one MMA's N)
constexpr int XS = 5;                     // ring of activation half-tiles
constexpr int WS = 4;                     // ring of weight tiles
constexpr int XBYTES = XH * 128;          // 32 KB
constexpr int WBYTES = BM * 128;          // 16 KB
constexpr int kWideDyn = XS * XBYTES + WS * WBYTES + 1024;

struct WideCtl {
  uint64_t x_full[XS], x_fixed[XS], x_empty[XS], w_full[WS], w_empty[WS], acc;
  uint32_t tmem_base;
};

__device__ __forceinline__ uint32_t cl_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cl_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cl_map(uint32_t local, uint32_t rank) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local), "r"(rank));
  return remote;
}
__device__ __forceinline__ void mbar_arrive_local(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// `bytes` of this CTA's shared memory -> the shared memory of another CTA of the cluster; completes (complete_tx) on
// that CTA's mbarrier
__device__ __forceinline__ void push_piece(uint32_t dst_cluster, uint32_t src_cta, uint32_t bytes, uint32_t bar_cluster) {
  asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst_cluster), "r"(src_cta), "r"(bytes), "r"(bar_cluster) : "memory");
}
// arrive on the mbarrier at this offset in every CTA of `mask` once all MMAs issued so far by this thread have completed
__device__ __forceinline__ void mma_commit_cluster(uint32_t bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ void tmem_ld32w(uint32_t taddr, float v[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// kDgrad = false: forward (A = W tile, rows = output features o, K = input features)
// kDgrad = true : dgrad   (A = W^T tile, rows = input features i, K = output features)
// CL: CTAs per cluster (1, 2 or 4), consecutive batch tiles
template <bool kDgrad, bool kLogProb, int CL>
__global__ void __launch_bounds__(WT, 1) wide_kernel(const __grid_constant__ CUtensorMap tm_act, const LinArgs a_in) {
  extern __shared__ uint8_t dsm[];
  __shared__ WideCtl ctl;
  __shared__ float red[64];
  LinArgs a = a_in;
  uint8_t *tiles = align1024(dsm);
  uint8_t *xs = tiles, *ws = tiles + XS * XBYTES;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool sample = a.flags & BBB_F_SAMPLE, relu = !kDgrad && (a.flags & BBB_F_RELU_IN);
  const int s = blockIdx.z;
  const int64_t m0 = (int64_t)blockIdx.x * BM, n0 = (int64_t)blockIdx.y * NBT;
  const int64_t Mdim = kDgrad ? a.in : a.out, Kdim = kDgrad ? a.out : a.in;
  const int nkb = (int)((Kdim + BK - 1) / BK);
  const uint32_t rank = CL > 1 ? cl_rank() : 0u;
  // the first cluster along the batch owns the log-prob terms: each of its CTAs those of the pieces it samples
  const bool lpcta = kLogProb && (int)blockIdx.y < CL;
  // sampler groups: with CL = 4 a CTA's piece of a stage is 256 quads, so the 512 sampler threads split into two
  // groups that take alternate k blocks
  constexpr int G = CL >= 4 ? CL / 2 : 1, T = STH / G, QP = 1024 / CL, QPT = QP / T, PIECE = WBYTES / CL;

  // ---- setup ----------------------------------------------------------------------------------------
  if (warp == SW) tmem_alloc(smem_u32(&ctl.tmem_base), 512);
  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < XS; ++i) {
      mbar_init(smem_u32(&ctl.x_full[i]), 1);
      mbar_init(smem_u32(&ctl.x_fixed[i]), SW / G);
      mbar_init(smem_u32(&ctl.x_empty[i]), 1);
    }
#pragma unroll
    for (int i = 0; i < WS; ++i) {
      mbar_init(smem_u32(&ctl.w_full[i]), 1);
      mbar_init(smem_u32(&ctl.w_empty[i]), CL);
    }
    mbar_init(smem_u32(&ctl.acc), 1);
    mbar_fence_init();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  if (CL > 1) cl_sync();                 // nobody pushes into a CTA whose barriers are not initialised yet
  const uint32_t tmem = ctl.tmem_base;
  pdl_wait();
  rng_resolve(a.rng);
  float lp = 0.0f, lq = 0.0f;

  if (warp == SW) {
    // ---- MMA warp ---------------------------------------------------------------------------
    if (lane == 0) {
      constexpr uint32_t idesc = kDgrad ? idesc_tf32_major(BM, XH, 1, 0) : idesc_tf32(BM, XH);
      for (int kb = 0; kb < nkb; ++kb) {
        const int wst = kb % WS;
        mbar_wait_parked(smem_u32(&ctl.w_full[wst]), (uint32_t)((kb / WS) & 1));
        const uint32_t As = smem_u32(ws + wst * WBYTES);
        const uint64_t da = smem_desc_sw128(As);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int xi = 2 * kb + h, xst = xi % XS;
          mbar_wait_parked(smem_u32(relu ? &ctl.x_fixed[xst] : &ctl.x_full[xst]), (uint32_t)((xi / XS) & 1));
          tc_fence_after_sync();
          const uint64_t db = smem_desc_sw128(smem_u32(xs + xst * XBYTES));
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            mma_tf32(tmem + h * XH, kDgrad ? smem_desc_mn32(As + kk * 1024, 4096) : da + 2u * kk, db + 2u * kk, idesc,
                     (kb == 0 && kk == 0) ? 0u : 1u);
          mma_commit(smem_u32(&ctl.x_empty[xst]));
        }
        if (CL > 1) mma_commit_cluster(smem_u32(&ctl.w_empty[wst]), (uint16_t)((1u << CL) - 1u));
        else mma_commit(smem_u32(&ctl.w_empty[wst]));
      }
      mma_commit(smem_u32(&ctl.acc));
    }
    __syncwarp();
  } else if (warp == SW + 1) {
    // ---- TMA warp: activation half-tiles, up to XS ahead of the MMAs ------------------------------
    if (lane == 0) {
      tma::prefetch_map(&tm_act);
      const int sa = kDgrad ? s : (a.x_sstride ? s : 0);
      for (int xi = 0; xi < 2 * nkb; ++xi) {
        const int xst = xi % XS;
        if (xi >= XS) mbar_wait(smem_u32(&ctl.x_empty[xst]), (uint32_t)(((xi / XS) - 1) & 1));
        const uint32_t bar = smem_u32(&ctl.x_full[xst]);
        tma::arrive_expect_tx(bar, (uint32_t)XBYTES);
        tma::load_3d(smem_u32(xs + xst * XBYTES), &tm_act, bar, (xi >> 1) * BK, (int)n0 + (xi & 1) * XH, sa);
      }
    }
    __syncwarp();
  } else {
    // ---- samplers ---------------------------------------------------------------------------------
    const int grp = tid / T, t = tid % T;
    for (int kb = grp; kb < nkb; kb += G) {
      const int wst = kb % WS;
      uint8_t *Wt = ws + wst * WBYTES;
      if (kb >= WS) mbar_wait(smem_u32(&ctl.w_empty[wst]), (uint32_t)(((kb / WS) - 1) & 1));
#pragma unroll
      for (int j = 0; j < QPT; ++j) {
        const int gq = (int)rank * QP + t + j * T;       // quad of the tile; this CTA's piece is the range [rank QP, +QP)
        float4 wv = make_float4(0.f, 0.f, 0.f, 0.f);
        uint32_t off;
        int64_t o, i;
        if (!kDgrad) {
          // [128 o][32 k] K-major: 8 quads per row, so the piece is 128 / CL consecutive rows
          const int row = gq >> 3, chunk = gq & 7;
          o = m0 + row; i = (int64_t)kb * BK + chunk * 4;
          off = sw128_off(row, chunk);
        } else {
          // W^T as an MN-major operand: 4 regions of [32 o rows][32 i], 256 quads each; a quad of 4 consecutive i of one
          // weight row o is ONE 16-byte store, nothing is transposed.  The piece is 4 / CL regions (or half of one)
          const int region = gq >> 8, kr = (gq & 255) >> 3, c16 = gq & 7;
          o = (int64_t)kb * BK + kr; i = m0 + 32 * region + 4 * c16;
          off = (uint32_t)region * 4096u + mn32_off(kr, c16);
        }
        if (o < a.out && i < a.in) {
          const int64_t e = o * a.in + i;
          Quad qd;
          load_quad(a, e, sample || lpcta, qd);
          float ep[4], w[4];
          sample_quad(a, s, e, qd, sample, ep, w);
          wv = make_float4(to_tf32(w[0]), to_tf32(w[1]), to_tf32(w[2]), to_tf32(w[3]));
          if (lpcta) {
            lp += logp_quad_fast(a.prior, w);
            lq += -4.0f * kHalfLog2Pi - logsigma_quad_fast(qd.sg) -
                  0.5f * (ep[0] * ep[0] + ep[1] * ep[1] + ep[2] * ep[2] + ep[3] * ep[3]);
          }
        }
        *reinterpret_cast<float4 *>(Wt + off) = wv;
      }
      fence_proxy_async_smem();
      asm volatile("bar.sync %0, %1;" ::"r"(1 + grp), "n"(T) : "memory");     // the group's piece is complete
      if (t == 0) {
        const uint32_t bar = smem_u32(&ctl.w_full[wst]);
        if (CL > 1) {
          tma::arrive_expect_tx(bar, (uint32_t)((CL - 1) * PIECE));
          const uint32_t src = smem_u32(Wt) + rank * PIECE;
#pragma unroll
          for (uint32_t p = 0; p < (uint32_t)CL; ++p)
            if (p != rank) push_piece(cl_map(src, p), src, (uint32_t)PIECE, cl_map(bar, p));
        } else {
          mbar_arrive_local(bar);
        }
      }
      if (relu) {
        // ReLU in place on the two activation half-tiles of this k block (the layer below stored pre-activations)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int xi = 2 * kb + h, xst = xi % XS;
          mbar_wait(smem_u32(&ctl.x_full[xst]), (uint32_t)((xi / XS) & 1));
          float4 *X = reinterpret_cast<float4 *>(xs + xst * XBYTES);
#pragma unroll
          for (int j = 0; j < XBYTES / 16 / T; ++j) X[t + j * T] = relu4(X[t + j * T]);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive_local(smem_u32(&ctl.x_fixed[xst]));
        }
      }
    }

    // ---- drain: warp w reads TMEM lanes 32 (w % 4) .. +31 (weight rows) and columns 128 (w / 4) .. +127 (batch) ----
    mbar_wait_parked(smem_u32(&ctl.acc), 0);
    tc_fence_after_sync();
    const int q4 = warp & 3, cq = warp >> 2;
    const int64_t m = m0 + q4 * 32 + lane;
    const bool m_ok = m < Mdim;
    float bias = 0.0f;
    if (!kDgrad && m_ok) {
      float sg, ep;
      const bool lpb = kLogProb && blockIdx.y == 0;
      bias_elem(a, s, m, sample, lpb, bias, sg, ep);
      if (lpb && cq == 0) { lp += logp_elem(a.prior, bias); lq += logq_elem(sg, ep); }
    }
    const float osc = (kDgrad && (a.flags & BBB_F_SCALE_DX) && a.out_scale_dev) ? __ldg(a.out_scale_dev) : 1.0f;
    const bool preact = kDgrad && (a.flags & BBB_F_DX_PREACT), relu_out = !kDgrad && (a.flags & BBB_F_RELU_OUT);
    float *dst = kDgrad ? a.dx + (int64_t)s * a.B * a.in : a.y + (int64_t)s * a.B * a.out;
    const float *msk = preact ? a.x + (int64_t)s * a.x_sstride : nullptr;
#pragma unroll 1
    for (int c0 = 0; c0 < 128; c0 += 32) {
      const int col = cq * 128 + c0;
      if (n0 + col >= a.B) break;                 // warp-uniform: the rest of this warp's columns are past the batch
      // the (x > 0) mask of these 32 batch columns first, all loads in flight at once (`dst` may alias nothing here, but
      // the compiler cannot know: interleaved with the stores they would be issued one L2 round trip at a time)
      float mk[32];
      if (preact) {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int64_t b = min(n0 + col + j, a.B - 1);
          mk[j] = m_ok ? __ldg(msk + b * Mdim + m) : 0.0f;
        }
      }
      float v[32];
      tmem_ld32w(tmem + ((uint32_t)(q4 * 32) << 16) + (uint32_t)col, v);
      if (m_ok) {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int64_t b = n0 + col + j;
          if (b < a.B) {
            float r = kDgrad ? osc * v[j] : v[j] + bias;
            if (relu_out) r = fmaxf(r, 0.0f);
            if (preact && !(mk[j] > 0.0f)) r = 0.0f;
            dst[b * Mdim + m] = r;
          }
        }
      }
    }
    tc_fence_before_sync();
  }
  pdl_launch_dependents();
  if (kLogProb) block_sum2_atomic(lp, lq, red, a.logp + s, a.logq + s);
  tc_fence_before_sync();
  __syncthreads();
  if (CL > 1) cl_sync();                 // peers may still be reading pieces pushed from this CTA's shared memory
  if (warp == SW) tmem_dealloc(tmem, 512);
}

inline int cdiv_w(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

template <bool kDgrad, bool kLogProb, int CL>
int launch_wide_cl(const CUtensorMap &tm, const LinArgs &a, dim3 grid, cudaStream_t st) {
  auto kern = wide_kernel<kDgrad, kLogProb, CL>;
  BBB_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kWideDyn));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(WT);
  cfg.dynamicSmemBytes = kWideDyn;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  attr[1].id = cudaLaunchAttributeClusterDimension;
  attr[1].val.clusterDim.x = 1;
  attr[1].val.clusterDim.y = CL;
  attr[1].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = CL > 1 ? 2 : 1;
  static const bool debug = getenv("BBB_DEBUG_WIDE") != nullptr;
  if (debug) {
    static bool said = false;
    if (!said) {
      said = true;
      int n = -1;
      cfg.attrs = attr + 1;      // (the occupancy query takes the cluster attribute only)
      cfg.numAttrs = CL > 1 ? 1 : 0;
      cudaOccupancyMaxActiveClusters(&n, kern, &cfg);
      fprintf(stderr, "[bbb] wide kernel: clusters of %d, %d co-resident clusters on this device, grid (%u, %u, %u)\n", CL, n,
              grid.x, grid.y, grid.z);
      cfg.attrs = attr;
      cfg.numAttrs = CL > 1 ? 2 : 1;
    }
  }
  BBB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, tm, a));
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}

template <bool kDgrad, bool kLogProb>
int launch_wide(const LinArgs &a, cudaStream_t st) {
  CUtensorMap tm;
  if (kDgrad) {
    if (int r = tma::make_map(&tm, a.dy, a.out, a.B, a.S, BK, XH, tma::kSw128)) return r;
  } else {
    if (int r = tma::make_map(&tm, a.x, a.in, a.B, a.x_sstride ? a.S : 1, BK, XH, tma::kSw128)) return r;
  }
  const int n_bt = cdiv_w(a.B, NBT);
  dim3 grid(cdiv_w(kDgrad ? a.in : a.out, BM), n_bt, (unsigned)a.S);
  // (clusters of 8 -- 15 co-resident on a B200 -- were tried for the energy they would save and did not complete: not
  // instantiated)
  if (n_bt % 4 == 0) return launch_wide_cl<kDgrad, kLogProb, 4>(tm, a, grid, st);
  if (n_bt % 2 == 0) return launch_wide_cl<kDgrad, kLogProb, 2>(tm, a, grid, st);
  return launch_wide_cl<kDgrad, kLogProb, 1>(tm, a, grid, st);
}

}  // namespace

int launch_linear_fwd_wide(const LinArgs &a, cudaStream_t st) {
  if (a.flags & BBB_F_LOGPROB) return launch_wide<false, true>(a, st);
  return launch_wide<false, false>(a, st);
}
int launch_linear_dgrad_wide(const LinArgs &a, cudaStream_t st) { return launch_wide<true, false>(a, st); }

}  // namespace bbb
