// Fused backward of the weight-sampling Bayesian linear layer for batches of at most 128 rows (tcgen05 kind::tf32):
// ONE kernel per layer does wgrad, the analytic mu/rho-gradient epilogue and dgrad, and regenerates eps once.
//
// A CTA owns a block of the weight matrix: rows [o_t0, o_t0 + rows) of one output-row tile (<= 128 rows) and a
// 4-aligned column range [i_lo, i_hi) of at most 88 columns.  Per Monte-Carlo sample it
//   1. stages the activation tiles in shared memory in their NATURAL row-major orientation, as stacked
//      [128 batch rows][128 B] swizzled regions:  dz_s[b][o_t0 .. +128)  and  x_s[b][i_lo .. +96);
//   2. MMA1  G[o][i] = sum_b dz[b][o] x[b][i]    -- both operands MN-major (the batch is K), accumulator in TMEM;
//   3. drains G to shared memory in the layout of an MN-major operand tile  Wt[o][i];
//   4. epilogue, one weight quad per thread-iteration, coalesced along i: regenerate eps (Philox), w = mu + sigma eps,
//      t = G - gp w R(w);  grad_mu += t;  grad_rho += sigmoid(rho) (t eps - gq / sigma)   (sums kept in registers
//      across samples), and overwrite the G quad IN PLACE by the TF32 weights w -- the tile is now the B operand
//      of dgrad, zero outside the CTA's own block;
//   5. MMA2  dX[b][i] = sum_o dz[b][o] Wt[o][i]  -- A = the same dz tile read K-major, B = Wt MN-major;
//   6. drains dX, optionally multiplied by (x > 0) (the ReLU that produced this layer's input), and adds the
//      partial sum over its o rows into dx with red.global.add.v4.f32.
// No transposes anywhere: a [rows = batch][32 floats] region is an MN-major operand as it stands.  MN-major TF32
// operands use the SWIZZLE_128B_BASE32B format and K-major ones SWIZZLE_128B (bbb_tc.cuh), so the dz tile is stored
// twice, once per swizzle, from the same registers.  eps is generated once per weight and sample for the whole
// backward, and W never leaves the SM.
//
// Work split: the output rows are cut into equal tiles of T_o <= 128 rows, each tile's input columns are divided
// evenly (granularity one quad) over grid.x CTAs; grid.x * grid.y is about one CTA per SM (launch_bwd_fused).
#include "bbb_tc_tiles.cuh"

namespace bbb {
namespace {

using namespace tc;
using namespace tcx;

constexpr int FT = 512;              // threads per CTA (16 warps, one CTA per SM)
constexpr int REG = 128 * 128;       // bytes of one [128 rows][128 B] swizzled region
constexpr int DZ_REGS = 4;           // dz tile: up to 128 o columns (only the regions the row tile needs are staged)
constexpr int XW_MAX = 3;            // x tile / Wt tile: XWR regions of 32 i columns, XWR = 1, 2 or 3 (template)
constexpr int QMAX = 6;              // weight quads per thread: 512 * 6 * 4 >= 128 * 88
constexpr uint32_t kFusedTmemCols = 256;  // G: columns [0, 32 XWR), dX: columns [128, 128 + 32 XWR)
// widest column range a CTA may own with XWR regions: the window is 32 XWR wide and starts at the range's first
// column, so the whole window could be owned; 8 columns are kept free so that ranges stay comfortably inside
constexpr int wmax_of(int xwr) { return 32 * xwr - 8; }
constexpr int fused_dyn(int xwr) { return (2 * DZ_REGS + 2 * xwr) * REG + 1024; }  // dz (MN) | dz (K) | x | Wt
static_assert(FT * QMAX * 4 >= 128 * wmax_of(XW_MAX), "every own weight needs a thread slot");

struct FCtl {
  uint64_t bar;
  uint32_t tmem_base;
};

// address of float4 column `col4` of row `row` in an MN-major (BASE32B) / a K-major (SWIZZLE_128B) tile
__device__ __forceinline__ uint8_t *mn_ptr(uint8_t *tile, int row, int col4) {
  return tile + (col4 >> 3) * REG + mn32_off(row, col4 & 7);
}
__device__ __forceinline__ uint8_t *k_ptr(uint8_t *tile, int row, int col4) {
  return tile + (col4 >> 3) * REG + sw128_off(row, col4 & 7);
}

template <bool kDx, int XWR>
__global__ void __launch_bounds__(FT, 1) bwd_fused_kernel(const LinArgs a_in, int T_o) {
  constexpr int NWIN = 32 * XWR;  // MMA N
  extern __shared__ uint8_t dsm[];
  __shared__ FCtl ctl;
  __shared__ float csum_part[2][128];   // (the dynamic tiles leave 2 KB of the 227 KB)
  LinArgs a = a_in;
  uint8_t *dz_t = align1024(dsm), *dzk_t = dz_t + DZ_REGS * REG, *x_t = dzk_t + DZ_REGS * REG, *w_t = x_t + XWR * REG;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool sample = a.flags & BBB_F_SAMPLE, relu = a.flags & BBB_F_RELU_IN, wgrad = !(a.flags & BBB_F_NO_WGRAD);
  const bool dx_preact = a.flags & BBB_F_DX_PREACT, accum = a.flags & BBB_F_ACCUM;
  const int B = (int)a.B;

  // this CTA's block
  const int64_t o_t0 = (int64_t)blockIdx.y * T_o;
  const int rows = (int)min((int64_t)T_o, a.out - o_t0);
  const int nq_i = (int)(a.in >> 2);
  const int q_lo = (int)((int64_t)blockIdx.x * nq_i / gridDim.x), q_hi = (int)((int64_t)(blockIdx.x + 1) * nq_i / gridDim.x);
  const int tq = q_hi - q_lo;                      // own quads per row (<= 22)
  const int64_t i_lo = (int64_t)q_lo * 4;
  const int nquad = rows * tq;
  const bool bias_cta = blockIdx.x == 0;
  const int nzr = (rows + 31) >> 5;                // dz regions (32 o columns each) this row tile needs
  const int st_row = tid >> 3, st_chunk = tid & 7; // staging: rows st_row + 64 h, chunk st_chunk of every region
  const uint32_t st_mn = mn32_off(st_row, st_chunk), st_k = sw128_off(st_row, st_chunk);

  if (warp == 0) tmem_alloc(smem_u32(&ctl.tmem_base), kFusedTmemCols);
  if (tid == 32) {
    mbar_init(smem_u32(&ctl.bar), 1);
    mbar_fence_init();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  pdl_wait();              // everything above is local; from here on global memory of earlier kernels is read
  rng_resolve(a.rng);
  const uint32_t tmem = ctl.tmem_base, tmem_g = tmem, tmem_dx = tmem + 128;
  constexpr uint32_t idesc1 = idesc_tf32_major(128, NWIN, 1, 1);  // MMA1: A = dz (MN-major), B = x (MN-major)
  constexpr uint32_t idesc2 = idesc_tf32_major(128, NWIN, 0, 1);  // MMA2: A = dz (K-major),  B = Wt (MN-major)
  const float osc = a.out_scale_dev ? __ldg(a.out_scale_dev) : 1.0f;
  const float dxs = ((a.flags & BBB_F_SCALE_DX) && a.out_scale_dev) ? osc : 1.0f;

  float gm[QMAX][4], gr[QMAX][4];
#pragma unroll
  for (int j = 0; j < QMAX; ++j)
#pragma unroll
    for (int c = 0; c < 4; ++c) gm[j][c] = gr[j][c] = 0.0f;
  float gbm = 0.0f, gbr = 0.0f;
  uint32_t phase = 0;

  for (int s = 0; s < a.S; ++s) {
    // ---- 1. stage dz_s [128 b][32 nzr o] and x_s [128 b][32 XWR i]: all loads first, then the swizzled stores.
    // Thread t handles rows t/8 + 64 h, 16-byte chunk t%8 of every region; rows r and r + 64 share (r & 7), so the
    // two shared-memory offsets (one per swizzle) are per-thread constants and the loops carry no index arithmetic.
    {
      const float *dys = a.dy + (int64_t)s * a.B * a.out + o_t0 + st_chunk * 4;
      const float *mks = a.mask ? a.mask + (int64_t)s * a.B * a.out + o_t0 + st_chunk * 4 : nullptr;
      float4 zv[2 * DZ_REGS];
#pragma unroll
      for (int g = 0; g < DZ_REGS; ++g) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (g < nzr) {
            const int b = st_row + 64 * h;
            const int64_t o = o_t0 + g * 32 + st_chunk * 4;
            if (a.vec_out) {
              const bool ok = b < B && o < a.out;
              const float4 t = __ldg(reinterpret_cast<const float4 *>(ok ? dys + (int64_t)b * a.out + g * 32 : a.dy));
              v = ok ? t : v;
              if (mks) v = mask4(v, ok ? __ldg(reinterpret_cast<const float4 *>(mks + (int64_t)b * a.out + g * 32)) : v);
            } else {
              v = ld_row4(a.dy + (int64_t)s * a.B * a.out, b, o, a.B, a.out, false);
              if (mks) v = mask4(v, ld_row4(a.mask + (int64_t)s * a.B * a.out, b, o, a.B, a.out, false));
            }
          }
          zv[2 * g + h] = v;
        }
      }
      const bool load_x = s == 0 || a.x_sstride != 0;
      float4 xv[2 * XWR];
      if (load_x) {
        const float *xs = a.x + (int64_t)s * a.x_sstride + i_lo + st_chunk * 4;
#pragma unroll
        for (int g = 0; g < XWR; ++g) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int b = st_row + 64 * h, c4 = g * 8 + st_chunk;
            const bool ok = b < B && c4 < tq;          // columns beyond the own range: zero
            const float4 t = __ldg(reinterpret_cast<const float4 *>(ok ? xs + (int64_t)b * a.in + g * 32 : a.x));
            xv[2 * g + h] = ok ? t : make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
      }
#pragma unroll
      for (int g = 0; g < DZ_REGS; ++g) {
        if (g < nzr) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            *reinterpret_cast<float4 *>(dz_t + g * REG + st_mn + h * 8192) = zv[2 * g + h];
            if (kDx) *reinterpret_cast<float4 *>(dzk_t + g * REG + st_k + h * 8192) = zv[2 * g + h];
          }
        }
      }
      if (load_x) {
#pragma unroll
        for (int g = 0; g < XWR; ++g) {
#pragma unroll
          for (int h = 0; h < 2; ++h)
            *reinterpret_cast<float4 *>(x_t + g * REG + st_mn + h * 8192) = relu ? relu4(xv[2 * g + h]) : xv[2 * g + h];
        }
      }
    }
    fence_proxy_async_smem();
    __syncthreads();

    // ---- 2. MMA1: G[o][i] = sum_b dz[b][o] x[b][i], K = batch in steps of 8 rows -------------------------------
    if (tid == 0) {
      tc_fence_after_sync();
      const int nk = (B + 7) >> 3;
      for (int k8 = 0; k8 < nk; ++k8)
        mma_tf32(tmem_g, smem_desc_mn32(smem_u32(dz_t) + k8 * 1024, REG), smem_desc_mn32(smem_u32(x_t) + k8 * 1024, REG),
                 idesc1, k8 > 0 ? 1u : 0u);
      mma_commit(smem_u32(&ctl.bar));
    }
    // the first weight quad's parameters travel while the tensor pipe works
    float4 nmu = make_float4(0.f, 0.f, 0.f, 0.f), nrho = nmu;
    if (tid < nquad) {
      const int r = tid / tq;
      const int64_t e = (o_t0 + r) * a.in + i_lo + (int64_t)(tid - r * tq) * 4;
      nmu = __ldg(reinterpret_cast<const float4 *>(a.w_mu + e));
      nrho = __ldg(reinterpret_cast<const float4 *>(a.w_rho + e));
    }
    mbar_wait_parked(smem_u32(&ctl.bar), phase);
    phase ^= 1u;
    tc_fence_after_sync();

    // ---- 3. G: TMEM [lane = o][column = i] -> Wt layout in shared memory ------------------------------------------
    {
      const int o_r = (warp & 3) * 32 + lane, cg = warp >> 2;   // 4 column groups of NWIN / 4
#pragma unroll
      for (int c0 = 0; c0 < NWIN / 4; c0 += 8) {
        const int col = cg * (NWIN / 4) + c0;
        float v[8];
        tmem_ld8(tmem_g + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)col, v);
        *reinterpret_cast<float4 *>(mn_ptr(w_t, o_r, col >> 2)) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4 *>(mn_ptr(w_t, o_r, (col >> 2) + 1)) = make_float4(v[4], v[5], v[6], v[7]);
      }
    }
    tc_fence_before_sync();
    __syncthreads();

    // ---- 4. epilogue over the CTA's own quads; G quad -> w quad in place ------------------------------------------
    const float gps = a.gp * (a.gp_dev ? __ldg(a.gp_dev + s * a.g_dev_stride) : 1.0f);
    const float gqs = a.gq * (a.gq_dev ? __ldg(a.gq_dev + s * a.g_dev_stride) : 1.0f);
#pragma unroll
    for (int j = 0; j < QMAX; ++j) {
      const int q = tid + FT * j;
      if (q < nquad) {
        const float4 cmu = nmu, crho = nrho;
        const int r = q / tq, iq = q - r * tq;
        const int64_t e = (o_t0 + r) * a.in + i_lo + (int64_t)iq * 4;
        if (j + 1 < QMAX && q + FT < nquad) {
          const int rn = (q + FT) / tq;
          const int64_t en = (o_t0 + rn) * a.in + i_lo + (int64_t)(q + FT - rn * tq) * 4;
          nmu = __ldg(reinterpret_cast<const float4 *>(a.w_mu + en));
          nrho = __ldg(reinterpret_cast<const float4 *>(a.w_rho + en));
        }
        Quad qd;
        qd.mu[0] = cmu.x; qd.mu[1] = cmu.y; qd.mu[2] = cmu.z; qd.mu[3] = cmu.w;
        qd.rho[0] = crho.x; qd.rho[1] = crho.y; qd.rho[2] = crho.z; qd.rho[3] = crho.w;
        float sgm[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) softplus_sigmoid_fast(qd.rho[c], qd.sg[c], sgm[c]);
        float ep[4], w[4];
        sample_quad(a, s, e, qd, sample, ep, w);
        float4 *slot = reinterpret_cast<float4 *>(mn_ptr(w_t, r, iq));
        if (wgrad) {
          const float4 G = *slot;
          const float Gv[4] = {G.x, G.y, G.z, G.w};
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            float t = Gv[c];
            if (gps != 0.0f) t = fmaf(-gps * w[c], prior_R_fast(a.prior, w[c]), t);
            gm[j][c] += t;
            gr[j][c] += sgm[c] * fmaf(t, ep[c], -gqs * __fdividef(1.0f, qd.sg[c]));
          }
        }
        if (kDx) *slot = make_float4(to_tf32(w[0]), to_tf32(w[1]), to_tf32(w[2]), to_tf32(w[3]));
      }
    }
    if (kDx) {  // everything in the 128 x 96 window that is not an own weight must not contribute to dX
      const int r_up = (rows + 7) & ~7;   // MMA2 reads Wt rows in steps of 8
      for (int idx = tid; idx < r_up * (NWIN / 4); idx += FT) {
        const int r = idx / (NWIN / 4), c4 = idx - r * (NWIN / 4);
        if (r >= rows || c4 >= tq) *reinterpret_cast<float4 *>(mn_ptr(w_t, r, c4)) = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    // bias gradients, part 1: column sums of the dz tile, 2 row groups x 128 columns over the first 256 threads
    if (wgrad && bias_cta && tid < 256) {
      const int o_l = tid & 127, grp = tid >> 7;
      const uint8_t *zp = dz_t + (o_l >> 5) * REG + (o_l & 3) * 4;
      const int b_end = min(B, grp * 64 + 64);
      float part = 0.0f;
#pragma unroll 8
      for (int b = grp * 64; b < b_end; ++b) part += *reinterpret_cast<const float *>(zp + mn32_off(b, (o_l >> 2) & 7));
      csum_part[grp][o_l] = part;
    }
    // part 2 (after the next CTA-wide barrier, overlapping MMA2): prior/posterior terms of the bias row
    auto bias_finish = [&]() {
      if (wgrad && bias_cta && tid < rows) {
        const float colsum = csum_part[0][tid] + csum_part[1][tid];
        const int64_t o = o_t0 + tid;
        float bv, sg, ep;
        bias_elem(a, s, o, sample, true, bv, sg, ep);
        float t = colsum;
        if (gps != 0.0f) t = fmaf(-gps * bv, prior_R(a.prior, bv), t);
        gbm += t;
        gbr += -expm1f(-sg) * (t * ep - gqs / sg);
      }
    };

    if (kDx) {
      fence_proxy_async_smem();
      __syncthreads();
      // ---- 5. MMA2: dX[b][i] = sum_o dz[b][o] Wt[o][i], K = o in steps of 8 rows of Wt ---------------------------
      if (tid == 0) {
        tc_fence_after_sync();
        const int nk = (rows + 7) >> 3;
        for (int k8 = 0; k8 < nk; ++k8)
          mma_tf32(tmem_dx, smem_desc_sw128(smem_u32(dzk_t) + (k8 >> 2) * REG + (k8 & 3) * 32),
                   smem_desc_mn32(smem_u32(w_t) + k8 * 1024, REG), idesc2, k8 > 0 ? 1u : 0u);
        mma_commit(smem_u32(&ctl.bar));
      }
      bias_finish();
      mbar_wait_parked(smem_u32(&ctl.bar), phase);
      phase ^= 1u;
      tc_fence_after_sync();
      // ---- 6. dX: TMEM [lane = b][column = i] -> (x > 0) mask -> red.add into dx --------------------------------
      {
        const int b = (warp & 3) * 32 + lane, cg = warp >> 2;
        float *drow = a.dx + ((int64_t)s * a.B + b) * a.in + i_lo;
#pragma unroll
        for (int c0 = 0; c0 < NWIN / 4; c0 += 8) {
          const int col = cg * (NWIN / 4) + c0;
          float v[8];
          tmem_ld8(tmem_dx + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)col, v);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int c4 = (col >> 2) + h;
            if (b < B && c4 < tq) {
              float4 d = make_float4(dxs * v[4 * h], dxs * v[4 * h + 1], dxs * v[4 * h + 2], dxs * v[4 * h + 3]);
              if (dx_preact) d = mask4(d, *reinterpret_cast<const float4 *>(mn_ptr(x_t, b, c4)));
              red_add_v4(drow + c4 * 4, d);
            }
          }
        }
      }
      tc_fence_before_sync();
    } else if (wgrad && bias_cta) {
      __syncthreads();
      bias_finish();
    }
    __syncthreads();  // the tiles and the accumulators are reused by the next sample
  }

  pdl_launch_dependents();   // the sample loop is done: let the next kernel of the chain become resident
  // ---- parameter gradients ----------------------------------------------------------------------------------------
  if (wgrad) {
#pragma unroll
    for (int j = 0; j < QMAX; ++j) {
      const int q = tid + FT * j;
      if (q < nquad) {
        const int r = q / tq, iq = q - r * tq;
        const int64_t e = (o_t0 + r) * a.in + i_lo + (int64_t)iq * 4;
        float g1[4], g2[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) { g1[c] = osc * gm[j][c]; g2[c] = osc * gr[j][c]; }
        float4 *pm = reinterpret_cast<float4 *>(a.g_w_mu + e), *pr = reinterpret_cast<float4 *>(a.g_w_rho + e);
        float4 om = make_float4(0.f, 0.f, 0.f, 0.f), orr = om;
        if (accum) { om = *pm; orr = *pr; }
        *pm = make_float4(g1[0] + om.x, g1[1] + om.y, g1[2] + om.z, g1[3] + om.w);
        *pr = make_float4(g2[0] + orr.x, g2[1] + orr.y, g2[2] + orr.z, g2[3] + orr.w);
      }
    }
    if (bias_cta && tid < rows) {
      const int64_t o = o_t0 + tid;
      a.g_b_mu[o] = accum ? fmaf(osc, gbm, a.g_b_mu[o]) : osc * gbm;
      a.g_b_rho[o] = accum ? fmaf(osc, gbr, a.g_b_rho[o]) : osc * gbr;
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, kFusedTmemCols);
}

inline int cdiv_i(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

}  // namespace

bool linear_bwd_fused_supported(const LinArgs &a) {
  return a.vec_in && a.in >= 4 && a.out >= 1 && a.B >= 1 && a.B <= 128 && a.S >= 1;
}

namespace {
template <bool kDx, int XWR>
int launch_one(const LinArgs &a, dim3 grid, int T_o, cudaStream_t st) {
  BBB_CHECK_CUDA(cudaFuncSetAttribute(bwd_fused_kernel<kDx, XWR>, cudaFuncAttributeMaxDynamicSharedMemorySize, fused_dyn(XWR)));
  BBB_CHECK_CUDA(launch_pdl(bwd_fused_kernel<kDx, XWR>, grid, dim3(FT), fused_dyn(XWR), st, a, T_o));
  BBB_CHECK_LAUNCH();
  return BBB_OK;
}
}  // namespace

int launch_linear_bwd_fused(const LinArgs &a, cudaStream_t st) {
  const bool want_dx = !(a.flags & BBB_F_NO_DX);
  const int n_ot = cdiv_i(a.out, 128);
  const int T_o = ((cdiv_i(a.out, n_ot) + 3) / 4) * 4;         // equal row tiles; a multiple of 4 keeps dz loads vectorised
  const int nq_i = (int)(a.in / 4);
  int n_c = sm_count() / n_ot;                                       // about one CTA per SM
  const int need = cdiv_i(nq_i, wmax_of(XW_MAX) / 4);          // every column range must fit the widest window
  if (n_c < need) n_c = need;
  if (n_c > nq_i) n_c = nq_i;
  if (n_c < 1) n_c = 1;
  const int width = cdiv_i(nq_i, n_c) * 4;                     // widest own column range
  dim3 grid(n_c, cdiv_i(a.out, T_o));
  if (want_dx && !(a.flags & BBB_F_OUT_ZEROED)) {
    BBB_CHECK_CUDA(cudaMemsetAsync(a.dx, 0, sizeof(float) * (size_t)a.S * a.B * a.in, st));
    note_launch();
  }
  if (width <= wmax_of(1)) return want_dx ? launch_one<true, 1>(a, grid, T_o, st) : launch_one<false, 1>(a, grid, T_o, st);
  if (width <= wmax_of(2)) return want_dx ? launch_one<true, 2>(a, grid, T_o, st) : launch_one<false, 2>(a, grid, T_o, st);
  return want_dx ? launch_one<true, 3>(a, grid, T_o, st) : launch_one<false, 3>(a, grid, T_o, st);
}

}  // namespace bbb
