// Network-level C-ABI entry points (include/bbb.h: bbb_mlp_supported / bbb_mlp_fwd / bbb_mlp_bwd): one call runs every
// layer of a weight-sampling BBB MLP for all S Monte-Carlo samples -- the body of BayesianNetwork.sample_elbo
// (networks.py:192-209) and of the autograd backward it triggers -- on the TMA-fed tcgen05 kernels of
// bbb_mlp_fwd.cu / bbb_mlp_bwd.cu, with the head (last layer + likelihood + ELBO assembly) on bbb_head.cu.
#include <mutex>
#include <string>
#include <vector>
#include <string.h>

#include "bbb_kernels.h"
#include "bbb_mlp.h"
#include "bbb_tma.cuh"

using namespace bbb;

namespace bbb {
namespace {
unsigned long long *g_timeline = nullptr;
int g_timeline_launch = 0;
}
// (every launch gets its own 160 x 16 slice of the buffer, 8 slices, in launch order)
unsigned long long *peer_timeline() { return g_timeline ? g_timeline + (size_t)8 * 2560 : nullptr; }
unsigned long long *debug_timeline() { return g_timeline ? g_timeline + (size_t)(g_timeline_launch++ % 8) * 2560 : nullptr; }
}  // namespace bbb

// debug aid (tools/kernel_timeline.py): every CTA of the NEXT network-level kernels writes 16 globaltimer stamps into buf
extern "C" int bbb_debug_set_timeline(unsigned long long *buf) {
  bbb::g_timeline = buf;
  bbb::g_timeline_launch = 0;
  return BBB_OK;
}

namespace bbb {
namespace tma {
EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &p, 12000, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}
}  // namespace tma
}  // namespace bbb

// ---- diagnostic: device time of every kernel launched by the network-level calls ------------------------------------
// (bench.py's roofline: the dominant kernel's duration, measured with CUDA events on the launching stream)
namespace {
struct TimedLaunch { char name[48]; cudaEvent_t e0, e1; };
std::mutex g_tmu;
bool g_timing = false;
std::vector<TimedLaunch> g_timed;

struct ScopedTimer {
  bool on = false;
  size_t idx = 0;
  cudaStream_t st;
  ScopedTimer(const char *fmt, long long a, long long b, cudaStream_t s) : st(s) {
    std::lock_guard<std::mutex> lk(g_tmu);
    if (!g_timing) return;
    TimedLaunch t{};
    snprintf(t.name, sizeof t.name, fmt, a, b);
    if (cudaEventCreate(&t.e0) != cudaSuccess || cudaEventCreate(&t.e1) != cudaSuccess) return;
    cudaEventRecord(t.e0, st);
    g_timed.push_back(t);
    idx = g_timed.size() - 1;
    on = true;
  }
  ~ScopedTimer() {
    if (!on) return;
    std::lock_guard<std::mutex> lk(g_tmu);
    if (idx < g_timed.size()) cudaEventRecord(g_timed[idx].e1, st);
  }
};
}  // namespace

extern "C" int bbb_timing_enable(int32_t on) {
  std::lock_guard<std::mutex> lk(g_tmu);
  for (auto &t : g_timed) { cudaEventDestroy(t.e0); cudaEventDestroy(t.e1); }
  g_timed.clear();
  g_timing = on != 0;
  return BBB_OK;
}

extern "C" int bbb_timing_report(char *buf, int64_t buf_bytes) {
  BBB_CHECK_ARG(buf && buf_bytes >= 64, "buffer too small");
  BBB_CHECK_CUDA(cudaDeviceSynchronize());
  std::lock_guard<std::mutex> lk(g_tmu);
  std::vector<std::string> names;
  std::vector<double> ms;
  std::vector<int> cnt;
  for (auto &t : g_timed) {
    float v = 0.0f;
    if (cudaEventElapsedTime(&v, t.e0, t.e1) != cudaSuccess) continue;
    size_t k = 0;
    while (k < names.size() && names[k] != t.name) ++k;
    if (k == names.size()) { names.push_back(t.name); ms.push_back(0.0); cnt.push_back(0); }
    ms[k] += v; cnt[k] += 1;
  }
  std::string out = "{";
  for (size_t k = 0; k < names.size(); ++k) {
    char item[128];
    snprintf(item, sizeof item, "%s\"%s\": [%.6f, %d]", k ? ", " : "", names[k].c_str(), ms[k], cnt[k]);
    out += item;
  }
  out += "}";
  if ((int64_t)out.size() + 1 > buf_bytes) return fail(BBB_EINVAL, "bbb_timing_report: buffer too small");
  memcpy(buf, out.c_str(), out.size() + 1);
  return BBB_OK;
}

namespace {

inline bool al16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// the shapes the network-level kernels cover: TF32 mode, batch <= 128, every hidden width a multiple of 4, a head
// (out <= 16) on top whose input width is a multiple of 4
bool dims_supported(const int64_t *dims, int n_layers, int64_t S, int64_t B) {
  if (n_layers < 2 || S < 1 || S > 65535 || B < 1 || B > 128) return false;
  const int groups = (int)((S + 1) / 2);
  for (int l = 0; l + 1 < n_layers; ++l) {
    const int64_t in = dims[l], out = dims[l + 1];
    if (in < 4 || in % 4 || out < 4 || out % 4) return false;
    if (((out + 127) / 128) * groups > sm_count() || in * out / 4 >= ((int64_t)1 << 32)) return false;
  }
  const int64_t in = dims[n_layers - 1], out = dims[n_layers];
  return out >= 1 && out <= 16 && in % 4 == 0 && in >= 4 && in <= 8192;
}

MlpLayerDesc make_desc(const bbb_mlp_layer &L, const float *x, bool x_shared) {
  MlpLayerDesc d{};
  d.x = x; d.x_shared = x_shared;
  d.w_mu = L.w_mu; d.w_rho = L.w_rho; d.b_mu = L.b_mu; d.b_rho = L.b_rho; d.eps_w = L.eps_w; d.eps_b = L.eps_b;
  d.in = L.in; d.out = L.out;
  d.y = L.y;
  d.dz = L.dz; d.g_w_mu = L.g_w_mu; d.g_w_rho = L.g_w_rho; d.g_b_mu = L.g_b_mu; d.g_b_rho = L.g_b_rho;
  return d;
}

}  // namespace

extern "C" int bbb_mlp_supported(const int64_t *dims, int32_t n_layers, int64_t S, int64_t B, int32_t flags) {
  if (!dims || !(flags & BBB_F_TF32)) return 0;
  return dims_supported(dims, n_layers, S, B) && tma::encode_fn() != nullptr ? 1 : 0;
}

extern "C" int bbb_mlp_fwd(const bbb_mlp_layer *layers, int32_t n_layers, const float *x, int64_t S, int64_t B,
                           const bbb_rng *rng, const bbb_prior *prior, int32_t flags, int32_t nll_kind,
                           const void *target, float sigma, float grad_scale, float *d_out, double *logp, double *logq,
                           double *nll, float beta, const float *beta_dev, float *out4, uint32_t *done_counter,
                           void *stream) {
  BBB_CHECK_ARG(layers && x && n_layers >= 2 && n_layers <= 64, "null pointer or bad layer count");
  BBB_CHECK_ARG(flags & BBB_F_TF32, "the network-level kernels are the tcgen05 kind::tf32 path: pass BBB_F_TF32");
  const bool sample = flags & BBB_F_SAMPLE, lpq = flags & BBB_F_LOGPROB;
  BBB_CHECK_ARG(!lpq || (prior && logp && logq), "log-prob outputs and prior required with BBB_F_LOGPROB");
  BBB_CHECK_ARG(!prior || prior->kind == BBB_PRIOR_GAUSSIAN || prior->kind == BBB_PRIOR_MIXTURE, "bad prior kind");
  int64_t dims[65];
  dims[0] = layers[0].in;
  for (int l = 0; l < n_layers; ++l) {
    const bbb_mlp_layer &L = layers[l];
    BBB_CHECK_ARG(L.w_mu && L.b_mu && L.y, "null layer pointer");
    BBB_CHECK_ARG(!(sample || lpq) || (L.w_rho && L.b_rho), "rho pointers required");
    BBB_CHECK_ARG(!sample || (L.eps_w && L.eps_b) || (!L.eps_w && !L.eps_b && rng), "give both eps pointers or an rng");
    BBB_CHECK_ARG(L.in == dims[l], "layer widths do not chain");
    dims[l + 1] = L.out;
  }
  if (!dims_supported(dims, n_layers, S, B) || !tma::encode_fn())
    return fail(BBB_EUNSUPPORTED, "bbb_mlp_fwd: needs batch <= 128, hidden widths that are multiples of 4 and a head of at "
                                  "most 16 outputs (see bbb_mlp_supported)");
  cudaStream_t st = (cudaStream_t)stream;
  PriorDev pd{};
  if (prior) pd = make_prior_dev(prior);
  const float *inp = x;
  for (int l = 0; l + 1 < n_layers; ++l) {
    bbb_rng r = rng ? *rng : bbb_rng{};
    r.layer = (uint32_t)l;
    MlpLayerDesc d = make_desc(layers[l], inp, l == 0);
    if (!mlp_fwd_layer_supported(d, S, B))
      return fail(BBB_EUNSUPPORTED, "bbb_mlp_fwd: layer %d needs 16-byte aligned tensors", l);
    {
      ScopedTimer tm("mlp_fwd[%lldx%lld]", (long long)d.in, (long long)d.out, st);
      const int32_t lf = (flags & (BBB_F_SAMPLE | BBB_F_LOGPROB | BBB_F_TF32)) | (l > 0 ? BBB_F_RELU_IN : 0);
      if (int rc = launch_mlp_fwd_layer(d, S, B, make_rng_dev(rng ? &r : nullptr), pd, lf, logp, logq, st)) return rc;
    }
    inp = layers[l].y;
  }
  const bbb_mlp_layer &H = layers[n_layers - 1];
  bbb_rng r = rng ? *rng : bbb_rng{};
  r.layer = (uint32_t)(n_layers - 1);
  const int32_t head_flags = (flags & (BBB_F_SAMPLE | BBB_F_LOGPROB)) | BBB_F_RELU_IN;    // its input is a pre-activation
  ScopedTimer tm("head_fwd[%lldx%lld]", (long long)H.in, (long long)H.out, st);
  return bbb_head_fwd(inp, B * H.in, H.w_mu, H.w_rho, H.b_mu, H.b_rho, H.eps_w, H.eps_b, rng ? &r : nullptr, prior, S, B,
                      H.in, H.out, head_flags, nll_kind, target, sigma, grad_scale, H.y, d_out, logp, logq, nll, beta,
                      beta_dev, out4, done_counter, stream);
}

extern "C" int bbb_mlp_bwd(const bbb_mlp_layer *layers, int32_t n_layers, const float *x, int64_t S, int64_t B,
                           const bbb_rng *rng, const bbb_prior *prior, int32_t flags, float gp, float gq,
                           const float *gp_dev, const float *gq_dev, int64_t g_dev_stride, const float *out_scale_dev,
                           void *stream) {
  BBB_CHECK_ARG(layers && x && n_layers >= 2 && n_layers <= 64, "null pointer or bad layer count");
  BBB_CHECK_ARG(flags & BBB_F_TF32, "the network-level kernels are the tcgen05 kind::tf32 path: pass BBB_F_TF32");
  BBB_CHECK_ARG(g_dev_stride == 0 || g_dev_stride == 1, "g_dev_stride must be 0 or 1");
  BBB_CHECK_ARG(((gp == 0.0f) && !gp_dev) || prior, "prior required when gp != 0");
  const bool sample = flags & BBB_F_SAMPLE;
  int64_t dims[65];
  dims[0] = layers[0].in;
  for (int l = 0; l < n_layers; ++l) {
    const bbb_mlp_layer &L = layers[l];
    BBB_CHECK_ARG(L.w_mu && L.w_rho && L.b_mu && L.b_rho && L.dz, "null layer pointer");
    BBB_CHECK_ARG(L.g_w_mu && L.g_w_rho && L.g_b_mu && L.g_b_rho, "null gradient pointer");
    BBB_CHECK_ARG(!sample || (L.eps_w && L.eps_b) || (!L.eps_w && !L.eps_b && rng), "give both eps pointers or an rng");
    BBB_CHECK_ARG(L.in == dims[l], "layer widths do not chain");
    BBB_CHECK_ARG(l + 1 == n_layers || L.y, "hidden layers need their stored pre-activation");
    dims[l + 1] = L.out;
  }
  if (!dims_supported(dims, n_layers, S, B) || !tma::encode_fn())
    return fail(BBB_EUNSUPPORTED, "bbb_mlp_bwd: needs batch <= 128, hidden widths that are multiples of 4 and a head of at "
                                  "most 16 outputs (see bbb_mlp_supported)");
  cudaStream_t st = (cudaStream_t)stream;
  PriorDev pd{};
  if (prior) pd = make_prior_dev(prior);
  const int32_t keep = flags & (BBB_F_SAMPLE | BBB_F_TF32 | BBB_F_ACCUM);
  // the head: dz of the last hidden layer = (d_out W_s) (y > 0), added into its zero-filled buffer
  {
    const bbb_mlp_layer &H = layers[n_layers - 1], &P = layers[n_layers - 2];
    bbb_rng r = rng ? *rng : bbb_rng{};
    r.layer = (uint32_t)(n_layers - 1);
    ScopedTimer tm("head_bwd[%lldx%lld]", (long long)H.in, (long long)H.out, st);
    if (int rc = bbb_linear_bwd(H.dz, nullptr, P.y, B * H.in, H.w_mu, H.w_rho, H.b_mu, H.b_rho, H.eps_w, H.eps_b,
                                rng ? &r : nullptr, prior, S, B, H.in, H.out,
                                keep | BBB_F_RELU_IN | BBB_F_DX_PREACT | BBB_F_OUT_ZEROED, gp, gq, gp_dev, gq_dev,
                                g_dev_stride, out_scale_dev, P.dz, H.g_w_mu, H.g_w_rho, H.g_b_mu, H.g_b_rho, stream))
      return rc;
  }
  for (int l = n_layers - 2; l >= 0; --l) {
    bbb_rng r = rng ? *rng : bbb_rng{};
    r.layer = (uint32_t)l;
    MlpLayerDesc d = make_desc(layers[l], l > 0 ? layers[l - 1].y : x, l == 0);
    d.dx = l > 0 ? layers[l - 1].dz : nullptr;
    if (!mlp_bwd_layer_supported(d, S, B))
      return fail(BBB_EUNSUPPORTED, "bbb_mlp_bwd: layer %d needs 16-byte aligned tensors", l);
    ScopedTimer tm("mlp_bwd[%lldx%lld]", (long long)d.in, (long long)d.out, st);
    if (int rc = launch_mlp_bwd_layer(d, S, B, make_rng_dev(rng ? &r : nullptr), pd, keep | (l > 0 ? BBB_F_RELU_IN : 0), gp, gq, gp_dev, gq_dev,
                                      (int)g_dev_stride, out_scale_dev, st))
      return rc;
  }
  return BBB_OK;
}
