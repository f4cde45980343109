"""torch.autograd glue between the nn.Module mirror of the reference API and the C-ABI kernels.

Every function here launches libbbb.so kernels on the current CUDA stream through ctypes
(_lib.py); PyTorch only owns the buffers and the autograd tape.  Nothing here computes on
the CPU and nothing imports oracle/.

Layer level  : bayes_linear / lr_linear          (one launch fwd, two bwd; S = 1)
Network level: mlp_forward / mlp_forward_lr      (all S samples per launch, ReLU fused into the
                                                  consumer's operand load, differentiable outputs)
               fused_elbo / fused_elbo_lr        (the above + likelihood + ELBO assembly, loss only
                                                  differentiable: what sample_elbo[_lr] call)
"""
import ctypes as C

import torch

from . import _lib as L
from . import rng as R


def make_prior(prior_init, mixture_prior):
    """prior_init -> bbb_prior (networks.py:61-68; mixture sigmas are exp(log sigma))."""
    import math
    if mixture_prior:
        assert len(prior_init) == 3, "Scale Mixture Prior requires three values in prior initialisation"
        return L.Prior(L.PRIOR_MIXTURE, float(prior_init[0]), math.exp(prior_init[1]), math.exp(prior_init[2]))
    assert len(prior_init) == 1, "Gaussian Prior requires one value in prior initialisation"
    return L.Prior(L.PRIOR_GAUSSIAN, 0.0, float(prior_init[0]), 0.0)


def _rng(layer, seed, step, sample_base, step_dev):
    return L.Rng(seed, step, sample_base, layer, L.ptr(step_dev))


def _f32c(t):
    """fp32, contiguous, detached.  The common case (an fp32 contiguous tensor seen inside autograd.Function.forward /
    backward, where nothing is recorded) costs no torch op at all: the eager call path is host-bound, and three ops per
    parameter tensor per pass were a third of it."""
    if t.dtype is torch.float32 and t.is_contiguous():
        return t if not t.requires_grad or not torch.is_grad_enabled() else t.detach()
    return t.detach().to(torch.float32).contiguous()


# Called as hook(layer_index, flat_gradient_slice) right after a layer's backward kernel has been launched (from the
# thread autograd runs the backward on).  parallel.OverlappedAllReduce installs it so that a layer's mu/rho gradients
# travel over NVLink while the layers below are still being differentiated.
grad_ready_hook = None


# Persistent flat gradient buckets, keyed by the address of the flat parameter buffer they belong to
# (optim.PeerShardedAdam registers one that the other ranks can read over NVLink): the network-level backward of a
# network whose parameters live in that buffer writes its gradients there instead of into a fresh allocation.
# Values are (flat bucket, owner): owner() (a weakref, or None) is the optimiser whose parameters the bucket serves.
grad_buckets = {}


def _bucket_for(params):
    """The registered bucket of this network, or None.  The bucket is handed to autograd as the gradient tensors
    themselves, and autograd installs them as p.grad WITHOUT a copy; if a p.grad from an earlier backward is still
    alive (zero_grad(set_to_none=False), gradient accumulation) it may BE the bucket, and the next backward would
    overwrite it before AccumulateGrad adds the new gradient to it (a silent 2x).  So the bucket is only used when
    every parameter of its owner has p.grad None; otherwise the gradients go to a fresh allocation and the owner's
    step() copies them in."""
    entry = grad_buckets.get(params[0][0].data_ptr())
    if entry is None:
        return None
    bucket, owner = entry
    opt = owner() if owner is not None else None
    if opt is not None and any(q.grad is not None for g in opt.param_groups for q in g['params']):
        return None
    return bucket


def _alloc_grads(params):
    """Gradient buffers for every layer as consecutive views of ONE flat tensor, in parameter order, so a
    multi-GPU step can all-reduce them with a single collective and no copies (parallel.py)."""
    total = sum(t.numel() for p in params for t in p)
    bucket = _bucket_for(params)
    if bucket is not None and bucket.numel() >= total and bucket.device == params[0][0].device:
        flat = bucket[:total]
    else:
        flat = torch.empty(total, dtype=torch.float32, device=params[0][0].device)
    out, off = [], 0
    for p in params:
        g, start = [], off
        for t in p:
            g.append(flat[off:off + t.numel()].view(t.shape))
            off += t.numel()
        out.append(_LayerGrads(g, flat[start:off]))
    return out


class _LayerGrads(tuple):
    """(grad_w_mu, grad_w_rho, grad_b_mu, grad_b_rho) of one layer + the flat slice of the bucket they live in"""

    def __new__(cls, grads, flat):
        self = super().__new__(cls, grads)
        self.flat = flat
        return self


def _split_beta(beta):
    """beta as a python number, or as a device tensor (read on the device: CUDA-graph replay can then follow
    the reference's per-minibatch schedule).  Returns (host multiplier, device scalar or None)."""
    if isinstance(beta, torch.Tensor):
        return 1.0, beta.detach().to(torch.float32).reshape(1)
    return float(beta), None


class _EpsPlan:
    """eps for one call: injected tensors (reference mode) or Philox coordinates."""

    def __init__(self, injected=None, seed=0, step=0):
        self.injected, self.seed, self.step = injected, seed, step
        # every RNG coordinate is pinned when the forward runs: the backward executes on autograd's own thread,
        # where the thread-local settings of rng.py (sample base, device step counter) are not the caller's
        self.sample_base, self.step_dev = R.get_sample_base(), R.device_step()

    def ptrs(self, l):
        if self.injected is None:
            return None, None
        return L.ptr(self.injected[l][0]), L.ptr(self.injected[l][1])

    def rng(self, l):
        return _rng(l, self.seed, self.step, self.sample_base, self.step_dev)

    def tensors(self):
        return [] if self.injected is None else [t for pair in self.injected.values() for t in pair]


def plan_eps(shapes, S, device, sample=True):
    """shapes: per layer (shape of the weight-like eps, shape of the bias eps).  In reference mode the
    draws follow SURVEY App. A-4: for s: for layer: weight eps, bias eps."""
    if not sample:
        return _EpsPlan()
    if R.get_eps_mode() in ('reference', 'injected'):
        draw = torch.randn if R.get_eps_mode() == 'reference' else R.pop_injected
        per = [([], []) for _ in shapes]
        for _ in range(S):
            for l, (sw, sb) in enumerate(shapes):
                per[l][0].append(draw(sw))
                per[l][1].append(draw(sb))
        inj = {l: (torch.stack(a).to(device), torch.stack(b).to(device)) for l, (a, b) in enumerate(per)}
        return _EpsPlan(inj)
    seed, step = R.next_step()
    return _EpsPlan(None, seed, step)


# =========================================================================================
# per-weight Gaussian priors p(w) = N(m, softplus(r)^2) (bbb_gauss_prior_*)
# =========================================================================================
def _gauss_prior_table(params, gauss, eps, sample, S, grads=None, layer_ids=None):
    """The tensor table of a bbb_gauss_prior_* call: every layer's weight and bias with its prior (gauss[l] =
    (weight m, weight r, bias m, bias r)), eps (injected, zeros for an unsampled call, or Philox: NULL) and, for a
    backward, the gradient views it adds into.  Returns (table, count, tensors the call must keep alive)."""
    n = 2 * len(params)
    if n > L.GAUSS_PRIOR_MAX_TENSORS:
        raise ValueError(f'a per-weight prior covers at most {L.GAUSS_PRIOR_MAX_TENSORS // 2} layers, got {n // 2}')
    tab, keep = (L.GaussPriorTensor * n)(), []
    for l, (p, pr) in enumerate(zip(params, gauss)):
        lid = l if layer_ids is None else layer_ids[l]
        inj = eps.ptrs(lid)
        for j in (0, 1):
            t = tab[2 * l + j]
            t.mu, t.rho = p[2 * j].data_ptr(), p[2 * j + 1].data_ptr()
            t.prior_mu, t.prior_rho = pr[2 * j].data_ptr(), pr[2 * j + 1].data_ptr()
            t.n, t.tensor_id = p[2 * j].numel(), 2 * lid + j
            if not sample:                   # w = mu: log-probs of the mean weights
                z = torch.zeros((S, t.n), dtype=torch.float32, device=p[0].device)
                keep.append(z)
                t.eps = z.data_ptr()
            else:
                t.eps = inj[j]
            if grads is not None:
                t.grad_mu, t.grad_rho = grads[l][2 * j].data_ptr(), grads[l][2 * j + 1].data_ptr()
    return tab, n, keep


# =========================================================================================
# the two estimators: everything that differs between their C-ABI families
# =========================================================================================
def _zeroed_views(shapes, device):
    """One zero-filled buffer carved into tensors of the given shapes (a single memset for all of them): the
    split-K tensor-core kernels add partial tiles into their output with red.add (BBB_F_OUT_ZEROED)."""
    sizes = [int(torch.Size(sh).numel()) for sh in shapes]
    padded = [(n + 63) // 64 * 64 for n in sizes]           # every view starts on a 256-byte boundary
    flat = torch.zeros(sum(padded), dtype=torch.float32, device=device)
    out, off = [], 0
    for sh, n, m in zip(shapes, sizes, padded):
        out.append(flat[off:off + n].view(sh))
        off += m
    return out


def _workspace(shapes, device, zero):
    if zero:
        return _zeroed_views(shapes, device)
    return [torch.empty(sh, dtype=torch.float32, device=device) for sh in shapes]


def head_eligible(p):
    """bbb_head_fwd's shape conditions (include/bbb.h): a narrow last layer whose rows are 16-byte multiples."""
    out, inn = p[0].shape
    return out <= 16 and inn % 4 == 0 and 4 <= inn <= 8192


def _dev_vec(g):
    """The gradient of a log-prob output as the fp32 device vector a backward kernel reads (a 0-d one as [1])."""
    if g is None:
        return None
    g = _f32c(g)
    return g.reshape(1) if g.dim() == 0 else g


def _prezero(B):
    """Only the kernels for batches of at most 128 rows combine split-K partial tiles with red.add into a zero-filled
    output (BBB_F_OUT_ZEROED).  Above that every kernel either writes its output with plain stores or zeroes it itself,
    so the per-step workspace (gigabytes at batch 4096) is allocated uninitialised."""
    return B <= 128


_relu_out_cache = {}


def _relu_out_layers(params, B, tf32):
    """Per layer: is its output stored POST-activation (BBB_F_RELU_OUT)?  The large-batch tensor kernels do that for
    hidden layers, so that nothing downstream passes over TMA-landed tiles to apply the ReLU; the consumers of such an
    output are called without BBB_F_RELU_IN (the (x > 0) mask of BBB_F_DX_PREACT is the same on either form)."""
    if not tf32:
        return [False] * len(params)
    key = (B, tuple(tuple(p[0].shape) for p in params))
    ro = _relu_out_cache.get(key)
    if ro is None:
        ro = [l < len(params) - 1 and
              bool(L.lib().bbb_linear_fwd_relu_out_supported(B, p[0].shape[1], p[0].shape[0], L.F_TF32))
              for l, p in enumerate(params)]
        _relu_out_cache[key] = ro
    return ro


def _mlp_layer_table(params, eps, ys, dzs, grads):
    tab = (L.MlpLayer * len(params))()
    for l, p in enumerate(params):
        t = tab[l]
        t.w_mu, t.w_rho, t.b_mu, t.b_rho = (q.data_ptr() for q in p)
        t.eps_w, t.eps_b = eps.ptrs(l)
        t.out, t.inn = p[0].shape
        t.y, t.dz = L.ptr(ys[l]), L.ptr(dzs[l])
        if grads is not None and grads[l] is not None:
            t.g_w_mu, t.g_w_rho, t.g_b_mu, t.g_b_rho = (g.data_ptr() for g in grads[l])
    return tab


def _mlp_forward_call(x2, target, params, eps, prior, S, B, sigma, mode, need_grad, beta_h, beta_d, out4,
                      gauss_fwd=None):
    """sample_elbo's forward as ONE C call (bbb_mlp_fwd): TMA-fed tcgen05 kernels for the hidden layers + the fused
    head.  Returns (ys, dxs, d_out): ys[l] the pre-activation output of layer l (the hidden ones live in the zero-filled
    workspace: their split-K partial tiles are reduce-added into it), dxs[l] the zero-filled gradient buffer w.r.t.
    layer l's pre-activation input.  gauss_fwd(logp, logq), when given, adds the per-weight prior terms to the zeroed
    accumulators before the call, which then runs without BBB_F_LOGPROB: its head assembles the four scalars from them."""
    dev = x2.device
    nl = len(params)
    hidden = [p[0].shape[0] for p in params[:-1]]
    # zero-filled (one memset): fp64 accumulators + the head's done counter | pre-activations of every hidden layer |
    # gradient w.r.t. every hidden layer's pre-activation output (the layer above adds its partial dx tiles into it)
    shapes = [(2 * (2 * S + 1) + 2,)] + [(S, B, h) for h in hidden]
    if need_grad:
        shapes += [(S, B, h) for h in hidden]
    ws = _zeroed_views(shapes, dev)
    acc = ws[0][:2 * (2 * S + 1)].view(torch.float64)
    done = ws[0][2 * (2 * S + 1):]
    Cc = params[-1][0].shape[0]
    ys = ws[1:1 + len(hidden)] + [torch.empty((S, B, Cc), dtype=torch.float32, device=dev)]
    dzs = (ws[1 + len(hidden):] if need_grad else [None] * len(hidden))
    logp, logq, nll = acc[:S], acc[S:2 * S], acc[2 * S:]
    d_out = torch.empty((S, B, Cc), dtype=torch.float32, device=dev) if need_grad else None
    tab = _mlp_layer_table(params, eps, ys, list(dzs) + [d_out], None)
    kind = L.NLL_CE if mode == 'classification' else L.NLL_GAUSS
    tgt = target if mode == 'classification' else _f32c(target)
    if gauss_fwd is not None:
        gauss_fwd(logp, logq)
    rng = eps.rng(0)
    L.check(L.lib().bbb_mlp_fwd(tab, nl, L.ptr(x2), S, B, C.byref(rng), C.byref(prior),
                                L.F_SAMPLE | (0 if gauss_fwd is not None else L.F_LOGPROB) | L.F_TF32, kind, L.ptr(tgt), float(sigma), 1.0 / S,
                                L.ptr(d_out), L.ptr(logp), L.ptr(logq), L.ptr(nll), beta_h, L.ptr(beta_d),
                                L.ptr(out4), L.ptr(done), L.stream()), 'bbb_mlp_fwd')
    return ys, ([None] + list(dzs) if need_grad else None), d_out


# sample_elbo in TF32 mode goes through ONE C call per network pass (bbb_mlp_fwd / bbb_mlp_bwd) when the library covers
# the network (bbb_mlp_supported); False forces the per-layer calls (A/B measurements, tools/check_mlp.py)
use_network_level_call = True


class _WeightSampling:
    """Weight sampling (networks.py:48-88, 192-209): weights [out, in] sampled per sample, log prior and log posterior
    of the sampled weights accumulated per sample (2S fp64 values), their gradient taken through the prior-gradient
    scalars gp / gq of the backward (BBB_F_LOGPROB is a forward flag only)."""
    __slots__ = ('prior', 'gauss')
    has_delta = False            # no per-layer buffer besides the output
    eps_per_row = False          # one eps per weight: every input row sees the same S networks
    reuse_error = ('sample_elbo: this graph was already differentiated (retain_graph=True is not supported by the '
                   'fused ELBO path: its backward workspace is single-use)')
    prezero = staticmethod(_prezero)
    relu_out = staticmethod(_relu_out_layers)

    def __init__(self, prior, gauss=None):
        self.prior = prior
        self.gauss = gauss       # per layer (weight m, weight r, bias m, bias r) of a per-weight prior, or None

    def with_gauss(self, gauss):
        """This estimator with the per-weight Gaussian prior `gauss` in place of the shared prior (None: as is)."""
        return self if gauss is None else _WeightSampling(self.prior, gauss)

    @staticmethod
    def layer_grad_args(pg):
        """The prior-gradient arguments of the layer calls when the per-weight prior kernels take the prior terms:
        gp = gq = 0, no device multipliers."""
        gflags, gargs = pg
        return gflags, (0.0, 0.0, None, None, gargs[4])

    def gauss_fwd(self, params, eps, S, sample, lp, layer_ids=None):
        tab, n, keep = _gauss_prior_table(params, self.gauss, eps, sample, S, layer_ids=layer_ids)
        rng = eps.rng(0)
        L.check(L.lib().bbb_gauss_prior_logprob(tab, n, S, C.byref(rng), L.ptr(lp[0]), L.ptr(lp[1]), L.stream()),
                'bbb_gauss_prior_logprob')

    def gauss_bwd(self, params, eps, S, sample, pg, out_scale, grads, layer_ids=None):
        gp, gq, gp_dev, gq_dev, g_stride = pg[1]
        if gp == 0.0 and gq == 0.0:
            return
        tab, n, keep = _gauss_prior_table(params, self.gauss, eps, sample, S, grads, layer_ids)
        rng = eps.rng(0)
        L.check(L.lib().bbb_gauss_prior_logprob_bwd(tab, n, S, C.byref(rng), gp, gq, L.ptr(gp_dev), L.ptr(gq_dev),
                                                    g_stride, L.ptr(out_scale), L.stream()),
                'bbb_gauss_prior_logprob_bwd')

    @staticmethod
    def shape(w):
        """(in, out) of a layer from its weight tensor."""
        out, inn = w.shape
        return inn, out

    @staticmethod
    def eps_shapes(params, B):
        return [(tuple(p[0].shape), (p[0].shape[0],)) for p in params]

    @staticmethod
    def acc_len(S):
        return 2 * S

    @staticmethod
    def lp(acc, S):
        """The log-prob accumulators the forward adds into: (log prior [S], log posterior [S])."""
        return acc[:S], acc[S:2 * S]

    @staticmethod
    def lp_outputs(lpq, S, scalars):
        """The log-prob outputs from the fp32 accumulators: per sample, or as two scalars when S = 1."""
        return (lpq[0], lpq[1]) if scalars else (lpq[:S], lpq[S:])

    @staticmethod
    def grad_args(gs, logprob, scalars):
        """(backward flags, prior-gradient arguments) from the gradients of the log-prob outputs (None: not used)."""
        gp, gq = (_dev_vec(g) for g in gs)
        return 0, (1.0 if gp is not None else 0.0, 1.0 if gq is not None else 0.0, gp, gq, 0 if scalars else 1)

    @staticmethod
    def elbo_grad_args(beta, beta_dev, S):
        """loss = beta (log q - log p) / S summed over the samples + nll: gp = -beta / S, gq = beta / S."""
        return 0, (-beta / S, beta / S, beta_dev, beta_dev, 0)

    def fwd(self, x, x_stride, p, eps, l, S, B, flags, y, delta, lp):
        wm, wr, bm, br = p
        out, inn = wm.shape
        ew, eb = eps.ptrs(l)
        rng = eps.rng(l)
        L.check(L.lib().bbb_linear_fwd(L.ptr(x), x_stride, L.ptr(wm), L.ptr(wr), L.ptr(bm), L.ptr(br), ew, eb,
                                       C.byref(rng), C.byref(self.prior), S, B, inn, out, flags, L.ptr(y),
                                       L.ptr(lp[0]), L.ptr(lp[1]), L.stream()), 'bbb_linear_fwd')

    def bwd(self, dy, x, x_stride, p, eps, l, delta, S, B, flags, gargs, out_scale, dx, grads):
        wm, wr, bm, br = p
        out, inn = wm.shape
        ew, eb = eps.ptrs(l)
        rng = eps.rng(l)
        gp, gq, gp_dev, gq_dev, g_stride = gargs
        L.check(L.lib().bbb_linear_bwd(L.ptr(dy), None, L.ptr(x), x_stride, L.ptr(wm), L.ptr(wr), L.ptr(bm),
                                       L.ptr(br), ew, eb, C.byref(rng), C.byref(self.prior), S, B, inn, out, flags,
                                       gp, gq, L.ptr(gp_dev), L.ptr(gq_dev), g_stride, L.ptr(out_scale), L.ptr(dx),
                                       L.ptr(grads[0]), L.ptr(grads[1]), L.ptr(grads[2]), L.ptr(grads[3]),
                                       L.stream()), 'bbb_linear_bwd')

    # ---- sample_elbo ------------------------------------------------------------------------------------------------
    @staticmethod
    def elbo_workspace(params, S, B, need_grad, dev):
        """ONE zero-filled workspace (one memset per step): fp64 accumulators + the head's completion counter |
        activations of every layer | dx of every layer above the first (the backward's split-K kernels add into them).
        Large batches zero only the accumulators.  Returns (lp, nll, done, ys, deltas, dxs, d_out)."""
        shapes = [(2 * (2 * S + 1) + 2,)] + [(S, B, p[0].shape[0]) for p in params]
        if need_grad:
            shapes += [(S, B, p[0].shape[1]) for p in params[1:]]
        if _prezero(B):
            ws = _zeroed_views(shapes, dev)
        else:
            ws = _zeroed_views(shapes[:1], dev) + _workspace(shapes[1:], dev, False)
        acc = ws[0][:2 * (2 * S + 1)].view(torch.float64)
        done = ws[0][2 * (2 * S + 1):]
        nl = len(params)
        ys, dxs = ws[1:1 + nl], ([None] + ws[1 + nl:] if need_grad else None)
        logp, logq, nll = acc[:S], acc[S:2 * S], acc[2 * S:]
        d_out = torch.empty((S, B, params[-1][0].shape[0]), dtype=torch.float32, device=dev) if need_grad else None
        return (logp, logq), nll, done, ys, [None] * nl, dxs, d_out

    def head(self, params, eps, S, B, mode, likelihood, target, sigma, d_out, lp, nll, beta_h, beta_d, out4, done):
        """The last layer, the likelihood with its gradient and the assembly of the four scalars in one launch
        (bbb_head_fwd), as head(inp, stride, flags, y) for the forward loop; None when it does not apply (the
        heteroscedastic likelihood has no fused head)."""
        if likelihood != 'gaussian' or not head_eligible(params[-1]):
            return None
        nl = len(params) - 1
        wm, wr, bm, br = params[nl]
        out, inn = wm.shape
        ew, eb = eps.ptrs(nl)
        kind = L.NLL_CE if mode == 'classification' else L.NLL_GAUSS
        tgt = target if mode == 'classification' else _f32c(target)

        def head(x, x_stride, flags, y):
            rng = eps.rng(nl)
            L.check(L.lib().bbb_head_fwd(L.ptr(x), x_stride, L.ptr(wm), L.ptr(wr), L.ptr(bm), L.ptr(br), ew, eb,
                                         C.byref(rng), C.byref(self.prior), S, B, inn, out, flags, kind, L.ptr(tgt),
                                         float(sigma), 1.0 / S, L.ptr(y), L.ptr(d_out), L.ptr(lp[0]), L.ptr(lp[1]),
                                         L.ptr(nll), beta_h, L.ptr(beta_d), L.ptr(out4), L.ptr(done), L.stream()),
                    'bbb_head_fwd')
        return head

    @staticmethod
    def finalize(lp, nll, S, beta_h, beta_d, out4):
        L.check(L.lib().bbb_elbo_finalize(L.ptr(lp[0]), L.ptr(lp[1]), None, L.ptr(nll), S, beta_h, L.ptr(beta_d),
                                          L.ptr(out4), L.stream()), 'bbb_elbo_finalize')

    @staticmethod
    def elbo_outputs(out4):
        """(loss [1], log_prior, log_variational_posterior, negative_log_likelihood [1])"""
        return out4[0:1], out4[1], out4[2], out4[3:4]

    @staticmethod
    def single_use(tf32):
        # the split-K backward kernels ADD into the dx workspace zero-filled by the forward (BBB_F_OUT_ZEROED)
        return True

    @staticmethod
    def network_call(params, S, B, mode, likelihood, tf32):
        """Does sample_elbo run as ONE C call per pass (bbb_mlp_fwd / bbb_mlp_bwd: TMA-fed tcgen05 kernels for the
        hidden layers + the fused head)?  Neither call implements the heteroscedastic likelihood."""
        dims = [params[0][0].shape[1]] + [p[0].shape[0] for p in params]
        return (likelihood == 'gaussian' and use_network_level_call and tf32 and
                mode in ('classification', 'regression') and L.mlp_supported(dims, S, B, L.F_TF32))

    def network_forward(self, x2, target, params, eps, S, B, sigma, mode, need_grad, beta_h, beta_d, out4):
        gauss_fwd = None
        if self.gauss is not None:
            def gauss_fwd(logp, logq):
                self.gauss_fwd(params, eps, S, True, (logp, logq))
        return _mlp_forward_call(x2, target, params, eps, self.prior, S, B, sigma, mode, need_grad, beta_h, beta_d,
                                 out4, gauss_fwd)

    def network_backward(self, x2, ys, dxs, d_out, params, S, eps, gargs, scale):
        """ONE C call for the whole backward (bbb_mlp_bwd): ys are the stored hidden pre-activations, dxs[l + 1] the
        zero-filled gradient w.r.t. hidden layer l's pre-activation output.  A per-weight prior's terms are added by
        their own kernel after it, before any layer's gradients are reported."""
        nl = len(params)
        grads = _alloc_grads(params)
        tab = _mlp_layer_table(params, eps, list(ys) + [None], list(dxs[1:nl]) + [d_out], grads)
        rng = eps.rng(0)
        pg = (0, gargs)
        gp, gq, gp_dev, gq_dev, g_stride = gargs if self.gauss is None else self.layer_grad_args(pg)[1]
        L.check(L.lib().bbb_mlp_bwd(tab, nl, L.ptr(x2), S, x2.shape[0], C.byref(rng), C.byref(self.prior),
                                    L.F_SAMPLE | L.F_TF32, gp, gq, L.ptr(gp_dev), L.ptr(gq_dev), g_stride,
                                    L.ptr(scale), L.stream()), 'bbb_mlp_bwd')
        if self.gauss is not None:
            self.gauss_bwd(params, eps, S, True, pg, scale, grads)
        if grad_ready_hook is not None:
            for l in reversed(range(nl)):
                grad_ready_hook(l, grads[l].flat)
        return grads


class _LocalReparam:
    """Local reparameterisation (networks.py:90-138, 211-225): weights [in, out], the pre-activation sampled per row
    from its mean x mu and variance delta = x^2 sigma^2 (kept per layer for the backward), one closed-form KL for the
    whole call, its gradient taken through BBB_F_LOGPROB in the backward."""
    __slots__ = ('sigma_p', 'gauss')
    has_delta = True
    eps_per_row = True           # the noise is drawn per input row: a chunked pass draws it chunk by chunk
    reuse_error = ('sample_elbo_lr: this graph was already differentiated (retain_graph=True is not supported by the '
                   'TF32 local-reparameterisation path: its saved state is single-use)')

    def __init__(self, sigma_p, gauss=None):
        self.sigma_p = float(sigma_p)
        self.gauss = gauss       # per layer (weight m, weight r, bias m, bias r) of a per-weight prior, or None

    def with_gauss(self, gauss):
        """This estimator with the per-weight Gaussian prior `gauss` in place of N(0, sigma_p) (None: as is)."""
        return self if gauss is None else _LocalReparam(self.sigma_p, gauss)

    @staticmethod
    def layer_grad_args(pg):
        """The layer calls run without BBB_F_LOGPROB when the per-weight prior kernels take the KL terms."""
        gflags, gargs = pg
        return gflags & ~L.F_LOGPROB, gargs

    def gauss_fwd(self, params, eps, S, sample, lp, layer_ids=None):
        tab, n, _ = _gauss_prior_table(params, self.gauss, _EpsPlan(), True, S, layer_ids=layer_ids)
        L.check(L.lib().bbb_gauss_prior_kl(tab, n, L.ptr(lp[0]), L.stream()), 'bbb_gauss_prior_kl')

    def gauss_bwd(self, params, eps, S, sample, pg, out_scale, grads, layer_ids=None):
        gflags, (g_kl, g_kl_dev) = pg
        if not gflags & L.F_LOGPROB:
            return
        tab, n, _ = _gauss_prior_table(params, self.gauss, _EpsPlan(), True, S, grads, layer_ids)
        L.check(L.lib().bbb_gauss_prior_kl_bwd(tab, n, g_kl, L.ptr(g_kl_dev), L.ptr(out_scale), L.stream()),
                'bbb_gauss_prior_kl_bwd')

    @staticmethod
    def shape(w):
        return tuple(w.shape)

    @staticmethod
    def eps_shapes(params, B):
        return [((B, p[0].shape[1]), (p[0].shape[1],)) for p in params]

    @staticmethod
    def prezero(B):
        # the tensor-core kernels add their split-K partial sums of x mu and x^2 sigma^2 into y and delta (and of dx)
        # before the epilogue turns them into the outputs, at every batch size
        return True

    @staticmethod
    def relu_out(params, B, tf32):
        return [False] * len(params)

    @staticmethod
    def acc_len(S):
        return 1

    @staticmethod
    def lp(acc, S):
        """The KL accumulator the forward adds into (evaluated once per call, not per sample: SURVEY B-8)."""
        return (acc,)

    @staticmethod
    def lp_outputs(lpq, S, scalars):
        return (lpq[0],)

    @staticmethod
    def grad_args(gs, logprob, scalars):
        use_kl = logprob and gs[0] is not None
        return (L.F_LOGPROB if use_kl else 0), (1.0, _dev_vec(gs[0]) if use_kl else None)

    @staticmethod
    def elbo_grad_args(beta, beta_dev, S):
        """loss = beta KL + nll"""
        return L.F_LOGPROB, (beta, beta_dev)

    def fwd(self, x, x_stride, p, eps, l, S, B, flags, y, delta, lp):
        wm, wr, bm, br = p
        inn, out = wm.shape
        ea, eb = eps.ptrs(l)
        rng = eps.rng(l)
        L.check(L.lib().bbb_lr_linear_fwd(L.ptr(x), x_stride, L.ptr(wm), L.ptr(wr), L.ptr(bm), L.ptr(br), ea, eb,
                                          C.byref(rng), self.sigma_p, S, B, inn, out, flags, L.ptr(y), L.ptr(delta),
                                          L.ptr(lp[0]), L.stream()), 'bbb_lr_linear_fwd')

    def bwd(self, dy, x, x_stride, p, eps, l, delta, S, B, flags, gargs, out_scale, dx, grads):
        """In TF32 mode the kernels overwrite the saved delta with dV (it has no other use in the backward)."""
        wm, wr, bm, br = p
        inn, out = wm.shape
        ea, eb = eps.ptrs(l)
        rng = eps.rng(l)
        g_kl, g_kl_dev = gargs
        L.check(L.lib().bbb_lr_linear_bwd(L.ptr(dy), None, L.ptr(x), x_stride, L.ptr(wm), L.ptr(wr), L.ptr(bm),
                                          L.ptr(br), ea, eb, C.byref(rng), L.ptr(delta), self.sigma_p, S, B, inn, out,
                                          flags, g_kl, L.ptr(g_kl_dev), L.ptr(out_scale), L.ptr(dx), L.ptr(grads[0]),
                                          L.ptr(grads[1]), L.ptr(grads[2]), L.ptr(grads[3]), L.stream()),
                'bbb_lr_linear_bwd')

    # ---- sample_elbo_lr ---------------------------------------------------------------------------------------------
    def elbo_workspace(self, params, S, B, need_grad, dev):
        """Returns (lp, nll, done, ys, deltas, dxs, d_out); the backward allocates its own dx buffers."""
        acc = torch.zeros(2, dtype=torch.float64, device=dev)
        kl, nll = acc[0:1], acc[1:2]
        ys, deltas = _activations(self, params, S, B, True, dev)
        d_out = torch.empty_like(ys[-1]) if need_grad else None
        return (kl,), nll, None, ys, deltas, None, d_out

    @staticmethod
    def head(*args):
        return None

    @staticmethod
    def finalize(lp, nll, S, beta_h, beta_d, out4):
        L.check(L.lib().bbb_elbo_finalize(None, None, L.ptr(lp[0]), L.ptr(nll), S, beta_h, L.ptr(beta_d), L.ptr(out4),
                                          L.stream()), 'bbb_elbo_finalize')

    @staticmethod
    def elbo_outputs(out4):
        """(loss [1], kl, negative_log_likelihood [1])"""
        return out4[0:1], out4[1], out4[2:3]

    @staticmethod
    def single_use(tf32):
        # the tcgen05 LR backward overwrites the saved delta buffers with dV
        return tf32

    @staticmethod
    def network_call(params, S, B, mode, likelihood, tf32):
        return False


# =========================================================================================
# one network pass, forward and backward, for either estimator
# =========================================================================================
def _activations(est, params, S, B, sample, dev):
    """Every layer's output [S,B,out] (and delta, when the estimator keeps one and the call samples): one buffer,
    zero-filled when the estimator's kernels add into it."""
    shapes = [(S, B, est.shape(p[0])[1]) for p in params]
    bufs = _workspace(shapes * (2 if sample and est.has_delta else 1), dev, est.prezero(B))
    n = len(params)
    return bufs[:n], (bufs[n:] or [None] * n)


def _forward(est, x2, params, S, eps, sample, logprob, tf32, lp, ys=None, deltas=None, head=None):
    """All layers, all S samples.  Returns (ys, deltas): ys[l] = [S,B,out_l] pre-activations, except the hidden
    layers est.relu_out names.  `ys`, `deltas` when the caller supplies them; `head(inp, stride, flags, y)`, when
    given, runs the last layer instead of the layer call (the fused ELBO tail)."""
    B = x2.shape[0]
    ro = est.relu_out(params, B, tf32)
    gauss = logprob and est.gauss is not None       # the per-weight prior kernel takes the log-prob terms
    base = ((L.F_SAMPLE if sample else 0) | (L.F_LOGPROB if logprob and not gauss else 0) | (L.F_TF32 if tf32 else 0) |
            (L.F_OUT_ZEROED if est.prezero(B) else 0))
    if ys is None:
        ys, deltas = _activations(est, params, S, B, sample, x2.device)
    if gauss:
        est.gauss_fwd(params, eps, S, sample, lp)
    inp, stride = x2, 0
    for l, p in enumerate(params):
        flags = base | (L.F_RELU_IN if l > 0 and not ro[l - 1] else 0) | (L.F_RELU_OUT if ro[l] else 0)
        if head is not None and l == len(params) - 1:
            head(inp, stride, flags, ys[l])
        else:
            est.fwd(inp, stride, p, eps, l, S, B, flags, ys[l], deltas[l], lp)
        inp, stride = ys[l], B * est.shape(p[0])[1]
    return ys, deltas


def _backward(est, x2, ys, deltas, d_out, params, S, eps, sample, tf32, pg, out_scale, need_dx0, dxs=None):
    """Backward of _forward; pg = (flags, arguments) of the prior gradient (est.grad_args / est.elbo_grad_args).
    Returns (dx0 or None, [grads per layer]).  Every layer above the first hands down the gradient w.r.t. the
    PRE-activation output of the layer below (BBB_F_DX_PREACT: the ReLU mask is applied where dx is produced), so no
    layer needs a separate mask pass over dy."""
    B = x2.shape[0]
    ro = est.relu_out(params, B, tf32)
    gflags, gargs = pg if est.gauss is None else est.layer_grad_args(pg)
    base = ((L.F_SAMPLE if sample else 0) | (L.F_TF32 if tf32 else 0) | (L.F_OUT_ZEROED if est.prezero(B) else 0) |
            gflags)
    grads = _alloc_grads(params)
    dy, dx0 = d_out, None
    first = 0 if need_dx0 else 1
    if dxs is None:
        dxs = [None] * first + _workspace([(S, B, est.shape(p[0])[0]) for p in params[first:]], x2.device,
                                          est.prezero(B))
    for l in reversed(range(len(params))):
        p = params[l]
        g = grads[l]
        flags = base | (L.F_DX_PREACT if l > 0 else 0) | (L.F_RELU_IN if l > 0 and not ro[l - 1] else 0)
        want_dx = l > 0 or need_dx0
        dx = dxs[l] if want_dx else None
        if not want_dx:
            flags |= L.F_NO_DX
        if l == 0 and need_dx0:
            flags |= L.F_SCALE_DX
        x_in, stride = (x2, 0) if l == 0 else (ys[l - 1], B * est.shape(p[0])[0])
        est.bwd(dy, x_in, stride, p, eps, l, deltas[l], S, B, flags, gargs, out_scale, dx, g)
        if grad_ready_hook is not None and est.gauss is None:
            grad_ready_hook(l, g.flat)
        dy = dx
        if l == 0:
            dx0 = dx
    if est.gauss is not None:
        # one launch adds the prior terms of every layer; only then are the gradients complete and reported
        est.gauss_bwd(params, eps, S, sample, pg, out_scale, grads)
        if grad_ready_hook is not None:
            for l in reversed(range(len(params))):
                grad_ready_hook(l, grads[l].flat)
    return dx0, grads


def _params(flat):
    return [tuple(_f32c(t) for t in flat[i:i + 4]) for i in range(0, len(flat), 4)]


def _save(ctx, **groups):
    """ctx.save_for_backward of named groups, each a tensor (or None) or a list of them; _saved(ctx) returns them by
    name."""
    layout, tensors = [], []
    for name, g in groups.items():
        is_list = isinstance(g, (list, tuple))
        layout.append((name, len(g) if is_list else None))
        tensors += g if is_list else [g]
    ctx.save_for_backward(*tensors)
    ctx.saved_layout = layout


def _saved(ctx):
    sv, out, i = ctx.saved_tensors, {}, 0
    for name, n in ctx.saved_layout:
        out[name] = sv[i] if n is None else list(sv[i:i + n])
        i += 1 if n is None else n
    return out


# =========================================================================================
# layer level: one sample of one layer
# =========================================================================================
class _Linear(torch.autograd.Function):
    """BayesianLinear.forward (networks.py:73-88) -> (y, log_prior, log_post), BayesianLinearLR.forward
    (networks.py:116-138) -> (y, kl), for one sample."""

    @staticmethod
    def forward(ctx, est, x, wm, wr, bm, br, sample, logprob, layer_id, tf32):
        L.require_cuda(x, wm, wr, bm, br)
        inn, out = est.shape(wm)
        x2 = _f32c(x).reshape(-1, inn)
        B = x2.shape[0]
        p = tuple(_f32c(t) for t in (wm, wr, bm, br))
        eps = plan_eps(est.eps_shapes([p], B), 1, x2.device, sample)
        if eps.injected is not None:            # re-key as layer `layer_id`
            eps.injected = {layer_id: eps.injected[0]}
        acc = torch.zeros(est.acc_len(1), dtype=torch.float64, device=x2.device)
        y = torch.empty((1, B, out), dtype=torch.float32, device=x2.device)
        delta = torch.empty_like(y) if sample and est.has_delta else None
        gauss = logprob and est.gauss is not None
        if gauss:
            est.gauss_fwd([p], eps, 1, sample, est.lp(acc, 1), [layer_id])
        flags = ((L.F_SAMPLE if sample else 0) | (L.F_LOGPROB if logprob and not gauss else 0) |
                 (L.F_TF32 if tf32 else 0))
        est.fwd(x2, 0, p, eps, layer_id, 1, B, flags, y, delta, est.lp(acc, 1))
        _save(ctx, x2=x2, p=p, delta=delta, eps=eps.tensors())
        ctx.est, ctx.sample, ctx.logprob, ctx.layer_id, ctx.tf32, ctx.eps = est, sample, logprob, layer_id, tf32, eps
        ctx.xshape, ctx.x_rg = x.shape, x.requires_grad
        ctx.set_materialize_grads(False)
        lpq = acc.to(torch.float32)
        return (y.view(*x.shape[:-1], out), *est.lp_outputs(lpq, 1, True))

    @staticmethod
    def backward(ctx, dy, *dlp):
        est, s = ctx.est, _saved(ctx)
        x2, p = s['x2'], tuple(s['p'])
        inn, out = est.shape(p[0])
        B = x2.shape[0]
        if dy is None:
            dy = torch.zeros((B, out), dtype=torch.float32, device=x2.device)
        dy = _f32c(dy).reshape(1, B, out)
        g = tuple(torch.empty_like(t) for t in p)
        dx = torch.empty((1, B, inn), dtype=torch.float32, device=x2.device) if ctx.x_rg else None
        pg = est.grad_args(dlp, ctx.logprob, True)
        gflags, gargs = pg if est.gauss is None else est.layer_grad_args(pg)
        flags = ((L.F_SAMPLE if ctx.sample else 0) | (L.F_TF32 if ctx.tf32 else 0) | (0 if ctx.x_rg else L.F_NO_DX) |
                 gflags)
        est.bwd(dy, x2, 0, p, ctx.eps, ctx.layer_id, s['delta'], 1, B, flags, gargs, None, dx, g)
        if est.gauss is not None:
            est.gauss_bwd([p], ctx.eps, 1, ctx.sample, pg, None, [g], [ctx.layer_id])
        return (None, dx.view(ctx.xshape) if ctx.x_rg else None, *g, None, None, None, None)


def bayes_linear(x, wm, wr, bm, br, prior, sample, logprob, layer_id=0, tf32=False, gauss=None):
    """gauss: (weight m, weight r, bias m, bias r) of a per-weight prior N(m, softplus(r)^2), replacing `prior`."""
    est = _WeightSampling(prior, None if gauss is None else [gauss])
    return _Linear.apply(est, x, wm, wr, bm, br, sample, logprob, layer_id, tf32)


def lr_linear(x, wm, wr, bm, br, sigma_p, sample, calc_kl, layer_id=0, gauss=None):
    """gauss: as bayes_linear's, replacing N(0, sigma_p)."""
    est = _LocalReparam(sigma_p, None if gauss is None else [gauss])
    return _Linear.apply(est, x, wm, wr, bm, br, sample, calc_kl, layer_id, False)


# =========================================================================================
# network level: S sampled forwards of the whole MLP, differentiable outputs
# =========================================================================================
class _NetworkForward(torch.autograd.Function):
    """(x, params) -> outputs [S,B,C] and the log-prob outputs: log_prior [S], log_post [S] (weight sampling), or kl []
    (local reparameterisation, computed once: SURVEY B-8)."""

    @staticmethod
    def forward(ctx, est, x2, S, sample, logprob, tf32, *flat):
        L.require_cuda(x2, *flat)
        x2 = _f32c(x2)
        params = _params(flat)
        eps = plan_eps(est.eps_shapes(params, x2.shape[0]), S, x2.device, sample)
        acc = torch.zeros(est.acc_len(S), dtype=torch.float64, device=x2.device)
        ys, deltas = _forward(est, x2, params, S, eps, sample, logprob, tf32, est.lp(acc, S))
        _save(ctx, x2=x2, flat=flat, ys=ys, deltas=deltas, eps=eps.tensors())
        ctx.est, ctx.S, ctx.sample, ctx.logprob, ctx.tf32, ctx.eps = est, S, sample, logprob, tf32, eps
        ctx.x_rg = x2.requires_grad
        ctx.set_materialize_grads(False)
        # the last layer's buffer is handed out; backward only needs the hidden pre-activations
        return (ys[-1], *est.lp_outputs(acc.to(torch.float32), S, False))

    @staticmethod
    def backward(ctx, d_out, *dlp):
        est, s = ctx.est, _saved(ctx)
        params = _params(s['flat'])
        if d_out is None:
            d_out = torch.zeros_like(s['ys'][-1])
        pg = est.grad_args(dlp, ctx.logprob, False)
        dx0, grads = _backward(est, s['x2'], s['ys'], s['deltas'], _f32c(d_out), params, ctx.S, ctx.eps, ctx.sample,
                               ctx.tf32, pg, None, ctx.x_rg)
        flat = [g for lg in grads for g in lg]
        return (None, dx0.sum(0) if ctx.x_rg else None, None, None, None, None, *flat)


def _network_forward(est, x2, layers, S, sample, logprob, tf32):
    return _NetworkForward.apply(est, x2, S, sample, logprob, tf32, *[t for layer in layers for t in layer])


def mlp_forward(x2, layers, prior, S, sample=True, logprob=True, tf32=False):
    return _network_forward(_WeightSampling(prior), x2, layers, S, sample, logprob, tf32)


def mlp_forward_lr(x2, layers, sigma_p, S, sample=True, calc_kl=True, tf32=False):
    return _network_forward(_LocalReparam(sigma_p), x2, layers, S, sample, calc_kl, tf32)


# =========================================================================================
# fused ELBO: the network pass + likelihood + ELBO assembly, loss only differentiable
# =========================================================================================
def _nll_launch(out, target, S, B, Cc, sigma, mode, likelihood, nll, d_out):
    """The likelihood and its gradient (scaled by 1/S) on the sampled outputs [S,B,Cc]: nll += ..., d_out written.
    The heteroscedastic likelihood reads `sigma` as sigma_min and Cc = 2D outputs per row."""
    if likelihood == 'heteroscedastic':
        tgt = _f32c(target)            # (held: a contiguous copy must outlive the call)
        L.check(L.lib().bbb_nll_gauss_het(L.ptr(out), L.ptr(tgt), float(sigma), S, B, Cc // 2, 1.0 / S, L.ptr(nll),
                                          L.ptr(d_out), L.stream()), 'bbb_nll_gauss_het')
    elif mode == 'classification':
        L.check(L.lib().bbb_nll_ce(L.ptr(out), L.ptr(target), S, B, Cc, 1.0 / S, L.ptr(nll), L.ptr(d_out),
                                   L.stream()), 'bbb_nll_ce')
    else:
        tgt = _f32c(target)
        L.check(L.lib().bbb_nll_gauss(L.ptr(out), L.ptr(tgt), float(sigma), S, B, Cc, 1.0 / S, L.ptr(nll),
                                      L.ptr(d_out), L.stream()), 'bbb_nll_gauss')


class _ELBO(torch.autograd.Function):
    """sample_elbo (networks.py:192-209) and sample_elbo_lr (networks.py:211-225): one launch per layer, then the
    likelihood and the assembly of the ELBO, or the estimator's fused tail: the head (last layer + likelihood +
    assembly in one launch) or ONE C call per pass (weight sampling, TF32, batch <= 128).  Only `loss` is
    differentiable.  likelihood 'heteroscedastic' (sigma is then sigma_min) always takes the per-layer calls."""

    @staticmethod
    def forward(ctx, est, x2, target, beta, S, sigma, mode, likelihood, tf32, *flat):
        L.require_cuda(x2, target, *flat)
        x2 = _f32c(x2)
        dev = x2.device
        params = _params(flat)
        B = x2.shape[0]
        eps = plan_eps(est.eps_shapes(params, B), S, dev, True)
        need_grad = any(t.requires_grad for t in flat)
        out4 = torch.empty(4, dtype=torch.float32, device=dev)
        beta_h, beta_d = _split_beta(beta)
        ctx.used_network_call = est.network_call(params, S, B, mode, likelihood, tf32)
        if ctx.used_network_call:
            ys, dxs, d_out = est.network_forward(x2, target, params, eps, S, B, sigma, mode, need_grad, beta_h, beta_d,
                                                 out4)
            deltas = [None] * len(params)
        else:
            lp, nll, done, ys, deltas, dxs, d_out = est.elbo_workspace(params, S, B, need_grad, dev)
            head = est.head(params, eps, S, B, mode, likelihood, target, sigma, d_out, lp, nll, beta_h, beta_d, out4,
                            done)
            _forward(est, x2, params, S, eps, True, True, tf32, lp, ys, deltas, head)
            if head is None:
                _nll_launch(ys[-1], target, S, B, ys[-1].shape[2], sigma, mode, likelihood, nll, d_out)
                est.finalize(lp, nll, S, beta_h, beta_d, out4)
        if need_grad:
            _save(ctx, x2=x2, d_out=d_out, flat=flat, ys=ys[:-1], deltas=deltas, eps=eps.tensors())
            ctx.dxs = dxs
        ctx.est, ctx.S, ctx.beta, ctx.beta_dev, ctx.tf32, ctx.eps = est, S, beta_h, beta_d, tf32, eps
        ctx.n_flat = len(flat)
        ctx.set_materialize_grads(False)      # no zero-filled gradients for the non-differentiable scalars
        outs = est.elbo_outputs(out4)
        ctx.mark_non_differentiable(*outs[1:])
        return outs

    @staticmethod
    def backward(ctx, g_loss, *unused):
        est = ctx.est
        if g_loss is None:
            return (None,) * (9 + ctx.n_flat)
        if est.single_use(ctx.tf32) and getattr(ctx, 'consumed', False):
            raise RuntimeError(est.reuse_error)
        ctx.consumed = True
        s = _saved(ctx)
        params = _params(s['flat'])
        scale = _f32c(g_loss).reshape(1)
        pg = est.elbo_grad_args(ctx.beta, ctx.beta_dev, ctx.S)
        if ctx.used_network_call:
            grads = est.network_backward(s['x2'], s['ys'], ctx.dxs, s['d_out'], params, ctx.S, ctx.eps, pg[1], scale)
        else:
            _, grads = _backward(est, s['x2'], s['ys'], s['deltas'], s['d_out'], params, ctx.S, ctx.eps, True,
                                 ctx.tf32, pg, scale, False, dxs=ctx.dxs)
        return (None,) * 9 + tuple(g for lg in grads for g in lg)


def _elbo(est, x2, target, beta, S, sigma, mode, layers, tf32, likelihood):
    return _ELBO.apply(est, x2, target, beta, S, sigma, mode, likelihood, tf32, *[t for layer in layers for t in layer])


def fused_elbo(x2, target, beta, S, sigma, mode, prior, layers, tf32=False, likelihood='gaussian'):
    return _elbo(_WeightSampling(prior), x2, target, beta, S, sigma, mode, layers, tf32, likelihood)


def fused_elbo_lr(x2, target, beta, S, sigma, mode, sigma_p, layers, tf32=False, likelihood='gaussian'):
    return _elbo(_LocalReparam(sigma_p), x2, target, beta, S, sigma, mode, layers, tf32, likelihood)


# =========================================================================================
# stand-alone reductions and the eps stream (tests, calculate_log_probs, diagnostics)
# =========================================================================================
def logprob_reduce(mu, rho, prior, eps=None, sample=True, seed=0, step=0, sample_idx=0, tensor_id=0,
                   return_w=False):
    L.require_cuda(mu, rho)
    mu, rho = _f32c(mu), _f32c(rho)
    n = mu.numel()
    acc = torch.zeros(2, dtype=torch.float64, device=mu.device)
    w = torch.empty_like(mu) if return_w else None
    e = _f32c(eps) if eps is not None else None
    L.check(L.lib().bbb_logprob_reduce(L.ptr(mu), L.ptr(rho), L.ptr(e), seed, step, sample_idx, tensor_id,
                                       C.byref(prior), n, L.F_SAMPLE if sample else 0, L.ptr(w), L.ptr(acc[0:1]),
                                       L.ptr(acc[1:2]), L.stream()), 'bbb_logprob_reduce')
    return acc[0], acc[1], w


def kl_gauss(mu, rho, sigma_p):
    L.require_cuda(mu, rho)
    mu, rho = _f32c(mu), _f32c(rho)
    acc = torch.zeros(1, dtype=torch.float64, device=mu.device)
    L.check(L.lib().bbb_kl_gauss(L.ptr(mu), L.ptr(rho), float(sigma_p), mu.numel(), L.ptr(acc), L.stream()),
            'bbb_kl_gauss')
    return acc[0]


def philox_normal(n, device, seed=0, step=0, sample_idx=0, tensor_id=0):
    out = torch.empty(n, dtype=torch.float32, device=device)
    L.require_cuda(out)
    L.check(L.lib().bbb_philox_fill_normal(L.ptr(out), n, seed, step, sample_idx, tensor_id, L.stream()),
            'bbb_philox_fill_normal')
    return out


# =========================================================================================
# consumers of the (mu, rho) stream and of the sampled outputs (SURVEY 8 f2 / f3)
# =========================================================================================
def compute_snr(mu, rho):
    """10 log10(|mu| / softplus(rho)) in decibels (weight_pruning.py:81-83), one kernel pass."""
    L.require_cuda(mu, rho)
    mu, rho = _f32c(mu), _f32c(rho)
    out = torch.empty_like(mu)
    L.check(L.lib().bbb_snr(L.ptr(mu), L.ptr(rho), mu.numel(), L.ptr(out), L.stream()), 'bbb_snr')
    return out


def snr_prune_(mu, rho, threshold_db):
    """In place: mu, rho *= (snr > threshold_db) (weight_pruning.py:101-115).  Returns the device count of kept entries."""
    L.require_cuda(mu, rho)
    if not (mu.dtype is torch.float32 and mu.is_contiguous() and rho.dtype is torch.float32 and rho.is_contiguous()):
        raise RuntimeError('snr_prune_ works in place on contiguous fp32 tensors')
    kept = torch.zeros(1, dtype=torch.int64, device=mu.device)
    L.check(L.lib().bbb_snr_prune(L.ptr(mu), L.ptr(rho), mu.numel(), float(threshold_db), L.ptr(kept), L.stream()),
            'bbb_snr_prune')
    return kept


def softmax_mean(logits):
    """[S,B,C] sampled logits -> [B,C] mean over the samples of softmax (class_task.py:84-86), one launch."""
    L.require_cuda(logits)
    z = _f32c(logits)
    S, B, Cc = z.shape
    out = torch.empty((B, Cc), dtype=torch.float32, device=z.device)
    L.check(L.lib().bbb_softmax_mean(L.ptr(z), S, B, Cc, L.ptr(out), L.stream()), 'bbb_softmax_mean')
    return out


# =========================================================================================
# posterior predictive: uncertainty and calibration of the sampled outputs (bbb_predictive_stats)
# =========================================================================================
PREDICTIVE_BUDGET_BYTES = 256 << 20      # bound on one chunk's fp32 activations, S * rows * sum of widths * 4 B
PREDICTIVE_MODES = ('classification', 'regression', 'heteroscedastic')
_PREDICTIVE_KIND = dict(classification=L.NLL_CE, regression=L.NLL_GAUSS, heteroscedastic=L.NLL_GAUSS_HET)


def _check_predictive_mode(mode):
    if mode not in PREDICTIVE_MODES:
        raise ValueError(f"mode must be one of {PREDICTIVE_MODES}, got {mode!r}")


def predictive_acc_len(mode, n_bins):
    """Length of the fp64 aggregate vector of bbb_predictive_stats (include/bbb.h)."""
    return 5 + 3 * n_bins if mode == 'classification' else 4


def _predictive_launch(out, target, mode, sigma, n_bins, mean, row_stats, pred, acc):
    S, B, Cc = out.shape
    kind = _PREDICTIVE_KIND[mode]
    L.check(L.lib().bbb_predictive_stats(L.ptr(out), L.ptr(target), S, B, Cc, kind, float(sigma), int(n_bins),
                                         L.ptr(mean), L.ptr(row_stats), L.ptr(pred), L.ptr(acc), L.stream()),
            'bbb_predictive_stats')


def _predictive_target(target, mode, B, Cc):
    """The target as the kernel reads it, row for row: int64 [B] labels, or float [B, D] ([B] when D = 1), where D = Cc
    except for the heteroscedastic likelihood's Cc = 2D outputs."""
    if target is None:
        return None
    L.require_cuda(target)
    if mode == 'heteroscedastic':
        Cc //= 2
    if mode == 'classification':
        if target.dtype != torch.int64 or tuple(target.shape) != (B,):
            raise ValueError(f'classification target must be int64 of shape ({B},), got {target.dtype} '
                             f'{tuple(target.shape)}')
        return target.contiguous()
    if not (tuple(target.shape) == (B, Cc) or (Cc == 1 and tuple(target.shape) == (B,))):
        raise ValueError(f'regression target must have shape ({B}, {Cc})' + (f' or ({B},)' if Cc == 1 else '') +
                         f', got {tuple(target.shape)}')
    return _f32c(target).reshape(B, Cc)


def _predictive_outputs(B, Cc, mode, n_bins, target, device):
    k = 5 if mode == 'classification' else Cc + 1
    mean = torch.empty((B, Cc // 2 if mode == 'heteroscedastic' else Cc), dtype=torch.float32, device=device)
    row_stats = torch.empty((B, k), dtype=torch.float32, device=device)
    pred = torch.empty(B, dtype=torch.int64, device=device) if mode == 'classification' else None
    acc = torch.zeros(predictive_acc_len(mode, n_bins), dtype=torch.float64, device=device) if target is not None \
        else None
    return mean, row_stats, pred, acc


def predictive_stats(out, target=None, mode='classification', sigma=1.0, n_bins=15):
    """[S,B,C] sampled outputs -> (mean [B,C], row_stats [B,K], pred [B] or None, acc or None), device tensors, one
    launch (bbb_predictive_stats; include/bbb.h gives every definition and the layout of row_stats and acc).
    mode 'classification': the outputs are logits and target int64 [B]; 'regression': a Gaussian likelihood with
    std `sigma` and target [B,D] ([B] when D = 1); 'heteroscedastic': the outputs are [f | r] (C = 2D), the likelihood
    N(f, (sigma + softplus(r))^2) with `sigma` as sigma_min, target as 'regression'.  acc (the aggregates) only with a
    target."""
    _check_predictive_mode(mode)
    L.require_cuda(out)
    z = _f32c(out)
    S, B, Cc = z.shape
    if mode == 'heteroscedastic' and Cc % 2:
        raise ValueError(f'heteroscedastic outputs are [f | r]: an even width, got {Cc}')
    tgt = _predictive_target(target, mode, B, Cc)
    mean, row_stats, pred, acc = _predictive_outputs(B, Cc, mode, n_bins, tgt, z.device)
    _predictive_launch(z, tgt, mode, sigma, n_bins, mean, row_stats, pred, acc)
    return mean, row_stats, pred, acc


def predictive_chunk_rows(S, widths, budget=PREDICTIVE_BUDGET_BYTES):
    """Rows per chunk that keep S * rows * sum(widths) * 4 bytes of activations under `budget`."""
    return max(1, budget // (4 * S * sum(widths)))


def predictive(x2, params, S, mode, target=None, sigma=1.0, n_bins=15, chunk_rows=None, prior=None, sigma_p=None,
               tf32=False):
    """Posterior predictive of a whole input set: the sampled forward (the kernels sample_predict runs) chunk by chunk,
    each chunk's [S, rows, C] outputs summarised by bbb_predictive_stats into one set of per-row outputs and one set of
    device aggregates.  Weight sampling when `prior` is given, local reparameterisation when `sigma_p` is.
    Returns (mean, row_stats, pred, acc) as predictive_stats does.  Nothing here waits for the device.

    Noise, and what chunking changes:
      * weight sampling: eps is planned ONCE per call and every chunk reuses the plan (the same injected tensors in
        the reference eps mode, the same Philox (seed, step) otherwise), so every row is scored by the same S posterior
        networks and the result does not depend on chunk_rows beyond the kernels' round-off.  The call consumes one
        Philox step, as sample_predict does.
      * local reparameterisation: the noise is per row by construction; each chunk draws its own, which equals calling
        the reference's predict chunk by chunk in order.  The call consumes one Philox step PER CHUNK.
    chunk_rows=None picks the largest row count whose activations, S * rows * sum of layer widths * 4 bytes, stay
    under PREDICTIVE_BUDGET_BYTES, and splits the rows into chunks of equal size.
    mode as in predictive_stats ('heteroscedastic': `sigma` is sigma_min)."""
    _check_predictive_mode(mode)
    if (prior is None) == (sigma_p is None):
        raise ValueError('give exactly one of prior (weight sampling) and sigma_p (local reparameterisation)')
    est = _WeightSampling(prior) if sigma_p is None else _LocalReparam(sigma_p)
    return _predictive(est, x2, params, S, mode, target, sigma, n_bins, chunk_rows, tf32)


def _predictive(est, x2, params, S, mode, target, sigma, n_bins, chunk_rows, tf32):
    L.require_cuda(x2, *[t for p in params for t in p])
    x2 = _f32c(x2)
    dev = x2.device
    B = x2.shape[0]
    params = [tuple(_f32c(t) for t in p) for p in params]
    widths = [est.shape(p[0])[1] for p in params]
    Cc = widths[-1]
    tgt = _predictive_target(target, mode, B, Cc)
    mean, row_stats, pred, acc = _predictive_outputs(B, Cc, mode, n_bins, tgt, dev)
    if B == 0:
        return mean, row_stats, pred, acc
    if chunk_rows is None:
        # (counting the delta buffer of each layer, where the estimator keeps one)
        n_chunks = -(-B // predictive_chunk_rows(S, widths * (2 if est.has_delta else 1)))
        chunk_rows = -(-B // n_chunks)
    chunk_rows = int(chunk_rows)
    if chunk_rows < 1:
        raise ValueError(f'chunk_rows must be >= 1, got {chunk_rows}')
    eps = None if est.eps_per_row else plan_eps(est.eps_shapes(params, B), S, dev, True)
    scratch = torch.zeros(2 * S, dtype=torch.float64, device=dev)    # log-prob slots the forward does not fill
    for r0 in range(0, B, chunk_rows):
        r1 = min(B, r0 + chunk_rows)
        xc = x2[r0:r1]
        if xc.data_ptr() % 16:     # keep the 16-byte row loads (and so the kernel family) of an unchunked call
            xc = xc.clone()
        ec = eps if eps is not None else plan_eps(est.eps_shapes(params, r1 - r0), S, dev, True)
        ys, _ = _forward(est, xc, params, S, ec, True, False, tf32, est.lp(scratch, S))
        _predictive_launch(ys[-1], None if tgt is None else tgt[r0:r1], mode, sigma, n_bins, mean[r0:r1],
                           row_stats[r0:r1], None if pred is None else pred[r0:r1], acc)
        del ys                     # free this chunk's activations before the next chunk allocates its own
    return mean, row_stats, pred, acc
