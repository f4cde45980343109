"""CPU TEST DOUBLE of the libbbb.so C ABI (include/bbb.h) -- test infrastructure only.

The product has no CPU path; this double exists so that the `-m "not gpu"` suite can exercise the
Python host (autograd plumbing, argument order, buffer shapes, mode logic) in a container without a
GPU.  It receives exactly the raw pointers / sizes / flags the ctypes layer would hand to the real
library, views them as numpy arrays over CPU tensor storage, and evaluates the documented semantics
with the float64 closed forms of oracle/closed_form.py.  Philox is not emulated: callers must inject
eps ('reference' eps mode).
"""
import ctypes as C

import numpy as np

from oracle import closed_form as CF

F_SAMPLE, F_LOGPROB, F_RELU_IN, F_ACCUM, F_TF32, F_NO_DX, F_SCALE_DX, F_NO_WGRAD = 1, 2, 4, 8, 16, 32, 64, 128
F_OUT_ZEROED, F_DX_PREACT, F_RELU_OUT = 256, 512, 1024


def _arr(ptr, ctype, *shape):
    n = int(np.prod(shape)) if shape else 1
    if n == 0:                      # an empty tensor may carry a null pointer
        return np.zeros(shape, dtype=np.dtype(ctype))
    if not ptr:
        return None
    return np.ctypeslib.as_array((ctype * n).from_address(ptr)).reshape(shape)


def _f(ptr, *shape):
    return _arr(ptr, C.c_float, *shape)


def _d(ptr, *shape):
    return _arr(ptr, C.c_double, *shape)


def _prior(pref):
    p = pref._obj
    return ('mixture', p.pi, p.sigma1, p.sigma2) if p.kind == 1 else ('gaussian', p.sigma1)


class FakeLib:
    calls = []

    def bbb_version(self):
        return 100

    def bbb_last_error_string(self):
        return b'fake'

    def bbb_launch_count(self):
        return len(self.calls)

    # ---------------------------------------------------------------- weight sampling
    def bbb_linear_fwd(self, x, xs, wm, wr, bm, br, ew, eb, rng, prior, S, B, inn, out, flags, y, logp, logq, st):
        self.calls.append('linear_fwd')
        if S == 0 or B == 0 or out == 0:       # an empty call launches nothing and touches no output (bbb.h)
            return 0
        sample, lpq, relu = flags & F_SAMPLE, flags & F_LOGPROB, flags & F_RELU_IN
        assert not sample or (ew and eb), 'fake lib: inject eps (reference eps mode)'
        X = _f(x, S if xs else 1, B, inn).astype(np.float64)
        WM, WR = _f(wm, out, inn).astype(np.float64), _f(wr, out, inn).astype(np.float64) if wr else None
        BM, BR = _f(bm, out).astype(np.float64), _f(br, out).astype(np.float64) if br else None
        EW, EB = _f(ew, S, out, inn), _f(eb, S, out)
        Y, LP, LQ = _f(y, S, B, out), _d(logp, S), _d(logq, S)
        pr = _prior(prior) if prior else None
        for s in range(S):
            xs_ = X[s if xs else 0]
            if relu:
                xs_ = np.maximum(xs_, 0)
            e_w = EW[s].astype(np.float64) if sample else np.zeros_like(WM)
            e_b = EB[s].astype(np.float64) if sample else np.zeros_like(BM)
            if sample or lpq:
                sw, sb = CF.softplus(WR), CF.softplus(BR)
            w = WM + sw * e_w if sample else WM
            b = BM + sb * e_b if sample else BM
            Y[s] = (xs_ @ w.T + b).astype(np.float32)
            if flags & F_RELU_OUT:
                Y[s] = np.maximum(Y[s], 0)
            if lpq:
                LP[s] += CF.prior_terms(w, pr)[0] + CF.prior_terms(b, pr)[0]
                LQ[s] += CF.log_q(sw, e_w) + CF.log_q(sb, e_b)
        return 0

    def bbb_linear_fwd_relu_out_supported(self, B, inn, out, flags):
        # as the library: TF32 mode, batches of >= 384 rows, 16-byte rows, not a head-sized layer
        return int(bool(flags & 16) and B >= 384 and inn % 4 == 0 and inn >= 32 and out >= 32)

    def bbb_linear_bwd(self, dy, mask, x, xs, wm, wr, bm, br, ew, eb, rng, prior, S, B, inn, out, flags, gp, gq,
                       gp_dev, gq_dev, gstride, oscale, dx, gwm, gwr, gbm, gbr, st):
        self.calls.append('linear_bwd')
        sample, relu = flags & F_SAMPLE, flags & F_RELU_IN
        assert not sample or (ew and eb)
        X = _f(x, S if xs else 1, B, inn).astype(np.float64)
        DY = _f(dy, S, B, out).astype(np.float64)
        MK = _f(mask, S, B, out)
        WM, WR = _f(wm, out, inn).astype(np.float64), _f(wr, out, inn).astype(np.float64)
        BM, BR = _f(bm, out).astype(np.float64), _f(br, out).astype(np.float64)
        EW, EB = _f(ew, S, out, inn), _f(eb, S, out)
        GPD, GQD = _f(gp_dev, max(1, S * gstride)), _f(gq_dev, max(1, S * gstride))
        osc = float(_f(oscale, 1)[0]) if oscale else 1.0
        pr = _prior(prior) if prior else None
        sw, sb = CF.softplus(WR), CF.softplus(BR)
        a_wm, a_wr, a_bm, a_br = (np.zeros_like(WM), np.zeros_like(WM), np.zeros_like(BM), np.zeros_like(BM))
        DX = _f(dx, S, B, inn) if not (flags & F_NO_DX) else None
        for s in range(S):
            gps = gp * (float(GPD[s * gstride]) if gp_dev else 1.0)
            gqs = gq * (float(GQD[s * gstride]) if gq_dev else 1.0)
            xs_ = X[s if xs else 0]
            x_pre = xs_
            if relu:
                xs_ = np.maximum(xs_, 0)
            dz = DY[s] * (MK[s] > 0) if mask else DY[s]
            e_w = EW[s].astype(np.float64) if sample else np.zeros_like(WM)
            e_b = EB[s].astype(np.float64) if sample else np.zeros_like(BM)
            w, b = WM + sw * e_w, BM + sb * e_b
            tw, tb = dz.T @ xs_, dz.sum(0)
            if gps != 0.0:
                tw = tw - gps * w * CF.prior_terms(w, pr)[1]
                tb = tb - gps * b * CF.prior_terms(b, pr)[1]
            a_wm += tw
            a_wr += CF.sigmoid(WR) * (tw * e_w - gqs / sw)
            a_bm += tb
            a_br += CF.sigmoid(BR) * (tb * e_b - gqs / sb)
            if DX is not None:
                d = (dz @ w) * (osc if flags & F_SCALE_DX else 1.0)
                if flags & F_DX_PREACT:      # x_pre: the stored input, pre- (with F_RELU_IN) or post-activation
                    d = d * (x_pre > 0)
                DX[s] = d.astype(np.float32)
        if flags & F_NO_WGRAD:                # the gradient buffers are not touched
            return 0
        for ptr, shape, val in ((gwm, (out, inn), a_wm), (gwr, (out, inn), a_wr), (gbm, (out,), a_bm),
                                (gbr, (out,), a_br)):
            G = _f(ptr, *shape)
            G[...] = (G + osc * val if flags & F_ACCUM else osc * val).astype(np.float32)
        return 0

    # ---------------------------------------------------------------- local reparameterisation
    def bbb_lr_linear_fwd(self, x, xs, wm, wr, bm, br, ea, eb, rng, sigma_p, S, B, inn, out, flags, y, delta, kl, st):
        self.calls.append('lr_fwd')
        if S == 0 or B == 0 or out == 0:
            return 0
        sample, calc, relu = flags & F_SAMPLE, flags & F_LOGPROB, flags & F_RELU_IN
        assert not sample or (ea and eb)
        X = _f(x, S if xs else 1, B, inn).astype(np.float64)
        WM, BM = _f(wm, inn, out).astype(np.float64), _f(bm, out).astype(np.float64)
        EA, EB = _f(ea, S, B, out), _f(eb, S, out)
        Y, DL = _f(y, S, B, out), _f(delta, S, B, out)
        if sample or calc:
            sw, sb = CF.softplus(_f(wr, inn, out).astype(np.float64)), CF.softplus(_f(br, out).astype(np.float64))
        for s in range(S):
            xs_ = X[s if xs else 0]
            if relu:
                xs_ = np.maximum(xs_, 0)
            if sample:
                d = np.sqrt((xs_ * xs_) @ (sw * sw))
                Y[s] = (xs_ @ WM + d * EA[s] + (BM + sb * EB[s])).astype(np.float32)
                if DL is not None:
                    DL[s] = d.astype(np.float32)
            else:
                Y[s] = (xs_ @ WM + BM).astype(np.float32)
        if calc:
            _d(kl, 1)[0] += CF.gaussian_kl(WM, sw, sigma_p) + CF.gaussian_kl(BM, sb, sigma_p)
        return 0

    def bbb_lr_linear_bwd(self, dy, mask, x, xs, wm, wr, bm, br, ea, eb, rng, delta, sigma_p, S, B, inn, out, flags,
                          g_kl, g_kl_dev, oscale, dx, gwm, gwr, gbm, gbr, st):
        self.calls.append('lr_bwd')
        sample, calc, relu = flags & F_SAMPLE, flags & F_LOGPROB, flags & F_RELU_IN
        X = _f(x, S if xs else 1, B, inn).astype(np.float64)
        DY, MK = _f(dy, S, B, out).astype(np.float64), _f(mask, S, B, out)
        WM, WR = _f(wm, inn, out).astype(np.float64), _f(wr, inn, out).astype(np.float64)
        BM, BR = _f(bm, out).astype(np.float64), _f(br, out).astype(np.float64)
        EA, EB, DL = _f(ea, S, B, out), _f(eb, S, out), _f(delta, S, B, out)
        osc = float(_f(oscale, 1)[0]) if oscale else 1.0
        gk = (g_kl * (float(_f(g_kl_dev, 1)[0]) if g_kl_dev else 1.0)) if calc else 0.0
        sw, sb = CF.softplus(WR), CF.softplus(BR)
        sp2 = sigma_p * sigma_p
        a_wm = gk * WM / sp2
        acc_v = np.zeros_like(WM)
        a_bm = gk * BM / sp2
        acc_b = np.zeros_like(BM)
        DX = _f(dx, S, B, inn) if not (flags & F_NO_DX) else None
        for s in range(S):
            xs_ = X[s if xs else 0]
            x_pre = xs_
            if relu:
                xs_ = np.maximum(xs_, 0)
            dz = DY[s] * (MK[s] > 0) if mask else DY[s]
            if sample:
                d = DL[s].astype(np.float64)
                with np.errstate(divide='ignore', invalid='ignore'):
                    dV = np.where(d > 0, dz * EA[s] / (2 * d), 0.0)
            else:
                dV = np.zeros_like(dz)
            a_wm = a_wm + xs_.T @ dz
            acc_v += (xs_ * xs_).T @ dV
            a_bm = a_bm + dz.sum(0)
            if sample:
                acc_b += dz.sum(0) * EB[s]
            if DX is not None:
                v = dz @ WM.T + 2 * xs_ * (dV @ (sw * sw).T)
                v = v * (osc if flags & F_SCALE_DX else 1.0)
                if flags & F_DX_PREACT:      # x_pre: the stored input, pre- (with F_RELU_IN) or post-activation
                    v = v * (x_pre > 0)
                DX[s] = v.astype(np.float32)
        a_wr = CF.sigmoid(WR) * (2 * sw * acc_v + gk * (sw / sp2 - 1 / sw))
        a_br = CF.sigmoid(BR) * (acc_b + gk * (sb / sp2 - 1 / sb))
        if flags & F_NO_WGRAD:
            return 0
        for ptr, shape, val in ((gwm, (inn, out), a_wm), (gwr, (inn, out), a_wr), (gbm, (out,), a_bm),
                                (gbr, (out,), a_br)):
            G = _f(ptr, *shape)
            G[...] = (G + osc * val if flags & F_ACCUM else osc * val).astype(np.float32)
        return 0

    # ---------------------------------------------------------------- reductions / likelihood
    def bbb_logprob_reduce(self, mu, rho, eps, seed, step, sample, tensor, prior, n, flags, w_out, logp, logq, st):
        M, Rr = _f(mu, n).astype(np.float64), _f(rho, n).astype(np.float64)
        sg = CF.softplus(Rr)
        if flags & F_SAMPLE:
            assert eps, 'fake lib: inject eps'
            E = _f(eps, n).astype(np.float64)
        else:
            E = np.zeros_like(M)
        w = M + sg * E
        if w_out:
            _f(w_out, n)[...] = w.astype(np.float32)
        _d(logp, 1)[0] += CF.prior_terms(w, _prior(prior))[0]
        _d(logq, 1)[0] += CF.log_q(sg, E)
        return 0

    def bbb_kl_gauss(self, mu, rho, sigma_p, n, kl, st):
        _d(kl, 1)[0] += CF.gaussian_kl(_f(mu, n).astype(np.float64), CF.softplus(_f(rho, n).astype(np.float64)), sigma_p)
        return 0

    def bbb_philox_fill_normal(self, *a):
        raise AssertionError('fake lib: Philox is not emulated')

    def bbb_nll_ce(self, logits, target, S, B, Cc, scale, nll, dlogits, st):
        self.calls.append('nll_ce')
        Z = _f(logits, S, B, Cc).astype(np.float64)
        T = _arr(target, C.c_int64, B)
        G = _f(dlogits, S, B, Cc)
        for s in range(S):
            v, g = CF.nll_and_grad(Z[s], T, 'classification', 1.0)
            _d(nll, 1)[0] += v
            if G is not None:
                G[s] = (scale * g).astype(np.float32)
        return 0

    def bbb_nll_gauss(self, out, target, sigma, S, B, D, scale, nll, dout, st):
        self.calls.append('nll_gauss')
        Z = _f(out, S, B, D).astype(np.float64)
        T = _f(target, B, D).astype(np.float64)
        G = _f(dout, S, B, D)
        for s in range(S):
            v, g = CF.nll_and_grad(Z[s], T, 'regression', sigma)
            _d(nll, 1)[0] += v
            if G is not None:
                G[s] = (scale * g).astype(np.float32)
        return 0

    def bbb_head_fwd(self, x, xs, wm, wr, bm, br, ew, eb, rng, prior, S, B, inn, out, flags, nll_kind, target, sigma,
                     scale, y, dy, logp, logq, nll, beta, beta_dev, out4, done, st):
        """last layer + likelihood + ELBO assembly: the composition of the three calls it replaces"""
        assert out <= 16 and inn % 4 == 0, 'fake lib: bbb_head_fwd shape conditions'
        self.bbb_linear_fwd(x, xs, wm, wr, bm, br, ew, eb, rng, prior, S, B, inn, out, flags, y, logp, logq, st)
        self.calls[-1] = 'head_fwd'
        if nll_kind == 1:
            self.bbb_nll_ce(y, target, S, B, out, scale, nll, dy, st)
            self.calls.pop()
        elif nll_kind == 2:
            self.bbb_nll_gauss(y, target, sigma, S, B, out, scale, nll, dy, st)
            self.calls.pop()
        if out4:
            assert done and _arr(done, C.c_uint32, 1)[0] == 0, 'fake lib: done counter must be zeroed'
            self.bbb_elbo_finalize(logp, logq, None, nll, S, beta, beta_dev, out4, st)
        return 0

    # ---------------------------------------------------------------- the whole network in one call
    def bbb_mlp_supported(self, dims, n_layers, S, B, flags):
        d = list(dims)
        if not (flags & F_TF32) or n_layers < 2 or not (1 <= B <= 128) or S < 1:
            return 0
        hidden_ok = all(d[l] >= 4 and d[l] % 4 == 0 and d[l + 1] >= 4 and d[l + 1] % 4 == 0 for l in range(n_layers - 1))
        return int(hidden_ok and 1 <= d[n_layers] <= 16 and d[n_layers - 1] % 4 == 0 and 4 <= d[n_layers - 1] <= 8192)

    def bbb_mlp_fwd(self, layers, n_layers, x, S, B, rng, prior, flags, nll_kind, target, sigma, scale, d_out, logp, logq,
                    nll, beta, beta_dev, out4, done, st):
        """hidden layers: y = x W_s^T + b_s ADDED into the zero-filled pre-activation buffer, ReLU applied by the consumer;
        last layer: bbb_head_fwd on the last pre-activation"""
        self.calls.append('mlp_fwd')
        n0 = len(self.calls)
        inp, xs = x, 0
        for l in range(n_layers - 1):
            t = layers[l]
            assert t.y and not np.any(_f(t.y, S, B, t.out)), 'fake lib: hidden pre-activation buffers must arrive zeroed'
            self.bbb_linear_fwd(inp, xs, t.w_mu, t.w_rho, t.b_mu, t.b_rho, t.eps_w, t.eps_b, rng, prior, S, B, t.inn,
                                t.out, (flags & (F_SAMPLE | F_LOGPROB)) | (F_RELU_IN if l > 0 else 0), t.y, logp, logq, st)
            inp, xs = t.y, B * t.out
        t = layers[n_layers - 1]
        self.bbb_head_fwd(inp, xs, t.w_mu, t.w_rho, t.b_mu, t.b_rho, t.eps_w, t.eps_b, rng, prior, S, B, t.inn, t.out,
                          (flags & (F_SAMPLE | F_LOGPROB)) | F_RELU_IN, nll_kind, target, sigma, scale, t.y, d_out, logp,
                          logq, nll, beta, beta_dev, out4, done, st)
        del self.calls[n0:]
        self.calls.append('head_fwd')
        return 0

    def bbb_mlp_bwd(self, layers, n_layers, x, S, B, rng, prior, flags, gp, gq, gp_dev, gq_dev, gstride, oscale, st):
        """backward of bbb_mlp_fwd: per layer bbb_linear_bwd on the stored pre-activations; the gradient w.r.t. a hidden
        layer's pre-activation output is ADDED into its (zero-filled) dz buffer"""
        self.calls.append('mlp_bwd')
        n0 = len(self.calls)
        for l in reversed(range(n_layers)):
            t = layers[l]
            inp, xs = (layers[l - 1].y, B * t.inn) if l > 0 else (x, 0)
            fl = (flags & (F_SAMPLE | F_ACCUM)) | ((F_RELU_IN | F_DX_PREACT) if l > 0 else F_NO_DX)
            dx = None
            if l > 0:
                assert not np.any(_f(layers[l - 1].dz, S, B, t.inn)), 'fake lib: hidden dz buffers must be zeroed'
                dx = layers[l - 1].dz
            self.bbb_linear_bwd(t.dz, None, inp, xs, t.w_mu, t.w_rho, t.b_mu, t.b_rho, t.eps_w, t.eps_b, rng, prior, S, B,
                                t.inn, t.out, fl, gp, gq, gp_dev, gq_dev, gstride, oscale, dx, t.g_w_mu, t.g_w_rho,
                                t.g_b_mu, t.g_b_rho, st)
        del self.calls[n0:]
        return 0

    def bbb_elbo_finalize(self, logp, logq, kl, nll, S, beta, beta_dev, out4, st):
        O = _f(out4, 4)
        if beta_dev:
            beta = beta * float(_f(beta_dev, 1)[0])
        nm = np.float32(_d(nll, 1)[0] / S)
        if kl:
            k = np.float32(_d(kl, 1)[0])
            O[:] = [np.float32(beta) * k + nm, k, nm, 0]
        else:
            lp = np.float32(_d(logp, S).astype(np.float32).astype(np.float64).mean())
            lq = np.float32(_d(logq, S).astype(np.float32).astype(np.float64).mean())
            O[:] = [np.float32(beta) * lq - np.float32(beta) * lp + nm, lp, lq, nm]
        return 0

    def bbb_adam_step(self, n, params, grads, exp_avg, exp_avg_sq, sizes, lr, b1, b2, eps, step, step_dev, lr_scale_dev, st):
        t = step + (int(_arr(step_dev, C.c_uint32, 1)[0]) if step_dev else 0)
        if lr_scale_dev:
            lr = lr * float(_f(lr_scale_dev, 1)[0])
        bc1, bc2 = 1 - b1 ** t, 1 - b2 ** t
        for i in range(n):
            k = sizes[i]
            p, g, m, v = (_f(tab[i], k) for tab in (params, grads, exp_avg, exp_avg_sq))
            m[...] = b1 * m + (1 - b1) * g
            v[...] = b2 * v + (1 - b2) * g * g
            p[...] = p - (lr / bc1) * m / (np.sqrt(v) / np.sqrt(bc2) + eps)
        return 0

    def bbb_enable_peer_access(self, dev):
        return 0

    def bbb_ipc_open(self, handle, off, out):
        raise AssertionError('fake lib: no CUDA IPC')

    def bbb_adam_step_peer(self, comm, exp_avg, exp_avg_sq, n, lr, b1, b2, eps, step, step_dev, lr_scale_dev, st):
        c = comm._obj
        assert c.world == 1 and c.rank == 0, 'fake lib: one rank only (peer memory needs GPUs)'
        t = step + (int(_arr(step_dev, C.c_uint32, 1)[0]) if step_dev else 0)
        if lr_scale_dev:
            lr = lr * float(_f(lr_scale_dev, 1)[0])
        bc1, bc2 = 1 - b1 ** t, 1 - b2 ** t
        p, g, m, v = _f(c.params[0], n), _f(c.grads[0], n), _f(exp_avg, n), _f(exp_avg_sq, n)
        m[...] = b1 * m + (1 - b1) * g
        v[...] = b2 * v + (1 - b2) * g * g
        p[...] = p - (lr / bc1) * m / (np.sqrt(v) / np.sqrt(bc2) + eps)
        return 0

    def bbb_snr(self, mu, rho, n, out, st):
        M, Rr = _f(mu, n).astype(np.float64), _f(rho, n).astype(np.float64)
        with np.errstate(divide='ignore'):
            _f(out, n)[...] = (10 * np.log10(np.abs(M) / CF.softplus(Rr))).astype(np.float32)
        return 0

    def bbb_snr_prune(self, mu, rho, n, thr, kept, st):
        M, Rr = _f(mu, n), _f(rho, n)
        with np.errstate(divide='ignore'):
            snr = (10 * np.log10(np.abs(M.astype(np.float64)) / CF.softplus(Rr.astype(np.float64)))).astype(np.float32)
        keep = snr > np.float32(thr)
        M[...] = M * keep
        Rr[...] = Rr * keep
        if kept:
            _arr(kept, C.c_int64, 1)[0] += int(keep.sum())
        return 0

    def bbb_softmax_mean(self, logits, S, B, Cc, probs, st):
        Z = _f(logits, S, B, Cc).astype(np.float64)
        E = np.exp(Z - Z.max(-1, keepdims=True))
        _f(probs, B, Cc)[...] = (E / E.sum(-1, keepdims=True)).mean(0).astype(np.float32)
        return 0

    def bbb_timing_enable(self, on):
        return 0

    def bbb_debug_wgrad_split(self, mode):
        return 0

    def bbb_debug_set_timeline(self, buf):
        return 0

    def bbb_timing_report(self, buf, n):
        raise AssertionError('fake lib: no device timing')

    def bbb_counter_add(self, counter, inc, st):
        _arr(counter, C.c_uint32, 1)[0] += inc
        return 0


def install(monkeypatch):
    """Route bnn_b200 through the double (pytest monkeypatch fixture)."""
    import bnn_b200
    fake = FakeLib()
    FakeLib.calls = []
    monkeypatch.setattr(bnn_b200._lib, 'lib', lambda: fake)
    monkeypatch.setattr(bnn_b200._lib, 'require_cuda', lambda *a: None)
    monkeypatch.setattr(bnn_b200._lib, 'stream', lambda: None)
    return fake
