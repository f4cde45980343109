"""The per-layer C ABI (include/bbb.h) against its float64 CPU double, call for call, family by family.

Each case of the table below calls one entry point of the real libbbb.so (bbb_linear_fwd, bbb_linear_bwd,
bbb_lr_linear_fwd, bbb_lr_linear_bwd) on CUDA tensors and tests.fake_bbb.FakeLib with the same sizes, flags and
scalars on CPU copies, and compares every output buffer.  The library runs with in-kernel Philox eps (and, for some
cases, with the same eps injected through the pointers); the double is handed that stream, materialised by
bbb_philox_fill_normal at the coordinates of bbb.h (weight eps: tensor id 2 layer, bias eps: 2 layer + 1, LR
activation eps: 2 layer; counter word 1 = sample_base + s).

Every case names the kernels it must launch, and torch.profiler confirms that exactly those layer kernels ran, so a
dispatch change that orphans a family fails here instead of silently losing coverage.  The contract is checked as
well as the values: buffers the call writes are pre-filled with NaN, accumulated ones (BBB_F_ACCUM) with random
values of the result's magnitude, and buffers a flag exempts (BBB_F_NO_DX, BBB_F_NO_WGRAD) with a sentinel that must
come back untouched.

Bounds (max-norm per tensor): exact-fp32 families 2e-5 on forward outputs, 5e-5 on dx and the gradients, 1e-5
relative on the log-prob / KL sums.  TF32 families: 5e-3 against the plain double, and a tight bound (TIGHT below)
against the double evaluated on operands rounded the way the kernel rounds them (TF32_ROUNDING).  What remains
after that emulation is fp32 accumulation and the SFU approximations of softplus; where those can tip an operand the
kernel computes itself (a sampled weight, sigma^2, dV) across a TF32 rounding boundary, or move the steep mixture-prior
term of the weight gradient, the element gets an explicit slack instead of a looser bound.  The largest tight errors
observed on a B200 are listed beside TIGHT; the emulation covers the GEMM outputs (y, delta, dx, grad_w_mu,
grad_w_rho), the bias gradients keep the plain bound.  Weights truncated instead of rounded (to_tf32 the identity)
pass the plain check and fail the tight one with errors of 1.3e-4 to 1.3e-3 of the max-norm.

The posterior scales are large here (rho in [-1.5, -0.5], sigma 0.2-0.5, against 0.007-0.02 in training): a wrong or
missing eps term in one K block, batch row or sample group then moves an output by several per cent of its max.
"""
import ctypes as C
import re
import zlib

import numpy as np
import pytest
import torch

from oracle import bbb_oracle as O
from oracle import closed_form as CF
from tests.fake_bbb import (FakeLib, F_SAMPLE, F_LOGPROB, F_RELU_IN, F_ACCUM, F_TF32, F_NO_DX, F_SCALE_DX, F_NO_WGRAD,
                            F_OUT_ZEROED, F_DX_PREACT, F_RELU_OUT)


MIX, GAUSS = ('mixture', 0.5, 1.0, float(np.exp(-6.0))), ('gaussian', 1.0)
RTOL_Y, RTOL_G, RTOL_SUM, RTOL_TF32 = 2e-5, 5e-5, 1e-5, 5e-3
SENTINEL = 7.25


# ---------------------------------------------------------------------------------------------------------------------
# TF32 operand rounding
# ---------------------------------------------------------------------------------------------------------------------
def tf32_rn(a):
    """fp32 -> TF32 as bbb_tc.cuh:to_tf32 does it: add half a TF32 ulp to the bit pattern, drop the low 13 mantissa
    bits (round to nearest, ties away from zero)."""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)
    return ((u + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def tf32_trunc(a):
    """what the tensor core makes of an fp32 operand it reads as it lies: the low 13 mantissa bits dropped"""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)
    return (u & np.uint32(0xFFFFE000)).view(np.float32)


def _exact(a):
    return np.asarray(a, dtype=np.float32)


RND = {'rn': tf32_rn, 'trunc': tf32_trunc, 'exact': _exact}


def tf32_ambiguity(a, mode, ulps=8):
    """For an operand the kernel computes itself (a sampled weight, sigma^2, dV), its fp32 value can differ from the
    emulation's by a few ulps (SFU softplus, fast divide).  Where that few-ulp window straddles a TF32 rounding
    boundary the kernel's TF32 operand may be one TF32 ulp away from the emulated one: returns that possible
    deviation per element (0 elsewhere)."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    low = (a.view(np.uint32) & np.uint32(0x1FFF)).astype(np.int64)
    edge = np.abs(low - 0x1000) <= ulps if mode == 'rn' else (low <= ulps) | (low >= 0x2000 - ulps)
    return np.where(edge, np.spacing(np.abs(a)).astype(np.float64) * 8192.0, 0.0)

# Operand rounding per family and GEMM, read from the kernels.  'rn': staged by a thread through to_tf32 (sampled
# weights; activation tiles of the batch-tiled kernels and of the LR forward).  'trunc': fp32 the tensor core reads
# as stored (TMA-landed tiles, tiles staged without conversion).  Pairs are (activation operand, weight operand) for
# fwd / dgrad and (dz, x) for wgrad; LR: 'mean' = x . mu, 'var' = x^2 . sigma^2 (both squares formed in fp32 first),
# in the backward (dz, mu) / (dV, sigma^2) for dgrad and (x, dz) / (x^2, dV) for wgrad.
TF32_ROUNDING = {
    'sk_fwd':     {'fwd': ('trunc', 'rn')},                        # bbb_linear_sk.cu: x raw, w to_tf32
    'tc_fwd':     {'fwd': ('rn', 'rn')},                           # bbb_linear_tc.cu: st_tile4 for both
    'tc_bwd':     {'dgrad': ('rn', 'rn'), 'wgrad': ('rn', 'rn')},
    'wide_fwd':   {'fwd': ('trunc', 'rn')},                        # bbb_wide.cu: x by TMA, w to_tf32
    'wide_bwd':   {'dgrad': ('trunc', 'rn'), 'wgrad': ('trunc', 'trunc')},   # big_wgrad_kernel: slabs as stored
    'fused_bwd':  {'dgrad': ('trunc', 'rn'), 'wgrad': ('trunc', 'trunc')},   # dz / x tiles raw, Wt to_tf32
    'lr_tc_fwd':  {'mean': ('rn', 'rn'), 'var': ('rn', 'rn')},     # bbb_lr_tc.cu: every operand to_tf32
    'lr_tc_bwd':  {'dgrad_mean': ('trunc', 'trunc'), 'dgrad_var': ('trunc', 'trunc'),
                   'wgrad_mean': ('trunc', 'trunc'), 'wgrad_var': ('trunc', 'trunc')},
}
# Tight bounds after emulation (max-norm per tensor, beyond the slack of tf32_ambiguity and of the mixture prior's
# conditioning, see _emu_linear_bwd): 10x the largest value observed over this table on a B200 (1000 W power limit),
# capped at 5e-5.  The observed maxima, all in the weight-sampling wgrad where they come with the mixture prior:
# wide_bwd 1.2e-5 and fused_bwd 6.4e-6 (headroom 4x and 8x under the cap).
TIGHT = {
    'sk_fwd': 3.2e-5,       # observed 3.2e-6
    'tc_fwd': 2e-5,         # 1.8e-6
    'tc_bwd': 3.5e-5,       # 3.3e-6
    'wide_fwd': 5e-5,       # 6.6e-6
    'wide_bwd': 5e-5,       # 1.2e-5
    'fused_bwd': 5e-5,      # 6.4e-6
    'lr_tc_fwd': 2e-6,      # 1.7e-7
    'lr_tc_bwd': 1e-5,      # 8.4e-7
}

# ---------------------------------------------------------------------------------------------------------------------
# the family table: entry point and the layer kernels a call of the family launches
# ---------------------------------------------------------------------------------------------------------------------
FAMILIES = {
    'head_fwd':       ('fwd', ['head_fwd_kernel']),
    'sk_fwd':         ('fwd', ['fwd_sk_kernel']),
    'wide_fwd':       ('fwd', ['wide_kernel']),
    'tc_fwd':         ('fwd', ['fwd_tc_kernel']),
    'narrow_fwd':     ('fwd', ['narrow_fwd_kernel']),
    'fma_fwd':        ('fwd', ['fwd_fma_kernel']),
    'head_bwd':       ('bwd', ['head_bwd_kernel']),
    'fused_bwd':      ('bwd', ['bwd_fused_kernel']),
    'wide_bwd':       ('bwd', ['wide_kernel', 'big_wgrad_kernel']),
    'tc_bwd':         ('bwd', ['dgrad_tc_kernel', 'wgrad_tc_kernel']),
    'narrow_bwd':     ('bwd', ['narrow_bwd_kernel']),
    'fma_bwd':        ('bwd', ['dgrad_fma_kernel', 'wgrad_fma_kernel']),
    'thin_bwd':       ('bwd', ['dgrad_fma_kernel', 'thin_wgrad_kernel']),
    'lr_tc_fwd':      ('lr_fwd', ['lr_fwd_sk_kernel', 'lr_epilogue_kernel']),
    'lr_narrow_fwd':  ('lr_fwd', ['lr_narrow_fwd_kernel']),
    'lr_fma_fwd':     ('lr_fwd', ['lr_fwd_kernel']),
    'lr_tc_bwd':      ('lr_bwd', ['lr_dv_kernel', 'lr_dgrad_sk_kernel', 'lr_wgrad_tc_kernel']),
    'lr_head_bwd':    ('lr_bwd', ['lr_head_bwd_kernel']),
    'lr_narrow_bwd':  ('lr_bwd', ['lr_narrow_bwd_kernel']),
    'lr_fma_bwd':     ('lr_bwd', ['lr_dgrad_kernel', 'lr_wgrad_kernel']),
}
EXTRA_KERNELS = ['wgrad_combine_kernel', 'lr_epilogue_scalar_kernel']   # reached by a flag or a layout within a family
ALL_KERNELS = sorted({k for _, ks in FAMILIES.values() for k in ks} | set(EXTRA_KERNELS))
DGRAD_KERNELS = {'dgrad_tc_kernel', 'dgrad_fma_kernel', 'lr_dgrad_sk_kernel', 'lr_dgrad_kernel'}
WGRAD_KERNELS = {'wgrad_tc_kernel', 'wgrad_fma_kernel', 'thin_wgrad_kernel', 'big_wgrad_kernel', 'wgrad_combine_kernel',
                 'lr_wgrad_tc_kernel', 'lr_wgrad_kernel'}
LARGE_BATCH = {'wide_fwd', 'wide_bwd'}


def _case(fam, S, B, inn, out, flags, **kw):
    entry = FAMILIES[fam][0]
    c = dict(fam=fam, entry=entry, S=S, B=B, inn=inn, out=out, flags=flags, mask=False, prior=MIX, gp=0.0, gq=0.0,
             gdev=None, oscale=False, xshared=False, sample_base=0, layer=0, inject=False, misalign=False, split=0,
             g_kl=0.0, g_kl_dev=False, kernels=None, tag='')
    c.update(kw)
    if c['kernels'] is None:
        ks = list(FAMILIES[fam][1])
        if entry in ('bwd', 'lr_bwd'):
            if flags & F_NO_DX:
                ks = [k for k in ks if k not in DGRAD_KERNELS and not (fam == 'wide_bwd' and k == 'wide_kernel')]
            if flags & F_NO_WGRAD:
                ks = [k for k in ks if k not in WGRAD_KERNELS]
        c['kernels'] = ks
    return c


def _cid(c):
    fl = '+'.join(n for n, f in (('S', F_SAMPLE), ('LP', F_LOGPROB), ('RI', F_RELU_IN), ('ACC', F_ACCUM), ('TF', F_TF32),
                                 ('NODX', F_NO_DX), ('SDX', F_SCALE_DX), ('NOWG', F_NO_WGRAD), ('OZ', F_OUT_ZEROED),
                                 ('PRE', F_DX_PREACT), ('RO', F_RELU_OUT)) if c['flags'] & f)
    extra = ''.join(['-mask' if c['mask'] else '', f"-gdev{c['gdev']}" if c['gdev'] is not None else '',
                     '-osc' if c['oscale'] else '', '-xsh' if c['xshared'] else '', '-inj' if c['inject'] else '',
                     '-mis' if c['misalign'] else '', f"-split{c['split']}" if c['split'] else '',
                     '-gauss' if c['prior'] is GAUSS else '', f"-{c['tag']}" if c['tag'] else ''])
    return f"{c['fam']}-S{c['S']}B{c['B']}i{c['inn']}o{c['out']}-{fl or 'none'}{extra}"


SL, TF = F_SAMPLE | F_LOGPROB, F_TF32


def _fwd_cases():
    cs = []
    # head: out <= 16, 16-byte rows, 4 <= in <= 8192, both modes, exact fp32
    cs += [_case('head_fwd', 1, 1, 64, 1, SL), _case('head_fwd', 3, 257, 64, 15, SL, layer=2, sample_base=5),
           _case('head_fwd', 3, 4, 36, 16, SL | TF, inject=True), _case('head_fwd', 2, 33, 64, 10, SL | F_RELU_IN,
                                                                         prior=GAUSS),
           _case('head_fwd', 2, 33, 64, 10, 0, tag='mean')]
    # stream-K forward: TF32, B <= 128, out > 16 (the K tail of in = 36; S = 1, 2, 3)
    for S, B, inn, out in ((1, 16, 36, 17), (2, 128, 64, 33), (3, 70, 36, 129)):
        cs.append(_case('sk_fwd', S, B, inn, out, SL | TF, layer=1, sample_base=3))
        cs.append(_case('sk_fwd', S, B, inn, out, SL | TF | F_OUT_ZEROED))
    cs += [_case('sk_fwd', 2, 100, 96, 40, SL | TF | F_RELU_IN, prior=GAUSS, inject=True),
           _case('sk_fwd', 2, 100, 96, 40, TF, tag='mean'), _case('sk_fwd', 2, 100, 96, 40, SL | TF, xshared=True)]
    # large batch: TF32, B >= 384, in, out >= 32 (ragged batch tiles, RELU_OUT, log-probs counted once per tile)
    fam = 'wide_fwd'
    cs += [_case(fam, 2, 384, 64, 33, SL | TF), _case(fam, 1, 513, 96, 129, SL | TF | F_RELU_OUT, layer=1),
           _case(fam, 3, 1030, 36, 129, SL | TF | F_RELU_IN, prior=GAUSS, sample_base=7),
           _case(fam, 2, 513, 64, 48, TF | F_RELU_OUT, tag='mean'), _case(fam, 2, 600, 64, 64, SL | TF, inject=True)]
    # batch-tiled TF32 forward: 128 < B < 384, or B >= 384 with out 17-31
    cs += [_case('tc_fwd', 2, 129, 64, 40, SL | TF), _case('tc_fwd', 3, 383, 36, 33, SL | TF | F_RELU_IN, layer=3),
           _case('tc_fwd', 2, 512, 64, 20, SL | TF, prior=GAUSS), _case('tc_fwd', 2, 200, 64, 40, TF, tag='mean')]
    # narrow: fp32, out <= 16, in > 8192
    cs += [_case('narrow_fwd', 2, 8, 8200, 6, SL), _case('narrow_fwd', 1, 20, 8200, 6, SL | F_RELU_IN, prior=GAUSS)]
    # FMA forward: fp32 with out > 16, or rows that are not 16-byte multiples
    cs += [_case('fma_fwd', 2, 5, 119, 17, SL), _case('fma_fwd', 2, 33, 64, 17, SL | F_RELU_IN, prior=GAUSS),
           _case('fma_fwd', 2, 9, 64, 8, SL, misalign=True), _case('fma_fwd', 3, 9, 119, 8, SL | TF, inject=True),
           _case('fma_fwd', 2, 33, 64, 17, 0, tag='mean'),
           _case('fma_fwd', 2, 0, 64, 17, SL, kernels=[], tag='empty')]     # B = 0: nothing launched, nothing touched
    return cs


def _bwd_matrix(fam, S, B, inn, out, base, **kw):
    """the backward flag matrix on one representative shape of a family"""
    G = dict(gp=0.3, gq=0.7)
    v = [_case(fam, S, B, inn, out, base, **G, **kw),
         _case(fam, S, B, inn, out, base | F_ACCUM, **G, **kw),
         _case(fam, S, B, inn, out, base | F_RELU_IN | F_DX_PREACT, **G, **kw),
         _case(fam, S, B, inn, out, base | F_DX_PREACT, **G, **kw),
         _case(fam, S, B, inn, out, base | F_SCALE_DX, oscale=True, **G, **kw),
         _case(fam, S, B, inn, out, base, gp=-0.4, gq=1.3, gdev=0, prior=GAUSS, **kw),
         _case(fam, S, B, inn, out, base, gp=-0.4, gq=1.3, gdev=1, oscale=True, **kw),
         _case(fam, S, B, inn, out, base | F_NO_DX, **G, **kw),
         _case(fam, S, B, inn, out, base | F_NO_WGRAD, **G, **kw),
         _case(fam, S, B, inn, out, base, xshared=True, **G, **kw),
         _case(fam, S, B, inn, out, base & ~F_SAMPLE, **G, **kw)]
    if fam not in LARGE_BATCH:      # a mask moves a large-batch call to the batch-tiled kernels (tc_bwd 'reroute')
        v.append(_case(fam, S, B, inn, out, base | F_ACCUM, mask=True, **G, **kw))
    return v


def _bwd_cases():
    cs = []
    cs += _bwd_matrix('head_bwd', 3, 33, 64, 10, F_SAMPLE, layer=1, sample_base=2)
    cs += [_case('head_bwd', 3, 5, 64, 16, F_SAMPLE | TF, mask=True, gp=0.3, gq=0.7, gdev=1),
           _case('head_bwd', 1, 257, 36, 1, F_SAMPLE, mask=True, gp=0.3, gq=0.7, inject=True)]
    cs += _bwd_matrix('fused_bwd', 2, 100, 96, 40, F_SAMPLE | TF, layer=2, sample_base=4)
    cs += [_case('fused_bwd', 3, 128, 64, 129, F_SAMPLE | TF, mask=True, gp=0.3, gq=0.7),
           _case('fused_bwd', 2, 64, 36, 33, F_SAMPLE | TF | F_OUT_ZEROED, gp=0.3, gq=0.7, inject=True),
           _case('fused_bwd', 1, 7, 400, 20, F_SAMPLE | TF | F_ACCUM, mask=True, gp=0.3, gq=0.7)]
    fam = 'wide_bwd'
    m = _bwd_matrix(fam, 3, 512, 64, 96, F_SAMPLE | TF, layer=1, sample_base=6)
    cs += [c for c in m if not (c['flags'] & F_DX_PREACT and not c['flags'] & F_RELU_IN)]
    split_ks = FAMILIES[fam][1] + ['wgrad_combine_kernel']
    cs += [_case(fam, 3, 512, 64, 96, F_SAMPLE | TF, gp=0.3, gq=0.7, split=1, kernels=split_ks),
           _case(fam, 4, 600, 64, 96, F_SAMPLE | TF | F_ACCUM, gp=0.3, gq=0.7, split=1, kernels=split_ks),
           _case(fam, 3, 512, 64, 96, F_SAMPLE | TF | F_ACCUM, gp=0.3, gq=0.7, split=-1),
           _case(fam, 2, 1030, 36, 132, F_SAMPLE | TF | F_RELU_IN | F_DX_PREACT, gp=0.3, gq=0.7, inject=True)]
    # the large-batch dgrad / wgrad do not take a dy mask: a masked call goes to the batch-tiled kernels
    cs += [_case('tc_bwd', 2, 600, 64, 96, F_SAMPLE | TF, mask=True, gp=0.3, gq=0.7, tag='reroute'),
           _case('tc_bwd', 2, 600, 64, 96, F_SAMPLE | TF | F_ACCUM, mask=True, gp=0.3, gq=0.7, tag='reroute'),
           # ... and so does a dy whose rows are not 16-byte multiples (out % 4 != 0)
           _case('tc_bwd', 2, 1030, 36, 129, F_SAMPLE | TF | F_RELU_IN | F_DX_PREACT, gp=0.3, gq=0.7, tag='reroute')]
    cs += _bwd_matrix('tc_bwd', 2, 129, 64, 40, F_SAMPLE | TF, layer=3, sample_base=1)
    cs += [_case('tc_bwd', 3, 300, 36, 33, F_SAMPLE | TF | F_ACCUM, mask=True, gp=0.3, gq=0.7),
           _case('tc_bwd', 2, 512, 64, 20, F_SAMPLE | TF, gp=0.3, gq=0.7, inject=True)]
    cs += _bwd_matrix('narrow_bwd', 2, 8, 8200, 6, F_SAMPLE)
    cs += _bwd_matrix('fma_bwd', 2, 9, 119, 17, F_SAMPLE, layer=1, sample_base=3)
    cs += [_case('fma_bwd', 2, 33, 64, 40, F_SAMPLE, mask=True, gp=0.3, gq=0.7, misalign=True),
           _case('fma_bwd', 3, 9, 119, 17, F_SAMPLE | TF | F_ACCUM, mask=True, gp=0.3, gq=0.7, inject=True),
           _case('fma_bwd', 2, 0, 64, 17, F_SAMPLE, gp=0.3, gq=0.7, kernels=['wgrad_fma_kernel'], tag='empty'),
           _case('fma_bwd', 2, 0, 64, 17, F_SAMPLE | F_ACCUM | F_NO_DX, gp=0.3, gq=0.7, gdev=1,
                 kernels=['wgrad_fma_kernel'], tag='empty')]
    cs += [_case('thin_bwd', 3, 40, 3, 20, F_SAMPLE, mask=True, gp=0.3, gq=0.7),
           _case('thin_bwd', 9, 40, 5, 33, F_SAMPLE | F_ACCUM, gp=0.3, gq=0.7, gdev=1)]
    return cs


def _lr_fwd_cases():
    LP = F_SAMPLE | F_LOGPROB
    cs = [_case('lr_tc_fwd', 2, 64, 36, 4, LP | TF), _case('lr_tc_fwd', 2, 128, 64, 132, LP | TF, layer=1, sample_base=2),
          _case('lr_tc_fwd', 2, 128, 64, 132, LP | TF | F_OUT_ZEROED), _case('lr_tc_fwd', 3, 33, 96, 40, LP | TF | F_RELU_IN,
                                                                             inject=True),
          _case('lr_tc_fwd', 2, 100, 64, 130, LP | TF, kernels=['lr_fwd_sk_kernel', 'lr_epilogue_scalar_kernel']),
          _case('lr_tc_fwd', 2, 100, 64, 40, F_LOGPROB | TF, kernels=['lr_fwd_sk_kernel'], tag='mean')]
    cs += [_case('lr_narrow_fwd', 2, 5, 64, 10, LP), _case('lr_narrow_fwd', 3, 33, 119, 16, LP | F_RELU_IN, layer=2),
           _case('lr_narrow_fwd', 2, 5, 64, 10, LP | TF, misalign=True)]   # a misaligned x leaves the tensor path
    cs += [_case('lr_fma_fwd', 2, 129, 64, 40, LP), _case('lr_fma_fwd', 2, 700, 64, 40, LP | TF, sample_base=9),
           _case('lr_fma_fwd', 2, 129, 64, 40, LP | TF | F_RELU_IN, xshared=True),
           _case('lr_fma_fwd', 2, 33, 119, 40, LP, inject=True), _case('lr_fma_fwd', 2, 33, 64, 40, F_LOGPROB, tag='mean')]
    return cs


def _lr_bwd_matrix(fam, S, B, inn, out, base, **kw):
    G = dict(g_kl=0.3)
    return [_case(fam, S, B, inn, out, base, **G, **kw),
            _case(fam, S, B, inn, out, base | F_ACCUM, **G, **kw),
            _case(fam, S, B, inn, out, base | F_RELU_IN | F_DX_PREACT, **G, **kw),
            _case(fam, S, B, inn, out, base | F_DX_PREACT, **G, **kw),
            _case(fam, S, B, inn, out, base | F_SCALE_DX, oscale=True, **G, **kw),
            _case(fam, S, B, inn, out, base, g_kl=-0.4, g_kl_dev=True, oscale=True, **kw),
            _case(fam, S, B, inn, out, base | F_NO_DX, **G, **kw),
            _case(fam, S, B, inn, out, base | F_NO_WGRAD, **G, **kw),
            _case(fam, S, B, inn, out, base, xshared=True, **G, **kw),
            _case(fam, S, B, inn, out, base & ~F_LOGPROB, **kw)] + (
        [] if fam == 'lr_tc_bwd' else          # a mask or SAMPLE off moves a tensor-path call to the exact kernels
        [_case(fam, S, B, inn, out, base | F_ACCUM, mask=True, **G, **kw),
         _case(fam, S, B, inn, out, base & ~F_SAMPLE, **G, **kw)])


def _lr_bwd_cases():
    LP = F_SAMPLE | F_LOGPROB
    cs = _lr_bwd_matrix('lr_tc_bwd', 2, 64, 64, 40, LP | TF, layer=1, sample_base=3)
    cs += [_case('lr_tc_bwd', 3, 128, 36, 132, LP | TF | F_ACCUM | F_SCALE_DX, g_kl=0.3, oscale=True, inject=True),
           _case('lr_tc_bwd', 2, 100, 64, 40, LP | TF | F_OUT_ZEROED, g_kl=0.3)]
    cs += _lr_bwd_matrix('lr_head_bwd', 2, 16, 64, 10, LP)
    cs += [_case('lr_head_bwd', 3, 33, 64, 10, LP | TF, mask=True, g_kl=0.3)]      # TF32 with a mask: exact head
    cs += _lr_bwd_matrix('lr_narrow_bwd', 2, 16, 119, 10, LP, layer=2)
    cs += _lr_bwd_matrix('lr_fma_bwd', 2, 33, 64, 40, LP)
    cs += [_case('lr_fma_bwd', 2, 129, 64, 40, LP | TF, mask=True, g_kl=0.3, tag='reroute'),
           _case('lr_fma_bwd', 2, 64, 64, 40, LP | TF | F_ACCUM, mask=True, g_kl=0.3, tag='reroute'),
           _case('lr_fma_bwd', 2, 64, 64, 40, F_LOGPROB | TF, g_kl=0.3, tag='mean'),
           _case('lr_fma_bwd', 2, 33, 119, 40, LP, mask=True, g_kl=0.3, inject=True),
           # B = 0: no dx; the gradients are the KL terms alone (null activation pointers, as for bbb_linear_bwd)
           _case('lr_fma_bwd', 2, 0, 64, 40, LP, g_kl=0.3, kernels=['lr_wgrad_kernel'], tag='empty'),
           _case('lr_fma_bwd', 2, 0, 64, 40, LP | F_ACCUM | F_NO_DX, g_kl=-0.4, g_kl_dev=True, oscale=True,
                 kernels=['lr_wgrad_kernel'], tag='empty')]
    return cs


def _with_rng_twins(cases):
    """every case runs with in-kernel Philox; a case that injects eps through the pointers gets an rng-mode twin"""
    out, ids = [], set()
    for c in cases:
        out.append(c)
        ids.add(_cid(c))
    for c in cases:
        if c['inject']:
            t = dict(c, inject=False)
            if _cid(t) not in ids:
                out.append(t)
                ids.add(_cid(t))
    return out


CASES = _with_rng_twins(_fwd_cases() + _bwd_cases() + _lr_fwd_cases() + _lr_bwd_cases())


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the table covers every family and every kernel, and the double it relies on is itself right
# ---------------------------------------------------------------------------------------------------------------------
def test_family_table_covers_every_kernel_family():
    fams = {c['fam'] for c in CASES}
    assert fams == set(FAMILIES), set(FAMILIES) - fams
    launched = {k for c in CASES for k in c['kernels']}
    assert launched == set(ALL_KERNELS), set(ALL_KERNELS) - launched
    assert len({_cid(c) for c in CASES}) == len(CASES), 'case ids must be unique'
    for fam in TF32_ROUNDING:
        assert any(c['flags'] & F_TF32 for c in CASES if c['fam'] == fam), fam
    # every backward family meets the flag matrix: ACCUM, mask, RELU_IN + DX_PREACT, SCALE_DX, gp_dev strides 0 / 1,
    # NO_DX, NO_WGRAD, shared x, SAMPLE off
    for fam, (entry, _) in FAMILIES.items():
        if entry != 'bwd' or fam == 'thin_bwd':
            continue
        cs = [c for c in CASES if c['fam'] == fam]
        want = [lambda c: c['flags'] & F_ACCUM, lambda c: c['flags'] & F_RELU_IN and c['flags'] & F_DX_PREACT,
                lambda c: c['flags'] & F_SCALE_DX and c['oscale'], lambda c: c['gdev'] == 0, lambda c: c['gdev'] == 1,
                lambda c: c['flags'] & F_NO_DX, lambda c: c['flags'] & F_NO_WGRAD, lambda c: c['xshared'],
                lambda c: not c['flags'] & F_SAMPLE]
        if fam not in LARGE_BATCH:
            want.append(lambda c: c['mask'])
        for i, w in enumerate(want):
            assert any(w(c) for c in cs), (fam, i)
    # ... and every LR backward family: ACCUM, mask, RELU_IN + DX_PREACT, DX_PREACT alone, SCALE_DX, g_kl_dev,
    # NO_DX, NO_WGRAD, shared x, LOGPROB off, SAMPLE off (the last two and the mask not on the tensor path, which
    # none of them reaches)
    for fam, (entry, _) in FAMILIES.items():
        if entry != 'lr_bwd':
            continue
        cs = [c for c in CASES if c['fam'] == fam]
        want = [lambda c: c['flags'] & F_ACCUM, lambda c: c['flags'] & F_RELU_IN and c['flags'] & F_DX_PREACT,
                lambda c: c['flags'] & F_DX_PREACT and not c['flags'] & F_RELU_IN,
                lambda c: c['flags'] & F_SCALE_DX and c['oscale'], lambda c: c['g_kl_dev'],
                lambda c: c['flags'] & F_NO_DX, lambda c: c['flags'] & F_NO_WGRAD, lambda c: c['xshared'],
                lambda c: not c['flags'] & F_LOGPROB]
        if fam != 'lr_tc_bwd':
            want += [lambda c: c['mask'], lambda c: not c['flags'] & F_SAMPLE]
        for i, w in enumerate(want):
            assert any(w(c) for c in cs), (fam, i)
    assert all(any(not c['inject'] and _cid(dict(c, inject=True)) == _cid(d) for c in CASES)
               for d in CASES if d['inject']), 'every injected case has an rng-mode twin'


def test_kernel_name_matching_is_exact():
    names = ['void bbb::(anonymous namespace)::lr_fwd_sk_kernel<true>(bbb::LrArgs, int, int, int)',
             'void bbb::(anonymous namespace)::lr_wgrad_tc_kernel(bbb::LrArgs, float const*, int)',
             '_ZN3bbb12_GLOBAL__N_116lr_narrow_fwd_kernelEN3bbb6LrArgsEi']
    assert _matched(names) == {'lr_fwd_sk_kernel', 'lr_wgrad_tc_kernel', 'lr_narrow_fwd_kernel'}
    assert _matched(['void bbb::fwd_sk_kernel<32, 2>(bbb::LinArgs)',
                     '_ZN3bbb16big_wgrad_kernelILb1EEEv14CUtensorMap_stS1_NS_7LinArgsENS_9WgradPartE']) == \
        {'fwd_sk_kernel', 'big_wgrad_kernel'}


def test_tf32_rounding_helpers_on_bit_patterns():
    def f(bits):
        return np.array([bits], dtype=np.uint32).view(np.float32)

    def bits(a):
        return int(np.asarray(a, np.float32).view(np.uint32)[0])
    lo = 0x3F800000                 # 1.0; TF32 ulp = 0x2000 in the fp32 bit pattern, halfway = 0x1000
    assert bits(tf32_rn(f(lo + 0x0FFF))) == lo             # just below the halfway point: down
    assert bits(tf32_rn(f(lo + 0x1000))) == lo + 0x2000    # exactly halfway: away from zero
    assert bits(tf32_rn(f(lo + 0x1001))) == lo + 0x2000    # just above: up
    assert bits(tf32_trunc(f(lo + 0x1FFF))) == lo
    neg = 0xBF800000                # -1.0: rounding acts on the magnitude
    assert bits(tf32_rn(f(neg + 0x1000))) == neg + 0x2000
    assert bits(tf32_rn(f(neg + 0x0FFF))) == neg
    assert bits(tf32_trunc(f(neg + 0x1FFF))) == neg
    x = np.float32(1.0) + np.float32(2.0 ** -11)           # exactly representable halfway value
    assert tf32_rn(np.array([x]))[0] == np.float32(1.0 + 2.0 ** -10)
    assert tf32_trunc(np.array([x]))[0] == np.float32(1.0)
    # a TF32 value is a fixed point of both
    v = tf32_rn(np.random.default_rng(0).standard_normal(1000).astype(np.float32))
    assert np.array_equal(tf32_rn(v), v) and np.array_equal(tf32_trunc(v), v)


def _f32(a):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32))


def _fake_linear(S, B, inn, out, flags, x, wm, wr, bm, br, ew, eb, prior, dy=None, mask=None, gp=0.0, gq=0.0,
                 gpd=None, gqd=None, gstride=0, osc=None, g0=None, dx0=None, fwd=False):
    """one call of FakeLib on CPU tensors; returns the written buffers"""
    fake = FakeLib()
    pr = _prior_struct(prior)
    P = lambda t: 0 if t is None else t.data_ptr()
    xs = B * inn if x.shape[0] == S and S > 1 else 0
    if fwd:
        y = torch.full((S, B, out), float('nan'))
        lp, lq = torch.zeros(S, dtype=torch.float64), torch.zeros(S, dtype=torch.float64)
        fake.bbb_linear_fwd(P(x), xs, P(wm), P(wr), P(bm), P(br), P(ew), P(eb), None, C.byref(pr), S, B, inn, out, flags,
                            P(y), P(lp), P(lq), None)
        return y, lp, lq
    dx = torch.full((S, B, inn), float('nan')) if dx0 is None else dx0.clone()
    g = [torch.full(sh, SENTINEL if flags & F_NO_WGRAD else float('nan')) for sh in ((out, inn), (out, inn), (out,), (out,))] \
        if g0 is None else [t.clone() for t in g0]
    fake.bbb_linear_bwd(P(dy), P(mask), P(x), xs, P(wm), P(wr), P(bm), P(br), P(ew), P(eb), None, C.byref(pr), S, B,
                        inn, out, flags, gp, gq, P(gpd), P(gqd), gstride, P(osc), P(dx), *[P(t) for t in g], None)
    return dx, g


def _prior_struct(prior):
    from bnn_b200 import _lib as L
    if prior[0] == 'mixture':
        return L.Prior(L.PRIOR_MIXTURE, prior[1], prior[2], prior[3])
    return L.Prior(L.PRIOR_GAUSSIAN, 0.0, prior[1], 0.0)


def _layer_np(gen, inn, out, lr=False):
    shp = (inn, out) if lr else (out, inn)
    wm = gen.uniform(-0.2, 0.2, shp).astype(np.float32)
    wr = gen.uniform(-1.5, -0.5, shp).astype(np.float32)
    bm = gen.uniform(-0.2, 0.2, out).astype(np.float32)
    br = gen.uniform(-1.5, -0.5, out).astype(np.float32)
    return wm, wr, bm, br


@pytest.mark.parametrize('flags,mask,gdev,osc,xshared,S,B', [
    (F_SAMPLE, False, None, False, False, 2, 5), (F_SAMPLE | F_ACCUM, True, None, False, False, 2, 5),
    (F_SAMPLE | F_RELU_IN | F_DX_PREACT, True, 0, True, False, 3, 4), (F_SAMPLE | F_DX_PREACT | F_SCALE_DX, False, 1, True,
                                                                    True, 3, 4),
    (F_SAMPLE | F_NO_DX, False, 1, False, False, 2, 3), (F_SAMPLE | F_NO_WGRAD, True, None, True, False, 2, 3),
    (0, True, 0, False, False, 2, 3), (F_SAMPLE, False, 1, True, False, 2, 0), (F_SAMPLE | F_ACCUM, False, 0, False,
                                                                             False, 3, 0)])
@pytest.mark.parametrize('prior', [MIX, GAUSS], ids=['mixture', 'gaussian'])
def test_fake_linear_matches_autograd_oracle(flags, mask, gdev, osc, xshared, S, B, prior):
    """FakeLib's bbb_linear_fwd / bbb_linear_bwd against float64 autograd through oracle.bayes_linear: the loss
    sum_s [ <dY_s, Y_s> + gp_s log p_s + gq_s log q_s ] (gp_s = gp gp_dev[s stride], ...) differentiated w.r.t. x and
    the four parameters gives dx (here the gradient of the ReLU'd input unless DX_PREACT) and grad_* times
    out_scale."""
    gen = np.random.default_rng(S * 100 + B + flags)
    inn, out = 7, 5
    wm, wr, bm, br = _layer_np(gen, inn, out)
    x = gen.standard_normal((1 if xshared else S, B, inn)).astype(np.float32)
    ew, eb = gen.standard_normal((S, out, inn)).astype(np.float32), gen.standard_normal((S, out)).astype(np.float32)
    dy = gen.standard_normal((S, B, out)).astype(np.float32)
    mk = gen.standard_normal((S, B, out)).astype(np.float32) if mask else None
    gp, gq = 0.3, -0.6
    gpd = gen.uniform(0.5, 1.5, S if gdev == 1 else 1).astype(np.float32) if gdev is not None else None
    gqd = gen.uniform(0.5, 1.5, S if gdev == 1 else 1).astype(np.float32) if gdev is not None else None
    oscv = np.array([0.7], np.float32) if osc else None
    g0 = [gen.standard_normal(s).astype(np.float32) for s in ((out, inn), (out, inn), (out,), (out,))]
    T = lambda a: None if a is None else _f32(a)
    dx, g = _fake_linear(S, B, inn, out, flags, T(x), T(wm), T(wr), T(bm), T(br), T(ew), T(eb), prior, dy=T(dy),
                         mask=T(mk), gp=gp, gq=gq, gpd=T(gpd), gqd=T(gqd), gstride=1 if gdev == 1 else 0, osc=T(oscv),
                         g0=[_f32(t) for t in g0] if flags & F_ACCUM else None,
                         dx0=torch.full((S, B, inn), SENTINEL))
    # float64 autograd; every sample has its own input leaf (the ABI writes one dx per sample even for a shared x),
    # holding the input as the layer uses it (ReLU'd under RELU_IN): dx is the gradient w.r.t. that input
    pri = O.make_prior([1.0], False) if prior is GAUSS else ('mixture', 0.5, 1.0, float(np.exp(-6.0)))
    D = lambda a: torch.tensor(np.asarray(a, np.float64), requires_grad=True)
    xin = [x[0 if xshared else s] for s in range(S)]
    Xs = [D(np.maximum(v, 0) if flags & F_RELU_IN else v) for v in xin]
    P = [D(t) for t in (wm, wr, bm, br)]
    loss = 0
    for s in range(S):
        if flags & F_SAMPLE:
            yv, lp, lq = O.bayes_linear(Xs[s], P, pri, torch.tensor(ew[s], dtype=torch.float64),
                                        torch.tensor(eb[s], dtype=torch.float64))
        else:
            yv, lp, lq = O.bayes_linear(Xs[s], P, pri)
        dz = torch.tensor(dy[s], dtype=torch.float64) * (torch.tensor(mk[s]) > 0 if mask else 1.0)
        gps = gp * (float(gpd[s if gdev == 1 else 0]) if gpd is not None else 1.0)
        gqs = gq * (float(gqd[s if gdev == 1 else 0]) if gqd is not None else 1.0)
        # gp, gq are d loss / d logp_s, d loss / d logq_s (bbb.h)
        loss = loss + (dz * yv).sum() + gps * lp + gqs * lq
    loss.backward()
    sc = float(oscv[0]) if osc else 1.0
    for got, p, base in zip(g, P, g0):
        if flags & F_NO_WGRAD:
            assert np.all(got.numpy() == SENTINEL)
            continue
        ref = sc * p.grad.numpy() + (base if flags & F_ACCUM else 0)
        assert np.abs(got.numpy() - ref).max() <= 1e-6 * max(1.0, np.abs(ref).max())
    if flags & F_NO_DX or B == 0:
        assert np.all(dx.numpy() == SENTINEL)
        return
    for s in range(S):
        ref = Xs[s].grad.numpy() * (sc if flags & F_SCALE_DX else 1.0)
        if flags & F_DX_PREACT:
            ref = ref * (xin[s] > 0)
        assert np.abs(dx.numpy()[s] - ref).max() <= 1e-6 * max(1.0, np.abs(ref).max())


@pytest.mark.parametrize('flags,mask,gkdev,osc,xshared,S,B', [
    (F_SAMPLE | F_LOGPROB, False, False, False, False, 2, 5), (F_SAMPLE | F_LOGPROB | F_ACCUM, True, False, False, False, 2, 5),
    (F_SAMPLE | F_LOGPROB | F_RELU_IN | F_DX_PREACT, True, True, True, False, 3, 4),
    (F_SAMPLE | F_LOGPROB | F_DX_PREACT | F_SCALE_DX, False, True, True, True, 3, 4),
    (F_SAMPLE | F_LOGPROB | F_RELU_IN, False, False, False, False, 2, 4),
    (F_SAMPLE | F_LOGPROB | F_NO_DX, False, True, False, False, 2, 3),
    (F_SAMPLE | F_LOGPROB | F_NO_WGRAD, True, False, True, False, 2, 3), (F_SAMPLE, True, False, False, False, 2, 3),
    (F_LOGPROB, True, True, True, False, 2, 3), (F_SAMPLE | F_LOGPROB, False, True, True, False, 2, 0),
    (F_SAMPLE | F_LOGPROB | F_ACCUM | F_NO_DX, False, False, False, False, 3, 0)])
def test_fake_lr_matches_autograd_oracle(flags, mask, gkdev, osc, xshared, S, B):
    """FakeLib's bbb_lr_linear_fwd / bbb_lr_linear_bwd against float64 autograd through oracle.lr_linear: the loss
    sum_s <dY_s, Y_s> + g_kl kl (g_kl times g_kl_dev; the KL with BBB_F_LOGPROB only, once per call) differentiated
    w.r.t. each sample's input (the ReLU'd input under RELU_IN, masked by the stored input > 0 under DX_PREACT) and the
    four parameters, times out_scale; the backward is handed the fp32 delta of the double's forward."""
    gen = np.random.default_rng(S * 100 + B + flags + 7 * mask)
    inn, out, sigma_p, g_kl = 7, 5, 0.8, 0.45
    lay = _layer_np(gen, inn, out, lr=True)
    x = gen.standard_normal((1 if xshared else S, B, inn)).astype(np.float32)
    x[..., 0] = np.abs(x[..., 0]) + 0.1           # no all-zero row after the ReLU: delta > 0 everywhere
    ea, eb = gen.standard_normal((S, B, out)).astype(np.float32), gen.standard_normal((S, out)).astype(np.float32)
    dy = gen.standard_normal((S, B, out)).astype(np.float32)
    mk = gen.standard_normal((S, B, out)).astype(np.float32) if mask else None
    gkd = np.array([1.3], np.float32) if gkdev else None
    oscv = np.array([0.7], np.float32) if osc else None
    g0 = [gen.standard_normal(sh).astype(np.float32) for sh in ((inn, out), (inn, out), (out,), (out,))]
    T = lambda a: None if a is None else _f32(a)
    yr, dl, kl = _lr_fake(S, B, inn, out, flags | F_SAMPLE, T(x), [T(t) for t in lay], T(ea), T(eb), sigma_p, fwd=True)
    gst = g0 if flags & F_ACCUM else [np.full(t.shape, SENTINEL if flags & F_NO_WGRAD else np.nan, np.float32) for t in g0]
    dx, g = _lr_fake(S, B, inn, out, flags, T(x), [T(t) for t in lay], T(ea), T(eb), sigma_p, dy=T(dy), mask=T(mk),
                     delta=dl, g_kl=g_kl, gkd=T(gkd), osc=T(oscv), g0=[_f32(t) for t in gst],
                     dx0=torch.full((S, B, inn), SENTINEL))
    D = lambda a: torch.tensor(np.asarray(a, np.float64), requires_grad=True)
    xin = [x[0 if xshared else s] for s in range(S)]
    Xs = [D(np.maximum(v, 0) if flags & F_RELU_IN else v) for v in xin]
    P = [D(t) for t in lay]
    loss = 0
    for s in range(S):
        if flags & F_SAMPLE:
            yv, _ = O.lr_linear(Xs[s], P, sigma_p, torch.tensor(ea[s], dtype=torch.float64),
                                torch.tensor(eb[s], dtype=torch.float64), calc_kl=False)
        else:
            yv, _ = O.lr_linear(Xs[s], P, sigma_p, calc_kl=False)
        dz = torch.tensor(dy[s], dtype=torch.float64) * (torch.tensor(mk[s]) > 0 if mask else 1.0)
        loss = loss + (dz * yv).sum()
    if flags & F_LOGPROB:
        _, klv = O.lr_linear(Xs[0][:0], P, sigma_p, calc_kl=True)
        loss = loss + g_kl * (float(gkd[0]) if gkdev else 1.0) * klv
    loss.backward()
    sc = float(oscv[0]) if osc else 1.0
    for got, p, base in zip(g, P, g0):
        if flags & F_NO_WGRAD:
            assert np.all(got.numpy() == SENTINEL)
            continue
        ref = sc * p.grad.numpy() + (base if flags & F_ACCUM else 0)
        assert np.abs(got.numpy() - ref).max() <= 1e-6 * max(1.0, np.abs(ref).max())
    if flags & F_NO_DX or B == 0:
        assert np.all(dx.numpy() == SENTINEL)
        return
    for s in range(S):
        ref = Xs[s].grad.numpy() * (sc if flags & F_SCALE_DX else 1.0)
        if flags & F_DX_PREACT:
            ref = ref * (xin[s] > 0)
        assert np.abs(dx.numpy()[s] - ref).max() <= 1e-6 * max(1.0, np.abs(ref).max())


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the drivers
# ---------------------------------------------------------------------------------------------------------------------
_NAME_RE = {k: re.compile(r'(?<![A-Za-z_])' + k + r'(?![a-z0-9_])') for k in ALL_KERNELS}


def _matched(names):
    """layer kernels of the table whose name occurs in the profiler's event names (demangled or mangled)"""
    return {k for k, rx in _NAME_RE.items() if any(rx.search(n) for n in names)}


def _profiled(fn):
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        rc = fn()
        torch.cuda.synchronize()
    return rc, _matched([e.name for e in prof.events()])


def _dev(a, misalign=False):
    """CUDA copy of a numpy array; misalign: its data pointer is one float past a 16-byte boundary"""
    t = torch.as_tensor(np.ascontiguousarray(a, dtype=a.dtype))
    if not misalign:
        return t.cuda()
    buf = torch.empty(t.numel() + 4, dtype=t.dtype, device='cuda')
    v = buf[1:1 + t.numel()].view(t.shape)
    v.copy_(t)
    return v


def _P(t):
    return None if t is None else t.data_ptr()


def _eps(c, lr):
    """the Philox stream the kernels generate, materialised at the coordinates of bbb.h"""
    from bnn_b200 import functional as F
    S, B, inn, out, l = c['S'], c['B'], c['inn'], c['out'], c['layer']
    seed, step = 1234 + l, 17
    ew = [F.philox_normal((B * out) if lr else (out * inn), 'cuda', seed, step, c['sample_base'] + s, 2 * l)
          for s in range(S)] if (B > 0 or not lr) else []
    eb = [F.philox_normal(out, 'cuda', seed, step, c['sample_base'] + s, 2 * l + 1) for s in range(S)]
    shape = (S, B, out) if lr else (S, out, inn)
    ew = torch.stack(ew).view(shape).cpu().numpy() if ew else np.zeros(shape, np.float32)
    return ew, torch.stack(eb).cpu().numpy(), seed, step


def _rng(c, seed, step):
    from bnn_b200 import _lib as L
    return L.Rng(seed, step, c['sample_base'], c['layer'], None)


def _err(got, ref):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    assert got.shape == ref.shape
    assert np.isfinite(got).all(), 'non-finite output'
    scale = np.abs(ref).max() if ref.size else 0.0
    d = np.abs(got - ref).max() if ref.size else 0.0
    return d / scale if scale > 0 else d


def _check(c, name, got, ref, bound, emu=None, tight=None):
    """emu: (emulated value, slack) -- the slack covers operands whose TF32 rounding is ambiguous (tf32_ambiguity)"""
    e = _err(got, ref)
    msg = f"ABI_ERR {c['fam']} {_cid(c)} {name} plain={e:.3e}"
    et = None
    if emu is not None:
        val, slack = emu
        scale = np.abs(np.asarray(ref, np.float64)).max()
        et = float(np.maximum(np.abs(np.asarray(got, np.float64) - val) - slack, 0).max() / scale)
        msg += f' tight={et:.3e}'
    print(msg)
    assert e <= bound, (name, e, bound)
    if et is not None:
        assert et <= tight, (name, 'TF32-emulated', et, tight)


def _is_tf32(c):
    return c['fam'] in TF32_ROUNDING and c['flags'] & F_TF32


def _w32(wm, wr, ew, sample):
    """sampled weights as the kernels form them in fp32: fl(mu + fl(sigma eps))"""
    if not sample:
        return np.broadcast_to(wm, ew.shape).astype(np.float32)
    sg = CF.softplus(wr.astype(np.float64)).astype(np.float32)
    return (wm + (sg * ew).astype(np.float32)).astype(np.float32)


def _run_fwd(c):
    from bnn_b200 import _lib as L
    S, B, inn, out, fl = c['S'], c['B'], c['inn'], c['out'], c['flags']
    gen = np.random.default_rng(zlib.crc32(_cid(c).encode()))
    wm, wr, bm, br = _layer_np(gen, inn, out)
    x = gen.standard_normal((1 if c['xshared'] else S, B, inn)).astype(np.float32)
    ew, eb, seed, step = _eps(c, False)
    lp0 = gen.standard_normal(S) * 10
    lq0 = gen.standard_normal(S) * 10
    # real library
    dx_ = _dev(x, c['misalign'])
    d = [_dev(t) for t in (wm, wr, bm, br)]
    y = torch.full((max(S * B * out, 16),), 0.0 if fl & F_OUT_ZEROED else float('nan'), device='cuda')
    if B == 0:
        y.fill_(SENTINEL)
    lp, lq = torch.tensor(lp0, device='cuda'), torch.tensor(lq0, device='cuda')
    inj = (_dev(ew), _dev(eb)) if c['inject'] else (None, None)
    rng, pr = _rng(c, seed, step), _prior_struct(c['prior'])
    xs = B * inn if not c['xshared'] else 0
    rc, ran = _profiled(lambda: L.lib().bbb_linear_fwd(
        _P(dx_), xs, *[_P(t) for t in d], _P(inj[0]), _P(inj[1]), C.byref(rng), C.byref(pr), S, B, inn, out, fl,
        _P(y), _P(lp), _P(lq), None))
    assert rc == 0, L.lib().bbb_last_error_string()
    assert ran == set(c['kernels']), (sorted(ran), c['kernels'])
    if B == 0:
        assert np.all(y.cpu().numpy() == SENTINEL) and np.array_equal(lp.cpu().numpy(), lp0)
        return
    # the double
    T = _f32
    yr, lpr, lqr = _fake_linear(S, B, inn, out, fl, T(x), T(wm), T(wr), T(bm), T(br), T(ew), T(eb), c['prior'], fwd=True)
    ygot = y[:S * B * out].view(S, B, out).cpu().numpy()
    exact = not _is_tf32(c)
    emu = None if exact else _emu_linear_fwd(c, x, wm, wr, bm, br, ew, eb)
    _check(c, 'y', ygot, yr.numpy(), RTOL_Y if exact else RTOL_TF32, emu, TIGHT.get(c['fam']))
    if fl & F_LOGPROB:
        for name, got, ref, v0 in (('logp', lp, lpr, lp0), ('logq', lq, lqr, lq0)):
            got, ref = got.cpu().numpy() - v0, ref.numpy()
            assert np.abs(got - ref).max() <= RTOL_SUM * np.abs(ref).max(), (name, got, ref)
    else:
        assert np.array_equal(lp.cpu().numpy(), lp0) and np.array_equal(lq.cpu().numpy(), lq0)


def _emu_linear_fwd(c, x, wm, wr, bm, br, ew, eb):
    """y on TF32-rounded operands: (value, slack for sampled weights whose rounding is ambiguous)"""
    S, B, out, fl = c['S'], c['B'], c['out'], c['flags']
    ra, rw = [RND[k] for k in TF32_ROUNDING[c['fam']]['fwd']]
    W = _w32(wm, wr, ew, fl & F_SAMPLE)
    bs = _w32(bm, br, eb, fl & F_SAMPLE)
    val, slack = np.empty((S, B, out)), np.zeros((S, B, out))
    wmode = TF32_ROUNDING[c['fam']]['fwd'][1]
    for s in range(S):
        xv = x[0 if c['xshared'] else s]
        xv = np.maximum(xv, 0) if fl & F_RELU_IN else xv
        val[s] = ra(xv).astype(np.float64) @ rw(W[s]).astype(np.float64).T + bs[s]
        if fl & F_SAMPLE:
            slack[s] = np.abs(ra(xv).astype(np.float64)) @ tf32_ambiguity(W[s], wmode).T
    if fl & F_RELU_OUT:
        val = np.maximum(val, 0)
    return val, slack


def _emu_linear_bwd(c, x, wm, wr, ew, dy, mk, gpd, oscv, g0):
    """dx, grad_w_mu, grad_w_rho on TF32-rounded GEMM operands (the rest as the double computes it)"""
    S, B, inn, out, fl = c['S'], c['B'], c['inn'], c['out'], c['flags']
    rnd = TF32_ROUNDING[c['fam']]
    W = _w32(wm, wr, ew, fl & F_SAMPLE).astype(np.float64)
    sw = CF.softplus(wr.astype(np.float64))
    pr = c['prior']
    a_wm, a_wr = np.zeros((out, inn)), np.zeros((out, inn))
    s_wm, s_wr = np.zeros((out, inn)), np.zeros((out, inn))
    dx, dx_slack = np.zeros((S, B, inn)), np.zeros((S, B, inn))
    osc = float(oscv[0]) if oscv is not None else 1.0
    for s in range(S):
        gps = c['gp'] * (float(gpd[0][s if c['gdev'] == 1 else 0]) if gpd else 1.0)
        gqs = c['gq'] * (float(gpd[1][s if c['gdev'] == 1 else 0]) if gpd else 1.0)
        xp = x[0 if c['xshared'] else s]
        xv = np.maximum(xp, 0) if fl & F_RELU_IN else xp
        dz = (dy[s] * (mk[s] > 0) if mk is not None else dy[s]).astype(np.float32)
        e = ew[s].astype(np.float64) if fl & F_SAMPLE else np.zeros((out, inn))
        ra, rb = [RND[k] for k in rnd['dgrad']] if 'dgrad' in rnd else (_exact, _exact)
        d = ra(dz).astype(np.float64) @ rb(W[s].astype(np.float32)).astype(np.float64)
        sl = np.abs(ra(dz).astype(np.float64)) @ tf32_ambiguity(W[s], rnd['dgrad'][1]) if fl & F_SAMPLE else 0.0
        d, sl = d * (osc if fl & F_SCALE_DX else 1.0), sl * (osc if fl & F_SCALE_DX else 1.0)
        if fl & F_DX_PREACT:
            d, sl = d * (xp > 0), sl * (xp > 0)
        dx[s], dx_slack[s] = d, sl
        ra, rb = [RND[k] for k in rnd['wgrad']]
        tw = ra(dz).astype(np.float64).T @ rb(xv).astype(np.float64)
        if gps != 0.0:
            tw = tw - gps * W[s] * CF.prior_terms(W[s], pr)[1]
            if pr[0] == 'mixture':
                # w = mu + sigma eps cancels where |w| << |sigma eps|: the kernel's softplus (a few 1e-7 relative) then
                # moves w by up to |sigma eps| 1e-6, and the mixture's d(w R(w))/dw (up to ~1/sigma2^2) amplifies that.
                # An fp32 effect of the prior term, not of TF32: it is granted as slack.  The 1e-6 is derived, not
                # measured: the PTX ISA bounds ex2.approx to 2^-22.5 relative and lg2.approx to 2^-22.6 absolute, so
                # sigma = ln2 lg2(1 + 2^(rho log2 e)) is within ~6e-7 relative for sigma >= 0.2 (rho >= -1.5 here).
                # For |w| within a few sigma2 of 0 this slack can exceed TIGHT; those elements keep the plain bound.
                h = 1e-7
                dwr = ((W[s] + h) * CF.prior_terms(W[s] + h, pr)[1] - (W[s] - h) * CF.prior_terms(W[s] - h, pr)[1]) / (2 * h)
                sl = abs(gps) * np.abs(dwr) * (np.abs(sw * e) * 1e-6 + 2 * np.spacing(np.abs(W[s]).astype(np.float32)))
                s_wm += sl
                s_wr += CF.sigmoid(wr.astype(np.float64)) * np.abs(e) * sl
        a_wm += tw
        a_wr += CF.sigmoid(wr.astype(np.float64)) * (tw * e - gqs / sw)
    g = [osc * a_wm, osc * a_wr]
    if fl & F_ACCUM:
        g = [g[0] + g0[0], g[1] + g0[1]]
    return (dx, dx_slack), [(g[0], abs(osc) * s_wm), (g[1], abs(osc) * s_wr)]


def _run_bwd(c):
    from bnn_b200 import _lib as L
    S, B, inn, out, fl = c['S'], c['B'], c['inn'], c['out'], c['flags']
    gen = np.random.default_rng(zlib.crc32(_cid(c).encode()))
    wm, wr, bm, br = _layer_np(gen, inn, out)
    x = gen.standard_normal((1 if c['xshared'] else S, B, inn)).astype(np.float32)
    dy = gen.standard_normal((S, B, out)).astype(np.float32)
    mk = gen.standard_normal((S, B, out)).astype(np.float32) if c['mask'] else None
    ew, eb, seed, step = _eps(c, False)
    gpd = None
    if c['gdev'] is not None:
        n = S if c['gdev'] == 1 else 1
        gpd = (gen.uniform(0.5, 1.5, n).astype(np.float32), gen.uniform(0.5, 1.5, n).astype(np.float32))
    oscv = np.array([0.7], np.float32) if c['oscale'] else None
    T = lambda a: None if a is None else _f32(a)
    fake_args = (S, B, inn, out, fl, T(x), T(wm), T(wr), T(bm), T(br), T(ew), T(eb), c['prior'])
    fkw = dict(dy=T(dy), mask=T(mk), gp=c['gp'], gq=c['gq'], gpd=T(gpd[0]) if gpd else None,
               gqd=T(gpd[1]) if gpd else None, gstride=1 if c['gdev'] == 1 else 0, osc=T(oscv))
    g0 = None
    if fl & F_ACCUM:          # accumulate onto values of the result's own magnitude
        _, gref = _fake_linear(*fake_args[:4], fl & ~(F_ACCUM | F_NO_WGRAD), *fake_args[5:], **fkw)
        g0 = [(gen.standard_normal(t.shape) * max(float(t.abs().max()), 1e-3)).astype(np.float32) for t in gref]
    dx0 = np.full((S, B, inn), SENTINEL if fl & F_NO_DX else (0.0 if fl & F_OUT_ZEROED else np.nan), np.float32)
    dxr, gr = _fake_linear(*fake_args, **fkw, g0=[_f32(t) for t in g0] if g0 else None, dx0=_f32(dx0))
    # real library
    shapes = ((out, inn), (out, inn), (out,), (out,))
    gfill = SENTINEL if fl & F_NO_WGRAD else np.nan
    gd = [_dev(g0[k]) if g0 else torch.full(sh, gfill, device='cuda') for k, sh in enumerate(shapes)]
    dxd = _dev(dx0, c['misalign'] and inn % 4 == 0)
    args = [_dev(dy), _dev(mk) if mk is not None else None, _dev(x, c['misalign'])]
    pd = [_dev(t) for t in (wm, wr, bm, br)]
    inj = (_dev(ew), _dev(eb)) if c['inject'] else (None, None)
    gdev = (_dev(gpd[0]), _dev(gpd[1])) if gpd else (None, None)
    osd = _dev(oscv) if oscv is not None else None
    rng, pr = _rng(c, seed, step), _prior_struct(c['prior'])
    xs = 0 if c['xshared'] else B * inn
    lib = L.lib()
    lib.bbb_debug_wgrad_split(c['split'])
    try:
        rc, ran = _profiled(lambda: lib.bbb_linear_bwd(
            _P(args[0]), _P(args[1]), _P(args[2]), xs, *[_P(t) for t in pd], _P(inj[0]), _P(inj[1]), C.byref(rng),
            C.byref(pr), S, B, inn, out, fl, c['gp'], c['gq'], _P(gdev[0]), _P(gdev[1]), 1 if c['gdev'] == 1 else 0,
            _P(osd), _P(dxd), *[_P(t) for t in gd], None))
    finally:
        lib.bbb_debug_wgrad_split(0)
    assert rc == 0, lib.bbb_last_error_string()
    assert ran == set(c['kernels']), (sorted(ran), c['kernels'])
    exact = not _is_tf32(c)
    emu_dx, emu_g = (None, [None, None])
    if not exact:
        emu_dx, emu_g = _emu_linear_bwd(c, x, wm, wr, ew, dy, mk, gpd, oscv, g0)
    tight = TIGHT.get(c['fam'])
    if fl & F_NO_DX:
        assert np.all(dxd.cpu().numpy() == SENTINEL), 'dx written under BBB_F_NO_DX'
    elif B > 0:
        _check(c, 'dx', dxd.cpu().numpy(), dxr.numpy(), RTOL_G if exact else RTOL_TF32, emu_dx, tight)
    for k, name in enumerate(('grad_w_mu', 'grad_w_rho', 'grad_b_mu', 'grad_b_rho')):
        got = gd[k].cpu().numpy()
        if fl & F_NO_WGRAD:
            assert np.array_equal(got, g0[k]) if g0 else np.all(got == SENTINEL), f'{name} written under NO_WGRAD'
            continue
        _check(c, name, got, gr[k].numpy(), RTOL_G if exact else RTOL_TF32, emu_g[k] if k < 2 else None, tight)


def _lr_fake(S, B, inn, out, fl, x, lay, ea, eb, sigma_p, dy=None, mask=None, delta=None, g_kl=0.0, gkd=None, osc=None,
             g0=None, dx0=None, fwd=False):
    fake = FakeLib()
    P = lambda t: 0 if t is None else t.data_ptr()
    xs = B * inn if x.shape[0] == S and S > 1 else 0
    if fwd:
        y, dl = torch.full((S, B, out), float('nan')), torch.full((S, B, out), float('nan'))
        kl = torch.zeros(1, dtype=torch.float64)
        fake.bbb_lr_linear_fwd(P(x), xs, *[P(t) for t in lay], P(ea), P(eb), None, sigma_p, S, B, inn, out, fl, P(y), P(dl),
                               P(kl), None)
        return y, dl, kl
    dx = dx0.clone()
    g = [t.clone() for t in g0]
    fake.bbb_lr_linear_bwd(P(dy), P(mask), P(x), xs, *[P(t) for t in lay], P(ea), P(eb), None, P(delta), sigma_p, S, B,
                           inn, out, fl, g_kl, P(gkd), P(osc), P(dx), *[P(t) for t in g], None)
    return dx, g


def _emu_lr(c, x, wm, wr, bm, br, ea, eb, dy=None, mk=None, delta=None, gk=0.0, oscv=None, g0=None):
    """LR forward (y, delta) or backward (dx, grad_w_mu, grad_w_rho) on TF32-rounded GEMM operands"""
    S, B, fl = c['S'], c['B'], c['flags']
    sg = CF.softplus(wr.astype(np.float64)).astype(np.float32)
    sg2 = (sg * sg).astype(np.float32)
    sp2 = 1.0
    r = TF32_ROUNDING[c['fam']]
    f64 = lambda a: np.asarray(a, np.float64)
    xin = [x[0 if c['xshared'] else s] for s in range(S)]
    xr = [np.maximum(v, 0) if fl & F_RELU_IN else v for v in xin]
    if dy is None:
        (ra, rb), (rc_, rd) = [[RND[k] for k in r[g]] for g in ('mean', 'var')]
        bs = _w32(bm, br, eb, True)
        y, dl = np.empty((S, B, c['out'])), np.empty((S, B, c['out']))
        sy, sd = np.zeros(y.shape), np.zeros(y.shape)
        for s in range(S):
            x2 = f64(rc_((xr[s] * xr[s]).astype(np.float32)))
            gam = f64(ra(xr[s])) @ f64(rb(wm))
            v = x2 @ f64(rd(sg2))
            dl[s] = np.sqrt(v)
            sd[s] = (x2 @ tf32_ambiguity(sg2, r['var'][1])) / (2 * np.maximum(dl[s], 1e-30))
            y[s] = gam + dl[s] * ea[s] + bs[s]
            sy[s] = sd[s] * np.abs(ea[s])
        return (y, sy), (dl, sd)
    osc = float(oscv[0]) if oscv is not None else 1.0
    a_wm = gk * f64(wm) / sp2
    acc_v, acc_vs = np.zeros(wm.shape), np.zeros(wm.shape)
    dx, dxs = np.empty((S, B, c['inn'])), np.empty((S, B, c['inn']))
    for s in range(S):
        dz = (dy[s] * (mk[s] > 0) if mk is not None else dy[s]).astype(np.float32)
        dV = np.where(delta[s] > 0, dz * ea[s] / (2 * delta[s]), 0).astype(np.float32)
        (ra, rb), (rc_, rd) = [[RND[k] for k in r[g]] for g in ('dgrad_mean', 'dgrad_var')]
        v = f64(ra(dz)) @ f64(rb(wm)).T + 2 * f64(xr[s]) * (f64(rc_(dV)) @ f64(rd(sg2)).T)
        sl = 2 * np.abs(f64(xr[s])) * (np.abs(f64(rc_(dV))) @ tf32_ambiguity(sg2, r['dgrad_var'][1]).T +
                                       tf32_ambiguity(dV, r['dgrad_var'][0]) @ np.abs(f64(rd(sg2))).T)
        v, sl = v * (osc if fl & F_SCALE_DX else 1.0), sl * (osc if fl & F_SCALE_DX else 1.0)
        if fl & F_DX_PREACT:
            v, sl = v * (xin[s] > 0), sl * (xin[s] > 0)
        dx[s], dxs[s] = v, sl
        (ra, rb), (rc_, rd) = [[RND[k] for k in r[g]] for g in ('wgrad_mean', 'wgrad_var')]
        a_wm = a_wm + f64(ra(xr[s])).T @ f64(rb(dz))
        acc_v += f64(rc_((xr[s] * xr[s]).astype(np.float32))).T @ f64(rd(dV))
        acc_vs += np.abs(f64(rc_((xr[s] * xr[s]).astype(np.float32)))).T @ tf32_ambiguity(dV, r['wgrad_var'][1])
    s64 = f64(sg)
    a_wr = CF.sigmoid(f64(wr)) * (2 * s64 * acc_v + gk * (s64 / sp2 - 1 / s64))
    g = [osc * a_wm, osc * a_wr]
    if fl & F_ACCUM:
        g = [g[0] + g0[0], g[1] + g0[1]]
    return (dx, dxs), [(g[0], 0.0), (g[1], abs(osc) * CF.sigmoid(f64(wr)) * 2 * s64 * acc_vs)]


def _run_lr(c):
    from bnn_b200 import _lib as L
    S, B, inn, out, fl = c['S'], c['B'], c['inn'], c['out'], c['flags']
    bwd = c['entry'] == 'lr_bwd'
    gen = np.random.default_rng(zlib.crc32(_cid(c).encode()))
    lay = _layer_np(gen, inn, out, lr=True)
    x = gen.standard_normal((1 if c['xshared'] else S, B, inn)).astype(np.float32)
    ea, eb, seed, step = _eps(c, True)
    sigma_p = 1.0
    T = lambda a: None if a is None else _f32(a)
    yr, dlr, klr = _lr_fake(S, B, inn, out, fl | F_SAMPLE if bwd else fl, T(x), [T(t) for t in lay], T(ea), T(eb),
                            sigma_p, fwd=True)
    pd = [_dev(t) for t in lay]
    inj = (_dev(ea), _dev(eb)) if c['inject'] else (None, None)
    rng = _rng(c, seed, step)
    xs = 0 if c['xshared'] else B * inn
    xd = _dev(x, c['misalign'])
    lib = L.lib()
    exact = not _is_tf32(c)
    tight = TIGHT.get(c['fam'])
    if not bwd:
        fill = 0.0 if fl & F_OUT_ZEROED else float('nan')
        y, dl = torch.full((S, B, out), fill, device='cuda'), torch.full((S, B, out), fill, device='cuda')
        kl0 = float(gen.standard_normal() * 10)
        kl = torch.tensor([kl0], dtype=torch.float64, device='cuda')
        rc, ran = _profiled(lambda: lib.bbb_lr_linear_fwd(
            _P(xd), xs, *[_P(t) for t in pd], _P(inj[0]), _P(inj[1]), C.byref(rng), sigma_p, S, B, inn, out, fl, _P(y),
            _P(dl), _P(kl), None))
        assert rc == 0, lib.bbb_last_error_string()
        assert ran == set(c['kernels']), (sorted(ran), c['kernels'])
        emu = (None, None)
        if not exact and fl & F_SAMPLE:
            emu = _emu_lr(c, x, *lay, ea, eb)
        bound = RTOL_Y if exact else RTOL_TF32
        _check(c, 'y', y.cpu().numpy(), yr.numpy(), bound, emu[0], tight)
        if fl & F_SAMPLE:
            _check(c, 'delta', dl.cpu().numpy(), dlr.numpy(), bound, emu[1], tight)
        if fl & F_LOGPROB:
            got = float(kl.cpu()[0]) - kl0
            assert abs(got - float(klr[0])) <= RTOL_SUM * abs(float(klr[0])), (got, float(klr[0]))
        else:
            assert float(kl.cpu()[0]) == kl0
        return
    # backward on the stored forward state of the double (delta in fp32)
    dy = gen.standard_normal((S, B, out)).astype(np.float32)
    mk = gen.standard_normal((S, B, out)).astype(np.float32) if c['mask'] else None
    delta = dlr.numpy()
    gkd = np.array([1.3], np.float32) if c['g_kl_dev'] else None
    oscv = np.array([0.7], np.float32) if c['oscale'] else None
    shapes = ((inn, out), (inn, out), (out,), (out,))
    g0 = None
    dxn = np.full((S, B, inn), np.nan, np.float32)
    base = dict(dy=T(dy), mask=T(mk), delta=T(delta), g_kl=c['g_kl'], gkd=T(gkd), osc=T(oscv))
    if fl & F_ACCUM:
        _, gref = _lr_fake(S, B, inn, out, fl & ~(F_ACCUM | F_NO_WGRAD), T(x), [T(t) for t in lay], T(ea), T(eb), sigma_p,
                           **base, g0=[torch.zeros(sh) for sh in shapes], dx0=_f32(dxn))
        g0 = [(gen.standard_normal(t.shape) * max(float(t.abs().max()), 1e-3)).astype(np.float32) for t in gref]
    gfill = SENTINEL if fl & F_NO_WGRAD else np.nan
    gstart = g0 if g0 else [np.full(sh, gfill, np.float32) for sh in shapes]
    dx0 = np.full((S, B, inn), SENTINEL if fl & F_NO_DX else (0.0 if fl & F_OUT_ZEROED else np.nan), np.float32)
    dxr, gr = _lr_fake(S, B, inn, out, fl, T(x), [T(t) for t in lay], T(ea), T(eb), sigma_p, **base,
                       g0=[_f32(t) for t in gstart], dx0=_f32(dx0))
    gd = [_dev(t) for t in gstart]
    dxd = _dev(dx0)
    dyd, mkd, dld = _dev(dy), _dev(mk) if mk is not None else None, _dev(delta)   # delta: a copy (TF32 overwrites it)
    gkdd, osd = (_dev(gkd) if gkd is not None else None), (_dev(oscv) if oscv is not None else None)
    rc, ran = _profiled(lambda: lib.bbb_lr_linear_bwd(
        _P(dyd), _P(mkd), _P(xd), xs, *[_P(t) for t in pd], _P(inj[0]), _P(inj[1]), C.byref(rng), _P(dld), sigma_p, S, B,
        inn, out, fl, c['g_kl'], _P(gkdd), _P(osd), _P(dxd), *[_P(t) for t in gd], None))
    assert rc == 0, lib.bbb_last_error_string()
    assert ran == set(c['kernels']), (sorted(ran), c['kernels'])
    emu_dx, emu_g = None, [None, None]
    if not exact:
        gk = c['g_kl'] * (float(gkd[0]) if gkd is not None else 1.0) if fl & F_LOGPROB else 0.0
        emu_dx, emu_g = _emu_lr(c, x, *lay, ea, eb, dy=dy, mk=mk, delta=delta, gk=gk, oscv=oscv, g0=g0)
    if fl & F_NO_DX:
        assert np.all(dxd.cpu().numpy() == SENTINEL), 'dx written under BBB_F_NO_DX'
    else:
        _check(c, 'dx', dxd.cpu().numpy(), dxr.numpy(), RTOL_G if exact else RTOL_TF32, emu_dx, tight)
    for k, name in enumerate(('grad_w_mu', 'grad_w_rho', 'grad_b_mu', 'grad_b_rho')):
        got = gd[k].cpu().numpy()
        if fl & F_NO_WGRAD:
            assert np.array_equal(got, gstart[k]), f'{name} written under NO_WGRAD'
            continue
        _check(c, name, got, gr[k].numpy(), RTOL_G if exact else RTOL_TF32, emu_g[k] if k < 2 else None, tight)
        if B == 0:      # an empty batch: the closed-form KL gradient alone (networks.py:109-114), times out_scale
            gk = c['g_kl'] * (float(gkd[0]) if gkd is not None else 1.0) if fl & F_LOGPROB else 0.0
            mu, rho = (lay[0], lay[1]) if k < 2 else (lay[2], lay[3])
            sg = CF.softplus(rho.astype(np.float64))
            kl_g = gk * mu / sigma_p ** 2 if k % 2 == 0 else CF.sigmoid(rho.astype(np.float64)) * gk * (
                sg / sigma_p ** 2 - 1 / sg)
            ref = (float(oscv[0]) if oscv is not None else 1.0) * kl_g + (g0[k] if g0 else 0.0)
            assert np.abs(got - ref).max() <= RTOL_G * np.abs(ref).max(), name


@pytest.mark.gpu
@pytest.mark.parametrize('c', CASES, ids=_cid)
def test_layer_call_matches_double(c):
    {'fwd': _run_fwd, 'bwd': _run_bwd, 'lr_fwd': _run_lr, 'lr_bwd': _run_lr}[c['entry']](c)


@pytest.mark.parametrize('fam', sorted(TF32_ROUNDING))
def test_tf32_emulation_without_rounding_is_the_double(fam, monkeypatch):
    """the emulated references, with every operand left exact, reproduce FakeLib: what the tight check adds is the
    operand rounding and nothing else"""
    monkeypatch.setitem(TF32_ROUNDING, fam, {k: ('exact', 'exact') for k in TF32_ROUNDING[fam]})
    entry = FAMILIES[fam][0]
    S, B, inn, out = 2, 6, 8, 5
    gen = np.random.default_rng(3)
    fl = F_SAMPLE | F_TF32 | F_RELU_IN | F_DX_PREACT | F_SCALE_DX | F_LOGPROB
    c = _case(fam, S, B, inn, out, fl, gp=0.3, gq=0.7, gdev=1, oscale=True, g_kl=0.4)
    lay = _layer_np(gen, inn, out, lr=entry.startswith('lr'))
    x = gen.standard_normal((S, B, inn)).astype(np.float32)
    dy = gen.standard_normal((S, B, out)).astype(np.float32)
    oscv = np.array([0.7], np.float32)
    T = _f32
    if entry.startswith('lr'):
        ea, eb = gen.standard_normal((S, B, out)).astype(np.float32), gen.standard_normal((S, out)).astype(np.float32)
        yr, dlr, _ = _lr_fake(S, B, inn, out, fl, T(x), [T(t) for t in lay], T(ea), T(eb), 1.0, fwd=True)
        if entry == 'lr_fwd':
            (y, _), (dl, _) = _emu_lr(c, x, *lay, ea, eb)
            assert np.abs(y - yr.numpy()).max() <= 1e-5 * np.abs(y).max()
            assert np.abs(dl - dlr.numpy()).max() <= 1e-5 * np.abs(dl).max()
            return
        shapes = ((inn, out), (inn, out), (out,), (out,))
        dxr, gr = _lr_fake(S, B, inn, out, fl, T(x), [T(t) for t in lay], T(ea), T(eb), 1.0, dy=T(dy), delta=dlr,
                           g_kl=0.4, osc=T(oscv), g0=[torch.zeros(sh) for sh in shapes],
                           dx0=torch.zeros(S, B, inn))
        (dx, _), g = _emu_lr(c, x, *lay, ea, eb, dy=dy, delta=dlr.numpy(), gk=0.4, oscv=oscv)
    else:
        ew, eb = gen.standard_normal((S, out, inn)).astype(np.float32), gen.standard_normal((S, out)).astype(np.float32)
        if entry == 'fwd':
            for fwd_flags in (F_SAMPLE | F_TF32 | F_RELU_IN, F_SAMPLE | F_TF32 | F_RELU_OUT, F_TF32 | F_RELU_OUT):
                cf = _case(fam, S, B, inn, out, fwd_flags)
                yr, _, _ = _fake_linear(S, B, inn, out, fwd_flags, T(x), *[T(t) for t in lay], T(ew), T(eb), MIX,
                                        fwd=True)
                val, _ = _emu_linear_fwd(cf, x, *lay, ew, eb)
                assert np.abs(val - yr.numpy()).max() <= 1e-5 * np.abs(val).max(), fwd_flags
            return
        gpd = (gen.uniform(0.5, 1.5, S).astype(np.float32), gen.uniform(0.5, 1.5, S).astype(np.float32))
        dxr, gr = _fake_linear(S, B, inn, out, fl, T(x), *[T(t) for t in lay], T(ew), T(eb), MIX, dy=T(dy), gp=0.3,
                               gq=0.7, gpd=T(gpd[0]), gqd=T(gpd[1]), gstride=1, osc=T(oscv))
        (dx, _), g = _emu_linear_bwd(c, x, lay[0], lay[1], ew, dy, None, gpd, oscv, None)
    assert np.abs(dx - dxr.numpy()).max() <= 1e-5 * np.abs(dx).max()
    for (v, _), r in zip(g, gr[:2]):
        assert np.abs(v - r.numpy()).max() <= 1e-5 * np.abs(v).max()


@pytest.mark.gpu
def test_network_level_backward_accum_adds_what_it_otherwise_writes():
    """bbb_mlp_bwd with BBB_F_ACCUM (kept for every layer, bbb_mlp.cu) adds into G0 exactly the gradients the same call
    writes without it: same forward state, eps and rng.  The hidden layers' dz are summed with red.add in an order that
    is not fixed, so the two calls may differ by fp32 round-off of those sums; beyond that the bound is one rounding of
    the addition G0 + G."""
    from bnn_b200 import _lib as L, functional as F
    torch.manual_seed(0)
    dims, S, B = (64, 96, 80, 10), 2, 64
    params = [tuple(t.cuda() for t in (torch.empty(o, i).uniform_(-0.2, 0.2), torch.empty(o, i).uniform_(-5, -4),
                                        torch.empty(o).uniform_(-0.2, 0.2), torch.empty(o).uniform_(-5, -4)))
              for i, o in zip(dims[:-1], dims[1:])]
    x = torch.randn(B, dims[0], device='cuda')
    target = torch.randint(0, dims[-1], (B,), device='cuda')
    prior = F.make_prior([0.5, 0, -6], True)
    assert L.mlp_supported(dims, S, B, L.F_TF32)
    eps = F._EpsPlan(None, 21, 4)
    ys, dxs, d_out = F._mlp_forward_call(x, target, params, eps, prior, S, B, 1.0, 'classification', True, 0.3, None,
                                         torch.empty(4, device='cuda'))
    nl = len(params)
    scale = torch.tensor([0.9], device='cuda')

    def backward(flags, grads):
        for dz in dxs[1:nl]:
            dz.zero_()                    # the layer above adds (dz W) (y > 0) into the hidden dz buffers
        tab = F._mlp_layer_table(params, eps, ys, list(dxs[1:nl]) + [d_out], grads)
        rng = eps.rng(0)
        rc, ran = _profiled(lambda: L.lib().bbb_mlp_bwd(tab, nl, L.ptr(x), S, B, C.byref(rng), C.byref(prior), flags,
                                                        -0.3 / S, 0.3 / S, None, None, 0, L.ptr(scale), L.stream()))
        assert rc == 0, L.lib().bbb_last_error_string()
        return ran

    g1 = [[torch.full_like(t, float('nan')) for t in p] for p in params]
    backward(L.F_SAMPLE | L.F_TF32, g1)
    g0 = [[torch.randn_like(t) * float(g.abs().max()) for t, g in zip(p, gp)] for p, gp in zip(params, g1)]
    g2 = [[t.clone() for t in p] for p in g0]
    backward(L.F_SAMPLE | L.F_TF32 | L.F_ACCUM, g2)
    for l in range(nl):
        for k in range(4):
            a, b, base = g2[l][k].double(), g1[l][k].double(), g0[l][k].double()
            assert torch.isfinite(b).all()
            ref = base + b
            tol = 2 * 2.0 ** -24 * (base.abs() + b.abs()) + (1e-6 * float(b.abs().max()) if l < nl - 1 else 0.0)
            assert bool(((a - ref).abs() <= tol).all()), (l, k, float((a - ref).abs().max()), float(b.abs().max()))
