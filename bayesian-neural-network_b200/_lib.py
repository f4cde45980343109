"""ctypes binding of libbbb.so (include/bbb.h).  There is NO fallback: if the shared library is
missing or a call fails, a RuntimeError is raised -- the CUDA path is the only path."""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('BBB_LIB') or os.path.join(_HERE, 'libbbb.so')   # BBB_LIB: A/B builds (tools/)

# flags (include/bbb.h)
F_SAMPLE, F_LOGPROB, F_RELU_IN, F_ACCUM, F_TF32, F_NO_DX, F_SCALE_DX, F_NO_WGRAD = 1, 2, 4, 8, 16, 32, 64, 128
F_OUT_ZEROED, F_DX_PREACT, F_RELU_OUT = 256, 512, 1024
PRIOR_GAUSSIAN, PRIOR_MIXTURE = 0, 1
NLL_NONE, NLL_CE, NLL_GAUSS, NLL_GAUSS_HET = 0, 1, 2, 3


class Rng(C.Structure):
    _fields_ = [('seed', C.c_uint64), ('step', C.c_uint32), ('sample_base', C.c_uint32),
                ('layer', C.c_uint32), ('step_dev', C.c_void_p)]


class Prior(C.Structure):
    _fields_ = [('kind', C.c_int32), ('pi', C.c_float), ('sigma1', C.c_float), ('sigma2', C.c_float)]


class PeerComm(C.Structure):
    """struct bbb_peer_comm: every rank's gradient bucket / parameter buffer / flag words as mapped in this process"""
    _fields_ = [('world', C.c_int32), ('rank', C.c_int32), ('grads', C.c_void_p * 8), ('params', C.c_void_p * 8),
                ('flags', C.c_void_p * 8), ('epoch', C.c_void_p), ('done_blocks', C.c_void_p),
                ('mc_grads', C.c_void_p), ('mc_params', C.c_void_p)]


class MlpLayer(C.Structure):
    """struct bbb_mlp_layer: one layer of a network-level call (bbb_mlp_fwd / bbb_mlp_bwd)"""
    _fields_ = [('w_mu', C.c_void_p), ('w_rho', C.c_void_p), ('b_mu', C.c_void_p), ('b_rho', C.c_void_p),
                ('eps_w', C.c_void_p), ('eps_b', C.c_void_p), ('inn', C.c_int64), ('out', C.c_int64),
                ('y', C.c_void_p), ('dz', C.c_void_p),
                ('g_w_mu', C.c_void_p), ('g_w_rho', C.c_void_p), ('g_b_mu', C.c_void_p), ('g_b_rho', C.c_void_p)]


class GaussPriorTensor(C.Structure):
    """struct bbb_gauss_prior_tensor: one weight or bias tensor of a per-weight Gaussian prior call"""
    _fields_ = [('mu', C.c_void_p), ('rho', C.c_void_p), ('prior_mu', C.c_void_p), ('prior_rho', C.c_void_p),
                ('eps', C.c_void_p), ('grad_mu', C.c_void_p), ('grad_rho', C.c_void_p), ('n', C.c_int64),
                ('tensor_id', C.c_uint32)]


GAUSS_PRIOR_MAX_TENSORS = 64

P, I64, I32, F32, F64, U32, U64 = C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_double, C.c_uint32, C.c_uint64
_SIGS = {
    'bbb_version': ([], C.c_int),
    'bbb_last_error_string': ([], C.c_char_p),
    'bbb_launch_count': ([], C.c_uint64),
    'bbb_linear_fwd': ([P, I64, P, P, P, P, P, P, P, P, I64, I64, I64, I64, I32, P, P, P, P], C.c_int),
    'bbb_linear_bwd': ([P, P, P, I64, P, P, P, P, P, P, P, P, I64, I64, I64, I64, I32, F32, F32, P, P, I64, P,
                        P, P, P, P, P, P], C.c_int),
    'bbb_lr_linear_fwd': ([P, I64, P, P, P, P, P, P, P, F32, I64, I64, I64, I64, I32, P, P, P, P], C.c_int),
    'bbb_lr_linear_bwd': ([P, P, P, I64, P, P, P, P, P, P, P, P, F32, I64, I64, I64, I64, I32, F32, P, P,
                           P, P, P, P, P, P], C.c_int),
    'bbb_logprob_reduce': ([P, P, P, U64, U32, U32, U32, P, I64, I32, P, P, P, P], C.c_int),
    'bbb_kl_gauss': ([P, P, F32, I64, P, P], C.c_int),
    'bbb_gauss_prior_logprob': ([P, I32, I64, P, P, P, P], C.c_int),
    'bbb_gauss_prior_logprob_bwd': ([P, I32, I64, P, F32, F32, P, P, I64, P, P], C.c_int),
    'bbb_gauss_prior_kl': ([P, I32, P, P], C.c_int),
    'bbb_gauss_prior_kl_bwd': ([P, I32, F32, P, P, P], C.c_int),
    'bbb_philox_fill_normal': ([P, I64, U64, U32, U32, U32, P], C.c_int),
    'bbb_snr': ([P, P, I64, P, P], C.c_int),
    'bbb_snr_prune': ([P, P, I64, F32, P, P], C.c_int),
    'bbb_softmax_mean': ([P, I64, I64, I64, P, P], C.c_int),
    'bbb_predictive_stats': ([P, P, I64, I64, I64, I32, F32, I32, P, P, P, P, P], C.c_int),
    'bbb_nll_ce': ([P, P, I64, I64, I64, F32, P, P, P], C.c_int),
    'bbb_nll_gauss': ([P, P, F32, I64, I64, I64, F32, P, P, P], C.c_int),
    'bbb_nll_gauss_het': ([P, P, F32, I64, I64, I64, F32, P, P, P], C.c_int),
    'bbb_head_fwd': ([P, I64, P, P, P, P, P, P, P, P, I64, I64, I64, I64, I32, I32, P, F32, F32, P, P, P, P, P, F32,
                      P, P, P, P], C.c_int),
    'bbb_mlp_supported': ([P, I32, I64, I64, I32], C.c_int),
    'bbb_linear_fwd_relu_out_supported': ([I64, I64, I64, I32], C.c_int),
    'bbb_mlp_fwd': ([P, I32, P, I64, I64, P, P, I32, I32, P, F32, F32, P, P, P, P, F32, P, P, P, P], C.c_int),
    'bbb_mlp_bwd': ([P, I32, P, I64, I64, P, P, I32, F32, F32, P, P, I64, P, P], C.c_int),
    'bbb_elbo_finalize': ([P, P, P, P, I64, F32, P, P, P], C.c_int),
    'bbb_adam_step': ([I32, P, P, P, P, P, F64, F64, F64, F64, U32, P, P, P], C.c_int),
    'bbb_enable_peer_access': ([I32], C.c_int),
    'bbb_ipc_open': ([C.c_char_p, I64, P], C.c_int),
    'bbb_adam_step_peer': ([P, P, P, I64, F64, F64, F64, F64, U32, P, P, P], C.c_int),
    'bbb_counter_add': ([P, U32, P], C.c_int),
    'bbb_timing_enable': ([I32], C.c_int),
    'bbb_debug_set_timeline': ([P], C.c_int),
    'bbb_debug_wgrad_split': ([C.c_int], C.c_int),
    'bbb_timing_report': ([C.c_char_p, I64], C.c_int),
}
EXPORTS = tuple(_SIGS)

_lib = None


def lib():
    """Load libbbb.so once.  Raises (never falls back) when it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f'{LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; '
                               f'g.build()"` (nvcc, sm_100a).  There is no CPU or PyTorch fallback.')
        l = C.CDLL(LIB_PATH)
        for name, (argtypes, restype) in _SIGS.items():
            fn = getattr(l, name)
            fn.argtypes, fn.restype = argtypes, restype
        _lib = l
    return _lib


_mlp_ok = {}


def mlp_supported(dims, S, B, flags):
    """bbb_mlp_supported, cached per (dims, S, B, flags)."""
    key = (tuple(dims), S, B, flags)
    ok = _mlp_ok.get(key)
    if ok is None:
        arr = (C.c_int64 * len(dims))(*dims)
        ok = _mlp_ok[key] = bool(lib().bbb_mlp_supported(arr, len(dims) - 1, S, B, flags))
    return ok


def check(status, what):
    if status != 0:
        raise RuntimeError(f'{what} failed ({status}): {lib().bbb_last_error_string().decode()}')


def ptr(t):
    """Device pointer of a tensor (or None)."""
    return None if t is None else t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError('bayesian-neural-network_b200 runs on CUDA tensors only (sm_100a kernels, no CPU '
                               'fallback); move the module and its inputs to a cuda device')
