"""ctypes binding of libfermiflow_b200.so (C ABI: include/fermiflow_b200.h).

torch is used only to own device memory and streams; every call below forwards raw device
pointers to the CUDA library.  There is no CPU fallback: if the shared library is missing
or the tensors are not CUDA float64, the call raises.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfermiflow_b200.so")


class FFModel(C.Structure):
    _fields_ = [("n_up", C.c_int), ("n_dn", C.c_int), ("H_eta", C.c_int), ("H_mu", C.c_int),
                ("eta_w1", C.c_void_p), ("eta_b1", C.c_void_p), ("eta_w2", C.c_void_p),
                ("mu_w1", C.c_void_p), ("mu_b1", C.c_void_p), ("mu_w2", C.c_void_p),
                ("t0", C.c_double), ("t1", C.c_double), ("nsteps", C.c_int)]


class FFObsGrid(C.Structure):
    _fields_ = [("extent", C.c_double), ("n_xy", C.c_int), ("n_rot", C.c_int),
                ("r_max", C.c_double), ("n_r", C.c_int)]


class FFMomGrid(C.Structure):
    _fields_ = [("k_max", C.c_double), ("n_k", C.c_int), ("n_kr", C.c_int),
                ("s_max", C.c_double), ("n_s", C.c_int)]


class FFSwapRegions(C.Structure):
    _fields_ = [("kind", C.c_int), ("Q", C.c_int), ("a", C.POINTER(C.c_double))]


_lib = None
_P, _LL, _I, _D = C.c_void_p, C.c_longlong, C.c_int, C.c_double
_M = C.POINTER(FFModel)

SIGNATURES = {
    "ff_version": ([], C.c_int),
    "ff_last_error": ([], C.c_char_p),
    "ff_launch_count": ([], C.c_longlong),
    "ff_set_option": ([C.c_char_p, _I], C.c_int),
    "ff_get_option": ([C.c_char_p, C.POINTER(_I)], C.c_int),
    "ff_backflow": ([_M, _P, _LL, _P, _P, _P], C.c_int),
    "ff_cnf_generate": ([_M, _P, _LL, _I, _P, _P], C.c_int),
    "ff_cnf_delta_logp": ([_M, _P, _LL, _P, _P, _P, _P, _P], C.c_int),
    "ff_stash_sizes": ([_M, _LL, C.POINTER(_LL), C.POINTER(_LL)], C.c_int),
    "ff_slater_logabsdet": ([_P, _LL, _I, _P, _P, _P, _P, _P, _P], C.c_int),
    "ff_free_fermion_logp": ([_P, _LL, _I, _I, _P, _P, _P, _P, _P], C.c_int),
    "ff_free_fermion_logp_lap": ([_P, _LL, _I, _I, _P, _P, _P, _P, _P, _P], C.c_int),
    "ff_slater_hvp": ([_P, _LL, _I, _I, _P, _P, _D, _P, _P, _P], C.c_int),
    "ff_metropolis": ([_LL, _I, _I, _P, _P, _I, _D, C.c_ulonglong, _LL, _P, _P, _P, _P, _P, _P], C.c_int),
    "ff_eloc": ([_M, _P, _LL, _P, _P, _D, _I] + [_P] * 10 + [_P], C.c_int),
    "ff_logp_backward": ([_M, _LL] + [_P] * 12 + [_P], C.c_int),
    "ff_backward_work_size": ([_M, _LL, C.POINTER(_LL)], C.c_int),
    "ff_potential": ([_P, _LL, _I, _D, _I, _P, _P], C.c_int),
    "ff_occupation_sample": ([_P, _I, _P, _LL, _P, _P, _P, _P], C.c_int),
    "ff_observables": ([_P, _LL, _I, _I, C.POINTER(FFObsGrid), _P, _LL, _P], C.c_int),
    "ff_wavefunction_ratio_work_size": ([_M, _LL, _I, C.POINTER(_LL)], C.c_int),
    "ff_wavefunction_ratio": ([_M, _P, _LL, _P, _P, _I, _P, _P, _P, _P, _P], C.c_int),
    "ff_momentum_accumulate": ([_P, _P, _P, _LL, _I, C.POINTER(FFMomGrid), _P, _LL, _P], C.c_int),
    "ff_density_matrix_accumulate": ([_P, _LL, _I, _I, _I, _P, _P, _P, _I, _P, _LL, _P], C.c_int),
    "ff_swap_ratio_work_size": ([_M, _LL, _I, C.POINTER(_LL)], C.c_int),
    "ff_swap_ratio": ([_M, _P, _LL, _P, _P, _LL, _P, C.POINTER(FFSwapRegions), _P, _P, _P, _P], C.c_int),
    "ff_swap_accumulate": ([_P, _P, _LL, _I, _I, _I, _P, _LL, _P], C.c_int),
    "ff_fp64_peak": ([_I, C.POINTER(_D), _P], C.c_int),
    "ff_fp64_mma_peak": ([_I, C.POINTER(_D), _P], C.c_int),
}


def lib():
    """Load the CUDA library once; raise if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "fermiflow_b200: %s is missing -- build it with "
                "`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
                "There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (args, res) in SIGNATURES.items():
            if os.environ.get('FF_DEV_PARTIAL') and not hasattr(L, name):
                continue
            fn = getattr(L, name)
            fn.argtypes, fn.restype = args, res
        _lib = L
    return _lib


def set_option(name, value):
    """Kernel-variant switch of the library (include/fermiflow_b200.h ff_set_option); 0 = default."""
    check(lib().ff_set_option(name.encode(), int(value)))


def get_option(name):
    v = C.c_int()
    check(lib().ff_get_option(name.encode(), C.byref(v)))
    return v.value


class options:
    """with options(flow_cta=1, ...): ... -- sets the switches and restores the previous values."""

    def __init__(self, **kw):
        self.kw = kw

    def __enter__(self):
        self.old = {k: get_option(k) for k in self.kw}
        for k, v in self.kw.items():
            set_option(k, v)
        return self

    def __exit__(self, *exc):
        for k, v in self.old.items():
            set_option(k, v)
        return False


# Python-side switch: keep the per-item radial functions (f, f', f'') in the adjoint stash (16x the memory of the
# stage inputs, 28 ms faster backward at 65536 walkers, N = 20).  Set to False to recompute them in the backward sweep.
STASH_RADIAL = True


def check(code):
    if code != 0:
        raise RuntimeError("fermiflow_b200 error %d: %s" % (code, lib().ff_last_error().decode()))


def ptr(t, dtype=torch.float64):
    """Device pointer of a tensor, validating device/dtype/layout.  None -> NULL."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("fermiflow_b200 kernels need CUDA tensors (got %s); no CPU fallback" % t.device)
    if t.dtype != dtype:
        raise TypeError("expected %s, got %s" % (dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError("tensor must be contiguous")
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def make_model(n_up, n_dn, eta, mu, t_span, nsteps):
    """eta / mu: (w1, b1, w2) CUDA float64 vectors (mu may be None).  The returned struct
    holds raw pointers: keep the tensors alive while it is in use."""
    m = FFModel()
    m.n_up, m.n_dn = int(n_up), int(n_dn)
    m.H_eta = int(eta[0].numel())
    m.eta_w1, m.eta_b1, m.eta_w2 = (ptr(t) for t in eta)
    if mu is not None:
        m.H_mu = int(mu[0].numel())
        m.mu_w1, m.mu_b1, m.mu_w2 = (ptr(t) for t in mu)
    else:
        m.H_mu = 0
    m.t0, m.t1, m.nsteps = float(t_span[0]), float(t_span[1]), int(nsteps)
    return m
