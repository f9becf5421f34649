"""ctypes binding of libmobocmf_b200.so (C ABI declared in include/mobocmf_b200.h).

The product path has no CPU fallback: importing this module without the built library, or calling a kernel
wrapper on a non-CUDA tensor, raises.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libmobocmf_b200.so")

_c_dp = ctypes.c_void_p
_c_i = ctypes.c_int
_c_ll = ctypes.c_longlong
_c_d = ctypes.c_double
_c_sz = ctypes.c_size_t

_SIGNATURES = {
    "mobo_abi_version": (_c_i, []),
    "mobo_launch_count": (_c_ll, []),
    "mobo_profile_enable": (None, [_c_i]),
    "mobo_profile_collect": (_c_i, [ctypes.c_char_p, _c_sz, ctypes.POINTER(ctypes.c_float), _c_i]),
    "mobo_padded_m": (_c_i, [_c_i]),
    "mobo_ops_doubles": (_c_sz, [_c_i]),
    "mobo_rows_save_doubles": (_c_sz, [_c_i, _c_ll]),
    "mobo_rows_bwd_work_doubles": (_c_sz, [_c_i, _c_ll]),
    "mobo_precompute_bwd_work_doubles": (_c_sz, [_c_i]),
    "mobo_layer_precompute": (_c_i, [_c_i, _c_i, _c_i, _c_dp, _c_dp, _c_dp, _c_dp, _c_dp, _c_d, _c_dp, _c_dp]),
    "mobo_layer_precompute_bwd": (_c_i, [_c_i, _c_i, _c_i] + [_c_dp] * 13),
    "mobo_layer_rows_fwd": (_c_i, [_c_i, _c_i, _c_i, _c_dp, _c_dp, _c_dp, _c_dp, _c_dp, _c_i, _c_dp, _c_dp, _c_i,
                                   _c_dp, _c_ll, _c_dp, _c_ll, _c_i, _c_dp, _c_dp, _c_dp, _c_dp, _c_dp, _c_dp,
                                   _c_dp]),
    "mobo_layer_rows_bwd": (_c_i, [_c_i, _c_i, _c_i, _c_dp, _c_dp, _c_dp, _c_dp, _c_dp, _c_i, _c_dp, _c_dp, _c_i,
                                   _c_dp, _c_ll, _c_dp, _c_ll, _c_i, _c_dp, _c_dp, _c_dp, _c_dp, _c_dp, _c_dp,
                                   _c_i, _c_dp, _c_dp, _c_dp, _c_dp, _c_dp, _c_dp, _c_dp]),
    # fused step / optimiser / acquisition chain (struct pointers travel as void*; see mobocmf_b200/fused.py)
    "mobo_elbo_step_workspace_doubles": (_c_sz, [_c_i, _c_i, _c_i, _c_i, _c_ll]),
    "mobo_elbo_step": (_c_i, [_c_dp, _c_dp]),
    "mobo_step_side_stream": (None, [_c_i]),
    "mobo_step_ctx_create": (_c_dp, []),
    "mobo_step_ctx_destroy": (None, [_c_dp]),
    "mobo_step_ctx_wait_layer": (_c_i, [_c_dp, _c_i, _c_dp]),
    "mobo_adam": (_c_i, [_c_i, _c_dp, _c_d, _c_d, _c_d, _c_d, _c_ll, _c_dp, _c_dp, _c_dp]),
    "mobo_adam_tick": (_c_i, [_c_dp, _c_dp, _c_dp]),
    "mobo_acq_moments": (_c_i, [_c_i, _c_i, _c_i, _c_i, _c_ll, _c_dp, _c_dp, _c_dp, _c_dp, _c_dp, _c_dp, _c_d, _c_d,
                                _c_dp, _c_dp, _c_dp, _c_dp, _c_dp]),
    "mobo_acq_bwd_work_doubles": (_c_sz, [_c_i, _c_i, _c_i, _c_i, _c_ll]),
    "mobo_acq_moments_bwd": (_c_i, [_c_i, _c_i, _c_i, _c_i, _c_ll, _c_dp, _c_dp, _c_dp, _c_dp, _c_dp, _c_dp, _c_d,
                                    _c_d, _c_dp, _c_dp, _c_dp, _c_i, _c_dp, _c_dp, _c_dp, _c_dp]),
    "mobo_jes": (_c_i, [_c_dp, _c_dp, _c_ll, _c_i, _c_dp, _c_dp]),
    # Pareto-sample generation
    "mobo_rff_eval": (_c_i, [_c_i, _c_i, _c_i, _c_dp, _c_dp, _c_dp, _c_ll, _c_dp, _c_dp, _c_dp]),
    "mobo_pareto_mask": (_c_i, [_c_dp, _c_ll, _c_i, _c_dp, _c_dp]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load():
    """Load the shared library (once).  Raises if it has not been built (``python -c 'import
    __graft_entry__ as g; g.build()'`` or ``python mobocmf_b200/build.py``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("mobocmf_b200: %s is missing - build it with mobocmf_b200/build.py; there is no "
                               "CPU fallback" % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def ptr(t):
    """Device pointer of a contiguous fp64 (or uint32) CUDA tensor; None -> NULL."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("mobocmf_b200 kernels need CUDA tensors (no CPU fallback)")
    if not t.is_contiguous():
        raise RuntimeError("mobocmf_b200 kernels need contiguous tensors")
    return ctypes.c_void_p(t.data_ptr())


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def check(code, what):
    if code != 0:
        raise RuntimeError("mobocmf_b200: %s failed with code %d (%s)" %
                           (what, code, {-1: "CUDA launch error", -2: "unsupported shape: M <= 256, d <= 8"}.get(
                               code, "unknown")))


def launch_count():
    return int(load().mobo_launch_count())


def profile_enable(on):
    load().mobo_profile_enable(1 if on else 0)


def profile_collect(max_records=200000):
    """[(kernel name, milliseconds)] of every launch since profiling was enabled (synchronises)."""
    names = ctypes.create_string_buffer(64 * max_records)
    ms = (ctypes.c_float * max_records)()
    n = load().mobo_profile_collect(names, len(names), ms, max_records)
    raw = names.raw.split(b"\0")
    return [(raw[i].decode(), float(ms[i])) for i in range(n)]


def ptr_array(tensors):
    """HOST array of device pointers (None -> NULL) for the batched entry points."""
    arr = (ctypes.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        p = ptr(t)
        arr[i] = None if p is None else p.value
    return arr


def int_array(values):
    return (ctypes.c_int * len(values))(*values)
