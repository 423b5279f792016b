"""ctypes binding of ``libpybold_b200.so`` (C ABI in ``include/pybold_b200.h``).

The library is the product: if it cannot be loaded this module raises ``ImportError``
and nothing in the package falls back to a CPU or PyTorch implementation.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_int, c_int64, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpybold_b200.so")

PB_OK = 0
PB_ERR_INVALID_ARG = -1
PB_ERR_UNSUPPORTED = -2
PB_ERR_NO_DEVICE = -3


class PyboldB200Error(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "pybold_b200: %s is missing -- build it with `python __graft_entry__.py` "
            "(or `make -C pybold_b200/csrc`); there is no CPU fallback." % LIB_PATH)
    try:
        return ctypes.CDLL(LIB_PATH)
    except OSError as exc:  # pragma: no cover - depends on the box
        raise ImportError("pybold_b200: cannot load %s: %s" % (LIB_PATH, exc)) from exc


lib = _load()

_P = c_void_p  # device pointers travel as integers (tensor.data_ptr())

# name -> argtypes (return type is always int unless noted); mirrors include/pybold_b200.h
_OPS = {
    "pb_integ_op": [_P, _P, c_int64, c_int, _P],
    "pb_integ_adj": [_P, _P, c_int64, c_int, _P],
    "pb_conv_op": [_P, c_int64, _P, _P, c_int64, c_int, c_int, _P],
    "pb_conv_adj": [_P, c_int64, _P, _P, c_int64, c_int, c_int, _P],
    "pb_hrfinteg_op": [_P, c_int64, _P, _P, c_int64, c_int, c_int, _P],
    "pb_hrfinteg_adj": [_P, c_int64, _P, _P, c_int64, c_int, c_int, _P],
    "pb_spm_hrf": [_P, c_double, c_double, c_int, _P, c_int64, c_int, _P],
    "pb_spm_hrf_ex": [_P, c_double, c_double, c_int, ctypes.POINTER(c_double), _P, c_int64, c_int, _P],
    "pb_lipschitz_power": [_P, c_int64, _P, c_int64, c_int, c_double, _P, c_int64, c_int, c_int, _P],
    "pb_lipschitz_frob": [_P, c_int64, _P, c_int64, c_int, c_int, _P],
    "pb_deconv": [_P, _P, c_int64, _P, c_int64, _P, c_int64, _P, c_int, c_int, c_int, c_double,
                  _P, _P, _P, _P, _P, c_int64, c_int, c_int, _P],
    "pb_deconv_masked": [_P, _P, c_int64, _P, c_int64, _P, c_int64, _P, _P, c_int, c_int, c_int, c_double,
                         _P, _P, _P, _P, _P, c_int64, c_int, c_int, _P],
    "pb_deconv_auto": [_P, _P, c_int64, _P, c_int64, _P, c_int64, c_int, c_int, c_int, c_int, c_double,
                       _P, _P, _P, _P, _P, _P, _P, _P, c_int64, c_int, c_int, _P],
    "pb_deconv_lbda_path": [_P, _P, _P, _P, c_int, c_int, _P, _P, _P, _P, _P, c_int64, c_int, c_int, _P],
    "pb_deconv_lbda_path_ex": [_P, _P, c_int64, _P, c_int64, _P, c_int, c_int, c_int, c_int, c_double,
                               _P, _P, _P, _P, _P, _P, _P, c_int64, c_int, c_int, _P],
    "pb_deconv_censored": [_P, _P, c_int64, _P, c_int64, _P, c_int64, _P, _P, c_int64, c_int, c_int, c_int,
                           c_double, _P, _P, _P, _P, _P, c_int64, c_int, c_int, _P],
    "pb_deconv_auto_censored": [_P, _P, c_int64, _P, c_int64, _P, c_int64, _P, c_int64, c_int, c_int, c_int, c_int,
                                c_double, _P, _P, _P, _P, _P, _P, _P, _P, c_int64, c_int, c_int, _P],
    "pb_deconv_lbda_path_censored": [_P, _P, c_int64, _P, c_int64, _P, c_int, _P, c_int64, c_int, c_int, c_int,
                                     c_double, _P, _P, _P, _P, _P, _P, _P, c_int64, c_int, c_int, _P],
    "pb_lipschitz_power_censored": [_P, c_int64, _P, c_int64, _P, c_int64, c_int, c_double, _P, c_int64, c_int,
                                    c_int, _P],
    "pb_mad_daub_noise_est_censored": [_P, _P, c_int64, c_double, _P, c_int64, c_int, _P],
    "pb_bd": [_P, c_double, c_double, _P, c_int64, _P, c_int64, _P, c_double, c_double,
              c_int, c_int, c_int, c_double, _P, _P, _P, _P, _P, _P, _P, _P, _P,
              c_int64, c_int, c_int, _P],
    "pb_transpose": [_P, _P, c_int64, c_int64, _P],
    "pb_noise_step": [_P, _P, _P, _P, _P, _P, c_double, _P, _P, _P, _P, _P, _P, _P, c_int64, c_int, _P],
    "pb_mad": [_P, c_double, _P, c_int64, c_int, _P],
    "pb_mad_daub_noise_est": [_P, c_double, _P, c_int64, c_int, _P],
    "pb_toeplitz": [_P, c_int, _P, c_int64, c_int64, _P],
    "pb_synth_voxels": [c_uint64, c_int64, c_double, c_double, c_double, c_int, c_int, c_double, c_double,
                        _P, _P, _P, c_int64, c_int, _P],
    "pb_inf_norm": [_P, _P, c_int64, c_int, _P],
    "pb_rel_l2_err": [_P, _P, c_int64, _P, c_int64, c_int, _P],
    "pb_hrf_estim": [_P, _P, c_double, c_double, _P, c_int64, c_double, c_double, _P, _P, _P,
                     c_int64, c_int, c_int, _P],
}
_PLAIN = {
    "pb_version": ([], c_int),
    "pb_max_T": ([], c_int),
    "pb_max_K": ([], c_int),
    "pb_max_iter": ([], c_int),
    "pb_error_string": ([c_int], c_char_p),
    "pb_solver_variant": ([c_int, c_int, c_int], c_int),
    "pb_hrf_len": ([c_double, c_double], c_int),
    "pb_hrf_len_ex": ([c_double, c_double, c_double], c_int),
    "pb_bd_wave_voxels": ([c_int, c_int, c_int, c_int], c_int),
    "pb_deconv_variant": ([c_int, c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_int)], c_int),
    "pb_deconv_censored_variant": ([c_int, c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_int)],
                                   c_int),
    "pb_bd_variant": ([c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_int)], c_int),
    "pb_bench_fma_f32": ([_P, c_int, c_int, _P], c_int),
    "pb_copy_async": ([_P, _P, ctypes.c_size_t, _P], c_int),
}

EXPORTED_SYMBOLS = sorted(list(_PLAIN) + [n + s for n in _OPS for s in ("_f32", "_f64")])

for _name, (_args, _res) in _PLAIN.items():
    _fn = getattr(lib, _name)
    _fn.argtypes = _args
    _fn.restype = _res
for _name, _args in _OPS.items():
    for _suf in ("_f32", "_f64"):
        _fn = getattr(lib, _name + _suf)
        _fn.argtypes = _args
        _fn.restype = c_int


def error_string(code):
    return lib.pb_error_string(int(code)).decode()


def check(code, what):
    """Map a C-ABI return code to the exception the reference-facing API raises."""
    if code == PB_OK:
        return
    msg = "%s failed: %s (code %d)" % (what, error_string(code), code)
    if code in (PB_ERR_INVALID_ARG, PB_ERR_UNSUPPORTED):
        raise ValueError(msg)
    raise PyboldB200Error(msg)


def fn(name, torch_dtype):
    """Return the ``_f32`` / ``_f64`` entry point for a torch dtype."""
    import torch
    if torch_dtype == torch.float32:
        return getattr(lib, name + "_f32")
    if torch_dtype == torch.float64:
        return getattr(lib, name + "_f64")
    raise TypeError("pybold_b200 supports float32 and float64 signals, got %s" % torch_dtype)
