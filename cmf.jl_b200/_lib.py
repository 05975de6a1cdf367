"""ctypes binding of libcmf_sm100 (include/cmf_sm100.h).  There is NO fallback: if the shared
library is missing or a call fails, an exception is raised."""
from __future__ import annotations

import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("CMF_SM100_LIB") or os.path.join(_HERE, "libcmf_sm100.so")   # override: A/B builds of the same ABI

F64, F32 = 0, 1
MULT, HALS, PGD = 0, 1, 2
_c = ctypes
_i64, _dbl, _int, _vp = _c.c_int64, _c.c_double, _c.c_int, _c.c_void_p
_h = _c.c_void_p

# every exported symbol of include/cmf_sm100.h with its argument types
SIGNATURES = {
    "cmf_create": [_c.POINTER(_h), _i64, _i64, _i64, _i64, _int, _int, _int],
    "cmf_create_shard": [_c.POINTER(_h), _i64, _i64, _i64, _i64, _i64, _i64, _int, _int, _int],
    "cmf_create_multi": [_c.POINTER(_h), _i64, _i64, _i64, _i64, _int, _int, _int, _c.POINTER(_int)],
    "cmf_comm_unique_id": [_vp],
    "cmf_create_rank": [_c.POINTER(_h), _i64, _i64, _i64, _i64, _int, _int, _int, _vp, _int, _int],
    "cmf_shard_range": [_i64, _int, _int, _c.POINTER(_i64), _c.POINTER(_i64)],
    "cmf_comm_info": [_h, _c.POINTER(_int), _c.POINTER(_int), _c.POINTER(_i64), _c.POINTER(_i64)],
    "cmf_exchange_halos": [_h],
    "cmf_destroy": [_h],
    "cmf_set_data": [_h, _vp, _i64],
    "cmf_synth_data": [_h, _c.c_uint64, _i64, _i64, _dbl, _dbl],
    "cmf_get_data": [_h, _vp, _int],
    "cmf_data_sumsq": [_h, _c.POINTER(_dbl)],
    "cmf_set_data_norm": [_h, _dbl],
    "cmf_set_factors": [_h, _vp, _vp, _i64],
    "cmf_init_rand": [_h, _c.c_uint64],
    "cmf_init_scale_partials": [_h, _c.POINTER(_dbl)],
    "cmf_scale_factors": [_h, _dbl],
    "cmf_get_factors": [_h, _vp, _vp],
    "cmf_update_motifs": [_h, _dbl, _dbl],
    "cmf_update_feature_maps": [_h, _dbl, _dbl, _c.POINTER(_dbl)],
    "cmf_loss": [_h, _c.POINTER(_dbl)],
    "cmf_fit": [_h, _i64, _dbl, _int, _int, _int, _dbl, _dbl, _dbl, _dbl, _dbl, _c.POINTER(_dbl),
                _c.POINTER(_dbl), _i64, _c.POINTER(_i64), _c.POINTER(_int)],
    "cmf_w_partials": [_h],
    "cmf_w_apply": [_h, _dbl, _dbl],
    "cmf_h_update": [_h, _dbl, _dbl],
    "cmf_loss_partial": [_h, _c.POINTER(_dbl)],
    "cmf_exchange_buffer": [_h, _int, _c.POINTER(_vp), _c.POINTER(_i64), _c.POINTER(_int)],
    "cmf_halo_buffers": [_h, _c.POINTER(_vp), _c.POINTER(_vp), _c.POINTER(_vp), _c.POINTER(_vp),
                         _c.POINTER(_i64)],
    "cmf_sync": [_h],
    "cmf_launch_count": [_h, _c.POINTER(_i64)],
    "cmf_stream": [_h, _c.POINTER(_vp)],
    "cmf_set_stream": [_h, _vp],
    "cmf_set_engine": [_h, _int],
    "cmf_get_engine": [_h, _c.POINTER(_int)],
    "cmf_get_fd_layout": [_h, _c.POINTER(_int), _c.POINTER(_int), _c.POINTER(_i64)],
    "cmf_set_loss_mode": [_h, _int],
    "cmf_get_loss_mode": [_h, _c.POINTER(_int)],
    "cmf_set_loss_guard": [_h, _dbl, _int],
    "cmf_get_loss_stats": [_h, _c.POINTER(_i64), _c.POINTER(_i64), _c.POINTER(_int), _c.POINTER(_dbl)],
    "cmf_profile": [_h, _int],
    "cmf_profile_read": [_h, _int, _c.POINTER(_dbl), _c.POINTER(_i64)],
    "cmf_set_pgd_loss": [_h, _int, _vp],
    "cmf_set_pgd_constraints": [_h, _int, _int],
    "cmf_tensor_conv": [_i64, _i64, _i64, _i64, _int, _vp, _vp, _vp],
    "cmf_tensor_transconv": [_i64, _i64, _i64, _i64, _int, _vp, _vp, _vp],
    "cmf_corr_w": [_i64, _i64, _i64, _i64, _int, _vp, _vp, _vp],
    "cmf_compute_resids": [_i64, _i64, _i64, _i64, _int, _vp, _vp, _vp, _vp],
    "cmf_shift_and_stack": [_i64, _i64, _i64, _int, _vp, _vp],
    "cmf_create_batch": [_c.POINTER(_h), _i64, _i64, _i64, _i64, _int, _int, _i64, _int],
    "cmf_create_batch_ranks": [_c.POINTER(_h), _i64, _i64, _c.POINTER(_i64), _i64, _int, _int, _i64, _int],
    "cmf_set_factors_batch": [_h, _vp, _vp],
    "cmf_get_factors_batch": [_h, _vp, _vp],
    "cmf_init_scale_partials_batch": [_h, _c.POINTER(_dbl)],
    "cmf_scale_factors_batch": [_h, _c.POINTER(_dbl)],
    "cmf_loss_batch": [_h, _c.POINTER(_dbl)],
    "cmf_create_sparse": [_c.POINTER(_h), _i64, _i64, _i64, _i64, _int, _int, _int],
    "cmf_create_batch_sparse": [_c.POINTER(_h), _i64, _i64, _c.POINTER(_i64), _i64, _int, _int, _i64, _int],
    "cmf_set_data_csc": [_h, _i64, _c.POINTER(_i64), _c.POINTER(_i64), _vp, _int],
    "cmf_fit_batch": [_h, _i64, _dbl, _int, _int, _int, _dbl, _c.POINTER(_dbl), _c.POINTER(_dbl), _c.POINTER(_dbl),
                      _c.POINTER(_dbl), _c.POINTER(_dbl), _c.POINTER(_dbl), _i64, _c.POINTER(_i64), _c.POINTER(_int)],
}

_LIB = None


class CMFError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libcmf_sm100 error {code}: {msg}")
        self.code = code


def load():
    """Loads the shared library (once).  Raises if it has not been built -- no fallback."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            raise ImportError(
                f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`"
                " (the CUDA path has no CPU fallback)")
        lib = ctypes.CDLL(SO_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = _int
        lib.cmf_last_error.argtypes = []
        lib.cmf_last_error.restype = _c.c_char_p
        _LIB = lib
    return _LIB


def check(code):
    if code != 0:
        raise CMFError(code, load().cmf_last_error().decode("utf-8", "replace"))


def np_dtype(dtype):
    return np.float64 if dtype == F64 else np.float32


def parse_dtype(d):
    if d in (F64, "f64", "float64", np.float64, "Float64"):
        return F64
    if d in (F32, "f32", "float32", np.float32, "Float32"):
        return F32
    raise ValueError(f"dtype must be f64 or f32, got {d!r}")


def fptr(a):
    return a.ctypes.data_as(_vp)


def julia_array(a, dtype):
    """Returns a Fortran-ordered (Julia column-major) array of the handle dtype (copy only if needed)."""
    return np.asfortranarray(a, dtype=np_dtype(dtype))
