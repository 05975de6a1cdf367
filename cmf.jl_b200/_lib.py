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


class Handle:
    """Owns one libcmf_sm100 handle and binds the calls every kind of handle takes.

    The arguments choose the create call: ``restarts=R`` a batch of R restarts (``K`` an int: cmf_create_batch; R ranks:
    cmf_create_batch_ranks, or cmf_create_batch_sparse with ``sparse``), ``sparse`` X held as compressed sparse columns
    (cmf_create_sparse), ``ngpu > 1`` one handle over that many GPUs (cmf_create_multi), ``comm=(unique_id, rank, world)``
    one rank with its NCCL communicator inside the library (cmf_create_rank; t0/t1 must be the balanced shard of that rank),
    columns [t0, t1) of a longer time axis (cmf_create_shard), otherwise cmf_create."""

    def __init__(self, N, T, K, L, dtype, alg, device=0, t0=0, t1=None, comm=None, ngpu=1, devices=None, sparse=False,
                 restarts=None):
        self._h = _vp()
        lib = load()
        t1 = T if t1 is None else t1
        ngpu = int(ngpu or 1)
        self.N, self.T, self.t0, self.t1, self.K, self.L, self.dtype = N, T, t0, t1, K, L, dtype
        out = _c.byref(self._h)
        if restarts is not None and not sparse and np.ndim(K) == 0:
            check(lib.cmf_create_batch(out, N, T, K, L, dtype, alg, restarts, device))
        elif restarts is not None:
            ranks = np.asarray([K] * restarts if np.ndim(K) == 0 else K, dtype=np.int64)
            create = lib.cmf_create_batch_sparse if sparse else lib.cmf_create_batch_ranks
            check(create(out, N, T, ranks.ctypes.data_as(_c.POINTER(_i64)), L, dtype, alg, restarts, device))
        elif sparse:
            check(lib.cmf_create_sparse(out, N, T, K, L, dtype, alg, device))
        elif ngpu > 1:
            devs = (_int * ngpu)(*(devices if devices is not None else range(ngpu)))
            check(lib.cmf_create_multi(out, N, T, K, L, dtype, alg, ngpu, devs))
            self.t0, self.t1 = 0, T
        elif comm is not None:
            uid, rank, world = comm      # uid None: reuse the communicator this process already built for (device, rank, world)
            buf = _c.create_string_buffer(bytes(uid), 128) if uid is not None else None
            check(lib.cmf_create_rank(out, N, T, K, L, dtype, alg, device, buf, rank, world))
            a, b = _i64(), _i64()
            check(lib.cmf_comm_info(self._h, None, None, _c.byref(a), _c.byref(b)))
            assert (a.value, b.value) == (t0, t1), "ShardPlan and cmf_shard_range disagree"
        elif t0 == 0 and t1 == T:
            check(lib.cmf_create(out, N, T, K, L, dtype, alg, device))
        else:
            check(lib.cmf_create_shard(out, N, T, t0, t1, K, L, dtype, alg, device))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            load().cmf_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # data ------------------------------------------------------------------------------------------
    def set_data(self, X, first_col=0):
        check(load().cmf_set_data(self._h, fptr(julia_array(X, self.dtype)), first_col))

    def synth_data(self, seed, K_true, L_true, p_h, noise):
        check(load().cmf_synth_data(self._h, int(seed), int(K_true), int(L_true), float(p_h), float(noise)))

    def data_sumsq(self):
        """||X||^2 of the owned columns; over ALL columns on handles whose collectives run inside the library."""
        out = _dbl()
        check(load().cmf_data_sumsq(self._h, _c.byref(out)))
        return out.value

    def set_data_norm(self, v):
        check(load().cmf_set_data_norm(self._h, float(v)))

    def get_data(self, out=None, with_halo=False):
        """Owned columns of X (plus the right halo, clipped to T, with ``with_halo``) as a
        Fortran-ordered N x cols array (optionally into a caller buffer)."""
        cols = (min(self.t1 + self.L - 1, self.T) if with_halo else self.t1) - self.t0
        if out is None:
            out = np.empty((self.N, cols), dtype=np_dtype(self.dtype), order="F")
        assert out.shape == (self.N, cols) and out.flags.f_contiguous
        check(load().cmf_get_data(self._h, fptr(out), int(with_halo)))
        return out

    # factors ---------------------------------------------------------------------------------------
    def set_factors(self, W, H, first_col=0):
        Wj, Hj = julia_array(W, self.dtype), julia_array(H, self.dtype)
        check(load().cmf_set_factors(self._h, fptr(Wj), fptr(Hj), first_col))

    def get_factors(self, out=None):
        """W (K x N x L) and the owned columns of H (K x Tl), Fortran order, handle dtype.  ``out=(W, H)`` downloads
        into caller-owned arrays of that shape/order/dtype (e.g. views of pinned buffers)."""
        dt = np_dtype(self.dtype)
        if out is not None:
            W, H = out
            for a, shp in ((W, (self.K, self.N, self.L)), (H, (self.K, self.t1 - self.t0))):
                if a.shape != shp or a.dtype != dt or not a.flags.f_contiguous:
                    raise ValueError("get_factors(out=...): need Fortran-ordered arrays of the handle dtype, shapes K x N x L and K x Tl")
        else:
            W = np.empty((self.K, self.N, self.L), dtype=dt, order="F")
            H = np.empty((self.K, self.t1 - self.t0), dtype=dt, order="F")
        check(load().cmf_get_factors(self._h, fptr(W), fptr(H)))
        return W, H            # handle dtype (no host-side conversion: H is 1 GiB at the benchmark size)

    def init_rand(self, seed):
        check(load().cmf_init_rand(self._h, seed))

    def init_scale_partials(self):
        """[<X, Xhat>, ||Xhat||^2] of the alpha rescale (src/model.jl:119-122)."""
        out = (_dbl * 2)()
        check(load().cmf_init_scale_partials(self._h, out))
        return [out[0], out[1]]

    def scale_factors(self, s):
        check(load().cmf_scale_factors(self._h, float(s)))

    # steps and loss --------------------------------------------------------------------------------
    def update_motifs(self, l1W=0.0, l2W=0.0):
        """One update_motifs! half-step (MU or HALS).  The update rules of model.py wrap it in the reference's signature."""
        check(load().cmf_update_motifs(self._h, float(l1W), float(l2W)))

    def update_feature_maps(self, l1H=0.0, l2H=0.0):
        """One update_feature_maps! half-step (MU or HALS); returns the relative loss."""
        out = _dbl()
        check(load().cmf_update_feature_maps(self._h, float(l1H), float(l2H), _c.byref(out)))
        return out.value

    def loss(self):
        out = _dbl()
        check(load().cmf_loss(self._h, _c.byref(out)))
        return out.value

    def launch_count(self):
        out = _i64()
        check(load().cmf_launch_count(self._h, _c.byref(out)))
        return out.value

    def sync(self):
        check(load().cmf_sync(self._h))

    # engine, loss path and diagnostics -------------------------------------------------------------
    def set_engine(self, engine):
        """0 = SIMT kernels, 1 = tcgen05 kernels in the time domain, 2 = frequency-domain engine (spectrum of X +
        per-frequency tcgen05 products); raises if the handle cannot use the engine."""
        check(load().cmf_set_engine(self._h, int(engine)))

    def get_engine(self):
        out = _int()
        check(load().cmf_get_engine(self._h, _c.byref(out)))
        return out.value

    def set_loss_mode(self, mode):
        """0 = direct residual pass, 1 = algebraic expansion on resident numH / C (tcgen05 engine only)."""
        check(load().cmf_set_loss_mode(self._h, int(mode)))

    @property
    def loss_mode(self):
        out = _int(0)
        check(load().cmf_get_loss_mode(self._h, _c.byref(out)))
        return out.value

    def set_loss_guard(self, guard=0.25, max_interval=16):
        """Relative loss at or below which loss mode 1 calibrates the expansion against the direct pass, and the
        longest stretch of evaluations between two direct passes (include/cmf_sm100.h)."""
        check(load().cmf_set_loss_guard(self._h, float(guard), int(max_interval)))

    def loss_stats(self):
        """dict(direct=, expansion=, interval=, last_err=): loss evaluations by path and the calibration state."""
        nd, ne, iv, le = _i64(), _i64(), _int(), _dbl()
        check(load().cmf_get_loss_stats(self._h, _c.byref(nd), _c.byref(ne), _c.byref(iv), _c.byref(le)))
        return dict(direct=nd.value, expansion=ne.value, interval=iv.value, last_err=le.value)

    def fd_layout(self):
        """(block length, hop, blocks) of the frequency-domain engine on this handle; zeros on the other engines."""
        b, v, n = _int(), _int(), _i64()
        check(load().cmf_get_fd_layout(self._h, _c.byref(b), _c.byref(v), _c.byref(n)))
        return b.value, v.value, n.value

    def profile(self, enable=True):
        check(load().cmf_profile(self._h, int(enable)))

    def profile_read(self):
        """{class: (total_ms, launches)} for conv / transconv / corr / sweep (HALS H sweep)."""
        res = {}
        for which, name in enumerate(("conv", "transconv", "corr", "sweep")):
            ms, n = _dbl(), _i64()
            check(load().cmf_profile_read(self._h, which, _c.byref(ms), _c.byref(n)))
            res[name] = (ms.value, n.value)
        return res
