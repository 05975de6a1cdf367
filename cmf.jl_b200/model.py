"""Host-side mirror of CMF.jl's public fit interface on top of libcmf_sm100.

Same names, argument meaning and error behaviour as the reference (file:line relative to
/root/reference):

    fit_cnmf(data; L, K, alg, max_itr, max_time, kwargs...)   src/model.jl:58-85
    init_rand(data, L, K)                                     src/model.jl:113-125
    converged(loss_hist, patience, tol)                       src/model.jl:91-107
    CNMF_results(data, W, H, time_hist, loss_hist)            src/model.jl:11-17 (+ accessors :21-30)
    AbstractCFUpdate / MultUpdate / HALSUpdate                src/algs/alternating.jl:8, mult.jl, hals.jl
    AlternatingOptimizer, fit(alg, data, L, K, W_init, H_init; kwargs...)   alternating.jl:10-71

All arithmetic runs in the CUDA library; nothing here computes on the CPU and nothing imports
``oracle/``.  If the shared library is missing or no GPU is visible, calls raise.
"""
from __future__ import annotations

import ctypes
import math
import time as _time
import warnings

import numpy as np

from . import _lib
from ._lib import HALS, MULT, PGD, CMFError, Handle, check, fptr, julia_array, np_dtype, parse_dtype

# kwargs the reference's methods read (src/algs/alternating.jl:23-31, mult.jl:23,42, hals.jl:31,37,
# src/model.jl:64,72-73) plus the README-generation spellings (README.md:44-52) and this library's own.
_REG_ALIASES = {"l1_W": "l1W", "l2_W": "l2W", "l1_H": "l1H", "l2_H": "l2H"}
_INIT_ALIASES = {"initW": "W_init", "initH": "H_init"}
_KNOWN = {"l1W", "l2W", "l1H", "l2H", "seed", "W_init", "H_init", "check_convergence", "patience",
          "eval_mode", "tol", "verbose", "dtype", "device", "layout", "printer", "engine", "loss_mode", "loss_guard", "ngpu", "devices", "loss_func", "mask", "constrW", "constrH"}


def _normalise_kwargs(kwargs):
    """README spellings -> current-src spellings; unknown keys are swallowed as the reference does
    (every method slurps ``kwargs...``) but, unlike the reference, with a warning."""
    out = {}
    for k, v in kwargs.items():
        k = _REG_ALIASES.get(k, _INIT_ALIASES.get(k, k))
        if k not in _KNOWN:
            warnings.warn(f"fit_cnmf: unknown keyword {k!r} ignored (the reference ignores it silently)")
            continue
        out[k] = v
    return out


class CNMF_results:
    """src/model.jl:11-17.  ``W`` is L x N x K by default (README / north-star layout) or K x N x L
    with ``layout="KNL"`` (current-src layout); ``W_LNK[l,n,k] == W_KNL[k,n,l]``."""

    def __init__(self, data, W, H, time_hist, loss_hist, layout="LNK"):
        self.data, self.W, self.H = data, W, H
        self.time_hist, self.loss_hist = time_hist, loss_hist
        self.layout = layout

    def _knl(self):
        return self.W if self.layout == "KNL" else self.W.transpose(2, 1, 0)


def num_lags(r):        # src/model.jl:21
    return r._knl().shape[2]


def num_units(r):       # src/model.jl:24
    return r._knl().shape[1]


def num_components(r):  # src/model.jl:27
    return r._knl().shape[0]


def num_iter(r):        # src/model.jl:30
    return len(r.loss_hist)


class SparseData:
    """X as canonical compressed sparse columns (column t = time bin t): ``colptr`` (T+1), ``rowval`` and ``nzval`` (nnz),
    0-based int64 indices, rows strictly increasing in every column, no explicit zeros, values of the handle dtype."""

    def __init__(self, shape, colptr, rowval, nzval):
        self.shape, self.colptr, self.rowval, self.nzval = shape, colptr, rowval, nzval
        self.ndim = 2

    @property
    def nnz(self):
        return len(self.nzval)


def _is_sparse(data):
    return isinstance(data, SparseData) or type(data).__module__.startswith("scipy.sparse")


def as_csc(data, dtype="f64"):
    """Any ``scipy.sparse`` matrix or array -> ``SparseData`` in the handle dtype: duplicates summed, indices sorted, explicit
    zeros dropped.  None for dense data (scipy is imported only here, so dense-only use does not need it)."""
    if isinstance(data, SparseData) or not _is_sparse(data):
        return data if isinstance(data, SparseData) else None
    import scipy.sparse as sp

    X = sp.csc_matrix(data, dtype=np.float64, copy=True)
    X.sum_duplicates()                    # also sorts the row indices of every column
    X = X.astype(np_dtype(parse_dtype(dtype)))
    X.eliminate_zeros()
    return SparseData(X.shape, X.indptr.astype(np.int64), X.indices.astype(np.int64), np.ascontiguousarray(X.data))


def _data_shape(data):
    """(N, T) of a dense or sparse ``data`` argument; ValueError when it is not a matrix."""
    shape = data.shape if _is_sparse(data) else np.shape(data)
    if len(shape) != 2:
        raise ValueError("data must be an N x T matrix")
    return tuple(int(d) for d in shape)


def _check_sparse_rule(sparse, rule_cls, ngpu):
    """Sparse data serve MultUpdate and HALSUpdate on one GPU: the same refusal (code 3) as the library's."""
    if not sparse:
        return
    if rule_cls is PGDUpdate:
        raise CMFError(3, "sparse data serve MultUpdate and HALSUpdate (PGD needs the dense X)")
    if int(ngpu or 1) > 1:
        raise CMFError(3, "sparse data run on one GPU")


def _set_csc(h, csc):
    i64 = ctypes.POINTER(ctypes.c_int64)
    check(_lib.load().cmf_set_data_csc(h, csc.nnz, csc.colptr.ctypes.data_as(i64), csc.rowval.ctypes.data_as(i64),
                                       fptr(csc.nzval), 0))


def _emit(printer, s, nl=True):
    if printer is print:
        print(s, end="\n" if nl else "", flush=True)
    else:
        printer(s)


def converged(loss_hist, patience, tol):
    """src/model.jl:91-107 (host control logic; the device loop in cmf_fit applies the same rule)."""
    if len(loss_hist) <= patience:
        return False
    d = np.diff(np.asarray(loss_hist[-(patience + 1):], dtype=np.float64))
    return bool(np.all(np.abs(d) < tol))


# ------------------------------------------------------------------------------------------
# update rules: the plugin boundary (abstract type AbstractCFUpdate, alternating.jl:8)
# ------------------------------------------------------------------------------------------
class AbstractCFUpdate(Handle):
    """A rule owns an opaque libcmf_sm100 handle: the constructor uploads (data, W, H) exactly like
    ``Rule(data, W, H)`` at src/model.jl:79; ``update_motifs`` / ``update_feature_maps`` run one
    device half-step each.  ``sync_host=True`` (default) copies the updated factor back into the
    caller's array after every call, reproducing the reference's in-place semantics; the driver
    loop turns it off and reads the factors once at the end."""

    _ALG = None

    def __init__(self, data, W, H, dtype="f64", device=0, sync_host=True, engine=None, loss_mode=None, ngpu=1,
                 devices=None, loss_guard=None):
        """``ngpu > 1``: the rule spans ``ngpu`` GPUs (time axis sharded inside the library, NCCL collectives driven
        from this one thread -- cmf_create_multi); every other argument and every method is unchanged.  ``data`` may be a
        ``scipy.sparse`` matrix or array (MultUpdate / HALSUpdate, one GPU): the handle then holds X as compressed sparse
        columns and never densifies it (cmf_create_sparse)."""
        dtype = parse_dtype(dtype)
        csc = as_csc(data, dtype)
        if csc is None:
            data = np.asarray(data)
        W = np.asarray(W)
        H = np.asarray(H)
        if len(data.shape) != 2 or W.ndim != 3 or H.ndim != 2:
            raise ValueError("expected data N x T, W K x N x L, H K x T")
        K, N, L = W.shape
        if data.shape[0] != N or H.shape[0] != K or H.shape[1] != data.shape[1]:
            raise ValueError(f"dimension mismatch: data {data.shape}, W {W.shape}, H {H.shape}")
        ngpu = int(ngpu or 1)
        _check_sparse_rule(csc is not None, type(self), ngpu)
        super().__init__(N, data.shape[1], K, L, dtype, self._ALG, device if devices is None else devices[0], ngpu=ngpu,
                         devices=devices, sparse=csc is not None)
        self.sync_host = sync_host
        if engine is not None:
            self.set_engine(engine)
        if loss_mode is not None:
            self.set_loss_mode(loss_mode)
        if loss_guard is not None:
            self.set_loss_guard(loss_guard, 16)
        if csc is not None:
            _set_csc(self._h, csc)
        else:
            self.set_data(data)
        self.set_factors(W, H)

    # -- the interface of src/algs/alternating.jl:52,54 ---------------------------------------
    def update_motifs(self, data, W, H, l1W=0.0, l2W=0.0, **kwargs):
        """update_motifs!(rule, data, W, H; l1W, l2W)  (mult.jl:23-39 / hals.jl:31-34)."""
        super().update_motifs(l1W, l2W)
        if self.sync_host and W is not None:
            Wn, _ = self.get_factors()
            W[...] = Wn

    def update_feature_maps(self, data, W, H, l1H=0.0, l2H=0.0, **kwargs):
        """loss = update_feature_maps!(rule, data, W, H; l1H, l2H)  (mult.jl:42-58 / hals.jl:37-42)."""
        loss = super().update_feature_maps(l1H, l2H)
        if self.sync_host and H is not None:
            _, Hn = self.get_factors()
            H[...] = Hn
        return loss

    # julia-style aliases
    update_motifs_ = update_motifs
    update_feature_maps_ = update_feature_maps


class MultUpdate(AbstractCFUpdate):
    """src/algs/mult.jl:1-58 on the GPU."""
    _ALG = MULT


class HALSUpdate(AbstractCFUpdate):
    """src/algs/hals.jl:6-154 on the GPU."""
    _ALG = HALS


class PGDUpdate(AbstractCFUpdate):
    """src/algs/pgd.jl:112-255 on the GPU for the SquareLoss / NonnegConstraint configuration.  The penalty lists
    of the reference are given as weights: ``l2W``/``l2H`` = SquarePenalty weight, ``l1W``/``l1H`` = AbsolutePenalty
    weight; the reference defaults are ``penaltiesW=[SquarePenalty(1)]`` and ``penaltiesH=[]`` (pgd.jl:161,185)."""
    _ALG = PGD

    def __init__(self, data, W, H, loss_func="square", mask=None, constrW="nonneg", constrH="nonneg", **kw):
        """``loss_func``: "square" (SquareLoss, pgd.jl:28-35) or "absolute" (AbsoluteLoss, :38-45); ``mask`` (N x T) wraps it in a
        MaskedLoss (:59-70).  Both run on the device (cmf_set_pgd_loss).  ``constrW`` / ``constrH``: "nonneg"
        (NonnegConstraint, :91-95) or "unitnorm" (UnitNormConstraint, :98-110) -- cmf_set_pgd_constraints."""
        super().__init__(data, W, H, **kw)
        cmap = {"nonneg": 0, "unitnorm": 1, 0: 0, 1: 1}
        if cmap[constrW] or cmap[constrH]:
            check(_lib.load().cmf_set_pgd_constraints(self._h, cmap[constrW], cmap[constrH]))
        lf = {"square": 0, "absolute": 1, 0: 0, 1: 1}[loss_func]
        if lf != 0 or mask is not None:
            m = None if mask is None else julia_array(np.asarray(mask), self.dtype)
            if m is not None and m.shape != (self.N, self.T):
                raise ValueError(f"mask must be {(self.N, self.T)}, got {m.shape}")
            check(_lib.load().cmf_set_pgd_loss(self._h, lf, None if m is None else fptr(m)))

    def update_motifs(self, data, W, H, l1W=0.0, l2W=1.0, **kwargs):
        return super().update_motifs(data, W, H, l1W=l1W, l2W=l2W, **kwargs)


_ALG_NAMES = {"mult": MultUpdate, ":mult": MultUpdate, "hals": HALSUpdate, ":hals": HALSUpdate,
              "pgd": PGDUpdate, ":pgd": PGDUpdate}


def _resolve_alg(alg):
    """Accepts the README symbols (:mult/:hals as strings) and the current-src rule types."""
    if isinstance(alg, str):
        try:
            return _ALG_NAMES[alg.lower()]
        except KeyError:
            raise ValueError(f"unknown alg {alg!r}: this path provides 'mult', 'hals' and 'pgd'") from None
    if isinstance(alg, type) and issubclass(alg, AbstractCFUpdate):
        return alg
    raise ValueError(f"alg must be 'mult', 'hals', MultUpdate or HALSUpdate, got {alg!r}")


# ------------------------------------------------------------------------------------------
# driver
# ------------------------------------------------------------------------------------------
class AlternatingOptimizer:
    """src/algs/alternating.jl:10-14."""

    def __init__(self, update_rule, max_itr=100, max_time=math.inf):
        self.update_rule, self.max_itr, self.max_time = update_rule, max_itr, max_time


def _alternate(loss, step, max_itr, max_time=math.inf, check_convergence=True, patience=3, tol=1e-4, tick=None):
    """The loop of src/algs/alternating.jl:37-66: ``loss`` before the first iteration, then ``step()`` (one iteration,
    returning its loss) until ``max_itr`` iterations, ``max_time`` seconds or convergence, with ``tick()`` after every
    iteration.  Returns (loss_hist, time_hist, stopped_early)."""
    loss_hist = [loss]                    # :37
    time_hist = [0.0]                     # :38
    itr = 1
    while itr <= max_itr and time_hist[-1] <= max_time:   # :45
        itr += 1
        t0 = _time.time()
        loss = step()
        time_hist.append(time_hist[-1] + (_time.time() - t0))
        loss_hist.append(loss)
        if tick is not None:
            tick()
        if check_convergence and converged(loss_hist, patience, tol):
            return loss_hist, time_hist, True
    return loss_hist, time_hist, False


def _results(data, W, H, time_hist, loss_hist, layout, engine_info=None):
    """CNMF_results from the factors as the library returns them: W (K x N x L) goes to ``layout``."""
    if layout == "LNK":
        W = np.ascontiguousarray(W.transpose(2, 1, 0))
    res = CNMF_results(data, W, H, list(time_hist), list(loss_hist), layout)
    if engine_info is not None:
        res.engine_info = engine_info      # not part of the reference struct: which engine / loss path produced loss_hist
    return res


def fit(alg, data, L, K, W_init, H_init, verbose=False, printer=print, layout="LNK", **kwargs):
    """src/algs/alternating.jl:16-71, stepping the rule from the host (one C-ABI call per
    half-step; factors stay on the device and are read back once at the end).  ``fit_cnmf`` uses
    the single-call device loop ``cmf_fit`` instead; both give identical histories."""
    check_convergence = kwargs.get("check_convergence", True)
    patience = kwargs.get("patience", 3)
    eval_mode = kwargs.get("eval_mode", False)
    assert patience >= 1
    tol = kwargs.get("tol", 1e-4)
    rule = alg.update_rule
    reg = {k: kwargs[k] for k in ("l1W", "l2W", "l1H", "l2H") if k in kwargs}

    def step():
        if not eval_mode:
            rule.update_motifs(data, None, None, **reg)
        return rule.update_feature_maps(data, None, None, **reg)

    rule.set_factors(W_init, H_init)      # alternating.jl:33-34 (deepcopy of the inits)
    old_sync, rule.sync_host = rule.sync_host, False
    try:
        loss0 = rule.loss()
        verbose and _emit(printer, "Starting ", False)
        loss_hist, time_hist, early = _alternate(loss0, step, alg.max_itr, alg.max_time, check_convergence, patience, tol,
                                                 tick=(lambda: _emit(printer, ".", False)) if verbose else None)
    finally:
        rule.sync_host = old_sync
    if early:
        _emit(printer, "Converged early.")   # :64, unconditional in the reference
    verbose and _emit(printer, " fit!")
    W, H = rule.get_factors()
    return _results(data, W, H, time_hist, loss_hist, layout)


def init_rand(data, L, K, seed=None, dtype="f64", device=0):
    """src/model.jl:113-125.  Uniform draws come from numpy's Generator (Julia's stream cannot be
    reproduced outside Julia; the Julia shim keeps its own ``rand``); the conv and the two
    reductions of the alpha rescale run on the GPU.  Returns (W K x N x L, H K x T).  ``data`` may be sparse."""
    if not _is_sparse(data):
        data = np.asarray(data)
    N, T = _data_shape(data)
    rng = np.random.default_rng(seed)
    W = rng.random((K, N, L))             # W drawn first (model.jl:116), then H (:117)
    H = rng.random((K, T))
    return _host_rescaled(data, W, H, dtype, device)


def _rescale(rule):
    dot, nrm2 = rule.init_scale_partials()
    alpha = dot / nrm2                    # model.jl:120
    s = math.sqrt(abs(alpha))             # model.jl:121-122
    rule.scale_factors(s)
    return s


class _FitCall:
    """What fit_cnmf and fit_cnmf_batch share: the keywords and the checks that come before their own, the data as a
    dense array or a ``scipy.sparse`` input, and the device loop (cmf_fit / cmf_fit_batch) with its history buffers and
    prints."""

    def __init__(self, data, alg, kwargs):
        self.kw = kw = _normalise_kwargs(kwargs)
        self.printer = kw.get("printer", print)
        self.verbose = kw.get("verbose", False)
        self.layout = kw.get("layout", "LNK")
        if self.layout not in ("LNK", "KNL"):
            raise ValueError("layout must be 'LNK' or 'KNL'")
        self.dtype = parse_dtype(kw.get("dtype", "f64"))
        self.device = kw.get("device", 0)
        self.rule_cls = _resolve_alg(alg)
        self.data_in = data
        self.sparse = _is_sparse(data)
        self.data = data if self.sparse else np.asarray(data)
        self.N, self.T = _data_shape(self.data)

    def run(self, entry, handle, regs, max_itr, max_time, R=1):
        """``entry(handle, <loop arguments>, *regs, <history buffers>)`` for a batch of R fits (R = 1: cmf_fit).  Returns
        (loss_hist R x cap, time_hist, iterations recorded per fit)."""
        kw = self.kw
        unbounded = not (max_itr < math.inf)
        cap = 1 + (int(max_itr) if not unbounded else 1_000_000)
        loss_hist = np.zeros(R * cap)
        time_hist = np.zeros(cap)
        n = np.zeros(R, dtype=np.int64)
        early = np.zeros(R, dtype=np.int32)
        self.verbose and _emit(self.printer, "Starting ", False)
        check(entry(
            handle._h, -1 if unbounded else int(max_itr), float(max_time),
            int(bool(kw.get("eval_mode", False))), int(bool(kw.get("check_convergence", True))),
            int(kw.get("patience", 3)), float(kw.get("tol", 1e-4)), *regs,
            _dptr(loss_hist), _dptr(time_hist), cap, n.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
            early.ctypes.data_as(ctypes.POINTER(ctypes.c_int))))
        self.verbose and _emit(self.printer, "." * (int(n.max()) - 1), False)
        for r in range(R):
            if early[r]:
                _emit(self.printer, "Converged early.")   # alternating.jl:64, once per fit that stopped early
        self.verbose and _emit(self.printer, " fit!")
        return loss_hist.reshape(R, cap), time_hist, n


def _dptr(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def fit_cnmf(data, L=10, K=5, alg=MultUpdate, max_itr=100, max_time=math.inf, **kwargs):
    """src/model.jl:58-85 as a drop-in: seeds, initialises (or takes W_init/H_init), constructs the
    rule and runs the alternating loop -- the loop itself is ONE call into the library (cmf_fit).

    Extra keywords of this implementation: ``dtype`` ("f64" default, "f32"), ``device``,
    ``layout`` ("LNK" default -- W returned as L x N x K as in the README -- or "KNL"), ``ngpu`` / ``devices``
    (the fit runs T-sharded over that many GPUs inside the same single library call; MultUpdate and HALSUpdate).
    ``data`` may be a ``scipy.sparse`` matrix or array (MultUpdate / HALSUpdate, one GPU): X is then never densified;
    ``CNMF_results.data`` is the caller's matrix."""
    fc = _FitCall(data, alg, kwargs)
    kw, dtype, device, rule_cls, N, T = fc.kw, fc.dtype, fc.device, fc.rule_cls, fc.N, fc.T
    L, K = int(L), int(K)
    _check_sparse_rule(fc.sparse, rule_cls, kw.get("ngpu", 1))
    data = fc.data
    if fc.sparse:
        W0, H0 = kw.get("W_init"), kw.get("H_init")
        if (W0 is not None and np.shape(W0) != (K, N, L)) or (H0 is not None and np.shape(H0) != (K, T)):
            raise ValueError(f"W_init must be {(K, N, L)} and H_init {(K, T)}; got {np.shape(W0)}, {np.shape(H0)}")
        data = as_csc(data, dtype)

    rng = np.random.default_rng(kw.get("seed"))      # model.jl:64-67
    W0 = kw.get("W_init")
    H0 = kw.get("H_init")
    need_rescale = W0 is None and H0 is None
    # model.jl:70-73: init_rand always runs, then either factor may be overridden
    Wr, Hr = rng.random((K, N, L)), rng.random((K, T))
    if W0 is None or H0 is None:
        if not need_rescale:
            Wr, Hr = _host_rescaled(data, Wr, Hr, dtype, device)
        W0 = Wr if W0 is None else W0
        H0 = Hr if H0 is None else H0
    W0, H0 = np.asarray(W0), np.asarray(H0)
    if W0.shape != (K, N, L) or H0.shape != (K, T):
        raise ValueError(f"W_init must be {(K, N, L)} and H_init {(K, T)}; got {W0.shape}, {H0.shape}")

    extra = {}
    if rule_cls is PGDUpdate:
        extra = dict(loss_func=kw.get("loss_func", "square"), mask=kw.get("mask"),
                     constrW=kw.get("constrW", "nonneg"), constrH=kw.get("constrH", "nonneg"))
    with rule_cls(data, W0, H0, dtype=dtype, device=device, sync_host=False,
                  engine=kw.get("engine"), loss_mode=kw.get("loss_mode"), loss_guard=kw.get("loss_guard"),
                  ngpu=kw.get("ngpu", 1), devices=kw.get("devices"), **extra) as rule:   # model.jl:79
        if need_rescale:
            _rescale(rule)
        regs = [float(kw.get("l1W", 0.0)), float(kw.get("l2W", 1.0 if rule_cls is PGDUpdate else 0.0)),
                float(kw.get("l1H", 0.0)), float(kw.get("l2H", 0.0))]
        loss_hist, time_hist, n = fc.run(_lib.load().cmf_fit, rule, regs, max_itr, max_time)
        W, H = rule.get_factors()
        engine_info = dict(rule.loss_stats(), engine=rule.get_engine(), loss_mode=rule.loss_mode)
    return _results(fc.data_in, W, H, time_hist[: n[0]], loss_hist[0, : n[0]], fc.layout, engine_info)


def _per_restart(name, v, R):
    a = np.asarray(v, dtype=np.float64)
    if a.ndim == 0:
        return np.full(R, float(a))
    if a.shape != (R,):
        raise ValueError(f"{name} must be a scalar or have one value per restart ({R}), got shape {a.shape}")
    return np.ascontiguousarray(a)


def _batch_ranks(K):
    ranks = list(K)
    for k in ranks:
        if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or k < 1:
            raise ValueError(f"every rank in K must be a positive integer; got {k!r}")
    if not ranks:
        raise ValueError("a batch needs at least one restart")
    return [int(k) for k in ranks]


def fit_cnmf_batch(data, L=10, K=5, alg=MultUpdate, max_itr=100, max_time=math.inf, *, seeds=None, **kwargs):
    """R MultUpdate fits of the same data in ONE library handle and one device loop (cmf_fit_batch).

    Restart r equals ``fit_cnmf(data, L, K, alg="mult", seed=seeds[r], l1W=l1W[r], ...)`` -- or the fit from
    ``W_init=W_init[r], H_init=H_init[r]`` -- with every other keyword the same: same initial draws and alpha rescale, same
    ``loss_hist`` and early stop.  ``seeds`` is a sequence of R seeds; otherwise ``W_init`` (R x K x N x L) and ``H_init``
    (R x K x T) are both given.  ``l1W``, ``l2W``, ``l1H``, ``l2H`` are scalars or length-R sequences.  A restart that meets
    the early stop is frozen while the others go on.  The one deliberate difference from R separate fits: ``max_time`` and
    ``time_hist`` use the batch's wall clock, so every restart has the same ``time_hist`` (cut to its own length).
    Returns a list of R ``CNMF_results``.  MultUpdate, fp64 / fp32, one GPU, the SIMT engine.

    ``K`` may also be a sequence of R positive ranks (a sweep over K in one handle, cmf_create_batch_ranks): restart r
    then has rank ``K[r]``, ``seeds`` has R entries, and ``W_init`` / ``H_init`` are sequences of R arrays of shapes
    ``K[r] x N x L`` and ``K[r] x T``.

    ``data`` may be a ``scipy.sparse`` matrix or array (cmf_create_batch_sparse): X is stored once as compressed sparse
    columns and never densified."""
    fc = _FitCall(data, alg, kwargs)
    kw, dtype, N, T = fc.kw, fc.dtype, fc.N, fc.T
    L = int(L)
    _check_sparse_rule(fc.sparse, fc.rule_cls, 1)
    ranks = None if np.ndim(K) == 0 else _batch_ranks(K)
    K = int(K) if ranks is None else None
    W0, H0 = kw.get("W_init"), kw.get("H_init")
    if seeds is not None:
        if W0 is not None or H0 is not None:
            raise ValueError("give either seeds or the W_init / H_init stacks, not both")
        seeds = list(seeds)
        R = len(seeds)
    elif W0 is not None and H0 is not None and ranks is not None:
        W0, H0 = [np.asarray(w) for w in W0], [np.asarray(x) for x in H0]
        R = len(ranks)
        if len(W0) != R or len(H0) != R:
            raise ValueError(f"W_init and H_init need one array per rank ({R}); got {len(W0)} and {len(H0)}")
        for r, (k, w, x) in enumerate(zip(ranks, W0, H0)):
            if w.shape != (k, N, L) or x.shape != (k, T):
                raise ValueError(f"W_init[{r}] must be {(k, N, L)} and H_init[{r}] {(k, T)}; got {w.shape}, {x.shape}")
    elif W0 is not None and H0 is not None:
        W0, H0 = np.asarray(W0), np.asarray(H0)
        if W0.ndim != 4 or H0.ndim != 3 or W0.shape[0] != H0.shape[0]:
            raise ValueError(f"W_init must be R x {(K, N, L)} and H_init R x {(K, T)}; got {W0.shape}, {H0.shape}")
        R = W0.shape[0]
        if W0.shape[1:] != (K, N, L) or H0.shape[1:] != (K, T):
            raise ValueError(f"W_init must be R x {(K, N, L)} and H_init R x {(K, T)}; got {W0.shape}, {H0.shape}")
    else:
        raise ValueError("fit_cnmf_batch needs seeds, or both the W_init and H_init stacks")
    if R < 1:
        raise ValueError("a batch needs at least one restart")
    if ranks is not None and len(ranks) != R:
        raise ValueError(f"K has {len(ranks)} ranks but the batch has {R} restarts")
    regs = {k: _per_restart(k, kw.get(k, 0.0), R) for k in ("l1W", "l2W", "l1H", "l2H")}
    if int(kw.get("ngpu", 1) or 1) > 1:
        raise CMFError(3, "batched restarts run on one GPU")

    Ks = [K] * R if ranks is None else ranks
    if seeds is not None:                                 # model.jl:64-67, 116-117: W drawn first, then H
        W0, H0 = [], []
        for k, seed in zip(Ks, seeds):
            rng = np.random.default_rng(seed)
            W0.append(rng.random((k, N, L)))
            H0.append(rng.random((k, T)))
    # restart-major host stacks, each block column-major (include/cmf_sm100.h)
    Wj = np.concatenate([julia_array(w, dtype).ravel(order="F") for w in W0])
    Hj = np.concatenate([julia_array(x, dtype).ravel(order="F") for x in H0])

    data = as_csc(fc.data, dtype) if fc.sparse else fc.data
    lib = _lib.load()
    with Handle(N, T, K if ranks is None else ranks, L, dtype, fc.rule_cls._ALG, fc.device, sparse=fc.sparse,
                restarts=R) as h:
        if kw.get("engine") is not None:
            h.set_engine(kw["engine"])
        if kw.get("loss_mode") is not None:
            h.set_loss_mode(kw["loss_mode"])
        if fc.sparse:
            _set_csc(h._h, data)
        else:
            h.set_data(data)
        check(lib.cmf_set_factors_batch(h._h, fptr(Wj), fptr(Hj)))
        if seeds is not None:                             # model.jl:119-122, per restart
            part = np.zeros(2 * R)
            check(lib.cmf_init_scale_partials_batch(h._h, _dptr(part)))
            s = np.sqrt(np.abs(part[0::2] / part[1::2]))
            check(lib.cmf_scale_factors_batch(h._h, _dptr(s)))
        loss_hist, time_hist, n = fc.run(lib.cmf_fit_batch, h, [_dptr(regs[k]) for k in ("l1W", "l2W", "l1H", "l2H")],
                                         max_itr, max_time, R)
        dt = np_dtype(dtype)
        Wo = np.empty(N * L * sum(Ks), dtype=dt)
        Ho = np.empty(T * sum(Ks), dtype=dt)
        check(lib.cmf_get_factors_batch(h._h, fptr(Wo), fptr(Ho)))
    out = []
    offs = np.concatenate([[0], np.cumsum(Ks)])
    for r in range(R):
        k, o = Ks[r], int(offs[r])
        W = Wo[N * L * o: N * L * (o + k)].reshape((k, N, L), order="F")
        H = Ho[T * o: T * (o + k)].reshape((k, T), order="F")
        nr = int(n[r])
        info = dict(direct=0 if fc.sparse else nr, expansion=nr if fc.sparse else 0, interval=0, last_err=0.0, engine=0,
                    loss_mode=int(fc.sparse), restarts=R)
        out.append(_results(fc.data_in, W, H, time_hist[:nr], loss_hist[r, :nr], fc.layout, info))
    return out


def _temporary_rule(data, W, H, dtype, device):
    """A MultUpdate rule for one computation on the device; use it as ``with _temporary_rule(...) as rule:``, which
    frees its handle."""
    return MultUpdate(data, W, H, dtype=dtype, device=device, sync_host=False)


def _host_rescaled(data, W, H, dtype, device):
    """(W, H) times the alpha rescale of src/model.jl:119-122, computed on the device."""
    with _temporary_rule(data, W, H, dtype, device) as rule:
        s = _rescale(rule)
    return W * s, H * s


# ------------------------------------------------------------------------------------------
# tensor primitives (src/common.jl) -- host in / host out, used by tests and notebooks
# ------------------------------------------------------------------------------------------
def tensor_conv(W, H, dtype="f64"):
    """src/common.jl:17-34."""
    dt = parse_dtype(dtype)
    K, N, L = W.shape
    T = H.shape[1]
    out = np.empty((N, T), dtype=np_dtype(dt), order="F")
    Wj, Hj = julia_array(W, dt), julia_array(H, dt)
    check(_lib.load().cmf_tensor_conv(N, T, K, L, dt, fptr(Wj), fptr(Hj), fptr(out)))
    return out


def tensor_transconv(W, X, dtype="f64"):
    """src/common.jl:62-81."""
    dt = parse_dtype(dtype)
    K, N, L = W.shape
    T = X.shape[1]
    out = np.empty((K, T), dtype=np_dtype(dt), order="F")
    Wj, Xj = julia_array(W, dt), julia_array(X, dt)
    check(_lib.load().cmf_tensor_transconv(N, T, K, L, dt, fptr(Wj), fptr(Xj), fptr(out)))
    return out


def corr_w(H, X, L, dtype="f64"):
    """numW of src/algs/mult.jl:31-34."""
    dt = parse_dtype(dtype)
    K, T = H.shape
    N = X.shape[0]
    out = np.empty((K, N, L), dtype=np_dtype(dt), order="F")
    Hj, Xj = julia_array(H, dt), julia_array(X, dt)
    check(_lib.load().cmf_corr_w(N, T, K, L, dt, fptr(Hj), fptr(Xj), fptr(out)))
    return out


def compute_resids(data, W, H, dtype="f64"):
    """src/common.jl:58-59: tensor_conv(W, H) - data."""
    dt = parse_dtype(dtype)
    K, N, L = W.shape
    T = H.shape[1]
    out = np.empty((N, T), dtype=np_dtype(dt), order="F")
    Xj, Wj, Hj = julia_array(data, dt), julia_array(W, dt), julia_array(H, dt)
    check(_lib.load().cmf_compute_resids(N, T, K, L, dt, fptr(Xj), fptr(Wj), fptr(Hj), fptr(out)))
    return out


def shift_and_stack(H, L, dtype="f64"):
    """src/common.jl:133-142: (K*L) x T matrix whose row l*K + k is H[k, :] shifted right by l columns."""
    dt = parse_dtype(dtype)
    K, T = H.shape
    out = np.empty((K * L, T), dtype=np_dtype(dt), order="F")
    Hj = julia_array(H, dt)
    check(_lib.load().cmf_shift_and_stack(K, T, L, dt, fptr(Hj), fptr(out)))
    return out


def compute_loss(data, W, H, dtype="f64", device=0):
    """src/common.jl:54-55."""
    with _temporary_rule(data, W, H, dtype, device) as rule:
        return rule.loss()
