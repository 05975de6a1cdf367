"""Sparse data (cmf_create_sparse / cmf_create_batch_sparse / cmf_set_data_csc): fits on CSC matrices without the dense X.

The two contractions that read X (numW, numH) are checked against a dense handle of the same data, the fits against the
dense fits and the C oracle at the bars of tests/test_gpu_batch.py, and the handle rules against the header."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

REG = dict(l1W=0.1, l2W=0.5, l1H=0.1, l2H=0.2)
NOREG = dict(l1W=0.0, l2W=0.0, l1H=0.0, l2H=0.0)


@pytest.fixture(scope="module")
def cmf():
    import __graft_entry__ as ge

    ge.build()
    import cmf_jl_b200

    return cmf_jl_b200


def thinned(N, T, L, density, seed=7, K_true=3):
    """Spike-like data: the convolutive model of synthetic_sequences, Bernoulli-thinned to the target density."""
    from oracle import cnmf_oracle as po

    rng = np.random.default_rng(seed)
    X, _, _ = po.synthetic_sequences(K=K_true, N=N, L=L, T=T, rng=rng)
    keep = rng.random(X.shape) < density / max(np.count_nonzero(X) / X.size, density)
    return sp.csc_matrix(np.where(keep, X, 0.0))


def exact_sparse(N, T, K, L, seed=3):
    """Data of the model with sparse W and H (about 1 % nonzeros, multiplicative noise on them) and a start near the factors."""
    rng = np.random.default_rng(seed)
    W = np.zeros((K, N, L))
    for k in range(K):
        units = rng.choice(N, size=max(N // 8, 1), replace=False)
        lags = rng.choice(L, size=min(3, L), replace=False)
        W[k][np.ix_(units, lags)] = rng.random((len(units), len(lags))) + 0.5
    H = np.where(rng.random((K, T)) < 0.01, rng.exponential(1.0, (K, T)), 0.0)
    from oracle import cnmf_oracle as po

    X = po.tensor_conv(W, H)
    X = np.where(X > 0, X * np.abs(1 + 0.06 * rng.standard_normal(X.shape)), 0.0)   # noise on the nonzeros: a loss floor of a few %
    W0 = W * (1 + 0.3 * rng.random(W.shape)) + 0.02
    H0 = H * (1 + 0.3 * rng.random(H.shape)) + 0.02
    return sp.csc_matrix(X), W0, H0


def _rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b) / np.abs(b)))


def _close(a, b, rtol, atol):
    np.testing.assert_allclose(np.asarray(a), np.asarray(b), rtol=rtol, atol=atol)


def _buffer(cmf, rule, which):
    """Device buffer `which` of a rule's handle (cmf_exchange_buffer) as a host array."""
    import torch

    from cmf_jl_b200.sharded import _CudaView

    lib = cmf._lib.load()
    p, n, dt = ctypes.c_void_p(), ctypes.c_int64(), ctypes.c_int()
    cmf._lib.check(lib.cmf_exchange_buffer(rule._h, which, ctypes.byref(p), ctypes.byref(n), ctypes.byref(dt)))
    cmf._lib.check(lib.cmf_sync(rule._h))
    ts = {0: "<f8", 1: "<f4"}[dt.value]
    return torch.as_tensor(_CudaView(p.value, n.value, ts), device="cuda").cpu().numpy().copy()


def _contractions(cmf, X, W, H, dtype):
    """(numW, numH) of a MultUpdate handle on X after one cmf_w_partials and one cmf_h_update from (W, H)."""
    lib = cmf._lib.load()
    rule = cmf.MultUpdate(X, W, H, dtype=dtype, sync_host=False)
    try:
        cmf._lib.check(lib.cmf_w_partials(rule._h))
        numW = _buffer(cmf, rule, 0)
        cmf._lib.check(lib.cmf_h_update(rule._h, 0.0, 0.0))
        numH = _buffer(cmf, rule, 2)
    finally:
        rule.close()
    return numW, numH


def _edge_cases():
    rng = np.random.default_rng(11)
    out = []
    # empty columns and empty rows
    D = rng.random((40, 333)) * (rng.random((40, 333)) < 0.05)
    D[:, 100:180] = 0.0
    D[7:15] = 0.0
    out.append(("empty_cols_rows", D, 4, 9))
    # nonzeros only in the last L-1 columns
    D = np.zeros((30, 257))
    D[:, -6:] = rng.random((30, 6)) * (rng.random((30, 6)) < 0.5)
    D[0, -1] = 1.0
    out.append(("last_L-1_cols", D, 3, 7))
    out.append(("K1", rng.random((50, 301)) * (rng.random((50, 301)) < 0.03), 1, 5))
    out.append(("L1", rng.random((50, 301)) * (rng.random((50, 301)) < 0.03), 4, 1))
    D = rng.random((1, 401)) * (rng.random((1, 401)) < 0.1)
    D[0, 3] = 1.0
    out.append(("N1", D, 3, 6))
    out.append(("odd_T", rng.random((37, 1237)) * (rng.random((37, 1237)) < 0.02), 6, 11))
    return out


@pytest.mark.parametrize("dtype,bar", [("f64", 1e-12), ("f32", 1e-5)])
def test_contractions_match_dense_handle(cmf, dtype, bar):
    cases = [("thinned_1pct", thinned(96, 1500, 12, 0.01).toarray(), 5, 12),
             ("thinned_5pct", thinned(64, 900, 9, 0.05, seed=2).toarray(), 7, 9)] + _edge_cases()
    for name, D, K, L in cases:
        N, T = D.shape
        rng = np.random.default_rng(5)
        W, H = rng.random((K, N, L)), rng.random((K, T))
        sW, sH = _contractions(cmf, sp.csc_matrix(D), W, H, dtype)
        dW, dH = _contractions(cmf, D, W, H, dtype)
        assert np.max(np.abs(sW - dW)) / np.max(np.abs(dW)) <= bar, name
        assert np.max(np.abs(sH - dH)) / np.max(np.abs(dH)) <= bar, name


@pytest.mark.parametrize("alg", ["mult", "hals"])
@pytest.mark.parametrize("layout", ["LNK", "KNL"])
def test_fp64_fits_match_dense_and_oracle(cmf, alg, layout):
    from oracle import c_oracle as co

    N, T, K, L, itr = 80, 700, 4, 9, 30
    Xs = thinned(N, T, L, 0.03, seed=4)
    X = Xs.toarray()
    rule = {"mult": co.MultUpdate, "hals": co.HALSUpdate}[alg]
    for reg in (NOREG, REG):
        s = cmf.fit_cnmf(Xs, L=L, K=K, alg=alg, max_itr=itr, seed=21, check_convergence=False, layout=layout, **reg)
        d = cmf.fit_cnmf(X, L=L, K=K, alg=alg, max_itr=itr, seed=21, check_convergence=False, layout=layout, **reg)
        assert s.data is Xs
        assert s.engine_info["engine"] == 0 and s.engine_info["loss_mode"] == 1 and s.engine_info["direct"] == 0
        assert len(s.loss_hist) == itr + 1
        assert _rel(s.loss_hist, d.loss_hist) < 1e-9
        _close(s.W, d.W, 1e-8, 1e-11)
        _close(s.H, d.H, 1e-8, 1e-11)
        init = cmf.fit_cnmf(Xs, L=L, K=K, max_itr=0, seed=21, check_convergence=False, layout="KNL")
        ref = co.fit(rule, X, init.W, init.H, itr, check_convergence=False, **reg)
        assert _rel(s.loss_hist, ref.loss_hist) < 1e-9
        Wk = s.W if layout == "KNL" else s.W.transpose(2, 1, 0)
        _close(Wk, ref.W, 1e-8, 1e-11)
        _close(s.H, ref.H, 1e-8, 1e-11)


@pytest.mark.parametrize("alg", ["mult", "hals"])
def test_fp32_fits_at_low_loss_match_fp64_oracle(cmf, alg):
    from oracle import c_oracle as co

    N, T, K, L, itr = 64, 2000, 3, 8, 100
    Xs, W0, H0 = exact_sparse(N, T, K, L)
    assert 0.002 < Xs.nnz / (N * T) < 0.05
    rule = {"mult": co.MultUpdate, "hals": co.HALSUpdate}[alg]
    ref = co.fit(rule, Xs.toarray(), W0, H0, itr, check_convergence=False)
    got = cmf.fit_cnmf(Xs, L=L, K=K, alg=alg, max_itr=itr, W_init=W0, H_init=H0, dtype="f32", check_convergence=False,
                       layout="KNL")
    assert ref.loss_hist[-1] < 0.1
    assert _rel(got.loss_hist, ref.loss_hist) < 1e-4


def test_helpers_take_sparse_data(cmf):
    N, T, K, L = 50, 400, 3, 6
    Xs = thinned(N, T, L, 0.04, seed=8)
    X = Xs.toarray()
    Ws, Hs = cmf.init_rand(Xs, L, K, seed=3)
    Wd, Hd = cmf.init_rand(X, L, K, seed=3)
    _close(Ws, Wd, 1e-10, 0)
    _close(Hs, Hd, 1e-10, 0)
    assert abs(cmf.compute_loss(Xs, Wd, Hd) / cmf.compute_loss(X, Wd, Hd) - 1) < 1e-10
    for alg in (cmf.MultUpdate, cmf.HALSUpdate):
        rs = cmf.fit(cmf.AlternatingOptimizer(alg(sp.coo_matrix(Xs), Wd, Hd), max_itr=5), sp.csr_array(Xs), L, K, Wd, Hd,
                     check_convergence=False)
        rd = cmf.fit(cmf.AlternatingOptimizer(alg(X, Wd, Hd), max_itr=5), X, L, K, Wd, Hd, check_convergence=False)
        assert _rel(rs.loss_hist, rd.loss_hist) < 1e-9


def test_determinism(cmf):
    Xs = thinned(128, 3000, 16, 0.02, seed=5)
    for alg, dtype in (("mult", "f32"), ("hals", "f32"), ("mult", "f64")):
        a = cmf.fit_cnmf(Xs, L=16, K=6, alg=alg, max_itr=15, seed=1, dtype=dtype, check_convergence=False)
        b = cmf.fit_cnmf(Xs, L=16, K=6, alg=alg, max_itr=15, seed=1, dtype=dtype, check_convergence=False)
        assert np.array_equal(a.W, b.W) and np.array_equal(a.H, b.H) and a.loss_hist == b.loss_hist


def test_batch_matches_single_sparse_fits(cmf):
    N, T, L, itr = 90, 800, 8, 40
    Xs = thinned(N, T, L, 0.03, seed=6)
    ranks = [1, 3, 5, 5, 8]
    R = len(ranks)
    regs = {k: np.zeros(R) for k in REG}
    for r in range(R):
        if r % 2 == 1:
            for k, v in REG.items():
                regs[k][r] = v
    seeds = [31 + r for r in range(R)]
    for K in (4, ranks):
        batch = cmf.fit_cnmf_batch(Xs, L=L, K=K, max_itr=itr, seeds=seeds, patience=3, tol=2e-4, layout="KNL", **regs)
        assert batch[0].data is Xs
        stopped = 0
        for r in range(R):
            k = K if np.ndim(K) == 0 else K[r]
            reg = {n: float(v[r]) for n, v in regs.items()}
            single = cmf.fit_cnmf(Xs, L=L, K=k, alg="mult", max_itr=itr, seed=seeds[r], patience=3, tol=2e-4, layout="KNL",
                                  **reg)
            b = batch[r]
            stopped += len(b.loss_hist) < itr + 1
            assert len(b.loss_hist) == len(single.loss_hist)
            assert _rel(b.loss_hist, single.loss_hist) < 1e-9
            _close(b.W, single.W, 1e-8, 1e-11)
            _close(b.H, single.H, 1e-8, 1e-11)
        assert stopped >= 1                   # the early stop of some restarts is exercised


def _batch_launches_per_iteration(cmf, Xs, K, L):
    """Kernel launches of one cmf_fit_batch iteration of a sparse batch with ranks K (difference of a 3- and a 1-iteration fit)."""
    lib = cmf._lib.load()
    c = cmf.as_csc(Xs, "f64")
    N, T = c.shape
    R = len(K)
    rk = np.asarray(K, dtype=np.int64)
    out = []
    for itr in (1, 3):
        h = ctypes.c_void_p()
        cmf._lib.check(lib.cmf_create_batch_sparse(ctypes.byref(h), N, T, rk.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), L,
                                                   0, 0, R, 0))
        try:
            cmf.model._set_csc(h, c)
            rng = np.random.default_rng(0)
            W = rng.random(N * L * int(rk.sum()))
            H = rng.random(T * int(rk.sum()))
            cmf._lib.check(lib.cmf_set_factors_batch(h, cmf._lib.fptr(W), cmf._lib.fptr(H)))
            z = np.zeros(R)
            dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))  # noqa: E731
            lh, th = np.zeros(R * 8), np.zeros(8)
            n, e = np.zeros(R, dtype=np.int64), np.zeros(R, dtype=np.int32)
            before = ctypes.c_int64()
            cmf._lib.check(lib.cmf_launch_count(h, ctypes.byref(before)))
            cmf._lib.check(lib.cmf_fit_batch(h, itr, 1e300, 0, 0, 3, 1e-4, dp(z), dp(z), dp(z), dp(z), dp(lh), dp(th), 8,
                                             n.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
                                             e.ctypes.data_as(ctypes.POINTER(ctypes.c_int))))
            after = ctypes.c_int64()
            cmf._lib.check(lib.cmf_launch_count(h, ctypes.byref(after)))
            out.append(after.value - before.value)
        finally:
            lib.cmf_destroy(h)
    return (out[1] - out[0]) / 2


def test_batch_launches_do_not_depend_on_R_or_nnz(cmf):
    L = 6
    a = _batch_launches_per_iteration(cmf, thinned(40, 500, L, 0.01, seed=1), [3] * 2, L)
    b = _batch_launches_per_iteration(cmf, thinned(40, 500, L, 0.01, seed=1), [3] * 64, L)
    c = _batch_launches_per_iteration(cmf, thinned(40, 500, L, 0.05, seed=1), [3] * 2, L)
    assert a == b == c and a > 0


def test_handle_rules(cmf):
    lib = cmf._lib.load()
    N, T, K, L = 30, 200, 3, 5
    Xs = thinned(N, T, L, 0.05, seed=2)
    c = cmf.as_csc(Xs, "f64")
    i64 = ctypes.POINTER(ctypes.c_int64)
    h = ctypes.c_void_p()
    cmf._lib.check(lib.cmf_create_sparse(ctypes.byref(h), N, T, K, L, 0, 1, 0))
    err = lambda: lib.cmf_last_error().decode()  # noqa: E731
    try:
        X = np.zeros((N, T))
        assert lib.cmf_set_data(h, cmf._lib.fptr(X), 0) == 1 and "cmf_set_data_csc" in err()
        assert lib.cmf_synth_data(h, 1, 2, 3, 0.1, 0.0) == 1 and "cmf_set_data_csc" in err()
        assert lib.cmf_get_data(h, cmf._lib.fptr(X), 0) == 1 and "cmf_set_data_csc" in err()
        assert lib.cmf_set_engine(h, 1) == 3 and lib.cmf_set_engine(h, 2) == 3
        assert lib.cmf_set_engine(h, 0) == 0
        eng, lm = ctypes.c_int(), ctypes.c_int()
        cmf._lib.check(lib.cmf_get_engine(h, ctypes.byref(eng)))
        cmf._lib.check(lib.cmf_get_loss_mode(h, ctypes.byref(lm)))
        assert eng.value == 0 and lm.value == 1
        assert lib.cmf_set_loss_mode(h, 0) == 3 and lib.cmf_set_loss_mode(h, 1) == 0
        assert lib.cmf_set_loss_guard(h, 0.5, 16) == 3

        def put(colptr, rowval, nzval, base=0, nnz=None):
            colptr, rowval = np.asarray(colptr, dtype=np.int64), np.asarray(rowval, dtype=np.int64)
            nzval = np.asarray(nzval, dtype=np.float64)
            return lib.cmf_set_data_csc(h, len(nzval) if nnz is None else nnz, colptr.ctypes.data_as(i64),
                                        rowval.ctypes.data_as(i64), cmf._lib.fptr(nzval), base)

        good = (c.colptr, c.rowval, c.nzval)
        assert put(*good, base=2) == 1 and "index_base" in err()
        assert put(*good, nnz=0) == 1 and "nnz" in err()
        bad = c.colptr.copy(); bad[0] = 1
        assert put(bad, c.rowval, c.nzval) == 1 and "colptr[0]" in err()
        bad = c.colptr.copy(); bad[-1] += 1
        assert put(bad, c.rowval, c.nzval) == 1 and "colptr[T]" in err()
        bad = c.colptr.copy(); j = int(np.argmax(np.diff(c.colptr) > 0)) + 1; bad[j] = bad[j - 1] - 1
        assert put(bad, c.rowval, c.nzval) == 1 and "column" in err()
        t = int(np.argmax(np.diff(c.colptr) >= 2))                       # a column with two entries
        i0 = int(c.colptr[t])
        bad = c.rowval.copy(); bad[i0] = N
        assert put(c.colptr, bad, c.nzval) == 1 and f"entry {i0}" in err() and f"column {t}" in err()
        bad = c.rowval.copy(); bad[i0 + 1] = bad[i0]
        assert put(c.colptr, bad, c.nzval) == 1 and "strictly increase" in err() and f"column {t}" in err()
        assert put(c.colptr + 1, c.rowval + 1, c.nzval, base=1) == 0      # Julia's 1-based arrays, unchanged
        ss = ctypes.c_double()
        cmf._lib.check(lib.cmf_data_sumsq(h, ctypes.byref(ss)))
        assert abs(ss.value - float(np.sum(c.nzval ** 2))) <= 1e-12 * ss.value
    finally:
        lib.cmf_destroy(h)
    # the dense handle refuses cmf_set_data_csc and names cmf_create_sparse
    cmf._lib.check(lib.cmf_create(ctypes.byref(h), N, T, K, L, 0, 0, 0))
    try:
        assert lib.cmf_set_data_csc(h, c.nnz, c.colptr.ctypes.data_as(i64), c.rowval.ctypes.data_as(i64),
                                    cmf._lib.fptr(c.nzval), 0) == 1 and "cmf_create_sparse" in err()
    finally:
        lib.cmf_destroy(h)


def test_beyond_dense_memory(cmf):
    """N = 4096, T = 2^24, fp32: the dense X would need 275 GB, more than the device has.  6 nonzeros per column (0.15 %)."""
    import torch

    lib = cmf._lib.load()
    N, T, K, L, per_col = 4096, 1 << 24, 16, 32, 6
    rng = np.random.default_rng(0)
    gaps = rng.integers(1, 600, size=(T, per_col))
    gaps[:, 0] = rng.integers(0, 600, size=T)
    rowval = np.cumsum(gaps, axis=1).ravel()                            # strictly increasing in every column, < 3600
    del gaps
    nzval = rng.random(T * per_col, dtype=np.float32)
    colptr = np.arange(0, T * per_col + 1, per_col, dtype=np.int64)
    dense_bytes = N * T * 4
    _, total = torch.cuda.mem_get_info()
    assert dense_bytes > total
    h = ctypes.c_void_p()
    i64 = ctypes.POINTER(ctypes.c_int64)
    cmf._lib.check(lib.cmf_create_sparse(ctypes.byref(h), N, T, K, L, 1, 0, 0))
    try:
        eng = ctypes.c_int()
        cmf._lib.check(lib.cmf_get_engine(h, ctypes.byref(eng)))
        assert eng.value == 0                                   # a dense fp32 handle of this shape would default to tcgen05
        cmf._lib.check(lib.cmf_set_data_csc(h, len(nzval), colptr.ctypes.data_as(i64), rowval.ctypes.data_as(i64),
                                            cmf._lib.fptr(nzval), 0))
        del rowval
        cmf._lib.check(lib.cmf_init_rand(h, 7))
        part = (ctypes.c_double * 2)()
        cmf._lib.check(lib.cmf_init_scale_partials(h, part))
        cmf._lib.check(lib.cmf_scale_factors(h, float(np.sqrt(abs(part[0] / part[1])))))
        lh, th = np.zeros(8), np.zeros(8)
        n, e = ctypes.c_int64(), ctypes.c_int()
        dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))  # noqa: E731
        cmf._lib.check(lib.cmf_fit(h, 3, 1e300, 0, 0, 3, 1e-4, 0.0, 0.0, 0.0, 0.0, dp(lh), dp(th), 8, ctypes.byref(n),
                                   ctypes.byref(e)))
        free, total = torch.cuda.mem_get_info()
        hist = lh[: n.value]
        assert n.value == 4 and np.all(np.isfinite(hist)) and np.all(np.diff(hist) < 0), hist
        assert total - free < dense_bytes
    finally:
        lib.cmf_destroy(h)
