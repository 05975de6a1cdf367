"""Batched restarts (cmf_create_batch / fit_cnmf_batch): R MultUpdate fits of one data set in one handle.

Restart r of a batch must equal fit_cnmf with seed seeds[r] (or W_init[r], H_init[r]) and its own regularisers.  The batch
stacks the restarts along the component axis, so numW and numH sum over the same terms in a different grouping: fp64 results
agree to ~1e-12, far inside the 1e-9 bar; with R = 1 the launches are the single handle's."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

REG = dict(l1W=0.1, l2W=0.5, l1H=0.1, l2H=0.2)


@pytest.fixture(scope="module")
def cmf():
    import __graft_entry__ as ge

    ge.build()
    import cmf_jl_b200

    return cmf_jl_b200


def _data(N, T, L, seed=7, K_true=3):
    from oracle import cnmf_oracle as po

    X, _, _ = po.synthetic_sequences(K=K_true, N=N, L=L, T=T, rng=np.random.default_rng(seed))
    return X


def _regs(R):
    # some restarts unregularised, some with the REG set, one with a mix
    out = {k: np.zeros(R) for k in REG}
    for r in range(R):
        if r % 3 == 1:
            for k, v in REG.items():
                out[k][r] = v
        elif r % 3 == 2:
            out["l1W"][r], out["l2H"][r] = 0.05, 0.3
    return out


def _rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b) / np.abs(b)))


def _close(a, b, rtol, atol):
    np.testing.assert_allclose(np.asarray(a), np.asarray(b), rtol=rtol, atol=atol)


@pytest.mark.parametrize("layout", ["LNK", "KNL"])
def test_fp64_parity_with_single_fits_and_oracle(cmf, layout):
    from oracle import c_oracle as co

    N, T, K, L, R, itr = 120, 600, 5, 10, 5, 30
    X = _data(N, T, L)
    seeds = [11, 12, 13, 14, 15]
    regs = _regs(R)
    batch = cmf.fit_cnmf_batch(X, L=L, K=K, max_itr=itr, seeds=seeds, check_convergence=False, layout=layout, **regs)
    assert len(batch) == R
    for r in range(R):
        reg = {k: float(v[r]) for k, v in regs.items()}
        single = cmf.fit_cnmf(X, L=L, K=K, alg="mult", max_itr=itr, seed=seeds[r], check_convergence=False, layout=layout, **reg)
        b = batch[r]
        assert len(b.loss_hist) == len(single.loss_hist) == itr + 1
        assert _rel(b.loss_hist, single.loss_hist) < 1e-9
        _close(b.W, single.W, 1e-8, 1e-11)
        _close(b.H, single.H, 1e-8, 1e-11)
        # the C oracle from the same (rescaled) initialisation
        init = cmf.fit_cnmf(X, L=L, K=K, max_itr=0, seed=seeds[r], check_convergence=False, layout="KNL")
        ref = co.fit(co.MultUpdate, X, init.W, init.H, itr, check_convergence=False, **reg)
        assert _rel(b.loss_hist, ref.loss_hist) < 1e-9
        Wk = b.W if layout == "KNL" else b.W.transpose(2, 1, 0)
        _close(Wk, ref.W, 1e-8, 1e-11)
        _close(b.H, ref.H, 1e-8, 1e-11)
        assert b.engine_info["engine"] == 0


def test_explicit_stacks_and_eval_mode(cmf):
    N, T, K, L, R, itr = 96, 500, 4, 8, 3, 12
    X = _data(N, T, L, seed=3)
    rng = np.random.default_rng(5)
    Wst, Hst = rng.random((R, K, N, L)), rng.random((R, K, T))
    for eval_mode in (False, True):
        batch = cmf.fit_cnmf_batch(X, L=L, K=K, max_itr=itr, W_init=Wst, H_init=Hst, eval_mode=eval_mode,
                                   check_convergence=False, layout="KNL", **REG)
        for r in range(R):
            single = cmf.fit_cnmf(X, L=L, K=K, max_itr=itr, W_init=Wst[r], H_init=Hst[r], eval_mode=eval_mode,
                                  check_convergence=False, layout="KNL", **REG)
            assert _rel(batch[r].loss_hist, single.loss_hist) < 1e-9
            _close(batch[r].W, single.W, 1e-8, 1e-11)
            _close(batch[r].H, single.H, 1e-8, 1e-11)
            if eval_mode:
                assert np.array_equal(batch[r].W, Wst[r])     # the W update is skipped


def _stop(hist, patience, tol):
    """Length of the history at which converged() first holds (None: never)."""
    for n in range(patience + 1, len(hist) + 1):
        if np.all(np.abs(np.diff(hist[n - patience - 1:n])) < tol):
            return n
    return None


def test_per_restart_early_stop_freezes_converged_restarts(cmf):
    N, T, K, L, R, itr, patience = 120, 600, 5, 10, 6, 80, 3
    X = _data(N, T, L, seed=9)
    seeds = list(range(40, 40 + R))
    regs = _regs(R)
    free = cmf.fit_cnmf_batch(X, L=L, K=K, max_itr=itr, seeds=seeds, check_convergence=False, **regs)
    hists = [np.asarray(f.loss_hist) for f in free]
    deltas = np.concatenate([np.abs(np.diff(h)) for h in hists])
    tol = None
    for cand in np.geomspace(1e-2, 1e-7, 400):
        stops = [_stop(h, patience, cand) for h in hists]
        borderline = np.any(np.abs(deltas - cand) <= 1e-8 * cand)
        if not borderline and all(s is not None for s in stops) and len(set(stops)) >= 2:
            tol = cand
            break
    assert tol is not None, "no tolerance separates the restarts' stopping iterations"
    assert not np.any(np.abs(deltas - tol) <= 1e-8 * tol)
    batch = cmf.fit_cnmf_batch(X, L=L, K=K, max_itr=itr, seeds=seeds, check_convergence=True, patience=patience, tol=tol,
                               printer=lambda s: None, **regs)
    lens = set()
    for r in range(R):
        reg = {k: float(v[r]) for k, v in regs.items()}
        single = cmf.fit_cnmf(X, L=L, K=K, max_itr=itr, seed=seeds[r], check_convergence=True, patience=patience, tol=tol,
                              printer=lambda s: None, **reg)
        assert len(batch[r].loss_hist) == len(single.loss_hist) < itr + 1
        assert _rel(batch[r].loss_hist, single.loss_hist) < 1e-9
        _close(batch[r].W, single.W, 1e-8, 1e-11)      # frozen at its own stop while the others went on
        _close(batch[r].H, single.H, 1e-8, 1e-11)
        assert batch[r].time_hist == batch[0].time_hist[: len(batch[r].time_hist)]
        lens.add(len(single.loss_hist))
    assert len(lens) >= 2


def test_fp32_against_fp64_oracle(cmf):
    from oracle import c_oracle as co

    N, T, K, L, R, itr = 256, 4096, 8, 10, 3, 6
    X = _data(N, T, L, seed=1234, K_true=4)
    seeds = [0, 1, 2]
    batch = cmf.fit_cnmf_batch(X, L=L, K=K, max_itr=itr, seeds=seeds, dtype="f32", check_convergence=False, layout="KNL", **REG)
    for r in range(R):
        init = cmf.fit_cnmf(X, L=L, K=K, max_itr=0, seed=seeds[r], check_convergence=False, layout="KNL")
        ref = co.fit(co.MultUpdate, X, init.W, init.H, itr, check_convergence=False, **REG)
        assert len(batch[r].loss_hist) == itr + 1
        assert np.max(np.abs(np.asarray(batch[r].loss_hist) - np.asarray(ref.loss_hist))) < 1e-4


def _handle(cmf, N, T, K, L, R, dtype=0, alg=0):
    lib = cmf._lib.load()
    h = ctypes.c_void_p()
    cmf._lib.check(lib.cmf_create_batch(ctypes.byref(h), N, T, K, L, dtype, alg, R, 0))
    return lib, h


def _fit_raw(cmf, lib, h, R, itr, cap):
    z = np.zeros(R)
    p = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))  # noqa: E731
    lh, th = np.zeros(R * cap), np.zeros(cap)
    n, e = np.zeros(R, dtype=np.int64), np.zeros(R, dtype=np.int32)
    cmf._lib.check(lib.cmf_fit_batch(h, itr, float("inf"), 0, 0, 3, 1e-4, p(z), p(z), p(z), p(z), p(lh), p(th), cap,
                                     n.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), e.ctypes.data_as(ctypes.POINTER(ctypes.c_int))))
    return lh, n


def test_launches_do_not_grow_with_R(cmf):
    N, T, K, L, itr = 120, 600, 5, 10, 5
    X = np.asfortranarray(_data(N, T, L))
    per = {}
    for R in (2, 64):
        lib, h = _handle(cmf, N, T, K, L, R)
        try:
            rng = np.random.default_rng(R)
            W = np.asfortranarray(rng.random((K, N, L, R)))
            H = np.asfortranarray(rng.random((K, T, R)))
            cmf._lib.check(lib.cmf_set_data(h, cmf._lib.fptr(X), 0))
            cmf._lib.check(lib.cmf_set_factors_batch(h, cmf._lib.fptr(W), cmf._lib.fptr(H)))
            a, b = ctypes.c_int64(), ctypes.c_int64()
            cmf._lib.check(lib.cmf_launch_count(h, ctypes.byref(a)))
            _fit_raw(cmf, lib, h, R, itr, itr + 1)
            cmf._lib.check(lib.cmf_launch_count(h, ctypes.byref(b)))
            per[R] = b.value - a.value
        finally:
            lib.cmf_destroy(h)
    assert per[2] == per[64], per


@pytest.mark.parametrize("N,T,K,L", [(120, 600, 1, 10), (120, 600, 5, 1), (121, 15, 3, 10), (77, 300, 4, 6)])
def test_edges_against_single_fits(cmf, N, T, K, L):
    X = _data(N, T, L, seed=21, K_true=2)
    seeds = [3, 4, 5]
    batch = cmf.fit_cnmf_batch(X, L=L, K=K, max_itr=10, seeds=seeds, check_convergence=False, layout="KNL", **REG)
    for r, seed in enumerate(seeds):
        single = cmf.fit_cnmf(X, L=L, K=K, max_itr=10, seed=seed, check_convergence=False, layout="KNL", **REG)
        assert _rel(batch[r].loss_hist, single.loss_hist) < 1e-9
        _close(batch[r].W, single.W, 1e-8, 1e-11)
        _close(batch[r].H, single.H, 1e-8, 1e-11)


def test_single_restart_equals_fit_cnmf(cmf):
    N, T, K, L = 120, 600, 5, 10
    X = _data(N, T, L)
    (b,) = cmf.fit_cnmf_batch(X, L=L, K=K, max_itr=20, seeds=[99], check_convergence=False, layout="KNL", **REG)
    s = cmf.fit_cnmf(X, L=L, K=K, max_itr=20, seed=99, check_convergence=False, layout="KNL", **REG)
    assert _rel(b.loss_hist, s.loss_hist) < 1e-12
    _close(b.W, s.W, 1e-12, 0)
    _close(b.H, s.H, 1e-12, 0)


def test_errors(cmf):
    lib = cmf._lib.load()
    h = ctypes.c_void_p()
    # footprint beyond the device: refused before anything is allocated, with the bytes named
    assert lib.cmf_create_batch(ctypes.byref(h), 500, 1_000_000, 5, 10, 0, 0, 4096, 0) == 1   # ~0.5 TB
    msg = lib.cmf_last_error().decode()
    assert "bytes" in msg and "4096 restarts need" in msg, msg
    # HALS / PGD are not batched
    assert lib.cmf_create_batch(ctypes.byref(h), 64, 200, 3, 5, 0, 1, 4, 0) == 3
    assert lib.cmf_create_batch(ctypes.byref(h), 64, 200, 3, 5, 0, 2, 4, 0) == 3
    lib, h = _handle(cmf, 64, 200, 3, 5, 4)
    try:
        buf = np.zeros(64 * 200)
        assert lib.cmf_set_factors(h, cmf._lib.fptr(buf), cmf._lib.fptr(buf), 0) == 1
        assert b"cmf_set_factors_batch" in lib.cmf_last_error()
        assert lib.cmf_get_factors(h, cmf._lib.fptr(buf), cmf._lib.fptr(buf)) == 1
        assert b"cmf_get_factors_batch" in lib.cmf_last_error()
        out = ctypes.c_double()
        assert lib.cmf_loss(h, ctypes.byref(out)) == 1
        assert b"cmf_loss_batch" in lib.cmf_last_error()
        assert lib.cmf_update_motifs(h, 0.0, 0.0) == 1
        assert lib.cmf_init_rand(h, 1) == 1
        assert lib.cmf_scale_factors(h, 1.0) == 1
        assert lib.cmf_w_partials(h) == 3
        assert lib.cmf_set_engine(h, 1) == 3
        assert lib.cmf_set_engine(h, 2) == 3
        assert lib.cmf_set_engine(h, 0) == 0
    finally:
        lib.cmf_destroy(h)
