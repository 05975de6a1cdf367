"""Rank sweeps in one batch (cmf_create_batch_ranks / fit_cnmf_batch with a sequence K): restart r has its own rank K[r].

Restart r must equal fit_cnmf with K = K[r], seed seeds[r] and its own regularisers, and the C oracle from the same
initialisation.  All ranks share one stacked component axis of width sum K[r]; with every K[r] equal, the handle is the
one cmf_create_batch makes and its results are the same bytes."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

REG = dict(l1W=0.1, l2W=0.5, l1H=0.1, l2H=0.2)
MIX = [1, 2, 3, 5, 8, 3]       # repeats and K = 1 included


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
    out = {k: np.zeros(R) for k in REG}
    for r in range(R):
        if r % 3 == 1:
            for k, v in REG.items():
                out[k][r] = v
        elif r % 3 == 2:
            out["l1W"][r], out["l2H"][r] = 0.05, 0.3
    return out


def _reg(regs, r):
    return {k: float(v[r]) for k, v in regs.items()}


def _rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b) / np.abs(b)))


def _close(a, b, rtol, atol):
    np.testing.assert_allclose(np.asarray(a), np.asarray(b), rtol=rtol, atol=atol)


def test_fp64_parity_with_single_fits_and_oracle(cmf):
    from oracle import c_oracle as co

    N, T, L, itr = 120, 600, 10, 30
    X = _data(N, T, L)
    R = len(MIX)
    seeds = list(range(21, 21 + R))
    regs = _regs(R)
    batch = cmf.fit_cnmf_batch(X, L=L, K=MIX, max_itr=itr, seeds=seeds, check_convergence=False, layout="KNL", **regs)
    assert len(batch) == R
    for r, k in enumerate(MIX):
        b = batch[r]
        assert b.W.shape == (k, N, L) and b.H.shape == (k, T)
        assert b.engine_info["restarts"] == R
        single = cmf.fit_cnmf(X, L=L, K=k, max_itr=itr, seed=seeds[r], check_convergence=False, layout="KNL", **_reg(regs, r))
        assert len(b.loss_hist) == len(single.loss_hist) == itr + 1
        assert _rel(b.loss_hist, single.loss_hist) < 1e-9
        _close(b.W, single.W, 1e-8, 1e-11)
        _close(b.H, single.H, 1e-8, 1e-11)
        init = cmf.fit_cnmf(X, L=L, K=k, max_itr=0, seed=seeds[r], check_convergence=False, layout="KNL")
        ref = co.fit(co.MultUpdate, X, init.W, init.H, itr, check_convergence=False, **_reg(regs, r))
        assert _rel(b.loss_hist, ref.loss_hist) < 1e-9
        _close(b.W, ref.W, 1e-8, 1e-11)
        _close(b.H, ref.H, 1e-8, 1e-11)


def test_lnk_layout_and_explicit_ragged_stacks(cmf):
    N, T, L, itr = 96, 500, 8, 12
    X = _data(N, T, L, seed=3)
    ks = [4, 1, 6]
    rng = np.random.default_rng(5)
    Ws, Hs = [rng.random((k, N, L)) for k in ks], [rng.random((k, T)) for k in ks]
    batch = cmf.fit_cnmf_batch(X, L=L, K=ks, max_itr=itr, W_init=Ws, H_init=Hs, check_convergence=False, **REG)
    for r, k in enumerate(ks):
        single = cmf.fit_cnmf(X, L=L, K=k, max_itr=itr, W_init=Ws[r], H_init=Hs[r], check_convergence=False, **REG)
        assert batch[r].W.shape == (L, N, k)
        assert _rel(batch[r].loss_hist, single.loss_hist) < 1e-9
        _close(batch[r].W, single.W, 1e-8, 1e-11)
        _close(batch[r].H, single.H, 1e-8, 1e-11)


def test_fp32_tracks_fp64(cmf):
    N, T, L, itr = 120, 600, 10, 100
    X = _data(N, T, L)
    R = len(MIX)
    seeds = list(range(31, 31 + R))
    regs = _regs(R)
    f32 = cmf.fit_cnmf_batch(X, L=L, K=MIX, max_itr=itr, seeds=seeds, dtype="f32", check_convergence=False, layout="KNL", **regs)
    for r, k in enumerate(MIX):
        ref = cmf.fit_cnmf(X, L=L, K=k, max_itr=itr, seed=seeds[r], check_convergence=False, layout="KNL", **_reg(regs, r))
        assert len(f32[r].loss_hist) == itr + 1
        assert np.max(np.abs(np.asarray(f32[r].loss_hist) - np.asarray(ref.loss_hist))) < 1e-4


def test_config1_rank_sweep_matches_single_fits(cmf):
    N, T, L, itr = 500, 2000, 10, 100
    X = _data(N, T, L, seed=11, K_true=4)
    ks = [k for k in range(1, 11) for _ in range(2)]               # R = 20, C = 110
    seeds = list(range(100, 100 + len(ks)))
    batch = cmf.fit_cnmf_batch(X, L=L, K=ks, max_itr=itr, seeds=seeds, check_convergence=False, layout="KNL")
    for r, k in enumerate(ks):
        single = cmf.fit_cnmf(X, L=L, K=k, max_itr=itr, seed=seeds[r], check_convergence=False, layout="KNL")
        assert _rel(batch[r].loss_hist, single.loss_hist) < 1e-9, (r, k)


@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_equal_ranks_are_the_uniform_batch(cmf, dtype):
    N, T, L, K, R, itr = 120, 600, 10, 5, 6, 25
    X = _data(N, T, L)
    seeds = list(range(50, 50 + R))
    regs = _regs(R)
    kw = dict(L=L, max_itr=itr, seeds=seeds, dtype=dtype, check_convergence=False, layout="KNL", **regs)
    ragged = cmf.fit_cnmf_batch(X, K=[K] * R, **kw)
    uniform = cmf.fit_cnmf_batch(X, K=K, **kw)
    for a, b in zip(ragged, uniform):
        assert a.W.tobytes() == b.W.tobytes()
        assert a.H.tobytes() == b.H.tobytes()
        assert np.asarray(a.loss_hist).tobytes() == np.asarray(b.loss_hist).tobytes()


def _stop(hist, patience, tol):
    for n in range(patience + 1, len(hist) + 1):
        if np.all(np.abs(np.diff(hist[n - patience - 1:n])) < tol):
            return n
    return None


def test_early_stop_freezes_each_rank_at_its_own_iteration(cmf):
    N, T, L, itr, patience = 120, 600, 10, 80, 3
    X = _data(N, T, L, seed=9)
    R = len(MIX)
    seeds = list(range(60, 60 + R))
    regs = _regs(R)
    free = cmf.fit_cnmf_batch(X, L=L, K=MIX, max_itr=itr, seeds=seeds, check_convergence=False, **regs)
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
    batch = cmf.fit_cnmf_batch(X, L=L, K=MIX, max_itr=itr, seeds=seeds, check_convergence=True, patience=patience, tol=tol,
                               printer=lambda s: None, **regs)
    lens = set()
    for r, k in enumerate(MIX):
        single = cmf.fit_cnmf(X, L=L, K=k, max_itr=itr, seed=seeds[r], check_convergence=True, patience=patience, tol=tol,
                              printer=lambda s: None, **_reg(regs, r))
        assert len(batch[r].loss_hist) == len(single.loss_hist) < itr + 1
        assert _rel(batch[r].loss_hist, single.loss_hist) < 1e-9
        _close(batch[r].W, single.W, 1e-8, 1e-11)      # frozen at its own stop while the others went on
        _close(batch[r].H, single.H, 1e-8, 1e-11)
        lens.add(len(single.loss_hist))
    assert len(lens) >= 2


def _launches_per_fit(cmf, X, L, ks, itr, uniform=False):
    from cmf_jl_b200._lib import check, fptr

    lib = cmf._lib.load()
    N, T = X.shape
    R, C = len(ks), sum(ks)
    h = ctypes.c_void_p()
    if uniform:
        check(lib.cmf_create_batch(ctypes.byref(h), N, T, ks[0], L, 0, 0, R, 0))
    else:
        rk = (ctypes.c_int64 * R)(*ks)
        check(lib.cmf_create_batch_ranks(ctypes.byref(h), N, T, rk, L, 0, 0, R, 0))
    try:
        rng = np.random.default_rng(R)
        W, H = rng.random(C * N * L), rng.random(C * T)
        check(lib.cmf_set_data(h, fptr(np.asfortranarray(X)), 0))
        check(lib.cmf_set_factors_batch(h, fptr(W), fptr(H)))
        z = np.zeros(R)
        p = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))  # noqa: E731
        cap = itr + 1
        lh, th = np.zeros(R * cap), np.zeros(cap)
        n, e = np.zeros(R, dtype=np.int64), np.zeros(R, dtype=np.int32)
        a, b = ctypes.c_int64(), ctypes.c_int64()
        check(lib.cmf_launch_count(h, ctypes.byref(a)))
        check(lib.cmf_fit_batch(h, itr, float("inf"), 0, 0, 3, 1e-4, p(z), p(z), p(z), p(z), p(lh), p(th), cap,
                                n.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), e.ctypes.data_as(ctypes.POINTER(ctypes.c_int))))
        check(lib.cmf_launch_count(h, ctypes.byref(b)))
        assert np.all(np.isfinite(lh)) and np.all(n == cap)
        return b.value - a.value
    finally:
        lib.cmf_destroy(h)


def test_launches_depend_neither_on_R_nor_on_the_ranks(cmf):
    """A ragged batch launches what a uniform batch of the same R launches, whatever its ranks.  Where the stacked numH
    leaves the device short of CTAs (config-1 shape, small R) its transposed convolution splits over units and adds one
    reduction launch, in the uniform batch as well; at T = 50 000 it never splits, and R = 4 and R = 64 launch the same."""
    N, L, itr = 500, 10, 5
    X = _data(N, 2000, L, seed=2)
    for R, mixes in ((4, ([1, 7, 3, 10], [2, 9, 4, 5])), (64, ([1 + r % 10 for r in range(64)], [10 - r % 3 for r in range(64)]))):
        per = {"uniform": _launches_per_fit(cmf, X, L, [5] * R, itr, uniform=True)}
        per.update({str(m[:4]): _launches_per_fit(cmf, X, L, m, itr) for m in mixes})
        assert len(set(per.values())) == 1, (R, per)
    X = _data(N, 50_000, L, seed=2)
    per = {
        "R=4": _launches_per_fit(cmf, X, L, [1, 7, 3, 10], 3),
        "R=64": _launches_per_fit(cmf, X, L, [1 + r % 10 for r in range(64)], 3),
        "R=64 uniform": _launches_per_fit(cmf, X, L, [5] * 64, 3, uniform=True),
    }
    assert len(set(per.values())) == 1, per


def test_footprint_refusal_names_the_bytes(cmf):
    lib = cmf._lib.load()
    h = ctypes.c_void_p()
    ks = [5 + r % 20 for r in range(2048)]
    rk = (ctypes.c_int64 * len(ks))(*ks)
    assert lib.cmf_create_batch_ranks(ctypes.byref(h), 500, 1_000_000, rk, 10, 0, 0, len(ks), 0) == 1   # ~0.6 TB
    msg = lib.cmf_last_error().decode()
    assert "bytes" in msg and "2048 restarts need" in msg and f"{sum(ks)} stacked components" in msg, msg
