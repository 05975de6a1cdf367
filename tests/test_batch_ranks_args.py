"""Argument checks of rank sweeps in one batch that run without a device: cmf_create_batch_ranks validates before it looks
for a GPU, and fit_cnmf_batch with a sequence of ranks validates the ranks, seeds and ragged stacks before it loads the
library."""
import ctypes

import numpy as np
import pytest


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge

    ge.build()
    from cmf_jl_b200 import _lib

    return _lib


def _ranks(*k):
    return (ctypes.c_int64 * len(k))(*k)


def test_create_batch_ranks_argument_validation(lib):
    L = lib.load()
    h = ctypes.c_void_p()
    K = _ranks(1, 3, 2)
    cases = [
        ((ctypes.byref(h), 8, 100, None, 5, 0, 0, 3, 0), 1, b"null rank array"),
        ((ctypes.byref(h), 8, 100, K, 5, 0, 0, 0, 0), 1, b"restarts"),                      # R < 1
        ((ctypes.byref(h), 8, 100, _ranks(2, 0, 3), 5, 0, 0, 3, 0), 1, b"K[1] = 0"),        # a rank < 1
        ((ctypes.byref(h), 8, 100, _ranks(2, 3, -4), 5, 0, 0, 3, 0), 1, b"K[2] = -4"),
        ((ctypes.byref(h), 8, 3, K, 5, 0, 0, 3, 0), 1, b"L <= T"),                          # L > T
        ((ctypes.byref(h), 8, 1000, K, 770, 0, 0, 3, 0), 3, b"L <= 769"),
        ((ctypes.byref(h), 8, 100, K, 5, 7, 0, 3, 0), 1, b"dtype"),                        # bad dtype
        ((ctypes.byref(h), 8, 100, K, 5, 0, 7, 3, 0), 1, b"alg"),                          # bad alg
        ((ctypes.byref(h), 8, 100, K, 5, 0, 1, 3, 0), 3, b"MultUpdate only"),              # HALS is not batched
        ((ctypes.byref(h), 8, 100, K, 5, 0, 2, 3, 0), 3, b"MultUpdate only"),              # nor PGD
        ((None, 8, 100, K, 5, 0, 0, 3, 0), 1, b"null output"),
    ]
    for args, code, msg in cases:
        assert L.cmf_create_batch_ranks(*args) == code, (args, L.cmf_last_error())
        assert msg in L.cmf_last_error(), (msg, L.cmf_last_error())
    # the ranks of all restarts together must fit one launch grid
    assert L.cmf_create_batch_ranks(ctypes.byref(h), 8, 100, _ranks(200_000, 200_000), 5, 0, 0, 2, 0) == 1
    assert b"R*K too large" in L.cmf_last_error()


def test_fit_cnmf_batch_rejects_bad_ranks_before_loading(monkeypatch):
    import cmf_jl_b200 as cmf
    from cmf_jl_b200 import _lib

    def boom():
        raise AssertionError("the library must not be loaded")

    monkeypatch.setattr(_lib, "load", boom)
    N, T, L = 6, 40, 3
    X = np.ones((N, T))
    ks = [1, 3, 2]
    rng = np.random.default_rng(0)
    W = [rng.random((k, N, L)) for k in ks]
    H = [rng.random((k, T)) for k in ks]
    with pytest.raises(ValueError):                                   # len(K) != R (seeds)
        cmf.fit_cnmf_batch(X, L=L, K=ks, seeds=[1, 2])
    with pytest.raises(ValueError):                                   # len(K) != R (stacks)
        cmf.fit_cnmf_batch(X, L=L, K=ks[:2], W_init=W, H_init=H)
    with pytest.raises(ValueError):                                   # a rank < 1
        cmf.fit_cnmf_batch(X, L=L, K=[2, 0, 1], seeds=[1, 2, 3])
    with pytest.raises(ValueError):                                   # a rank that is not an integer
        cmf.fit_cnmf_batch(X, L=L, K=[2, 1.5, 1], seeds=[1, 2, 3])
    with pytest.raises(ValueError):                                   # no ranks at all
        cmf.fit_cnmf_batch(X, L=L, K=[], seeds=[])
    with pytest.raises(ValueError):                                   # W_init[1] has another restart's rank
        cmf.fit_cnmf_batch(X, L=L, K=ks, W_init=[W[0], W[2], W[1]], H_init=H)
    with pytest.raises(ValueError):                                   # H_init[2] has the wrong length
        cmf.fit_cnmf_batch(X, L=L, K=ks, W_init=W, H_init=H[:2] + [rng.random((2, T - 1))])
    with pytest.raises(ValueError):                                   # W_init with the wrong L
        cmf.fit_cnmf_batch(X, L=L, K=ks, W_init=[w[:, :, :2] for w in W], H_init=H)
    with pytest.raises(ValueError):                                   # one array short
        cmf.fit_cnmf_batch(X, L=L, K=ks, W_init=W[:2], H_init=H)
    with pytest.raises(ValueError):                                   # only one stack
        cmf.fit_cnmf_batch(X, L=L, K=ks, W_init=W)
    with pytest.raises(ValueError):                                   # seeds and stacks
        cmf.fit_cnmf_batch(X, L=L, K=ks, seeds=[1, 2, 3], W_init=W, H_init=H)
    with pytest.raises(ValueError):                                   # regulariser length != R
        cmf.fit_cnmf_batch(X, L=L, K=ks, seeds=[1, 2, 3], l1W=[0.1, 0.2])
