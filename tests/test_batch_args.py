"""Argument checks of the batched-restart path that run without a device: cmf_create_batch validates before it looks for
a GPU, and fit_cnmf_batch validates the stacks and per-restart regularisers before it loads the library."""
import ctypes

import numpy as np
import pytest


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge

    ge.build()
    from cmf_jl_b200 import _lib

    return _lib


def test_create_batch_argument_validation(lib):
    L = lib.load()
    h = ctypes.c_void_p()
    assert L.cmf_create_batch(ctypes.byref(h), 8, 100, 2, 5, 0, 0, 0, 0) == 1     # R < 1
    assert b"restarts" in L.cmf_last_error()
    assert L.cmf_create_batch(ctypes.byref(h), 8, 100, 2, 5, 0, 7, 4, 0) == 1     # bad alg
    assert L.cmf_create_batch(ctypes.byref(h), 8, 100, 2, 5, 0, 1, 4, 0) == 3     # HALS is not batched
    assert L.cmf_create_batch(ctypes.byref(h), 8, 100, 2, 5, 0, 2, 4, 0) == 3     # nor PGD
    assert L.cmf_create_batch(ctypes.byref(h), 8, 3, 2, 5, 0, 0, 4, 0) == 1       # L > T
    assert L.cmf_create_batch(ctypes.byref(h), 8, 100, 2, 5, 7, 0, 4, 0) == 1     # bad dtype
    assert L.cmf_fit_batch(None, 1, 1.0, 0, 0, 3, 1e-4, None, None, None, None, None, None, 2, None, None) == 1
    assert L.cmf_set_factors_batch(None, None, None) == 1


def test_fit_cnmf_batch_rejects_bad_stacks_before_loading(monkeypatch):
    import cmf_jl_b200 as cmf
    from cmf_jl_b200 import _lib

    def boom():
        raise AssertionError("the library must not be loaded")

    monkeypatch.setattr(_lib, "load", boom)
    X = np.ones((6, 40))
    K, N, L, T = 2, 6, 3, 40
    rng = np.random.default_rng(0)
    W, H = rng.random((3, K, N, L)), rng.random((3, K, T))
    with pytest.raises(ValueError):                                   # R differs between the stacks
        cmf.fit_cnmf_batch(X, L=L, K=K, W_init=W, H_init=H[:2])
    with pytest.raises(ValueError):                                   # wrong block shape
        cmf.fit_cnmf_batch(X, L=L, K=K, W_init=W[:, :, :, :2], H_init=H)
    with pytest.raises(ValueError):                                   # only one stack
        cmf.fit_cnmf_batch(X, L=L, K=K, W_init=W)
    with pytest.raises(ValueError):                                   # seeds and stacks
        cmf.fit_cnmf_batch(X, L=L, K=K, seeds=[1, 2, 3], W_init=W, H_init=H)
    with pytest.raises(ValueError):                                   # neither
        cmf.fit_cnmf_batch(X, L=L, K=K)
    with pytest.raises(ValueError):                                   # regulariser length != R
        cmf.fit_cnmf_batch(X, L=L, K=K, seeds=[1, 2, 3], l1W=[0.1, 0.2])
    with pytest.raises(ValueError):                                   # README spelling goes through the same check
        cmf.fit_cnmf_batch(X, L=L, K=K, seeds=[1, 2, 3], l2_H=np.zeros(4))
    with pytest.raises(ValueError):
        cmf.fit_cnmf_batch(X, L=L, K=K, seeds=[])
