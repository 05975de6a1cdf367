"""Checks of the sparse-data path that run without a device: cmf_create_sparse / cmf_create_batch_sparse validate before
they look for a GPU, the Python helper canonicalises any scipy.sparse input to CSC, and fit_cnmf / fit_cnmf_batch refuse
bad sparse calls before they load the library."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge

    ge.build()
    from cmf_jl_b200 import _lib

    return _lib


@pytest.fixture
def no_load(monkeypatch):
    from cmf_jl_b200 import _lib

    def boom():
        raise AssertionError("the library must not be loaded")

    monkeypatch.setattr(_lib, "load", boom)


def _ranks(*k):
    a = np.asarray(k, dtype=np.int64)
    return a, a.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))


def test_create_sparse_argument_validation(lib):
    L = lib.load()
    h = ctypes.c_void_p()
    assert L.cmf_create_sparse(ctypes.byref(h), 8, 100, 2, 5, 7, 0, 0) == 1            # bad dtype
    assert L.cmf_create_sparse(ctypes.byref(h), 8, 3, 2, 5, 0, 0, 0) == 1              # L > T
    assert b"L <= T" in L.cmf_last_error()
    assert L.cmf_create_sparse(ctypes.byref(h), 2**31, 100, 2, 5, 0, 0, 0) == 1        # N > INT32_MAX
    assert b"INT32_MAX" in L.cmf_last_error()
    assert L.cmf_create_sparse(ctypes.byref(h), 8, 100, 2, 5, 0, 2, 0) == 3            # PGD
    assert L.cmf_create_sparse(ctypes.byref(h), 8, 100, 2, 5, 0, 9, 0) == 1            # bad alg
    assert L.cmf_create_sparse(None, 8, 100, 2, 5, 0, 0, 0) == 1


def test_create_batch_sparse_argument_validation(lib):
    L = lib.load()
    h = ctypes.c_void_p()
    k, kp = _ranks(2, 3, 0)
    assert L.cmf_create_batch_sparse(ctypes.byref(h), 8, 100, kp, 5, 0, 0, 3, 0) == 1   # a rank < 1
    assert b"K[2]" in L.cmf_last_error()
    assert L.cmf_create_batch_sparse(ctypes.byref(h), 8, 100, None, 5, 0, 0, 3, 0) == 1  # null rank array
    k, kp = _ranks(2, 3)
    assert L.cmf_create_batch_sparse(ctypes.byref(h), 8, 100, kp, 5, 0, 0, 0, 0) == 1    # R < 1
    assert L.cmf_create_batch_sparse(ctypes.byref(h), 8, 100, kp, 5, 7, 0, 2, 0) == 1    # bad dtype
    assert L.cmf_create_batch_sparse(ctypes.byref(h), 8, 3, kp, 5, 0, 0, 2, 0) == 1      # L > T
    assert L.cmf_create_batch_sparse(ctypes.byref(h), 2**31, 100, kp, 5, 0, 0, 2, 0) == 1  # N > INT32_MAX
    assert L.cmf_create_batch_sparse(ctypes.byref(h), 8, 100, kp, 5, 0, 2, 2, 0) == 3    # PGD
    assert L.cmf_create_batch_sparse(ctypes.byref(h), 8, 100, kp, 5, 0, 1, 2, 0) == 3    # HALS is not batched
    assert L.cmf_set_data_csc(None, 1, None, None, None, 0) == 1


def test_as_csc_canonicalises_coo_and_csr():
    from cmf_jl_b200 import as_csc

    # COO with a duplicate (1, 2) summed to 5, an entry whose duplicates cancel (0, 0), an explicit zero (3, 1),
    # unsorted entries
    rows = np.array([3, 1, 0, 2, 1, 0, 3])
    cols = np.array([4, 2, 0, 4, 2, 0, 1])
    vals = np.array([1.5, 2.0, 1.0, -4.0, 3.0, -1.0, 0.0])
    coo = sp.coo_matrix((vals, (rows, cols)), shape=(4, 6))
    dense = np.zeros((4, 6))
    np.add.at(dense, (rows, cols), vals)
    want_colptr = np.array([0, 0, 0, 1, 1, 3, 3])
    want_rowval = np.array([1, 2, 3])
    want_nzval = np.array([5.0, -4.0, 1.5])
    for X in (coo, coo.tocsr(), sp.csr_array(coo), sp.csc_matrix(coo)):
        for dtype, npdt in (("f64", np.float64), ("f32", np.float32)):
            c = as_csc(X, dtype)
            assert c.shape == (4, 6) and c.nnz == 3
            assert c.colptr.dtype == np.int64 and c.rowval.dtype == np.int64 and c.nzval.dtype == npdt
            assert np.array_equal(c.colptr, want_colptr) and np.array_equal(c.rowval, want_rowval)
            assert np.array_equal(c.nzval, want_nzval.astype(npdt))
            back = sp.csc_matrix((c.nzval, c.rowval, c.colptr), shape=c.shape).toarray()
            assert np.array_equal(back, dense.astype(npdt))
    # a CSR matrix with unsorted column indices inside a row and a duplicate
    csr = sp.csr_matrix((np.array([1.0, 2.0, 3.0]), np.array([3, 0, 3]), np.array([0, 3, 3])), shape=(2, 5))
    c = as_csc(csr)
    assert np.array_equal(c.colptr, [0, 1, 1, 1, 2, 2]) and np.array_equal(c.rowval, [0, 0])
    assert np.array_equal(c.nzval, [2.0, 4.0])
    assert as_csc(np.ones((2, 3))) is None


def test_fit_cnmf_sparse_rejects_bad_calls_before_loading(no_load):
    import cmf_jl_b200 as cmf

    N, T, K, L = 6, 40, 2, 3
    X = sp.random(N, T, density=0.2, random_state=0, format="csc")
    rng = np.random.default_rng(0)
    W, H = rng.random((K, N, L)), rng.random((K, T))
    with pytest.raises(ValueError):                                          # wrong W_init shape
        cmf.fit_cnmf(X, L=L, K=K, W_init=W[:, :, :2], H_init=H)
    with pytest.raises(ValueError):                                          # wrong H_init shape, only H given
        cmf.fit_cnmf(X, L=L, K=K, H_init=H[:, :-1])
    with pytest.raises(cmf.CMFError) as ei:
        cmf.fit_cnmf(X, L=L, K=K, alg="pgd", W_init=W, H_init=H)
    assert ei.value.code == 3
    with pytest.raises(cmf.CMFError) as ei:
        cmf.fit_cnmf(X, L=L, K=K, ngpu=2, W_init=W, H_init=H)
    assert ei.value.code == 3
    with pytest.raises(cmf.CMFError) as ei:
        cmf.MultUpdate(X, W, H, ngpu=2)
    assert ei.value.code == 3
    with pytest.raises(cmf.CMFError) as ei:
        cmf.PGDUpdate(X, W, H)
    assert ei.value.code == 3
    with pytest.raises(ValueError):                                          # shape mismatch in the rule constructor
        cmf.MultUpdate(X, W[:, :5], H)


def test_fit_cnmf_batch_sparse_rejects_bad_calls_before_loading(no_load):
    import cmf_jl_b200 as cmf

    N, T, K, L = 6, 40, 2, 3
    X = sp.random(N, T, density=0.2, random_state=0, format="coo")
    rng = np.random.default_rng(0)
    W, H = rng.random((3, K, N, L)), rng.random((3, K, T))
    with pytest.raises(ValueError):                                          # wrong block shape
        cmf.fit_cnmf_batch(X, L=L, K=K, W_init=W[:, :, :, :2], H_init=H)
    with pytest.raises(ValueError):                                          # ragged: wrong W_init[1]
        cmf.fit_cnmf_batch(X, L=L, K=[1, 2], W_init=[W[0, :1], W[0, :1]], H_init=[H[0, :1], H[0]])
    with pytest.raises(cmf.CMFError) as ei:
        cmf.fit_cnmf_batch(X, L=L, K=K, alg="pgd", seeds=[1, 2])
    assert ei.value.code == 3
    with pytest.raises(cmf.CMFError) as ei:
        cmf.fit_cnmf_batch(X, L=L, K=K, seeds=[1, 2], ngpu=2)
    assert ei.value.code == 3
