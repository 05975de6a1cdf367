"""oracle/lagged_ref.py (the chunked float64 contractions the long-T GPU tests compare with) against the literal oracles:
cnmf_oracle (NumPy, one product per lag), c_oracle (plain C loops) and restructured.gram_R, to 1e-12 of the output scale.
Shapes include L = 1, T < 2L, T < L (lags past the end of H), ragged N, K and T, and T longer than one stacked chunk."""
import numpy as np
import pytest

from oracle import c_oracle as co
from oracle import cnmf_oracle as po
from oracle import lagged_ref as lr
from oracle import restructured as rs

# (N, T, K, L)
DIMS = [(7, 50, 3, 1), (13, 29, 5, 20), (9, 12, 4, 20), (33, 301, 7, 9), (64, 1000, 1, 33), (5, 3, 2, 4),
        (17, 4099, 3, 100), (20, 2000, 128, 32)]


def _rand(N, T, K, L, seed):
    rng = np.random.default_rng(seed)
    return rng.random((K, N, L)), rng.random((K, T)), rng.random((N, T))


def _close(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape and a.dtype == np.float64
    scale = max(float(np.max(np.abs(b))), 1e-300)
    assert float(np.max(np.abs(a - b))) <= 1e-12 * scale


@pytest.mark.parametrize("dims", DIMS)
def test_lagged_ref_matches_literal_oracles(dims, monkeypatch):
    N, T, K, L = dims
    W, H, X = _rand(*dims, seed=sum(dims))
    # chunks of 7 columns, so that every shape here crosses chunk boundaries, with chunks shorter than L
    monkeypatch.setattr(lr, "_chunk_len", lambda rows: 7)
    est = po.tensor_conv(W, H)
    _close(lr.conv(W, H), est)
    _close(lr.conv(W, H), co.tensor_conv(W, H))
    _close(lr.transconv(W, X), po.tensor_transconv(W, X))
    _close(lr.transconv(W, X), co.tensor_transconv(W, X))
    _close(lr.corr_w(H, X, L), po.corr_w(H, X, L))
    _close(lr.corr_w(H, X, L), co.corr_w(H, X, L))
    _close(lr.gram_R(H, L), rs.gram_R(H, L))
    _close(lr.denom_h(W, H), po.tensor_transconv(W, est))
    ss = float(np.sum((est - X) ** 2))
    assert abs(lr.sumsq_resid(W, H, X) - ss) <= 1e-12 * ss


def test_lagged_ref_default_chunks_and_float32_inputs():
    # the default chunk length at a long T, and float32 inputs taken exactly as given (upcast, not rounded again)
    N, T, K, L = 24, 20011, 6, 7
    W, H, X = (a.astype(np.float32) for a in _rand(N, T, K, L, seed=3))
    W64, H64, X64 = (a.astype(np.float64) for a in (W, H, X))
    assert lr._chunk_len(L * K) < T
    _close(lr.conv(W, H), po.tensor_conv(W64, H64))
    _close(lr.transconv(W, X), po.tensor_transconv(W64, X64))
    _close(lr.corr_w(H, X, L), po.corr_w(H64, X64, L))
    _close(lr.denom_h(W, H), po.tensor_transconv(W64, po.tensor_conv(W64, H64)))
