"""Float64 contractions of the MU half-steps that stay fast at T ~ 2e5  --  TEST INFRASTRUCTURE ONLY.

Same access contract as oracle/cnmf_oracle.py.  The literal oracles take O(L) passes over X (one product per lag, each
reading or writing an N x T array); at T ~ 2e5 and L ~ 100 that is tens of GB of memory traffic per contraction.  Here t is
cut into chunks and, per chunk, the lags are stacked (the tconv3 identity, ``cnmf_oracle.shift_and_stack``) so that each
contraction is one BLAS GEMM per chunk with an inner dimension of L*K, N or the chunk length:

    Hs[l*K + k, t] = H[k, t - l]  (zero for t < l)
    conv      est[:, c]                 = Wu @ Hs[:, c]                      Wu[n, l*K + k] = W[k, n, l]
    corr_w    numW[k, n, l]             = sum_c (Hs[:, c] @ X[:, c]')[l*K + k, n]
    transconv out[k, t]                 = sum_l (Wu' @ X)[l*K + k, t + l]    (t + l < T)

Inputs are upcast to float64 (the GPU tests draw them in float32 so that the device and this reference see the same
values).  Truncation follows cnmf_oracle: lags >= T contribute nothing, transconv drops t + l >= T.
tests/test_lagged_ref.py pins every function to cnmf_oracle, c_oracle and restructured.gram_R.
"""
from __future__ import annotations

import numpy as np

_CHUNK_ELEMS = 1 << 22          # doubles of one stacked chunk Hs[:, c] (32 MB) ...
_CHUNK_MAX = 16384              # ... and at most this many columns, so that the X columns of a chunk stay small too


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _chunk_len(rows):
    return min(_CHUNK_MAX, max(256, _CHUNK_ELEMS // max(1, rows)))


def _stacked(H, L, t0, t1):
    """Hs[:, t0:t1] of cnmf_oracle.shift_and_stack(H, L)."""
    K = H.shape[0]
    Hs = np.zeros((L * K, t1 - t0))
    for lag in range(L):
        a = max(t0, lag)                 # first column t with t - lag >= 0
        if a < t1:
            Hs[lag * K : (lag + 1) * K, a - t0 :] = H[:, a - lag : t1 - lag]
    return Hs


def _unfold(W):
    """Wu[n, l*K + k] = W[k, n, l]."""
    K, N, L = W.shape
    return np.ascontiguousarray(W.transpose(1, 2, 0).reshape(N, L * K))


def conv(W, H):
    """cnmf_oracle.tensor_conv: est[n, t] = sum_{l <= t} sum_k W[k, n, l] H[k, t - l]."""
    W, H = _f64(W), _f64(H)
    K, N, L = W.shape
    T = H.shape[1]
    Wu = _unfold(W)
    est = np.empty((N, T))
    step = _chunk_len(L * K)
    for t0 in range(0, T, step):
        t1 = min(T, t0 + step)
        np.matmul(Wu, _stacked(H, L, t0, t1), out=est[:, t0:t1])
    return est


def corr_w(H, X, L):
    """cnmf_oracle.corr_w: numW[k, n, l] = sum_{t=l}^{T-1} H[k, t - l] X[n, t]."""
    H, X = _f64(H), _f64(X)
    K, T = H.shape
    N = X.shape[0]
    acc = np.zeros((L * K, N))
    step = _chunk_len(L * K)
    for t0 in range(0, T, step):
        t1 = min(T, t0 + step)
        acc += _stacked(H, L, t0, t1) @ X[:, t0:t1].T
    return np.ascontiguousarray(acc.reshape(L, K, N).transpose(1, 2, 0))


def gram_R(H, L):
    """restructured.gram_R: R[k, k', d] = sum_{u=0}^{T-1-d} H[k, u] H[k', u + d], i.e. corr_w(H, H, L)."""
    return corr_w(H, H, L)


def transconv(W, X):
    """cnmf_oracle.tensor_transconv: out[k, t] = sum_{l < T - t} sum_n W[k, n, l] X[n, t + l]."""
    W, X = _f64(W), _f64(X)
    K, N, L = W.shape
    T = X.shape[1]
    WuT = np.ascontiguousarray(_unfold(W).T)
    out = np.zeros((K, T))
    step = _chunk_len(L * K)
    for t0 in range(0, T, step):
        t1 = min(T, t0 + step)
        e = min(T, t1 + L - 1)           # X columns t0 .. t1 + L - 2 feed the outputs t0 .. t1 - 1
        M = WuT @ X[:, t0:e]
        for lag in range(L):
            n = min(t1, e - lag) - t0    # outputs t with t + lag < e
            if n <= 0:
                break
            out[:, t0 : t0 + n] += M[lag * K : (lag + 1) * K, lag : lag + n]
    return out


def denom_h(W, H):
    """denomH = transconv(W, conv(W, H)) (mult.jl:44,48), truncated tail included."""
    return transconv(W, conv(W, H))


def sumsq_resid(W, H, X):
    """||conv(W, H) - X||_F^2 (src/common.jl:54-59)."""
    r = conv(W, H)
    r -= _f64(X)
    return float(np.einsum("nt,nt->", r, r))
