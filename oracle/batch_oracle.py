"""Float64 reference for R MultUpdate restarts of one data set  --  TEST INFRASTRUCTURE ONLY.

The batch handle (cmf_create_batch) fits R factor sets over one X.  This module is the checker for it: the operations of
``cnmf_oracle.MultUpdate`` (src/algs/mult.jl) with a leading restart axis and per-restart regularisers.  The three
contractions are products with ``cnmf_oracle.shift_and_stack(H)`` (the tconv3 identity), so that BLAS runs them with an inner
dimension of L*K, N or T rather than K.  Stacks are ``W[R, K, N, L]`` and ``H[R, K, T]``; ``X[N, T]`` is shared.
Restarts are processed in chunks so that the N x T estimates of a chunk stay within a few hundred MB.
"""
from __future__ import annotations

import numpy as np

from .cnmf_oracle import EPSILON

_CHUNK_ELEMS = 1 << 25          # doubles of R_chunk x N x T estimate held at once (256 MB)


def shift_and_stack(H, L):
    """Hs[r] = cnmf_oracle.shift_and_stack(H[r], L):  Hs[r][l*K + k, t] = H[r][k, t - l], zero for t < l."""
    R, K, T = H.shape
    Hs = np.zeros((R, L * K, T))
    for lag in range(min(L, T)):
        Hs[:, lag * K : (lag + 1) * K, lag:] = H[:, :, : T - lag]
    return Hs


def _unfold(W):
    """Wu[r][n, l*K + k] = W[r][k, n, l] (the unfolded motifs of src/common.jl:24-34)."""
    R, K, N, L = W.shape
    return W.transpose(0, 2, 3, 1).reshape(R, N, L * K)


def tensor_conv(W, H):
    """est[r] = cnmf_oracle.tensor_conv(W[r], H[r]) = Wu[r] @ shift_and_stack(H[r]) (the tconv3 identity)."""
    return np.matmul(_unfold(W), shift_and_stack(H, W.shape[3]))


def tensor_transconv(W, X):
    """out[r] = cnmf_oracle.tensor_transconv(W[r], X or X[r]):  out[r][k, t] = sum_l (Wu[r]' Y)[l*K + k, t + l]."""
    R, K, N, L = W.shape
    T = X.shape[-1]
    WuT = _unfold(W).transpose(0, 2, 1)
    if X.ndim == 2:             # shared data: one product over all R*L*K rows
        M = (WuT.reshape(R * L * K, N) @ X).reshape(R, L * K, T)
    else:
        M = np.matmul(WuT, X)
    out = np.zeros((R, K, T))
    for lag in range(min(L, T)):
        out[:, :, : T - lag] += M[:, lag * K : (lag + 1) * K, lag:]
    return out


def corr_w(H, X, L):
    """out[r] = cnmf_oracle.corr_w(H[r], X or X[r], L):  out[r][k, n, l] = (shift_and_stack(H[r]) X')[l*K + k, n]."""
    R, K, T = H.shape
    N = X.shape[-2]
    Hs = shift_and_stack(H, L)
    if X.ndim == 2:
        C = (Hs.reshape(R * L * K, T) @ X.T).reshape(R, L, K, N)
    else:
        C = np.matmul(Hs, X.transpose(0, 2, 1)).reshape(R, L, K, N)
    return C.transpose(0, 2, 3, 1).copy()


def _chunks(R, N, T):
    step = max(1, _CHUNK_ELEMS // max(1, N * T))
    return [slice(r0, min(R, r0 + step)) for r0 in range(0, R, step)]


def _per_restart(v, R):
    a = np.asarray(v, dtype=np.float64)
    return np.full(R, float(a)) if a.ndim == 0 else a.reshape(R)


def losses(X, W, H):
    """||conv(W[r], H[r]) - X||_F / ||X||_F for every restart (src/common.jl:54-55)."""
    X = np.asarray(X, dtype=np.float64)
    R, N, T = W.shape[0], X.shape[0], X.shape[1]
    out = np.empty(R)
    for c in _chunks(R, N, T):
        out[c] = np.sqrt(np.sum((tensor_conv(W[c], H[c]) - X) ** 2, axis=(1, 2)))
    return out / np.linalg.norm(X)


def scale_partials(X, W, H):
    """(<X, est_r>, ||est_r||^2) per restart, the two sums of the init_rand rescale (src/model.jl:119-120); shape (R, 2)."""
    X = np.asarray(X, dtype=np.float64)
    R, N, T = W.shape[0], X.shape[0], X.shape[1]
    out = np.empty((R, 2))
    for c in _chunks(R, N, T):
        est = tensor_conv(W[c], H[c])
        out[c, 0] = np.einsum("rnt,nt->r", est, X)
        out[c, 1] = np.einsum("rnt,rnt->r", est, est)
    return out


def mu_step(X, W, H, l1W=0.0, l2W=0.0, l1H=0.0, l2H=0.0, eval_mode=False):
    """One MultUpdate iteration of every restart (src/algs/alternating.jl:46-50): update_motifs! (mult.jl:23-39, skipped
    with ``eval_mode``), then update_feature_maps! (mult.jl:42-58).  Regularisers are scalars or one value per restart.
    Returns (W1, H1, loss1) with loss1 the relative loss after the step.  The inputs are not modified."""
    X = np.asarray(X, dtype=np.float64)
    W = np.array(W, dtype=np.float64)
    H = np.array(H, dtype=np.float64)
    R, K, N, L = W.shape
    T = X.shape[1]
    reg = [_per_restart(v, R) for v in (l1W, l2W, l1H, l2H)]
    loss = np.empty(R)
    for c in _chunks(R, N, T):
        Wc, Hc = W[c], H[c]
        a1W, a2W, a1H, a2H = (v[c] for v in reg)
        if not eval_mode:
            est = tensor_conv(Wc, Hc)
            numW = corr_w(Hc, X, L)
            denW = corr_w(Hc, est, L)
            Wc *= numW / (denW + a1W[:, None, None, None] + 2 * a2W[:, None, None, None] * Wc + EPSILON)
            np.maximum(Wc, EPSILON, out=Wc)
        est = tensor_conv(Wc, Hc)
        numH = tensor_transconv(Wc, X)
        denH = tensor_transconv(Wc, est)
        Hc *= numH / (denH + a1H[:, None, None] + 2 * a2H[:, None, None] * Hc + EPSILON)
        np.maximum(Hc, EPSILON, out=Hc)
        loss[c] = np.sqrt(np.sum((tensor_conv(Wc, Hc) - X) ** 2, axis=(1, 2)))
    return W, H, loss / np.linalg.norm(X)
