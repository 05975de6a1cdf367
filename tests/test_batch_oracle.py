"""The float64 batch reference (oracle/batch_oracle.py) against the per-restart oracles, without a device.

tests/test_gpu_batch_regimes.py checks the batch handle against this reference, so it is pinned here first: each restart's
MultUpdate step must equal the C oracle's (oracle/cnmf_oracle.c) from the same factors and regularisers, and the loss and
rescale partials must equal the NumPy oracle's."""
import numpy as np
import pytest

from oracle import batch_oracle as bo
from oracle import c_oracle as co
from oracle import cnmf_oracle as po


def _stacks(R, N, T, K, L, seed):
    rng = np.random.default_rng(seed)
    X = rng.random((N, T)) * (rng.random((N, T)) < 0.7)
    return X, rng.random((R, K, N, L)), rng.random((R, K, T))


def _regs(R):
    rng = np.random.default_rng(R)
    regs = {k: rng.random(R) * s for k, s in (("l1W", 0.2), ("l2W", 0.5), ("l1H", 0.2), ("l2H", 0.3))}
    for v in regs.values():
        v[0] = 0.0                  # restart 0 unregularised
    return regs


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


@pytest.mark.parametrize("N,T,K,L", [(23, 120, 3, 7), (17, 60, 4, 1), (9, 10, 2, 10)])
@pytest.mark.parametrize("eval_mode", [False, True])
def test_mu_step_matches_c_oracle_per_restart(N, T, K, L, eval_mode):
    R = 4
    X, W, H = _stacks(R, N, T, K, L, seed=N + T)
    regs = _regs(R)
    W1, H1, loss1 = bo.mu_step(X, W, H, eval_mode=eval_mode, **regs)
    for r in range(R):
        Wr, Hr = np.asfortranarray(W[r]), np.asfortranarray(H[r])
        rule = co.MultUpdate(X, Wr, Hr)
        reg = {k: float(v[r]) for k, v in regs.items()}
        if not eval_mode:
            rule.update_motifs(X, Wr, Hr, **reg)
        loss = rule.update_feature_maps(X, Wr, Hr, **reg)
        assert _rel(W1[r], Wr) < 1e-12
        assert _rel(H1[r], Hr) < 1e-12
        assert abs(loss1[r] - loss) < 1e-12 * loss
        if eval_mode:
            assert np.array_equal(W1[r], W[r])


def test_inputs_are_not_modified_and_restarts_do_not_mix():
    X, W, H = _stacks(5, 11, 50, 3, 4, seed=3)
    W0, H0 = W.copy(), H.copy()
    W1, H1, loss1 = bo.mu_step(X, W, H, l1W=0.1, l2H=0.2)
    assert np.array_equal(W, W0) and np.array_equal(H, H0)
    W2, H2, loss2 = bo.mu_step(X, W[::-1], H[::-1], l1W=0.1, l2H=0.2)
    # BLAS may block the stacked products differently, so equal to rounding rather than bitwise
    assert _rel(W2[::-1], W1) < 1e-14 and _rel(H2[::-1], H1) < 1e-14 and _rel(loss2[::-1], loss1) < 1e-14


def test_loss_partials_and_primitives_match_numpy_oracle(monkeypatch):
    R, N, T, K, L = 6, 13, 80, 3, 5
    X, W, H = _stacks(R, N, T, K, L, seed=8)
    monkeypatch.setattr(bo, "_CHUNK_ELEMS", 2 * N * T)      # several chunks, the last one short
    loss = bo.losses(X, W, H)
    part = bo.scale_partials(X, W, H)
    conv, trans, corr = bo.tensor_conv(W, H), bo.tensor_transconv(W, X), bo.corr_w(H, X, L)
    trans_r, corr_r = bo.tensor_transconv(W, conv), bo.corr_w(H, conv, L)
    for r in range(R):
        est = po.tensor_conv(W[r], H[r])
        assert abs(loss[r] - po.compute_loss(X, W[r], H[r])) < 1e-13 * loss[r]
        assert _rel(part[r], np.array([np.vdot(X, est), np.vdot(est, est)])) < 1e-13
        assert np.array_equal(bo.shift_and_stack(H, L)[r], po.shift_and_stack(H[r], L))
        assert _rel(conv[r], est) < 1e-13
        assert _rel(trans[r], po.tensor_transconv(W[r], X)) < 1e-13
        assert _rel(corr[r], po.corr_w(H[r], X, L)) < 1e-13
        assert _rel(trans_r[r], po.tensor_transconv(W[r], est)) < 1e-13
        assert _rel(corr_r[r], po.corr_w(H[r], est, L)) < 1e-13
