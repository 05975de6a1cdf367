"""A call that replaces X, W or H must leave nothing stale behind: after it, a handle that has already iterated (its cached
operands -- numH, W W', the Gram partial, the bf16 planes and spectra of X, W and H -- all resident) computes bit for bit
what a fresh handle with the same host state computes.  Covered for set_factors, init_rand, scale_factors and set_data on
every engine (SIMT fp64 / fp32, time-domain and frequency-domain tcgen05) and MultUpdate (both loss modes), HALSUpdate and
PGDUpdate.  PGD gets set_factors only: init_rand, scale_factors and set_data deliberately keep its step sizes."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N, T, K, L = 96, 1200, 6, 9          # N % 8 == 0: engines 1 and 2 are available
REG_W = dict(l1W=0.05, l2W=0.1)
REG_H = dict(l1H=0.05, l2H=0.1)

ENGINES = [("f64", 0), ("f32", 0), ("f32", 1), ("f32", 2)]
RULES = [("mult", 0), ("mult", 1), ("hals", 0), ("pgd", 0)]
EVENTS = ["set_factors", "init_rand", "scale_factors", "set_data"]
CASES = [(dt, eng, alg, lm, ev) for dt, eng in ENGINES for alg, lm in RULES for ev in EVENTS
         if alg != "pgd" or ev == "set_factors"]


@pytest.fixture(scope="module")
def cmf():
    import __graft_entry__ as ge

    ge.build()
    import cmf_jl_b200

    return cmf_jl_b200


def _host(seed):
    rng = np.random.default_rng(seed)
    return rng.random((N, T)), rng.random((K, N, L)), rng.random((K, T))


def _rule(cmf, alg, dtype, engine, loss_mode, X, W, H):
    cls = {"mult": cmf.MultUpdate, "hals": cmf.HALSUpdate, "pgd": cmf.PGDUpdate}[alg]
    return cls(X, W, H, dtype=dtype, engine=engine, loss_mode=loss_mode, sync_host=False)


def _step(rule):
    loss0 = rule.loss()
    rule.update_motifs(None, None, None, **REG_W)
    loss1 = rule.update_feature_maps(None, None, None, **REG_H)
    W, H = rule.get_factors()
    return loss0, loss1, W, H


@pytest.mark.parametrize("dtype,engine,alg,loss_mode,event", CASES)
def test_used_handle_matches_fresh_after_state_change(cmf, dtype, engine, alg, loss_mode, event):
    from cmf_jl_b200 import _lib

    lib = _lib.load()
    X, W0, H0 = _host(1)
    a = _rule(cmf, alg, dtype, engine, loss_mode, X, W0, H0)
    for _ in range(2):                                  # fills every cache the handle keeps
        a.update_motifs(None, None, None, **REG_W)
        a.update_feature_maps(None, None, None, **REG_H)
    if event == "set_factors":
        _, W1, H1 = _host(2)
        a.set_factors(W1, H1)
        b = _rule(cmf, alg, dtype, engine, loss_mode, X, W1, H1)
    elif event == "init_rand":
        _lib.check(lib.cmf_init_rand(a._h, 77))
        b = _rule(cmf, alg, dtype, engine, loss_mode, X, W0, H0)
        _lib.check(lib.cmf_init_rand(b._h, 77))
    elif event == "scale_factors":
        Wa, Ha = a.get_factors()                        # handle dtype: the host product rounds like the device's
        s = Wa.dtype.type(0.75)
        _lib.check(lib.cmf_scale_factors(a._h, 0.75))
        b = _rule(cmf, alg, dtype, engine, loss_mode, X, Wa * s, Ha * s)
    else:
        Wa, Ha = a.get_factors()
        X2, _, _ = _host(3)
        _lib.check(lib.cmf_set_data(a._h, _lib.fptr(_lib.julia_array(X2, a.dtype)), 0))
        b = _rule(cmf, alg, dtype, engine, loss_mode, X2, Wa, Ha)
    try:
        la0, la1, Wa, Ha = _step(a)
        lb0, lb1, Wb, Hb = _step(b)
    finally:
        a.close()
        b.close()
    assert la0 == lb0 and la1 == lb1, (la0, lb0, la1, lb1)
    assert np.array_equal(Wa, Wb)
    assert np.array_equal(Ha, Hb)
