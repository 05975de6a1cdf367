"""Batched restarts and the SIMT contractions at the tilings R*K stacked components select, against float64 references.

A batch handle runs numW and numH as ONE correlation and ONE transposed convolution over R*K components, so at R = 64 and
K = 5 (Kout = 320) `launch_transconv` picks tilings, k-tile counts and unit splits that no single fit of a few components
reaches, and in fp32 at large T the correlations flush their fp32 accumulators into fp64 partials several times per split.
The tests below reach those regimes twice:

- through the primitives (cmf_tensor_transconv, cmf_corr_w, cmf_tensor_conv), which run the same kernels as the batch's stacked
  numH, numW and loss conv when their K is R*K, against float64 NumPy;
- through the batch handle, against oracle/batch_oracle.py (pinned to the C oracle in tests/test_batch_oracle.py), against
  single fits, and against itself with the restarts reordered or a neighbour rescaled.

The plan mirrors below restate the host arithmetic that picks each regime, so every case is labelled with the regime it
reaches and test_case_lists_reach_every_regime fails if a change to the plan leaves a regime untested.  Tests that need no
device (the mirrors and the argument guards) carry no gpu marker.  The gpu tests of this file take about 35 s on one B200.
"""
import ctypes

import numpy as np
import pytest

from oracle import batch_oracle as bo

gpu = pytest.mark.gpu


def cdiv(a, b):
    return -(-a // b)


# ------------------------------------------------------------------------------------------ plan mirrors
def transconv_plan(Nin, Kout, Lin, t_out, nrest=1):
    """Tile choice of launch_transconv (cmf.jl_b200/csrc/cmf_sm100.cu:1110-1151): TK and k-groups with the least padding
    of Kout, t-groups halved while the (t, k) grid is short of 296 CTAs, and the split over units (unit split) when a single
    restart's grid is still short and Nin >= 64."""
    best = None
    for tk in (8, 5, 4):
        kg = 1
        while kg < 16 and kg * tk < Kout:
            kg *= 2
        kp = kg * tk
        waste = (cdiv(Kout, kp) * kp - Kout) / Kout
        if best is None or waste < best[0] - 1e-9:
            best = (waste, tk, kg)
    _, tk, kg = best
    tg0 = tg = max(128 // kg, 8)
    while tg * kg > 32 and cdiv(t_out, tg * 8) < 296:
        tg //= 2
    ctas = cdiv(t_out, tg * 8) * cdiv(Kout, kg * tk)
    nsplit = 1
    if nrest == 1 and ctas < 296 and Nin >= 64:
        want = min(cdiv(Nin, 32), cdiv(296, ctas), 32)
        nsplit = cdiv(Nin, cdiv(cdiv(Nin, want), 16) * 16)      # TR_NC = 16
    return dict(tk=tk, kg=kg, ktiles=cdiv(Kout, kg * tk), halved=tg < tg0, ctas=ctas, nsplit=nsplit)


def corr_plan(Nin, tau_hi, Kc, L, nrest=1):
    """plan_split (cmf_sm100.cu:1015-1022): (nsplit, split_len) of corr_kernel's tau sum; CORR_PB = 16, CORR_BTAU = 32.
    fp32 accumulators are flushed into the fp64 partial every CORR_FLUSH = 2048 columns (kernels_simt.cuh:459-463), so a
    split longer than 2048 columns takes the flush-and-accumulate branch."""
    bxy = cdiv(Nin, 128) * cdiv(Kc * cdiv(L, 8), 16) * nrest
    ns = min(max(cdiv(592, bxy), 1), 64)
    split_len = max(cdiv(cdiv(tau_hi, ns), 32) * 32, 32)
    return cdiv(tau_hi, split_len), split_len


CORR_FLUSH = 2048


def conv_kc(K, L, itemsize):
    """Components per shared-memory H window of conv_kernel (launch_conv, cmf_sm100.cu:1074-1080): a 160 KiB budget less
    the W chunk (CONV_LC = 32 lags x BN units, BN = 64 in fp64 and 128 in fp32), over BT + Lpad - 1 = 127 + Lpad columns."""
    bn = 64 if itemsize == 8 else 128
    hw = 128 + cdiv(L, 8) * 8 - 1
    return min(K, (160 * 1024 - 32 * bn * itemsize) // (hw * itemsize))


# ------------------------------------------------------------------------------------------ cases
# transconv (N, T, K, L): Kout = K output components; N = 40 keeps the unit split off (Nin < 64), K >= 129 fills the device
# with k-tiles, T = 20000 with 16 k-groups leaves the t-groups unhalved.
TRANSCONV_CASES = (
    [(200, 3000, K, 10) for K in (1, 3, 8, 13, 20, 40, 64, 65, 128, 129, 320, 321)]
    + [(40, 3000, K, 10) for K in (5, 64, 320)]
    + [(128, 20000, K, 10) for K in (128, 320, 321)]
    + [(500, 2000, 320, 10), (500, 2000, 91, 10), (77, 999, 13, 1), (150, 1500, 40, 17)]
)
# corr (N, T, K, L): K = 320, N = 500, L = 10, T = 30000 is numW of the R = 64 batch below (4 splits of 7520 columns)
CORR_CASES = [(500, 30000, 320, 10), (500, 2000, 320, 10), (130, 9000, 13, 17), (64, 5000, 3, 1)]
# conv (N, T, K, L): K beyond one H window (two kc0 passes) in each dtype
CONV_CASES = [(64, 1000, 130, 100), (100, 700, 200, 100), (150, 900, 5, 10)]


def _transconv_regimes():
    out = []
    for N, T, K, L in TRANSCONV_CASES:
        p = transconv_plan(N, K, L, T)
        out.append(dict(p, unit_split=p["nsplit"] > 1, few_ctas=p["ctas"] < 296, small_nin=N < 64))
    return out


def test_case_lists_reach_every_regime():
    regs = _transconv_regimes()
    assert {p["tk"] for p in regs} == {8, 5, 4}
    assert {p["kg"] for p in regs} == {1, 2, 4, 8, 16}
    assert any(p["ktiles"] == 1 for p in regs) and any(p["ktiles"] >= 3 for p in regs)
    assert any(p["unit_split"] for p in regs)                                       # Nin >= 64, few CTAs
    assert any(p["small_nin"] and p["few_ctas"] and not p["unit_split"] for p in regs)
    assert any(not p["few_ctas"] and not p["unit_split"] and not p["small_nin"] for p in regs)
    assert any(p["halved"] for p in regs) and any(not p["halved"] for p in regs)
    # corr: a split of several flush intervals in fp32
    nsplit, split_len = corr_plan(500, 30000 + 9, 320, 10)
    assert (nsplit, split_len) == (4, 7520) and split_len > 3 * CORR_FLUSH
    # conv: more components than one H window holds, in each dtype
    assert conv_kc(130, 100, 8) == 79 and conv_kc(200, 100, 4) < 200
    assert all(conv_kc(K, L, 4) < K or conv_kc(K, L, 8) < K for _, _, K, L in CONV_CASES[:2])
    # the batch shapes below: config 1 at R = 64 stacks Kout = 320 (TK = 5, 16 k-groups, 4 k-tiles, no unit split); the fp32
    # R = 64, T = 30000 batch flushes in its per-restart Gram and in numW, while T = 20000 would not flush the Gram
    assert transconv_plan(500, 320, 10, 2000) == dict(tk=5, kg=16, ktiles=4, halved=True, ctas=500, nsplit=1)
    assert transconv_plan(500, 7 * 13, 10, 2000)["nsplit"] > 1                     # R = 7, K = 13: ragged R*K, split on
    assert corr_plan(5, 30000 + 9, 5, 10, nrest=64) == (10, 3008)
    assert corr_plan(500, 30000 + 9, 320, 10) == (4, 7520)
    assert corr_plan(5, 20000 + 9, 5, 10, nrest=64)[1] < CORR_FLUSH


# ------------------------------------------------------------------------------------------ fixtures and helpers
@pytest.fixture(scope="module")
def cmf():
    import __graft_entry__ as ge

    ge.build()
    import cmf_jl_b200

    return cmf_jl_b200


def _round(a, dtype):
    """The inputs as the device sees them, back in float64."""
    return np.asarray(a, dtype=np.float32 if dtype == "f32" else np.float64).astype(np.float64)


def _scale_err(got, ref):
    return float(np.max(np.abs(np.asarray(got, dtype=np.float64) - ref)) / np.max(np.abs(ref)))


TOL = {"f64": 1e-12, "f32": 2e-5}


def _data(N, T, L, seed):
    from oracle import cnmf_oracle as po

    X, _, _ = po.synthetic_sequences(K=3, N=N, L=L, T=T, rng=np.random.default_rng(seed))
    return X


def _stacks(X, R, K, L, seed):
    """Uniform draws, each restart rescaled by its own alpha (src/model.jl:119-122) so that est is on the scale of X."""
    rng = np.random.default_rng(seed)
    N, T = X.shape
    W, H = rng.random((R, K, N, L)), rng.random((R, K, T))
    part = bo.scale_partials(X, W, H)
    s = np.sqrt(np.abs(part[:, 0] / part[:, 1]))
    return W * s[:, None, None, None], H * s[:, None, None]


def _regs(R, seed=0):
    """Different regularisers per restart; restart 0 unregularised."""
    rng = np.random.default_rng(seed)
    regs = {k: rng.random(R) * s for k, s in (("l1W", 0.2), ("l2W", 0.6), ("l1H", 0.2), ("l2H", 0.4))}
    for v in regs.values():
        v[0] = 0.0
    return regs


def _open(cmf, X, W, H, dtype):
    from cmf_jl_b200._lib import check, fptr, julia_array, parse_dtype

    lib = cmf._lib.load()
    dt = parse_dtype(dtype)
    R, K, N, L = W.shape
    h = ctypes.c_void_p()
    check(lib.cmf_create_batch(ctypes.byref(h), N, X.shape[1], K, L, dt, 0, R, 0))
    try:
        check(lib.cmf_set_data(h, fptr(julia_array(X, dt)), 0))
        check(lib.cmf_set_factors_batch(h, fptr(julia_array(np.moveaxis(W, 0, -1), dt)),
                                        fptr(julia_array(np.moveaxis(H, 0, -1), dt))))
    except Exception:
        lib.cmf_destroy(h)
        raise
    return lib, h


def _fit(cmf, X, W, H, itr, dtype="f64", **kw):
    """fit_cnmf_batch from explicit stacks, no early stop; returns (W [R,K,N,L], H [R,K,T], loss [R, itr+1])."""
    R, K, N, L = W.shape
    res = cmf.fit_cnmf_batch(X, L=L, K=K, max_itr=itr, W_init=W, H_init=H, dtype=dtype, check_convergence=False,
                             layout="KNL", **kw)
    assert len(res) == R and all(len(r.loss_hist) == itr + 1 for r in res)
    return (np.stack([r.W for r in res]), np.stack([r.H for r in res]), np.array([r.loss_hist for r in res]))


# ------------------------------------------------------------------------------------------ 2. primitives
@gpu
@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("N,T,K,L", TRANSCONV_CASES)
def test_transconv_tilings(cmf, N, T, K, L, dtype):
    rng = np.random.default_rng(N * 7 + K)
    W, X = _round(rng.random((K, N, L)), dtype), _round(rng.random((N, T)), dtype)
    got = cmf.tensor_transconv(W, X, dtype=dtype)
    ref = bo.tensor_transconv(W[None], X)[0]
    assert _scale_err(got, ref) < TOL[dtype], transconv_plan(N, K, L, T)


@gpu
@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("N,T,K,L", CORR_CASES)
def test_corr_splits_and_flush(cmf, N, T, K, L, dtype):
    rng = np.random.default_rng(N + T + K)
    H, X = _round(rng.random((K, T)), dtype), _round(rng.random((N, T)), dtype)
    got = cmf.corr_w(H, X, L, dtype=dtype)
    ref = bo.corr_w(H[None], X, L)[0]
    assert _scale_err(got, ref) < TOL[dtype], corr_plan(N, T + L - 1, K, L)


@gpu
@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("N,T,K,L", CONV_CASES)
def test_conv_component_windows(cmf, N, T, K, L, dtype):
    rng = np.random.default_rng(N + K)
    W, H = _round(rng.random((K, N, L)), dtype), _round(rng.random((K, T)), dtype)
    got = cmf.tensor_conv(W, H, dtype=dtype)
    ref = bo.tensor_conv(W[None], H[None])[0]
    assert _scale_err(got, ref) < TOL[dtype], conv_kc(K, L, 8 if dtype == "f64" else 4)


# ------------------------------------------------------------------------------------------ 3. batch handle
@gpu
@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("R", [1, 7, 64, 256])
def test_loss_and_scale_partials_batch(cmf, R, dtype):
    N, T, K, L = 150, 700, 5, 10
    X = _round(_data(N, T, L, seed=R), dtype)
    rng = np.random.default_rng(R)
    W = _round(rng.random((R, K, N, L)) * rng.random((R, 1, 1, 1)) * 0.3, dtype)   # a different scale per restart
    H = _round(rng.random((R, K, T)), dtype)
    lib, h = _open(cmf, X, W, H, dtype)
    try:
        loss, part = np.zeros(R), np.zeros(2 * R)
        dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))  # noqa: E731
        cmf._lib.check(lib.cmf_loss_batch(h, dp(loss)))
        cmf._lib.check(lib.cmf_init_scale_partials_batch(h, dp(part)))
    finally:
        lib.cmf_destroy(h)
    ref_loss, ref_part = bo.losses(X, W, H), bo.scale_partials(X, W, H)
    tol = TOL[dtype]
    np.testing.assert_allclose(loss, ref_loss, rtol=tol, atol=0)
    np.testing.assert_allclose(part.reshape(R, 2), ref_part, rtol=tol, atol=0)


STEP_CASES = {
    "config1_R64": (500, 2000, 5, 10, 64),      # R*K = 320: TK = 5, 16 k-groups, 4 k-tiles
    "R7_K13": (300, 1500, 13, 10, 7),           # R*K = 91: ragged k-tile, unit split on
    "R3_L1": (120, 600, 4, 1, 3),
    "R3_T_eq_L": (60, 12, 3, 12, 3),            # T = L: the denomH tail covers every column
}


@gpu
@pytest.mark.parametrize("eval_mode", [False, True])
@pytest.mark.parametrize("case", list(STEP_CASES))
def test_one_step_fp64(cmf, case, eval_mode):
    N, T, K, L, R = STEP_CASES[case]
    X = _data(N, T, L, seed=N + R)
    W, H = _stacks(X, R, K, L, seed=R)
    regs = _regs(R, seed=K)
    Wg, Hg, lg = _fit(cmf, X, W, H, 1, eval_mode=eval_mode, **regs)
    W1, H1, loss1 = bo.mu_step(X, W, H, eval_mode=eval_mode, **regs)
    np.testing.assert_allclose(lg[:, 0], bo.losses(X, W, H), rtol=1e-12, atol=0)
    np.testing.assert_allclose(lg[:, 1], loss1, rtol=1e-12, atol=0)
    for r in range(R):
        np.testing.assert_allclose(Wg[r], W1[r], rtol=1e-11, atol=1e-11 * np.max(W1[r]), err_msg=f"W of restart {r}")
        np.testing.assert_allclose(Hg[r], H1[r], rtol=1e-11, atol=1e-11 * np.max(H1[r]), err_msg=f"H of restart {r}")
    if eval_mode:
        assert np.array_equal(Wg, W)


def test_t_below_l_is_refused(cmf):
    # the batch keeps the reference's L <= T (src/common.jl:28-31), so T = L above is the shortest series it fits
    lib = cmf._lib.load()
    h = ctypes.c_void_p()
    assert lib.cmf_create_batch(ctypes.byref(h), 60, 11, 3, 12, 0, 0, 3, 0) == 1


@pytest.fixture(scope="module")
def long_fp32(cmf):
    """R = 64, K = 5, L = 10, N = 500, T = 30000: the per-restart Gram runs 10 splits of 3008 columns and numW 4 splits of
    7520, both longer than CORR_FLUSH, so the fp32 correlations flush and accumulate."""
    N, T, K, L, R = 500, 30000, 5, 10, 64
    assert corr_plan(K, T + L - 1, K, L, nrest=R)[1] > CORR_FLUSH and corr_plan(N, T + L - 1, R * K, L)[1] > CORR_FLUSH
    X = _round(_data(N, T, L, seed=5), "f32")
    W, H = _stacks(X, R, K, L, seed=6)
    return X, _round(W, "f32"), _round(H, "f32"), _regs(R, seed=3)


@gpu
def test_fp32_long_one_step(cmf, long_fp32):
    """The fp32 step against the float64 reference from the same fp32 inputs.  Each accumulation runs in fp32 over at most
    2048 columns (correlations) or N*L = 5000 terms (transposed convolution) before it is carried in fp64, so the step's
    relative error is a few 1e-6 for sums of like-signed terms (measured on a B200: 7e-7 for W, 3e-6 for H, worst restart);
    the bar, 5e-5 of each factor's scale, leaves 10x of margin and is still 4 orders below what a lost flush (3/4 of a
    split dropped) would give."""
    X, W, H, regs = long_fp32
    Wg, Hg, lg = _fit(cmf, X, W, H, 1, dtype="f32", **regs)
    W1, H1, loss1 = bo.mu_step(X, W, H, **regs)
    for r in range(W.shape[0]):
        assert _scale_err(Wg[r], W1[r]) < 5e-5, r
        assert _scale_err(Hg[r], H1[r]) < 5e-5, r
    np.testing.assert_allclose(lg[:, 1], loss1, rtol=2e-5, atol=0)


@gpu
def test_fp32_long_twenty_iterations_track_fp64(cmf, long_fp32):
    X, W, H, regs = long_fp32
    _, _, l32 = _fit(cmf, X, W, H, 20, dtype="f32", **regs)
    _, _, l64 = _fit(cmf, X, W, H, 20, dtype="f64", **regs)
    assert np.max(np.abs(l32 - l64)) < 1e-4


@pytest.fixture(scope="module")
def config1(cmf):
    N, T, K, L, R = 500, 2000, 5, 10, 64
    X = _data(N, T, L, seed=1234)
    W, H = _stacks(X, R, K, L, seed=77)
    return X, W, H, _regs(R, seed=9)


@gpu
def test_config1_hundred_iterations_match_single_fits_and_c_oracle(cmf, config1):
    from oracle import c_oracle as co

    X, W, H, regs = config1
    R, K, N, L = W.shape
    itr = 100
    Wg, Hg, lg = _fit(cmf, X, W, H, itr, **regs)
    for r in range(R):
        reg = {k: float(v[r]) for k, v in regs.items()}
        single = cmf.fit_cnmf(X, L=L, K=K, max_itr=itr, W_init=W[r], H_init=H[r], check_convergence=False, layout="KNL", **reg)
        np.testing.assert_allclose(lg[r], single.loss_hist, rtol=1e-12, atol=0, err_msg=f"restart {r}")
    for r in (0, R // 2, R - 1):
        reg = {k: float(v[r]) for k, v in regs.items()}
        ref = co.fit(co.MultUpdate, X, W[r], H[r], itr, check_convergence=False, **reg)
        np.testing.assert_allclose(lg[r], ref.loss_hist, rtol=1e-9, atol=0, err_msg=f"restart {r}")
        np.testing.assert_allclose(Wg[r], ref.W, rtol=1e-8, atol=1e-11)
        np.testing.assert_allclose(Hg[r], ref.H, rtol=1e-8, atol=1e-11)


@gpu
@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_restart_order_does_not_change_results(cmf, config1, dtype):
    """No output element's summation order depends on its column's position in the stack, so reversing the restarts
    reverses the results bit for bit."""
    X, W, H, regs = config1
    a = _fit(cmf, X, W, H, 10, dtype=dtype, **regs)
    b = _fit(cmf, X, W[::-1], H[::-1], 10, dtype=dtype, **{k: v[::-1] for k, v in regs.items()})
    for x, y in zip(a, b):
        assert np.array_equal(x, y[::-1])


@gpu
@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_rescaled_neighbour_does_not_change_others(cmf, config1, dtype):
    X, W, H, regs = config1
    j = 37
    W2, H2 = W.copy(), H.copy()
    W2[j] *= 1e4
    H2[j] *= 1e4
    a = _fit(cmf, X, W, H, 10, dtype=dtype, **regs)
    b = _fit(cmf, X, W2, H2, 10, dtype=dtype, **regs)
    keep = np.arange(W.shape[0]) != j
    for x, y in zip(a, b):
        assert np.array_equal(x[keep], y[keep])
    assert not np.array_equal(a[2][j], b[2][j])


@gpu
def test_max_restarts(cmf):
    N, T, K, L, R = 4, 40, 7, 3, 32768
    X = _data(N, T, L, seed=2)
    rng = np.random.default_rng(3)
    W, H = rng.random((R, K, N, L)) * 0.3, rng.random((R, K, T))
    regs = _regs(R, seed=4)
    Wg, Hg, lg = _fit(cmf, X, W, H, 1, **regs)
    W1, H1, loss1 = bo.mu_step(X, W, H, **regs)
    np.testing.assert_allclose(lg[:, 0], bo.losses(X, W, H), rtol=1e-12, atol=0)
    np.testing.assert_allclose(lg[:, 1], loss1, rtol=1e-12, atol=0)
    np.testing.assert_allclose(Wg, W1, rtol=1e-11, atol=1e-11 * np.max(W1))
    np.testing.assert_allclose(Hg, H1, rtol=1e-11, atol=1e-11 * np.max(H1))


def test_restart_grid_guards(cmf):
    """cmf_create_batch refuses R*K past what one launch grid holds (R*K <= 4*65535) and R past 32768 before it looks
    for a device."""
    lib = cmf._lib.load()
    h = ctypes.c_void_p()
    assert lib.cmf_create_batch(ctypes.byref(h), 4, 40, 8, 3, 0, 0, 32768, 0) == 1
    assert b"R*K too large" in lib.cmf_last_error()
    assert lib.cmf_create_batch(ctypes.byref(h), 4, 40, 1, 3, 0, 0, 32769, 0) == 1
    assert b"restarts" in lib.cmf_last_error()
