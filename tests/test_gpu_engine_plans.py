"""The two tensor-core engines at the plans the benchmarks run, against float64 references.

The host code of each engine picks a plan from the shape: `fd_setup` the block length B, the hop and the column tiles of the
frequency-domain engine (engine 2), `tc_setup` the t-splits of the time-domain correlation (engine 1), whose `TC_CORR` kernel
flushes its fp32 registers into an fp64 partial every FLUSH_T = 65536 columns.  Small test shapes land on the simplest plans
(B <= 512, one split, one flush segment), so the cases below are chosen to reach the plans of the c3 / c4 / c5 workloads:
B = 1024 with its 8-column tiles and trailing radix-2 pass, Kq = 128 at B = 256 .. 1024, L = 256, more than 256 blocks,
several splits of several segments, a segment of a single k-block, and the 100-iteration fixtures at the block lengths the
benchmark runs.

`fd_plan` and `tc_plan` restate the host arithmetic in plain Python; `test_case_lists_reach_every_regime` (no GPU) fails if a
change to the plan or to the case lists leaves a regime untested.  The references come from oracle/lagged_ref.py (pinned to
the literal oracles in tests/test_lagged_ref.py); inputs are drawn in float32 and upcast, so device and reference see the
same values.
"""
import os
import sys

import numpy as np
import pytest

from oracle import lagged_ref as lr

gpu = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")

NUM_SMS = 148          # B200
FLUSH_T = 65536        # kernels_tc.cuh: TC_CORR columns per fp64 flush segment
BK, BM, BN = 32, 128, 256
LOSS_TOL, CONTRACTION_TOL = 2e-5, 3e-5


def cdiv(a, b):
    return -(-a // b)


# ------------------------------------------------------------------------------------------ plan mirrors
def fd_plan(N, T, K, L, forced=0):
    """fd_setup (cmf_sm100.cu) for one shard of T columns with room for the first-choice block length: Kq, the block length
    B0 (smallest power of two >= 8L, at most 1024, >= 4L), the short-shard rule (halve B0 when the longer block does not win
    3 % on the product work F * (ceil(blocks / 256) * 256 + ceil(blocks / 16) * 16)), the CMF_FD_B acceptance rule, the hops
    V and V2, the block counts and the column tiles of fd_cols_h / fd_cols_w."""
    Kq = 64 if K <= 64 else 128
    B0 = 64
    while B0 < 8 * L and B0 < 1024:
        B0 *= 2
    while B0 < 4 * L:
        B0 *= 2
    natural = B0
    eligible = B0 // 2 >= 4 * L and B0 // 2 >= 64

    def work(B):
        nb = cdiv(T, B - L + 1)
        return (B // 2 + 1) * (cdiv(nb, BN) * BN + cdiv(nb, 16) * 16)

    halved = eligible and work(B0) > 0.97 * work(B0 // 2)
    if halved:
        B0 //= 2
    accepted = forced >= 4 * L and forced >= 64 and forced <= 1024 and forced & (forced - 1) == 0
    B = forced if accepted else B0
    V, V2 = B - L + 1, B - 2 * L + 2
    nblk = cdiv(T, V)
    cols = 8 if B >= 1024 else 16
    return dict(Kq=Kq, B0=natural, eligible=eligible, halved=halved, natural=B0, forced=accepted, B=B, V=V, V2=V2,
                nblk=nblk, nblkp=cdiv(nblk, 16) * 16, nblk2=cdiv(T, V2), cols_h=cols, cols_w=cols,
                numH_tiles=cdiv(cdiv(nblk, 16) * 16, BN))


def tc_plan(N, T, K, L, num_sms=NUM_SMS):
    """tc_setup (cmf_sm100.cu) for one shard of T columns: Kp, G, KLp, the tiles of the correlation, its split (the most
    even fill of num_sms persistent CTAs over 1..16 splits of >= FLUSH_T columns), the Gram's split (enough to fill the
    machine twice, at most tau / FLUSH_T) and, per split, the flush segments of n_segments / segment_kb (kernels_tc.cuh)."""
    Kp = cdiv(K, 8) * 8
    G = 128 // Kp
    KLp = cdiv(L * Kp, 64) * 64
    tiles_m, tiles_n = cdiv(KLp, BM), cdiv(N, BN)
    tau = T + L - 1
    best, nsplit, split_len = -1.0, 1, tau
    for ns in range(1, 17):
        sl = cdiv(cdiv(tau, ns), BK) * BK
        if ns > 1 and sl < FLUSH_T:
            break
        units = tiles_m * tiles_n * cdiv(tau, sl)
        eff = units / (cdiv(units, num_sms) * num_sms)
        if eff > best + 1e-9:
            best, nsplit, split_len = eff, cdiv(tau, sl), sl
    ns_g = min(max(1, cdiv(2 * num_sms, tiles_m)), max(1, tau // FLUSH_T))
    split_len_g = cdiv(cdiv(tau, ns_g), BK) * BK

    def segments(nsp, sl):
        out = []
        for sp in range(nsp):
            ta, tb = sp * sl, min(tau, (sp + 1) * sl)
            out.append([min(FLUSH_T, tb - a) for a in range(ta, tb, FLUSH_T)])
        return out

    return dict(Kp=Kp, G=G, KLp=KLp, tiles_m=tiles_m, tiles_n=tiles_n, nsplit=nsplit, split_len=split_len,
                nsplit_g=cdiv(tau, split_len_g), split_len_g=split_len_g, segments=segments(nsplit, split_len),
                segments_g=segments(cdiv(tau, split_len_g), split_len_g))


# ------------------------------------------------------------------------------------------ cases
# engine 2: (N, T, K, L, CMF_FD_B or 0)
FD_CASES = [
    (264, 230000, 16, 100, 0),     # B 1024 kept by the short-shard rule, Kq 64, 8-column tiles, two N tiles
    (136, 240000, 8, 150, 0),      # B 1024, 275 blocks (two block tiles of the numH product), V2 726
    (256, 20000, 100, 200, 0),     # B 1024, Kq 128
    (128, 20000, 8, 256, 0),       # L 256: B 1024 = 4L, V 769, V2 514
    (256, 40000, 128, 32, 0),      # config-5 components: B 256, Kq 128
    (200, 60000, 72, 64, 0),       # B 512 kept by the short-shard rule, Kq 128
    (200, 60000, 72, 64, 256),     # forced B 256 = 4L instead of 512: V2 130, 311 blocks
]
# engine 1: (N, T, K, L).  T = 200023 rather than a T that leaves a data k-block of a few columns: the last k-block holds
# 23 columns of data, enough for its loss to stand above the bar (test_case_lists_reach_every_regime).
TC_CASES = [
    (264, 200023, 20, 7),          # 3 splits x 2 segments, last segment 1117 columns, G 5, N ragged over two tiles
    (136, 140000, 128, 32),        # config-5 components: G 1, 2 splits x 2 segments
    (128, 131100, 64, 4),          # split_len 65568: split 0 ends in a one-k-block segment, split 1 has one segment
    (512, 150000, 8, 33),          # G 16, 2 splits
]
FIXTURE_FORCED_B = {"c4shape": 1024, "c3shape": 512}     # the block lengths the benchmark runs at c4 / c3
FIXTURE_DIMS = {"c4shape": (256, 8192, 64, 100), "c3shape": (256, 16384, 20, 50)}
HALS_C5 = (136, 3000, 128, 32)
HALS_C5_B = 256                                          # the block length config 5 runs at


def case_data(N, T, K, L):
    """W, H, X drawn in float32 (then held as float64: the values both sides see)."""
    rng = np.random.default_rng(N * 7 + T * 3 + K * 5 + L)
    return tuple(rng.random(shape, dtype=np.float32).astype(np.float64) for shape in ((K, N, L), (K, T), (N, T)))


def kblock_sensitivity(H, X, numW_max):
    """Lower bound, over the data-bearing 32-column k-blocks b of the correlation's t range, of the change of the float64
    numW if k-block b were left out, relative to max |numW|: the lag-0 part sum_{s in b} H[k, s] X[n, s], max over (k, n)."""
    K, T = H.shape
    worst = np.inf
    nb = cdiv(T, BK)
    Hp = np.zeros((K, nb * BK)); Hp[:, :T] = H
    Xp = np.zeros((X.shape[0], nb * BK)); Xp[:, :T] = X
    for b0 in range(0, nb, 512):
        b1 = min(nb, b0 + 512)
        Hb = Hp[:, b0 * BK : b1 * BK].reshape(K, b1 - b0, BK).transpose(1, 0, 2)
        Xb = Xp[:, b0 * BK : b1 * BK].reshape(-1, b1 - b0, BK).transpose(1, 2, 0)
        d = np.matmul(Hb, Xb)                                     # [block][k][n]
        worst = min(worst, float(np.abs(d).reshape(b1 - b0, -1).max(axis=1).min()))
    return worst / numW_max


def test_case_lists_reach_every_regime():
    fd = [fd_plan(*c) for c in FD_CASES]
    # engine 2: Kq 128 at B 256 / 512 / 1024, Kq 64 at 1024, both column tiles, L = 256 at B = 4L
    assert {p["B"] for p in fd if p["Kq"] == 128} >= {256, 512, 1024}
    assert any(p["B"] == 1024 and p["Kq"] == 64 for p in fd)
    assert {p["cols_h"] for p in fd} == {8, 16}
    assert any(L == 256 and p["B"] == 4 * L and (p["V"], p["V2"]) == (769, 514) for (_, _, _, L, _), p in zip(FD_CASES, fd))
    # more than 256 blocks (two block tiles of the numH product) at B 1024, and at Kq 128
    assert any(p["B"] == 1024 and p["nblk"] > 256 and p["numH_tiles"] == 2 for p in fd)
    assert any(p["Kq"] == 128 and p["nblk"] > 256 for p in fd)
    # the short-shard rule: eligible and keeping B0; a forced B that differs from the natural one
    assert any(p["eligible"] and not p["halved"] and p["B"] == p["B0"] == 1024 for p in fd)
    assert any(p["eligible"] and not p["halved"] and p["B"] == p["B0"] == 512 and p["Kq"] == 128 for p in fd)
    forced = [p for p in fd if p["forced"]]
    assert forced and all(p["B"] != p["natural"] for p in forced)
    assert fd_plan(200, 60000, 72, 64, 256)["V2"] == 130 and fd_plan(200, 60000, 72, 64, 256)["nblk"] == 311
    # ... and halving the fixture dims: the fits at the benchmark's block length must force it
    for name, B in FIXTURE_FORCED_B.items():
        p = fd_plan(*FIXTURE_DIMS[name])
        assert p["halved"] and p["natural"] == B // 2 and p["B0"] == B and fd_plan(*FIXTURE_DIMS[name], B)["B"] == B
    assert fd_plan(*HALS_C5)["natural"] == HALS_C5_B // 2 and fd_plan(*HALS_C5, HALS_C5_B)["B"] == HALS_C5_B
    # CMF_FD_B values outside the acceptance rule are ignored
    assert not fd_plan(128, 20000, 8, 256, 512)["forced"] and not fd_plan(64, 5000, 4, 5, 96)["forced"]
    # engine 1: several splits of the correlation and of the Gram, every split of several segments, a one-k-block segment
    tc = [tc_plan(*c) for c in TC_CASES]
    assert all(p["nsplit"] >= 2 and p["nsplit_g"] >= 2 for p in tc)
    assert any(all(len(s) >= 2 for s in p["segments"]) for p in tc)
    assert any(s[-1] == BK and len(s) >= 2 for p in tc for s in p["segments"])
    assert {p["G"] for p in tc} >= {1, 5, 16}
    assert any(N > BN and N % BN and p["tiles_n"] == 2 for (N, _, _, _), p in zip(TC_CASES, tc))
    assert tc[0]["nsplit"] == 3 and [len(s) for s in tc[0]["segments"]] == [2, 2, 2]
    assert tc_plan(128, 131100, 64, 4)["split_len"] == 65568
    assert [len(s) for s in tc_plan(128, 131100, 64, 4)["segments"]] == [2, 1]
    # sensitivity: leaving out any data-bearing k-block moves the reference numW by more than 3x the bar
    for dims in TC_CASES:
        W, H, X = case_data(*dims)
        numW_max = float(np.abs(lr.corr_w(H, X, dims[3])).max())
        assert kblock_sensitivity(H, X, numW_max) > 3 * CONTRACTION_TOL, dims


# ------------------------------------------------------------------------------------------ GPU fixtures and helpers
@pytest.fixture(scope="module")
def cmf():
    import __graft_entry__ as ge

    ge.build()
    import cmf_jl_b200

    return cmf_jl_b200


@pytest.fixture(scope="module")
def refs():
    """float64 references per shape, each computed once: sum of squared residuals, numW, Gram partial, numH, denomH."""
    cache = {}

    def get(dims):
        if dims not in cache:
            N, T, K, L = dims
            W, H, X = case_data(*dims)
            cache[dims] = dict(W=W, H=H, X=X, ss=lr.sumsq_resid(W, H, X), numW=lr.corr_w(H, X, L), gram=lr.gram_R(H, L),
                               numH=lr.transconv(W, X), denH=lr.denom_h(W, H))
        return cache[dims]

    return get


def _scale_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


def _numW(s, N, K, L):
    import torch

    torch.cuda.synchronize()
    return s.exchange[0].cpu().numpy().reshape(L, K, N).transpose(1, 2, 0).copy()


def _check_contractions(s, ref, dims, numW_again):
    """Loss, numW (and its repeats, bitwise), Gram partial, numH and denomH of one handle against the reference."""
    import torch

    N, T, K, L = dims
    s.set_data(ref["X"], 0)
    s.set_factors(ref["W"], ref["H"], 0)
    s.set_data_norm(1.0)
    s.set_loss_mode(0)
    got_ss = s.loss_partial()
    assert abs(got_ss - ref["ss"]) < LOSS_TOL * ref["ss"], (got_ss, ref["ss"])
    s.w_partials()
    numW = _numW(s, N, K, L)
    assert _scale_err(numW, ref["numW"]) < CONTRACTION_TOL
    Rg = s.exchange[1].cpu().numpy()[: L * K * K].reshape(L, K, K).transpose(1, 2, 0)
    assert _scale_err(Rg, ref["gram"]) < CONTRACTION_TOL
    for setup in numW_again:
        setup()
        s.w_partials()
        assert np.array_equal(_numW(s, N, K, L), numW), setup.__doc__
    s.h_update(0.0, 0.0)
    torch.cuda.synchronize()
    numH = s.exchange[2].cpu().numpy().reshape(T, K).T
    assert _scale_err(numH, ref["numH"]) < CONTRACTION_TOL
    denH = s.exchange[3].cpu().numpy().reshape(T, K).T
    assert _scale_err(denH, ref["denH"]) < CONTRACTION_TOL
    if L > 1:    # the truncated tail on its own scale
        assert _scale_err(denH[:, T - L + 1 :], ref["denH"][:, T - L + 1 :]) < CONTRACTION_TOL


# ------------------------------------------------------------------------------------------ contractions
@gpu
@pytest.mark.parametrize("case", FD_CASES, ids=["x".join(map(str, c[:4])) + (f"-B{c[4]}" if c[4] else "") for c in FD_CASES])
def test_fd_contractions_at_plan(cmf, refs, case, monkeypatch):
    dims, forced = case[:4], case[4]
    if forced:
        monkeypatch.setenv("CMF_FD_B", str(forced))
    else:
        monkeypatch.delenv("CMF_FD_B", raising=False)
    p = fd_plan(*case)
    ref = refs(dims)
    s = cmf.DeviceShard(*dims[:2], 0, dims[1], *dims[2:], dtype="f32", device=0)
    try:
        s.set_engine(2)
        assert s.get_engine() == 2
        assert s.fd_layout() == (p["B"], p["V"], p["nblkp"])

        def again():
            """numW on a second run"""

        _check_contractions(s, ref, dims, [again])
    finally:
        s.close()


@gpu
@pytest.mark.parametrize("dims", TC_CASES, ids=lambda d: "x".join(map(str, d)))
def test_tc_contractions_at_plan(cmf, refs, dims, monkeypatch):
    monkeypatch.delenv("CMF_LOCKSTEP", raising=False)
    ref = refs(dims)
    s = cmf.DeviceShard(*dims[:2], 0, dims[1], *dims[2:], dtype="f32", device=0)
    try:
        s.set_engine(1)
        assert s.get_engine() == 1 and s.fd_layout() == (0, 0, 0)

        def again():
            """numW on a second run"""

        def no_lockstep():
            """numW without the lock-step window (CMF_LOCKSTEP=0)"""
            monkeypatch.setenv("CMF_LOCKSTEP", "0")

        _check_contractions(s, ref, dims, [again, no_lockstep])
    finally:
        s.close()


# ------------------------------------------------------------------------------------------ whole fits
def _fixture(case):
    if GOLD not in sys.path:
        sys.path.insert(0, GOLD)
    import make_golden_bench_shape as mg

    g = np.load(os.path.join(GOLD, f"mu_bench_{case}.npz"))
    X, W0, H0 = mg.inputs(case)
    assert abs(float(np.linalg.norm(X)) - float(g["X_norm"])) < 1e-9 * float(g["X_norm"])
    return g, X, W0, H0


def _forced_layout(cmf, dims, B):
    N, T, K, L = dims
    s = cmf.DeviceShard(N, T, 0, T, K, L, dtype="f32", device=0)
    try:
        s.set_engine(2)
        return s.fd_layout()
    finally:
        s.close()


@gpu
@pytest.mark.parametrize("case", ["c4shape_dense", "c4shape_sparse", "c3shape_dense", "c3shape_sparse"])
@pytest.mark.parametrize("loss_mode", [1, 0])
def test_mu_100_iterations_at_benchmark_block_length(cmf, case, loss_mode, monkeypatch):
    shape = case.split("_")[0]
    B = FIXTURE_FORCED_B[shape]
    monkeypatch.setenv("CMF_FD_B", str(B))
    g, X, W0, H0 = _fixture(case)
    N, T, K, L = (int(v) for v in g["dims"])
    assert (N, T, K, L) == FIXTURE_DIMS[shape]
    p = fd_plan(N, T, K, L, B)
    assert _forced_layout(cmf, (N, T, K, L), B) == (B, p["V"], p["nblkp"])
    ref = np.asarray(g["loss_hist"])
    r = cmf.fit_cnmf(X, L=L, K=K, alg="mult", max_itr=int(g["iters"]), W_init=W0, H_init=H0, check_convergence=False,
                     layout="KNL", dtype="f32", engine=2, loss_mode=loss_mode)
    assert r.engine_info["engine"] == 2
    got = np.asarray(r.loss_hist)
    assert got.shape == ref.shape
    rel = np.abs(got - ref) / ref
    assert rel.max() < 1e-4, (case, loss_mode, int(rel.argmax()), float(rel.max()))


@gpu
def test_calibrated_expansion_at_block_length_1024(cmf, monkeypatch):
    monkeypatch.setenv("CMF_FD_B", "1024")
    g, X, W0, H0 = _fixture("c4shape_sparse")
    N, T, K, L = (int(v) for v in g["dims"])
    assert _forced_layout(cmf, (N, T, K, L), 1024)[0] == 1024
    ref = np.asarray(g["loss_hist"])
    r = cmf.fit_cnmf(X, L=L, K=K, alg="mult", max_itr=int(g["iters"]), W_init=W0, H_init=H0, check_convergence=False,
                     layout="KNL", dtype="f32", engine=2, loss_mode=1, loss_guard=1e30)
    rel = np.abs(np.asarray(r.loss_hist) - ref) / ref
    info = r.engine_info
    assert rel.max() < 1e-4, (int(rel.argmax()), float(rel.max()), info)
    assert info["loss_mode"] == 1 and info["engine"] == 2, info
    assert info["direct"] <= 0.5 * info["expansion"], info
    assert info["last_err"] < 1e-4 and info["interval"] >= 2, info


@pytest.fixture(scope="module")
def hals_c5():
    """HALS at the config-5 component shape, data built as in test_gpu_parity.py's c5shape, 10 iterations of the C oracle."""
    from oracle import c_oracle as co
    from oracle import cnmf_oracle as po

    N, T, K, L = HALS_C5
    X, _, _ = po.synthetic_sequences(K=6, N=N, L=L, T=T, p_h=0.3, noise_scale=0.5, rng=np.random.default_rng(5))
    W0, H0 = po.init_rand(X, L, K, np.random.default_rng(6))
    reg = dict(l1W=0.05, l2W=0.1, l1H=0.05, l2H=0.1)
    ref = co.fit(co.HALSUpdate, X, W0, H0, 10, check_convergence=False, **reg)
    return X, W0, H0, reg, ref


@gpu
@pytest.mark.parametrize("engine", [1, 2])
def test_hals_c5_component_shape_on_tensor_engines(cmf, hals_c5, engine, monkeypatch):
    X, W0, H0, reg, ref = hals_c5
    N, T, K, L = HALS_C5
    if engine == 2:
        monkeypatch.setenv("CMF_FD_B", str(HALS_C5_B))
        p = fd_plan(N, T, K, L, HALS_C5_B)
        assert _forced_layout(cmf, HALS_C5, HALS_C5_B) == (HALS_C5_B, p["V"], p["nblkp"])
    r = cmf.fit_cnmf(X, L=L, K=K, alg="hals", max_itr=10, W_init=W0, H_init=H0, check_convergence=False, layout="KNL",
                     dtype="f32", engine=engine, **reg)
    assert r.engine_info["engine"] == engine
    rel = np.abs(np.asarray(r.loss_hist) - np.asarray(ref.loss_hist)) / np.asarray(ref.loss_hist)
    assert rel.max() < 1e-4, rel
