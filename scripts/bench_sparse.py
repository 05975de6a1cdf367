"""Sparse data against dense: MultUpdate / HALS fits on CSC matrices (cmf_create_sparse) and on the same data as a dense
array (cmf_create), at spike-like densities.  Writes one JSON file.

Data: the convolutive model with sparse ground truth (K_true = 8 components, each on a quarter of the units at 4 random lags,
Bernoulli activations), computed as a sparse product on the host from a fixed seed, then Bernoulli-thinned to the target
density rho.  Case 3 (a shape whose dense X does not fit one GPU) draws a spike raster directly instead (a fixed number of
distinct random units per bin): the host product would need more memory than the measurement.

Cases:
  1. c3 shape (N=1024, T=2^20, K=20, L=50), fp32 and fp64, rho in {0.1 %, 1 %, 5 %}: ms per MU and per HALS iteration of the
     sparse handle; the mean PROF_CORR (numW) and PROF_TRANSCONV (numH) launch times of the sparse handle and of a dense
     handle of the same data on engine 0 and, for fp32, on engine 2; device memory in use with the sparse handle alone; the
     largest relative loss_hist difference between the sparse and dense (engine 0) MU fits from the same start.
  2. config-1 shape at T = 50 000 (N=500, L=10), fp64, rho = 1 %: fit_cnmf_batch rank sweep K = 1..10 x 8 seeds, sparse
     against dense, wall time and the largest relative loss_hist difference.
  3. N=4096, T=2^24, K=16, L=32, fp32, ~0.15 %: ms per MU iteration and device memory in use (dense X: 275 GB).
The card's name and power limit are read in the same run."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as ge  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clk = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def model_data(N, T, rho, seed=1234, K_true=8, L_true=4, Lmax=50):
    """Sparse conv(W, H) of a sparse ground truth, thinned to density rho (scipy CSC, float64)."""
    import scipy.sparse as sp

    rng = np.random.default_rng(seed)
    p_h = -np.log(1 - min(2.5 * rho, 0.5)) / (K_true * 0.25 * L_true)   # raw density ~2.5 rho before the thinning
    H = sp.random(K_true, T, density=p_h, random_state=rng, format="csc", data_rvs=lambda n: rng.exponential(1.0, n))
    X = None
    for k in range(K_true):
        units = rng.choice(N, size=N // 4, replace=False)
        for lag in rng.choice(Lmax, size=L_true, replace=False):
            Wl = sp.csc_matrix((rng.random(len(units)) + 0.2, (units, np.zeros(len(units), dtype=np.int64))), shape=(N, 1))
            Hk = H[k:k + 1, : T - lag]
            Hs = sp.hstack([sp.csc_matrix((1, lag)), Hk], format="csc") if lag else H[k:k + 1]
            term = (Wl @ Hs).tocsc()
            X = term if X is None else X + term
    X = X.tocsc()
    X.sum_duplicates()
    keep = rng.random(X.nnz) < rho / (X.nnz / (N * T))
    X.data = np.where(keep, X.data, 0.0)
    X.eliminate_zeros()
    return X


def raster(N, T, per_col, seed=0):
    """per_col distinct random units per bin (CSC arrays, 0-based)."""
    rng = np.random.default_rng(seed)
    gaps = rng.integers(1, max(2, (N - 1) // per_col), size=(T, per_col))
    gaps[:, 0] = rng.integers(0, max(2, (N - 1) // per_col), size=T)
    rowval = np.cumsum(gaps, axis=1).ravel()
    colptr = np.arange(0, T * per_col + 1, per_col, dtype=np.int64)
    return colptr, rowval, rng.random(T * per_col, dtype=np.float32)


def mem_in_use():
    import torch

    free, total = torch.cuda.mem_get_info()
    return int(total - free)


class Handle:
    """A single-handle fit through the C ABI with device-side uniform init and the alpha rescale."""

    def __init__(self, cmf, N, T, K, L, dtype, alg, sparse_csc=None, dense=None):
        self.cmf, self.lib, self._l = cmf, cmf._lib.load(), cmf._lib
        self.dt = self._l.parse_dtype(dtype)
        self.h = ctypes.c_void_p()
        if sparse_csc is not None:
            self._l.check(self.lib.cmf_create_sparse(ctypes.byref(self.h), N, T, K, L, self.dt, alg, 0))
            i64 = ctypes.POINTER(ctypes.c_int64)
            colptr, rowval, nzval = sparse_csc
            nz = np.ascontiguousarray(nzval, dtype=self._l.np_dtype(self.dt))
            self._l.check(self.lib.cmf_set_data_csc(self.h, len(nz), colptr.ctypes.data_as(i64), rowval.ctypes.data_as(i64),
                                                    self._l.fptr(nz), 0))
        else:
            self._l.check(self.lib.cmf_create(ctypes.byref(self.h), N, T, K, L, self.dt, alg, 0))
            self._l.check(self.lib.cmf_set_data(self.h, self._l.fptr(self._l.julia_array(dense, self.dt)), 0))

    def engine(self, e):
        self._l.check(self.lib.cmf_set_engine(self.h, e))
        if e == 0:
            self._l.check(self.lib.cmf_set_loss_mode(self.h, 0))   # engine 0 of a dense handle: the direct loss

    def init(self, seed=7):
        self._l.check(self.lib.cmf_init_rand(self.h, seed))
        part = (ctypes.c_double * 2)()
        self._l.check(self.lib.cmf_init_scale_partials(self.h, part))
        self._l.check(self.lib.cmf_scale_factors(self.h, float(np.sqrt(abs(part[0] / part[1])))))

    def fit(self, itr, profile=False):
        """(loss_hist, ms per iteration, {class: mean ms per launch})."""
        if profile:
            self._l.check(self.lib.cmf_profile(self.h, 1))
        lh, th = np.zeros(itr + 1), np.zeros(itr + 1)
        n, e = ctypes.c_int64(), ctypes.c_int()
        dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))  # noqa: E731
        self._l.check(self.lib.cmf_sync(self.h))
        t0 = time.perf_counter()
        self._l.check(self.lib.cmf_fit(self.h, itr, 1e300, 0, 0, 3, 1e-4, 0.0, 0.0, 0.0, 0.0, dp(lh), dp(th), itr + 1,
                                       ctypes.byref(n), ctypes.byref(e)))
        self._l.check(self.lib.cmf_sync(self.h))
        ms = (time.perf_counter() - t0) * 1e3 / itr
        prof = {}
        if profile:
            for name, which in (("numH", 1), ("numW", 2)):
                tot, cnt = ctypes.c_double(), ctypes.c_int64()
                self._l.check(self.lib.cmf_profile_read(self.h, which, ctypes.byref(tot), ctypes.byref(cnt)))
                prof[name] = tot.value / max(cnt.value, 1)
            self._l.check(self.lib.cmf_profile(self.h, 0))
        return lh[: n.value].tolist(), ms, prof

    def close(self):
        self.lib.cmf_destroy(self.h)


def case_c3(cmf, dtype, rho, itr):
    N, T, K, L = 1024, 1 << 20, 20, 50
    X = model_data(N, T, rho)
    csc = (X.indptr.astype(np.int64), X.indices.astype(np.int64), X.data)
    out = {"case": "c3", "dtype": dtype, "rho": X.nnz / (N * T), "nnz": int(X.nnz), "N": N, "T": T, "K": K, "L": L}
    base = mem_in_use()
    for alg, name in ((0, "mu"), (1, "hals")):
        h = Handle(cmf, N, T, K, L, dtype, alg, sparse_csc=csc)
        if alg == 0:
            out["device_bytes_sparse_handle"] = mem_in_use() - base
        h.init()
        h.fit(1)                                                     # warm-up
        h.init()
        lh, ms, prof = h.fit(itr, profile=(alg == 0))
        out[f"sparse_{name}_ms_per_iter"] = ms
        if alg == 0:
            out["sparse_numW_ms"], out["sparse_numH_ms"] = prof["numW"], prof["numH"]
            sparse_hist = lh
        h.close()
    D = X.toarray()
    del X
    engines = (0, 2) if dtype == "f32" else (0,)
    h = Handle(cmf, N, T, K, L, dtype, 0, dense=D)
    del D
    for e in engines:
        h.engine(e)
        h.init()
        h.fit(1)
        h.init()
        lh, ms, prof = h.fit(itr, profile=True)
        out[f"dense_e{e}_mu_ms_per_iter"] = ms
        out[f"dense_e{e}_numW_ms"], out[f"dense_e{e}_numH_ms"] = prof["numW"], prof["numH"]
        if e == 0:
            out["max_rel_loss_diff_vs_dense_e0"] = float(np.max(np.abs(np.array(sparse_hist) - lh) / np.array(lh)))
    h.close()
    return out


def case_sweep(cmf, itr):
    N, T, L = 500, 50_000, 10
    X = model_data(N, T, 0.01, Lmax=L)
    ranks = [k for k in range(1, 11) for _ in range(8)]
    seeds = list(range(len(ranks)))
    out = {"case": "config1_T50k_rank_sweep", "dtype": "f64", "rho": X.nnz / (N * T), "N": N, "T": T, "L": L, "R": len(ranks)}
    kw = dict(L=L, K=ranks, seeds=seeds, max_itr=itr, check_convergence=False, dtype="f64")
    cmf.fit_cnmf_batch(X, **dict(kw, max_itr=1))                    # warm-up
    t0 = time.perf_counter()
    s = cmf.fit_cnmf_batch(X, **kw)
    out["sparse_s"] = time.perf_counter() - t0
    D = X.toarray()
    cmf.fit_cnmf_batch(D, **dict(kw, max_itr=1))
    t0 = time.perf_counter()
    d = cmf.fit_cnmf_batch(D, **kw)
    out["dense_s"] = time.perf_counter() - t0
    out["speedup"] = out["dense_s"] / out["sparse_s"]
    out["max_rel_loss_diff"] = max(float(np.max(np.abs(np.array(a.loss_hist) - b.loss_hist) / np.array(b.loss_hist)))
                                   for a, b in zip(s, d))
    return out


def case_big(cmf, itr):
    N, T, K, L, per_col = 4096, 1 << 24, 16, 32, 6
    csc = raster(N, T, per_col)
    out = {"case": "beyond_dense", "dtype": "f32", "N": N, "T": T, "K": K, "L": L, "nnz": int(len(csc[2])),
           "rho": per_col / N, "dense_X_bytes": N * T * 4}
    base = mem_in_use()
    h = Handle(cmf, N, T, K, L, "f32", 0, sparse_csc=csc)
    del csc
    h.init()
    out["device_bytes_sparse_handle"] = mem_in_use() - base
    h.fit(1)
    h.init()
    lh, ms, prof = h.fit(itr, profile=True)
    out.update(mu_ms_per_iter=ms, numW_ms=prof["numW"], numH_ms=prof["numH"], loss_hist=lh)
    h.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--itr", type=int, default=5)
    ap.add_argument("--cases", default="c3,sweep,big")
    ap.add_argument("--rhos", default="0.001,0.01,0.05")
    args = ap.parse_args()
    ge.build()
    import cmf_jl_b200 as cmf

    res = {"card": card(), "itr": args.itr, "runs": []}

    def save():
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)

    cases = args.cases.split(",")
    if "c3" in cases:
        for dtype in ("f32", "f64"):
            for rho in (float(r) for r in args.rhos.split(",")):
                res["runs"].append(case_c3(cmf, dtype, rho, args.itr))
                print(json.dumps(res["runs"][-1]), flush=True)
                save()
    if "sweep" in cases:
        res["runs"].append(case_sweep(cmf, 20))
        print(json.dumps(res["runs"][-1]), flush=True)
        save()
    if "big" in cases:
        res["runs"].append(case_big(cmf, 3))
        print(json.dumps(res["runs"][-1]), flush=True)
        save()


if __name__ == "__main__":
    main()
