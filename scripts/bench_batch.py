"""Batched restarts against serial fits: R MultUpdate fits of one data set as R separate fit_cnmf calls and as one
fit_cnmf_batch call, at the config-1 shape (N=500, T=2000, K=5, L=10) and at the top of the reference's T sweep
(N=500, T=50 000), fp64 and fp32, R in {1, 8, 64, 256}, 100 iterations without early stop.  Writes one JSON file.

Per run: fits/s of both arms and the speed-up; device time per batched iteration (CUDA events on the handle's stream around
cmf_fit_batch, so it includes the per-iteration loss read-back); launches per iteration; the largest relative loss_hist
difference between batched and serial restarts with the same seeds.  The serial arm times min(R, --serial-max) fits (fits/s
is a rate; the cap keeps the large shape's R = 256 run short).  The card's name and power limit are read in the same run.

--ranks K1,K2,... runs a rank sweep instead: --per-rank seeds for every rank (default K = 1..10 x 8 seeds, R = 80,
sum K = 440), all of them as serial fit_cnmf calls (no cap) against one fit_cnmf_batch(K=[...]) call."""
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

SHAPES = {"config1": dict(N=500, T=2000, K=5, L=10), "T50k": dict(N=500, T=50_000, K=5, L=10)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power}


def device_run(cmf, X, K, L, R, dtype, itr):
    """Device time and launches per iteration of one batch handle (random factors; the arithmetic does not depend on them).
    K: one rank for every restart (cmf_create_batch), or a list of R ranks (cmf_create_batch_ranks)."""
    import torch

    lib, _lib = cmf._lib.load(), cmf._lib
    N, T = X.shape
    dt = _lib.parse_dtype(dtype)
    h = ctypes.c_void_p()
    if isinstance(K, int):
        _lib.check(lib.cmf_create_batch(ctypes.byref(h), N, T, K, L, dt, 0, R, 0))
        C = K * R
    else:
        _lib.check(lib.cmf_create_batch_ranks(ctypes.byref(h), N, T, (ctypes.c_int64 * R)(*K), L, dt, 0, R, 0))
        C = sum(K)
    try:
        rng = np.random.default_rng(0)
        _lib.check(lib.cmf_set_data(h, _lib.fptr(_lib.julia_array(X, dt)), 0))
        W = _lib.julia_array(rng.random(C * N * L), dt)
        H = _lib.julia_array(rng.random(C * T), dt)
        _lib.check(lib.cmf_set_factors_batch(h, _lib.fptr(W), _lib.fptr(H)))
        sp = ctypes.c_void_p()
        _lib.check(lib.cmf_stream(h, ctypes.byref(sp)))
        stream = torch.cuda.ExternalStream(sp.value)
        z = np.zeros(R)
        p = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))  # noqa: E731
        cap = itr + 1
        lh, th = np.zeros(R * cap), np.zeros(cap)
        n, e = np.zeros(R, dtype=np.int64), np.zeros(R, dtype=np.int32)

        def fit(k):
            _lib.check(lib.cmf_fit_batch(h, k, float("inf"), 0, 0, 3, 1e-4, p(z), p(z), p(z), p(z), p(lh), p(th), cap,
                                         n.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), e.ctypes.data_as(ctypes.POINTER(ctypes.c_int))))

        c = [ctypes.c_int64() for _ in range(3)]
        _lib.check(lib.cmf_launch_count(h, ctypes.byref(c[0])))
        fit(1)
        _lib.check(lib.cmf_launch_count(h, ctypes.byref(c[1])))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fit(itr)
        b.record(stream)
        b.synchronize()
        _lib.check(lib.cmf_launch_count(h, ctypes.byref(c[2])))
        launches = ((c[2].value - c[1].value) - (c[1].value - c[0].value)) / (itr - 1)
        return a.elapsed_time(b) / itr, launches
    finally:
        lib.cmf_destroy(h)


def sweep(cmf, X, sname, N, T, L, dtype, args):
    """One rank sweep: every (rank, seed) pair as a serial fit_cnmf call and all of them as one fit_cnmf_batch call."""
    ranks = [int(k) for k in args.ranks.split(",")]
    ks = [k for k in ranks for _ in range(args.per_rank)]
    seeds = list(range(len(ks)))
    R = len(ks)
    kw = dict(L=L, max_itr=args.itr, check_convergence=False, dtype=dtype)
    for k in sorted(set(ks)):                                                                   # warm-up of every shape
        cmf.fit_cnmf(X, K=k, seed=0, **{**kw, "max_itr": 3})
    cmf.fit_cnmf_batch(X, K=ks[:2], seeds=[0, 1], **{**kw, "max_itr": 3})
    t0 = time.perf_counter()
    serial = [cmf.fit_cnmf(X, K=k, seed=sd, **kw) for k, sd in zip(ks, seeds)]
    t_serial = time.perf_counter() - t0
    t0 = time.perf_counter()
    batch = cmf.fit_cnmf_batch(X, K=ks, seeds=seeds, **kw)
    t_batch = time.perf_counter() - t0
    diff = max(float(np.max(np.abs(np.asarray(b.loss_hist) - np.asarray(a.loss_hist)) / np.asarray(a.loss_hist)))
               for a, b in zip(serial, batch))
    ms_it, launches = device_run(cmf, X, ks, L, R, dtype, args.itr)
    run = dict(shape=sname, N=N, T=T, L=L, dtype=dtype, ranks=ranks, per_rank=args.per_rank, R=R, C=sum(ks),
               serial_fits_timed=R, serial_fits_per_s=R / t_serial, batched_fits_per_s=R / t_batch,
               speedup=t_serial / t_batch, batched_device_ms_per_iter=ms_it, launches_per_iter=launches,
               max_rel_loss_diff=diff)
    print(json.dumps(run), flush=True)
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--itr", type=int, default=100)
    ap.add_argument("--restarts", default="1,8,64,256")
    ap.add_argument("--shapes", default="config1,T50k")
    ap.add_argument("--dtypes", default="f64,f32")
    ap.add_argument("--serial-max", type=int, default=64)
    ap.add_argument("--ranks", help="comma-separated ranks: run a rank sweep (e.g. 1,2,3,4,5,6,7,8,9,10)")
    ap.add_argument("--per-rank", type=int, default=8, help="seeds per rank of --ranks")
    args = ap.parse_args()
    ge.build()
    import cmf_jl_b200 as cmf
    from oracle import cnmf_oracle as po

    out = {"card": card(), "iterations": args.itr, "serial_max": args.serial_max, "runs": []}
    for sname in args.shapes.split(","):
        s = SHAPES[sname]
        N, T, K, L = s["N"], s["T"], s["K"], s["L"]
        X, _, _ = po.synthetic_sequences(K=3, N=N, L=20, T=T, rng=np.random.default_rng(1234))   # as scripts/configs12.py
        for dtype in args.dtypes.split(","):
            if args.ranks:
                out["runs"].append(sweep(cmf, X, sname, N, T, L, dtype, args))
                continue
            kw = dict(L=L, K=K, max_itr=args.itr, check_convergence=False, dtype=dtype)
            cmf.fit_cnmf(X, seed=0, **{**kw, "max_itr": 3})                                         # warm-up of the shape
            cmf.fit_cnmf_batch(X, seeds=[0, 1], **{**kw, "max_itr": 3})
            for R in [int(r) for r in args.restarts.split(",")]:
                seeds = list(range(R))
                ns = min(R, args.serial_max)
                t0 = time.perf_counter()
                serial = [cmf.fit_cnmf(X, seed=sd, **kw) for sd in seeds[:ns]]
                t_serial = time.perf_counter() - t0
                t0 = time.perf_counter()
                batch = cmf.fit_cnmf_batch(X, seeds=seeds, **kw)
                t_batch = time.perf_counter() - t0
                diff = max(float(np.max(np.abs(np.asarray(b.loss_hist) - np.asarray(a.loss_hist)) / np.asarray(a.loss_hist)))
                           for a, b in zip(serial, batch))
                ms_it, launches = device_run(cmf, X, K, L, R, dtype, args.itr)
                run = dict(shape=sname, N=N, T=T, K=K, L=L, dtype=dtype, R=R, serial_fits_timed=ns,
                           serial_fits_per_s=ns / t_serial, batched_fits_per_s=R / t_batch,
                           speedup=(R / t_batch) / (ns / t_serial), batched_device_ms_per_iter=ms_it,
                           launches_per_iter=launches, max_rel_loss_diff=diff)
                print(json.dumps(run), flush=True)
                out["runs"].append(run)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
