#!/usr/bin/env python
"""bench.py -- CNMF iterations/s of the B200 fit path on BASELINE.json's headline workload.

    python bench.py --gpus N --steps K --warmup W            (this repo's CUDA path)
    python bench.py --impl reference --gpus N --steps K ...  (the reference's CPU algorithm, oracle port)
    python bench.py ... --dump-outputs DIR                   (also write W, H and the losses of the timed steps as .npy)

One "step" = one full MU iteration (update_motifs! + update_feature_maps! incl. the loss,
src/algs/alternating.jl:51-54) over the whole synthetic data set.  N > 1 shards the time axis
(strong scaling: the workload is fixed, SURVEY.md section 8e).  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json configs (fp32 MU).  "c4" is the configuration the metric is quoted on; it fits
# one B200 (X = 64 GiB fp32), so it is the N=1 workload too.
CONFIGS = {
    "c4": dict(N=4096, T=1 << 22, K=64, L=100),
    "c3": dict(N=1024, T=1 << 20, K=20, L=50),
    "c1": dict(N=500, T=2000, K=5, L=10),
    "c5": dict(N=512, T=1 << 24, K=128, L=32),     # spectrogram-shaped, HALS (--alg hals)
}
SEED_DATA, SEED_INIT, P_H, NOISE = 1234, 0, 0.05, 0.1
# --dump-outputs: each factor is written whole up to DUMP_ELEMS values (24 MiB in fp32), else as a fixed, seeded sample of
# units (W) or columns (H), so that two builds run with the same arguments can be compared entry for entry
DUMP_ELEMS, DUMP_SEED = 6 << 20, 2024


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tensor_burst=d["bf16_tflops"], tensor=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor=1400.0, src="fallback")


def flops_contraction(N, T, K, L):
    return 2.0 * N * K * (L * T - L * (L - 1) / 2.0)          # SURVEY.md section 8d  F_c


def bytes_iteration(N, T, K, L, s=4):
    return s * (2.0 * N * T + 4.0 * K * T + 6.0 * K * N * L)  # SURVEY.md section 8d  B_alg


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc = gpu, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm (oracle port, NumPy/OpenBLAS per-lag GEMMs like src/common.jl)
# ------------------------------------------------------------------------------------------------
def cpu_iteration_time(cfg, T_sample, steps, warmup, threads=None):
    """Seconds per literal MU iteration (src/algs/mult.jl:23-58) on a T_sample-column slice of the
    workload (same N, K, L), Float64 like the reference, on `threads` BLAS threads (default: every host
    core, set explicitly -- launchers such as torch.distributed.run export OMP_NUM_THREADS=1)."""
    import numpy as np
    from threadpoolctl import threadpool_limits

    from oracle import cnmf_oracle as po

    with threadpool_limits(limits=threads or host_cores(), user_api="blas"):
        return _cpu_iteration_time(np, po, cfg, T_sample, steps, warmup)


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def _cpu_iteration_time(np, po, cfg, T_sample, steps, warmup):

    N, K, L = cfg["N"], cfg["K"], cfg["L"]
    rng = np.random.default_rng(SEED_DATA)
    X = rng.random((N, T_sample))
    W = rng.random((K, N, L))
    H = rng.random((K, T_sample))
    rule = po.MultUpdate.__new__(po.MultUpdate)     # skip the ctor's extra conv: we time the iteration only
    rule.data_norm = float(np.linalg.norm(X))
    rule.est = np.zeros_like(X)
    rule.resids = None
    for _ in range(warmup):
        rule.update_motifs(X, W, H)
        rule.update_feature_maps(X, W, H)
    t0 = time.perf_counter()
    for _ in range(steps):
        rule.update_motifs(X, W, H)
        rule.update_feature_maps(X, W, H)
    return (time.perf_counter() - t0) / steps


def cpu_iteration_time_hals(cfg, T_sample):
    """Seconds per literal HALS iteration (src/algs/hals.jl:31-154: rank-1 sweeps on a persistent residual) of the plain-C
    restatement (oracle/cnmf_oracle.c, OpenMP where the reference's BLAS would thread) on a T_sample-column slice."""
    import numpy as np

    from oracle import c_oracle as co

    N, K, L = cfg["N"], cfg["K"], cfg["L"]
    rng = np.random.default_rng(SEED_DATA)
    X = np.asfortranarray(rng.random((N, T_sample)))
    W = np.asfortranarray(rng.random((K, N, L)))
    H = np.asfortranarray(rng.random((K, T_sample)))
    rule = co.HALSUpdate(X, W, H)
    t0 = time.perf_counter()
    rule.update_motifs(X, W, H)
    rule.update_feature_maps(X, W, H)
    return time.perf_counter() - t0


def cpu_threads(threads=None):
    """BLAS threads actually in use inside a `threadpool_limits(threads or all cores)` region."""
    try:
        import numpy  # noqa: F401  (loads the BLAS that threadpoolctl inspects)
        from threadpoolctl import threadpool_info, threadpool_limits

        with threadpool_limits(limits=threads or host_cores(), user_api="blas"):
            return max([p.get("num_threads", 1) for p in threadpool_info() if p.get("user_api") == "blas"] or [1])
    except Exception:
        return 1


def cpu_sample_T(cfg):
    # ~10-30 s of CPU work per bounded sample: 7 contractions of 2*N*K*L*T_sample FLOP at O(100) GFLOP/s
    target_flops = 1.0e12
    per_col = 7 * 2.0 * cfg["N"] * cfg["K"] * cfg["L"]
    Ts = int(max(4 * cfg["L"], min(cfg["T"], target_flops / per_col)))
    return max(cfg["L"], (Ts // 256) * 256 or Ts)


def run_reference(args, cfg, name):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    Ts = cpu_sample_T(cfg)
    sec = cpu_iteration_time(cfg, Ts, max(args.steps, 1), max(args.warmup, 1))
    its = 1.0 / (sec * cfg["T"] / Ts)                 # cost is exactly linear in T (SURVEY.md section 8d)
    sample = f"literal MU iteration timed on a T={Ts} slice (same N,K,L), extrapolated x{cfg['T'] / Ts:.0f} to T={cfg['T']}"
    cores = cpu_threads()
    # the reference's own SLURM jobs asked for 2 CPUs (figures/fast_bcd/synthetic_run.sh:7): the same sample on 2 threads
    sec2 = cpu_iteration_time(cfg, Ts, 1, 1, threads=2)
    its2 = 1.0 / (sec2 * cfg["T"] / Ts)
    line = {
        "impl": "reference", "metric": "CNMF iterations/sec", "value": its, "unit": "iterations/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / its,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{name}: MU N={cfg['N']} T={cfg['T']} K={cfg['K']} L={cfg['L']}", "alg": "mult"},
        "cpu_baseline": {"value": its, "unit": "iterations/s", "cores": cores, "kind": "port", "sample": sample,
                         "two_threads": {"value": its2, "cores": cpu_threads(2)}},
        "e2e": {"value": its, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "Julia is not installed in this image, so the reference itself cannot run; this is the "
                "NumPy/OpenBLAS restatement of src/algs/mult.jl (oracle/cnmf_oracle.py), same per-lag GEMM structure",
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_ours(args, cfg, name):
    import numpy as np
    import torch

    import __graft_entry__ as ge

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch multi-GPU runs with torch.distributed.run (one rank per GPU)")
    if rank == 0:
        ge.build()
    dist = None
    if world > 1:
        # keep stdout to the one JSON line: NCCL writes its version banner / warnings to stdout unless told otherwise
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        # NCCL prints its version banner to stdout while the communicator is set up: point fd 1 at stderr for that part
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    torch.cuda.set_device(local_rank)
    import cmf_jl_b200 as cmf

    N, T, K, L = cfg["N"], cfg["T"], cfg["K"], cfg["L"]
    plan = cmf.ShardPlan(T, world, L)
    t0, t1 = plan.ranges[rank]
    # collectives: "lib" = NCCL inside libcmf_sm100 (the reference-facing calls drive all ranks; one process per GPU under
    # torchrun, the 128-byte NCCL id travels over torch.distributed), "host" = the older split-phase calls with
    # torch.distributed doing the collectives between them
    def new_uid():      # an NCCL id builds ONE communicator: a fresh one per handle
        box = [cmf.DeviceShard.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        return box[0]

    have_comm = []

    def make_shard():
        if world > 1 and args.collectives == "lib":
            uid = None if have_comm else new_uid()      # later handles reuse the process's communicator
            have_comm.append(True)
            sh = cmf.DeviceShard(N, T, t0, t1, K, L, dtype="f32", device=local_rank, alg=args.alg, comm=(uid, rank, world))
        else:
            sh = cmf.DeviceShard(N, T, t0, t1, K, L, dtype="f32", device=local_rank, alg=args.alg)
        if args.engine is not None:
            sh.set_engine(args.engine)
        if args.alg == "mult":
            sh.set_loss_mode(args.loss_mode)
        if world > 1 and args.collectives == "host":
            return sh, cmf.ShardedMultFit(sh, rank, world, dist)
        return sh, cmf.LibraryFit(sh)

    shard, fitter = make_shard()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # synthetic data of BASELINE's shape, generated in HBM; random-init factors + alpha rescale
    shard.synth_data(SEED_DATA, K, L, P_H, NOISE)
    fitter.setup_data_norm()
    shard.init_rand(SEED_INIT)
    fitter.rescale_init()
    loss0 = fitter.loss()

    for _ in range(args.warmup):
        fitter.iterate()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    shard.profile(True)
    launches0 = shard.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    losses = []
    for _ in range(args.steps):
        losses.append(fitter.iterate())
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    prof = shard.profile_read()
    shard.profile(False)
    launches = shard.launch_count() - launches0
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        lt = torch.tensor([launches], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(lt)
        launches = int(lt.item())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, shard, losses, rank, world, dist)
    ms_per_step = ms / args.steps
    value = 1e3 / ms_per_step
    engine = shard.get_engine()
    fd_layout = shard.fd_layout()

    # secondary: the same iteration with the loss evaluated by the direct conv + residual pass (mult.jl:55-57 literally)
    value_direct = None
    if args.loss_mode == 1 and args.alg == "mult" and not args.no_direct:
        shard.set_loss_mode(0)
        fitter.iterate()
        barrier()
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record()
        for _ in range(args.steps):
            fitter.iterate()
        d1.record()
        barrier()
        dms = d0.elapsed_time(d1)
        if world > 1:
            t = torch.tensor([dms], dtype=torch.float64, device=f"cuda:{local_rank}")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dms = float(t.item())
        value_direct = args.steps / (dms / 1e3)
        shard.set_loss_mode(1)

    # third figure: the regime at or below the 25 % guard, where the library calibrates the expansion against the direct pass
    # every `interval` evaluations (include/cmf_sm100.h, cmf_set_loss_guard).  The guard is lifted above any loss so that this
    # workload is in that regime from the first evaluation; the interval ramps 1, 2, 4, 8, 16 over the first 31 iterations
    # (untimed), then 32 iterations = two full calibration periods are timed.
    calibrated = None
    if args.loss_mode == 1 and args.alg == "mult" and engine == 2 and not args.no_calibrated:
        shard.set_loss_guard(1e30, 16)
        for _ in range(31):
            fitter.iterate()
        barrier()
        st0 = shard.loss_stats()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(32):
            fitter.iterate()
        c1.record()
        barrier()
        cms = c0.elapsed_time(c1)
        if world > 1:
            t = torch.tensor([cms], dtype=torch.float64, device=f"cuda:{local_rank}")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            cms = float(t.item())
        st1 = shard.loss_stats()
        calibrated = {"value": 32 / (cms / 1e3), "unit": "iterations/s", "iterations": 32,
                      "direct_passes": st1["direct"] - st0["direct"], "expansion_evaluations": st1["expansion"] - st0["expansion"],
                      "interval": st1["interval"], "last_checked_prediction_rel_err": st1["last_err"],
                      "note": "loss mode 1 below the guard: expansion minus a bias measured against the direct pass every `interval` "
                              "iterations; each direct pass checks the previous bias's prediction (interval halves above 2e-5)"}
        shard.set_loss_guard(0.25, 16)

    # ---- end-to-end through the public API with HOST buffers (upload inside the timed region)
    e2e = None
    if not args.no_e2e:
        hi = min(t1 + (L - 1), T)                 # owned columns + the static right halo of X
        host = torch.empty((hi - t0, N), dtype=torch.float32, pin_memory=True)   # [t][n] == Julia N x cols
        Xh = host.numpy().T                       # N x cols, Fortran-ordered view of the pinned buffer
        shard.get_data(Xh, with_halo=True)
        # the caller's factors, also in pinned host memory: W (K x N x L) and H over this rank's columns + halos (the halo
        # columns are filled by exchange, not uploaded), Fortran-ordered float32 (what a Julia caller holds)
        lo_h, hi_h = max(t0 - (L - 1), 0), min(t1 + (L - 1), T)
        w_pin = torch.empty((L, N, K), dtype=torch.float32, pin_memory=True)
        h_pin = torch.zeros((hi_h - lo_h, K), dtype=torch.float32, pin_memory=True)
        W0, Hbuf = w_pin.numpy().T, h_pin.numpy().T          # K x N x L and K x cols, Fortran-ordered views
        shard.get_factors(out=(W0, Hbuf[:, t0 - lo_h : t0 - lo_h + (t1 - t0)]))
        we_pin = torch.empty((L, N, K), dtype=torch.float32, pin_memory=True)
        he_pin = torch.empty((t1 - t0, K), dtype=torch.float32, pin_memory=True)
        We, He = we_pin.numpy().T, he_pin.numpy().T
        shard.close()
        del shard, fitter
        torch.cuda.empty_cache()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        marks = [time.perf_counter()]

        def mark():
            torch.cuda.synchronize()
            marks.append(time.perf_counter())

        sh2, f2 = make_shard()
        sh2.set_data(Xh, t0)                      # H2D of this rank's columns from pinned host memory
        f2.setup_data_norm()
        mark()
        # factors: host W (replicated) and this rank's columns of H (+ halos are exchanged, not uploaded)
        sh2.set_factors(W0, Hbuf, lo_h)
        f2.exchange_halos()
        el = [f2.loss()]
        mark()
        for _ in range(args.steps):
            el.append(f2.iterate())               # each iteration reads its loss back (8 bytes D2H)
        mark()
        sh2.get_factors(out=(We, He))             # D2H of the result into pinned host memory
        mark()
        e1.record()
        barrier()
        ems = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ems], dtype=torch.float64, device=f"cuda:{local_rank}")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ems = float(t.item())
        h2d = (Xh.nbytes + W0.size * 4 + Hbuf.size * 4) * world / args.steps
        d2h = ((We.size + He.size) * 4 * world + 8 * (args.steps + 1)) / args.steps
        e2e = {"value": args.steps / (ems / 1e3), "unit": "iterations/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "iterations": args.steps,
               "note": "fit through the public API from pinned host buffers: one upload of X/W/H, K iterations "
                       "each reading its loss back, one download of W/H; bytes are totals divided by K",
               "final_loss": el[-1],
               "phases_s": dict(zip(("create+upload_X+norm", "upload_factors+first_loss", "iterations", "download_W_H"),
                                    [round(y - x, 4) for x, y in zip(marks[:-1], marks[1:])]))}
        sh2.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()
    Fc = flops_contraction(N, T, K, L)
    # dominant kernel = the contraction class with the largest device time in the timed region
    sweep_ms, sweep_n = prof.pop("sweep", (0.0, 0))
    dom = max(prof, key=lambda k: prof[k][0])
    dom_ms, dom_n = prof[dom]
    per_launch_ms = dom_ms / max(dom_n, 1)
    Fc_rank = Fc / world
    achieved_tf = Fc_rank / (per_launch_ms * 1e-3) / 1e12
    contr_share = sum(v[0] for v in prof.values()) / (ms_per_step * args.steps) if ms > 0 else None
    Tl = t1 - t0
    if engine == 2:
        # frequency-domain engine: the dominant kernel streams the spectrum of X once per launch and is HBM-bound.
        # Algorithmic bytes per launch (SURVEY.md section 8d, one contraction): X once + the small operand + the output,
        # in fp32; the bytes actually moved are the bf16 hi/lo spectrum planes (B/V * (B/2+1)/(B/2) ~ 1.25x of X).
        Bfft, V, nblkp = fd_layout             # asked from the library (cmf_get_fd_layout) before the handle was closed
        F = Bfft // 2 + 1
        alg_bytes = 4.0 * (N * Tl + K * Tl + K * N * L)
        moved_bytes = 4.0 * F * nblkp * 2 * N
        exec_flops = 3.0 * 2.0 * 128 * (2 * N) * nblkp * F
        achieved_gbs = alg_bytes / (per_launch_ms * 1e-3) / 1e9
        # dram__bytes_read.sum + dram__bytes_write.sum per launch from one `ncu --set full` capture of this workload
        traffic, traffic_note = None, "no ncu capture for this workload / kernel"
        if name == "c4" and world == 1 and (dom, Bfft) in NCU_TRAFFIC_C4_FD:
            traffic, traffic_note = NCU_TRAFFIC_C4_FD[(dom, Bfft)]
        roofline = {
            "bound": "hbm", "kernel": dom + (" (TC_FQT: per-frequency conj(W^) X^)" if dom == "transconv" else " (TC_FQC: per-frequency conj(H^) X^)"),
            "achieved": achieved_gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": achieved_gbs / pk["hbm"],
            "traffic": traffic, "traffic_note": traffic_note, "peak_source": f"{pk['src']} HBM copy bandwidth",
            "bytes_per_launch": alg_bytes, "ms_per_launch": per_launch_ms,
            "moved": {"bytes_per_launch": moved_bytes, "gbs": moved_bytes / (per_launch_ms * 1e-3) / 1e9,
                      "frac": moved_bytes / (per_launch_ms * 1e-3) / 1e9 / pk["hbm"],
                      "note": "size of the spectrum planes the kernel streams (block length %d, hop %d, %d blocks)" % (Bfft, V, nblkp)},
            "tensor": {"executed_tflops": exec_flops / (per_launch_ms * 1e-3) / 1e12,
                       "frac": exec_flops / (per_launch_ms * 1e-3) / 1e12 / pk["tensor"],
                       "equivalent_time_domain_tflops": achieved_tf,
                       "note": "bf16 MMAs issued (3 per product) vs sustained bf16 peak; 'equivalent' = the time-domain "
                               "2*N*K*L*T FLOPs this launch replaces"},
            "note": "overlap-save spectrum of X (constant over the fit) turns the shifted contraction into one 128 x 2N (resp. "
                    "2nblk) real GEMM per frequency: ~8.5 instead of 2*L flops per element of X, so HBM binds",
            "kernel_ms": {k: {"total_ms": v[0], "launches": v[1]} for k, v in prof.items()},
            "contraction_share_of_step": contr_share,
        }
    else:
        roofline = _tensor_roofline(name, world, dom, engine, achieved_tf, pk, Fc_rank, per_launch_ms, K, L, prof, contr_share)
    B = bytes_iteration(N, T, K, L) / world
    hbm = {"achieved": B / (ms_per_step * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
           "frac": B / (ms_per_step * 1e-3) / 1e9 / pk["hbm"],
           "note": "whole-iteration algorithmic bytes s*(2NT + 4KT + 6KNL) per GPU over the step time (the % HBM figure the metric asks for)"}

    cpu = None
    if world == 1 and not args.no_cpu and args.alg == "hals":
        Ts = int(min(T, 4096))
        sec = cpu_iteration_time_hals(cfg, Ts)
        cpu = {"value": 1.0 / (sec * T / Ts), "unit": "iterations/s", "cores": int(os.environ.get("OMP_NUM_THREADS", host_cores())),
               "kind": "port", "sample": f"one literal Float64 HALS iteration (plain-C restatement of hals.jl) on a T={Ts} slice (same N,K,L), extrapolated x{T / Ts:.0f}"}
    elif world == 1 and not args.no_cpu:
        Ts = cpu_sample_T(cfg)
        sec = cpu_iteration_time(cfg, Ts, 1, 1)
        cpu = {"value": 1.0 / (sec * T / Ts), "unit": "iterations/s", "cores": cpu_threads(), "kind": "port",
               "sample": f"one literal Float64 MU iteration on a T={Ts} slice (same N,K,L), extrapolated x{T / Ts:.0f}"}

    critical = None
    if args.alg == "hals":
        # the H sweep (hals.jl:121-154) is a chain of T dependent steps per component: neither HBM nor tensor bound, and no
        # GPU count shortens it; on a sharded fit it runs on rank 0 over all T columns (gather Q / scatter H around it)
        per_sweep = sweep_ms / max(sweep_n, 1)
        critical = {"kernel": "hals2_sweep_kernel (cooperative launch in rounds: recurrence warps with lane = component, 8x8 pull blocks, "
                              "diagonal items; one 1024-column chunk per component per round)",
                    "dependent_column_steps": T + (K - 1) * L, "ms_per_sweep": per_sweep, "sweeps": sweep_n,
                    "us_per_1024_columns": per_sweep * 1e3 / (T / 1024.0) if sweep_n else None,
                    "ns_per_column": per_sweep * 1e6 / T if sweep_n else None,
                    "share_of_step": sweep_ms / (ms_per_step * args.steps) if ms > 0 else None,
                    "note": "measured on rank 0 (the sweep runs there over all T columns); exact reference order k outer / t inner"}
    line = {
        "metric": "CNMF iterations/sec", "value": value, "unit": "iterations/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{name}: {'MU' if args.alg == 'mult' else 'HALS'} N={N} T={T} K={K} L={L}", "alg": args.alg,
                   "parallelism": f"T-shard x{world}", "collectives": ("NCCL inside libcmf_sm100 (cmf_create_rank)" if args.collectives == "lib" else "torch.distributed between the split-phase calls") if world > 1 else "none",
                   "l2": "inputs (X = %.1f GiB per GPU) exceed the 126 MB L2" % (4.0 * N * (t1 - t0) / 2 ** 30),
                   "seeds": {"data": SEED_DATA, "init": SEED_INIT}, "p_h": P_H, "noise": NOISE,
                   "engine": {0: "SIMT fp32", 1: "tcgen05 split-bf16, time domain (3 MMAs per product, fp32 accumulate)",
                              2: "tcgen05 split-bf16, frequency domain (overlap-save spectrum of X, SIMT FFTs, per-frequency "
                                 "complex products with 3 MMAs per product)"}[engine],
                   "loss": ("algebraic expansion ||X||^2 - 2<numH,H> + <WW',HtHt'> (exact identity; at or below 25% loss it is "
                            "calibrated against the direct pass every 1..16 evaluations, see value_calibrated_loss)" if (args.loss_mode == 1 and args.alg == "mult") else "direct conv + residual pass")},
        "value_direct_loss": value_direct, "value_calibrated_loss": calibrated,
        "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "roofline_hbm": hbm, "cpu_baseline": cpu,
        "clocks": clocks, "loss": {"initial": loss0, "final": losses[-1] if losses else None},
    }
    if critical is not None:
        line["critical_path"] = critical
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_sample(n, keep, seed):
    """Sorted indices of a fixed, seeded sample of `keep` out of range(n); all of range(n) when keep >= n."""
    import numpy as np

    if keep >= n:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, size=keep, replace=False))


def dump_outputs(outdir, shard, losses, rank, world, dist):
    """Writes what the timed loop leaves its caller as OUTDIR/W.npy (K x N x L), H.npy (K x T) in the fit's float32 and
    loss.npy (the loss of every timed step, float64).  A factor larger than DUMP_ELEMS keeps a seeded sample of its units
    (W) or columns (H); the columns of H are gathered over the ranks, so the files do not depend on the GPU count."""
    import numpy as np

    K, N, L = shard.K, shard.N, shard.L
    W, H_own = shard.get_factors()
    cols = dump_sample(shard.T, DUMP_ELEMS // K, DUMP_SEED)
    mine = np.ascontiguousarray(H_own[:, cols[(cols >= shard.t0) & (cols < shard.t1)] - shard.t0])
    parts = [mine]
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, mine)
    if rank != 0:
        return
    units = dump_sample(N, DUMP_ELEMS // (K * L), DUMP_SEED + 1)
    os.makedirs(outdir, exist_ok=True)
    np.save(os.path.join(outdir, "W.npy"), np.ascontiguousarray(W[:, units, :]))
    np.save(os.path.join(outdir, "H.npy"), np.concatenate(parts, axis=1))      # ranks own ascending column ranges
    np.save(os.path.join(outdir, "loss.npy"), np.asarray(losses, dtype=np.float64))


def _tensor_roofline(name, world, dom, engine, achieved_tf, pk, Fc_rank, per_launch_ms, K, L, prof, contr_share):
    # dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from one `ncu --set full` capture of this very
    # workload (profiles/r1_ncu_full_corr_c4_lockstep.md); only known for the 1-GPU c4 correlation launch
    traffic, traffic_note = None, "no ncu capture for this workload / kernel"
    if name == "c4" and world == 1 and dom == "corr":
        traffic = 128.9e9
        traffic_note = ("ncu --set full, c4, 1 GPU, per launch: 113.9 GB read + 15.1 GB written vs 68.7 GB algorithmic "
                        "(X hi/lo planes once); profiles/r1_ncu_full_corr_c4_lockstep.md")
    return {
        "bound": "tensor", "kernel": dom, "achieved": achieved_tf, "peak": pk["tensor"], "unit": "TFLOP/s",
        "frac": achieved_tf / pk["tensor"], "traffic": traffic, "traffic_note": traffic_note,
        "peak_source": f"{pk['src']} bf16 sustained",
        "flops_per_launch": Fc_rank, "ms_per_launch": per_launch_ms,
        "executed": {"tflops": 3.0 * achieved_tf if engine == 1 else achieved_tf,
                     "frac": (3.0 * achieved_tf if engine == 1 else achieved_tf) / pk["tensor"],
                     "note": "bf16 tensor FLOPs actually issued: every fp32 product is 3 bf16 MMAs (hi*hi + hi*lo + lo*hi)"},
        "note": "arithmetic intensity K*L/2 = %d FLOP/B >> machine balance: the contraction is tensor/FMA bound, "
                "not HBM bound (SURVEY.md section 8d); algorithmic FLOPs 2*N*K*(L*T - L(L-1)/2) per contraction launch" % (K * L // 2),
        "kernel_ms": {k: {"total_ms": v[0], "launches": v[1]} for k, v in prof.items()},
        "contraction_share_of_step": contr_share,
    }


# per-launch DRAM traffic of the frequency-domain kernels at c4 on one GPU, from `ncu --set full` (profiles/); filled per round
NCU_TRAFFIC_C4_FD = {
    ("transconv", 1024): (82.01e9, "ncu --set full, c4, 1 GPU, block length 1024, per launch: 80.82 GB read + 1.20 GB written vs 76.38 GB of spectrum planes + "
                                   "1.08 GB operand that must be read and 69.9 GB algorithmic; profiles/r2_ncu_full_products_c4.md"),
    ("corr", 1024): (81.82e9, "ncu --set full, c4, 1 GPU, block length 1024, per launch: 80.74 GB read + 1.08 GB written vs 76.38 GB of spectrum planes + "
                              "2.4 GB operand that must be read and 69.9 GB algorithmic; profiles/r2_ncu_full_products_c4.md"),
    ("transconv", 512): (89.76e9, "ncu --set full, c4, 1 GPU, per launch: 88.42 GB read + 1.34 GB written vs 85.56 GB of spectrum planes + 1.08 GB "
                           "operand that must be read and 69.9 GB algorithmic; profiles/r1_ncu_full_fd_kernels.md"),
    ("corr", 512): (90.11e9, "ncu --set full, c4, 1 GPU, per launch: 89.57 GB read + 0.54 GB written vs 85.56 GB of spectrum planes + 2.67 GB "
                      "operand that must be read and 69.9 GB algorithmic; profiles/r1_ncu_full_fd_kernels.md"),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c4", choices=sorted(CONFIGS))
    ap.add_argument("--T", type=int, default=None, help="override T (development only; reported in config.workload)")
    ap.add_argument("--loss-mode", type=int, default=1, choices=[0, 1],
                    help="1: loss by the algebraic expansion on resident numH / W W' (default); 0: direct residual pass")
    ap.add_argument("--engine", type=int, default=None, choices=[0, 1, 2],
                    help="contraction engine (default: the library's choice): 0 SIMT, 1 tcgen05 time domain, 2 tcgen05 frequency domain")
    ap.add_argument("--alg", default="mult", choices=["mult", "hals"])
    ap.add_argument("--collectives", default="lib", choices=["lib", "host"],
                    help="multi-GPU: NCCL inside the library behind the reference-facing calls (default) or torch.distributed between the split-phase calls")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-direct", action="store_true", help="skip the direct-loss figure")
    ap.add_argument("--no-calibrated", action="store_true", help="skip the calibrated-expansion figure (63 more iterations)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write W.npy, H.npy (float32; a seeded sample of units / columns where a "
                         "factor exceeds 24 MiB) and loss.npy (every timed step, float64) to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    cfg = dict(CONFIGS[args.config])
    name = args.config
    if args.T:
        cfg["T"] = args.T
        name += f"(T overridden to {args.T})"
    if args.impl == "reference":
        run_reference(args, cfg, name)
    else:
        run_ours(args, cfg, name)


if __name__ == "__main__":
    main()
