"""bench.py's command line: the reference arm (CPU only: the oracle port timed on the host cores) prints one JSON line with
the keys a reader of the result needs; --dump-outputs writes what the timed steps computed, as a fixed sample that does not
depend on the GPU count; the GPU arm's dump on a small configuration."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "c1",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "CNMF iterations/sec" and d["unit"] == "iterations/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_zero_steps_is_rejected():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 2 and "--steps" in out.stderr


class _Shard:
    """The part of DeviceShard that bench.dump_outputs reads, over host arrays."""

    def __init__(self, W, H, t0, t1):
        (self.K, self.N, self.L), self.T = W.shape, H.shape[1]
        self.W, self.H, self.t0, self.t1 = W, H, t0, t1

    def get_factors(self):
        return self.W, self.H[:, self.t0 : self.t1]


class _TwoRanks:
    """all_gather_object of a two-rank group whose rank 1 calls first."""

    from_rank1 = None

    def all_gather_object(self, out, obj):
        if self.from_rank1 is None:
            self.from_rank1 = obj
        else:
            out[:] = [obj, self.from_rank1]


def _load(d):
    return {n: np.load(os.path.join(d, n + ".npy")) for n in ("W", "H", "loss")}


def test_dump_outputs_is_a_fixed_bounded_sample_independent_of_the_gpu_count(tmp_path):
    sys.path.insert(0, ROOT)
    import bench

    rng = np.random.default_rng(0)
    K, N, L, T = 64, 300, 400, 120000                 # 7.7 M values per factor: both are sampled
    W = rng.random((K, N, L), dtype=np.float32)
    H = rng.random((K, T), dtype=np.float32)
    losses = [0.5, 0.4]
    bench.dump_outputs(str(tmp_path / "one"), _Shard(W, H, 0, T), losses, 0, 1, None)
    bench.dump_outputs(str(tmp_path / "again"), _Shard(W, H, 0, T), losses, 0, 1, None)
    two = _TwoRanks()
    for rank, (t0, t1) in ((1, (50001, T)), (0, (0, 50001))):
        bench.dump_outputs(str(tmp_path / "two"), _Shard(W, H, t0, t1), losses, rank, 2, two)
    one = _load(tmp_path / "one")
    for other in (_load(tmp_path / "again"), _load(tmp_path / "two")):
        for name in one:
            assert np.array_equal(one[name], other[name]), name
    cols = bench.dump_sample(T, bench.DUMP_ELEMS // K, bench.DUMP_SEED)
    units = bench.dump_sample(N, bench.DUMP_ELEMS // (K * L), bench.DUMP_SEED + 1)
    assert len(np.unique(cols)) == len(cols) < T and len(np.unique(units)) == len(units) < N
    assert np.array_equal(one["H"], H[:, cols]) and np.array_equal(one["W"], W[:, units, :])
    assert one["W"].dtype == one["H"].dtype == np.float32 and one["loss"].dtype == np.float64
    assert np.array_equal(one["loss"], losses)
    assert sum(p.stat().st_size for p in (tmp_path / "one").iterdir()) <= 64 * 2 ** 20


def test_dump_outputs_writes_small_factors_whole(tmp_path):
    sys.path.insert(0, ROOT)
    import bench

    rng = np.random.default_rng(1)
    W, H = rng.random((5, 50, 10), dtype=np.float32), rng.random((5, 2000), dtype=np.float32)
    bench.dump_outputs(str(tmp_path), _Shard(W, H, 0, 2000), [0.3], 0, 1, None)
    got = _load(tmp_path)
    assert np.array_equal(got["W"], W) and np.array_equal(got["H"], H)


@pytest.mark.gpu
def test_gpu_arm_dumps_the_outputs_of_its_timed_steps(tmp_path):
    # config c1 (both factors written whole); the same arguments give the same inputs, so a run of 3 timed steps repeats
    # the 2 of a shorter run before taking its third
    loss = {}
    for steps in (2, 3):
        out_dir = tmp_path / str(steps)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "c1", "--steps", str(steps),
                              "--warmup", "1", "--no-e2e", "--no-cpu", "--no-direct", "--no-calibrated",
                              "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
        assert len(lines) == 1, lines
        d = json.loads(lines[0])
        got = _load(out_dir)
        assert d["steps"] == steps and got["loss"].shape == (steps,) and got["loss"][-1] == d["loss"]["final"]
        assert got["W"].shape == (5, 500, 10) and got["H"].shape == (5, 2000)
        assert got["W"].dtype == got["H"].dtype == np.float32
        assert np.all(np.isfinite(got["W"])) and np.all(np.isfinite(got["H"]))
        loss[steps] = got["loss"]
    assert np.allclose(loss[3][:2], loss[2], rtol=1e-6, atol=0), (loss[2], loss[3])
