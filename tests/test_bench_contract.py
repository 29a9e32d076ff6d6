"""`bench.py --impl reference` prints one JSON line with the contract's keys (runs on CPU); `--dump-outputs`
writes the state the timed steps left."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    out = subprocess.run(
        [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "3",
         "--nwalkers", "512", "--ndim", "16"],
        capture_output=True, text=True, timeout=300, cwd=ROOT,
    )
    assert out.returncode == 0, out.stderr
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["dtype"] == "f64" and d["vs_baseline"] is None
    assert d["steps"] == 3 and d["warmup"] == 3
    # the unmodified reference whenever build() packaged it (oracle/make_ref.py), else the port, named as such
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "emcee_reference.zip"))
    assert d["cpu_baseline"]["kind"] == ("reference" if have_ref else "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["port"] > 0
    if have_ref:
        assert d["cpu_baseline"]["reference_vectorize"] > 0 and d["cpu_baseline"]["reference_pool"] > 0
        # every arm timed over exactly --steps steps
        assert "vectorize=True 3 steps x3" in d["cpu_baseline"]["sample"]
        assert "BLAS threads=1, 3 steps x3" in d["cpu_baseline"]["sample"]
    else:
        assert "oracle/_ref/emcee_reference.zip absent" in d["cpu_baseline"]["sample"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"] > 0
    assert "workload" in d["config"]


def test_dump_outputs_sample_is_capped_and_fixed(tmp_path):
    import bench

    rng = np.random.default_rng(3)
    n, d = 70000, 128  # 72 MB of coordinates: above the cap
    coords, log_prob, nacc = rng.standard_normal((n, d)), rng.standard_normal(n), rng.integers(0, 9, n).astype(np.uint64)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), coords, log_prob, nacc)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["coords.npy", "log_prob.npy", "naccepted.npy", "walkers.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) <= bench.DUMP_BYTES
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in names}
    rows = got["walkers"].astype(np.int64)
    assert len(rows) > n // 2 and np.all(np.diff(rows) > 0) and np.array_equal(rows, got["walkers"])
    assert np.array_equal(got["coords"], coords[rows]) and np.array_equal(got["log_prob"], log_prob[rows])
    assert np.array_equal(got["naccepted"], nacc[rows].astype(np.float64))
    assert all(a.dtype == np.float64 for a in got.values())
    for f in names:
        assert np.array_equal(np.load(tmp_path / "b" / f), got[f[:-4]])
    # below the cap everything is written, unsampled
    bench.dump_outputs(str(tmp_path / "small"), coords[:100], log_prob[:100], nacc[:100])
    assert sorted(os.listdir(tmp_path / "small")) == ["coords.npy", "log_prob.npy", "naccepted.npy"]
    assert np.array_equal(np.load(tmp_path / "small" / "coords.npy"), coords[:100])


def test_dump_outputs_needs_the_gpu_arm(tmp_path):
    out = subprocess.run(
        [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
        capture_output=True, text=True, timeout=300, cwd=ROOT,
    )
    assert out.returncode != 0 and "--dump-outputs" in out.stderr and not os.listdir(tmp_path)


@pytest.mark.gpu
def test_dump_outputs_hold_the_state_after_the_timed_steps(tmp_path):
    import bench

    warmup, steps, n, d = 3, 4, 512, 16
    out = subprocess.run(
        [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
         "--nwalkers", str(n), "--ndim", str(d), "--no-configs", "--cpu-steps", "2", "--cpu-pool-steps", "1",
         "--no-microbench", "--dump-outputs", str(tmp_path)],
        capture_output=True, text=True, timeout=600, cwd=ROOT,
    )
    assert out.returncode == 0, out.stderr
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    assert line["steps"] == steps and line["warmup"] == warmup
    # the CPU baseline beside the GPU line is the unmodified reference whenever build() packaged it
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "emcee_reference.zip"))
    assert line["cpu_baseline"]["kind"] == ("reference" if have_ref else "port"), line["cpu_baseline"]["sample"]
    assert sorted(os.listdir(tmp_path)) == ["coords.npy", "log_prob.npy", "naccepted.npy"]
    o = bench.oracle_sampler(bench.make_workload("gauss_dense", n, d), bench.SAMPLER_SEED)
    o.run(warmup + steps)
    assert np.array_equal(np.load(tmp_path / "coords.npy"), o.coords)
    np.testing.assert_allclose(np.load(tmp_path / "log_prob.npy"), o.log_prob, rtol=1e-11, atol=1e-11)
    assert np.array_equal(np.load(tmp_path / "naccepted.npy"), o.naccepted.astype(np.float64))
