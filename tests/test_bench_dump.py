"""bench.py --dump-outputs: what the last timed step returned, as float64 .npy files under a size budget, the same for the same
arguments from run to run (to the rounding of reordered sums)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_writes_float64_and_samples_over_budget(tmp_path, monkeypatch):
    small = {"a": np.arange(5, dtype=np.int32), "b": [1.5, 2.5]}
    bench.dump_outputs(str(tmp_path / "small"), small)
    for k, v in small.items():
        got = np.load(tmp_path / "small" / (k + ".npy"))
        assert got.dtype == np.float64 and np.array_equal(got, np.asarray(v, dtype=np.float64))
    monkeypatch.setattr(bench, "DUMP_BYTES", 8 * 100)
    big = {"x": np.linspace(0.0, 1.0, 1000), "y": np.ones(10)}
    for d in ("big1", "big2"):
        bench.dump_outputs(str(tmp_path / d), big)
    x1, x2 = np.load(tmp_path / "big1" / "x.npy"), np.load(tmp_path / "big2" / "x.npy")
    assert x1.size == 50 and np.array_equal(x1, x2) and np.all(np.diff(x1) > 0) and np.isin(x1, big["x"]).all()
    assert np.array_equal(np.load(tmp_path / "big1" / "y.npy"), big["y"])


def test_dump_refused_outside_the_default_path(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "--dump-outputs" in out.stderr


@pytest.mark.gpu
def test_dump_is_the_last_timed_step_and_the_same_from_run_to_run(tmp_path):
    """Warm-up and timed steps advance one chain, so (warmup 1, steps 2) and (warmup 2, steps 1) both end on the chain's third
    step and must dump the same arrays, while (warmup 1, steps 1) ends on its second step and must dump other alms."""
    runs = {}
    for name, warmup, steps in (("w1s2", 1, 2), ("w2s1", 2, 1), ("w1s1", 1, 1)):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--nside", "16", "--lmax", "32", "--steps", str(steps),
                              "--warmup", str(warmup), "--no-cpu-baseline", "--no-other-mask", "--no-chain-batch",
                              "--dump-outputs", str(tmp_path / name)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and len(line["pcg_iterations_per_step"]) == steps
        files = {n[:-4]: np.load(tmp_path / name / n) for n in os.listdir(tmp_path / name)}
        assert sorted(files) == ["accept_BB", "accept_EE", "alm_BB", "alm_EE", "binned_dl_BB", "binned_dl_EE", "pcg_iterations"]
        assert all(a.dtype == np.float64 for a in files.values()) and files["alm_EE"].size == 33 ** 2
        assert files["pcg_iterations"][0] == line["pcg_iterations_per_step"][-1]
        runs[name] = files
    for n, a in runs["w1s2"].items():
        b = runs["w2s1"][n]
        assert a.shape == b.shape and np.allclose(a, b, rtol=1e-10, atol=0), n
    assert not np.allclose(runs["w1s2"]["alm_EE"], runs["w1s1"]["alm_EE"], rtol=1e-6, atol=0)
