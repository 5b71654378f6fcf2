"""bench.py contract checks that need no GPU: the reference arm runs on the host cores and prints ONE JSON line with
the keys the driver reads; the product arm refuses to run without a CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, timeout=600, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          timeout=timeout, cwd=ROOT, env=env)


def test_reference_arm_json_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-sample", "8"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, "exactly one JSON line on stdout"
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "filter-steps/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("filter-steps/s at N=100 features")
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and "workload" in d["config"]
    assert d["value"] > 0 and d["cpu_baseline"]["value"] == d["value"]
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0
    # the Octave probe never invents a number
    assert "octave" in d and (d["octave"]["octave"] is not None or "ABSENT" in d["octave"]["note"])


def test_product_arm_needs_a_gpu():
    r = _run(["--steps", "1", "--warmup", "1"], timeout=300, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode != 0
    assert not [ln for ln in r.stdout.splitlines() if ln.strip().startswith("{")], "no metric line without a GPU"


class _HostBank:
    """Stands in for FilterBank in dump_outputs: the download calls of the real one, on host arrays."""

    def __init__(self, B, N):
        self.B, self.N, self.n_max = B, N, 13 + 6 * N
        self.x = np.random.default_rng(1).standard_normal((B, self.n_max))

    def P(self, b):
        return np.arange(self.n_max ** 2, dtype=np.float64).reshape(self.n_max, self.n_max) + 1e7 * b

    def download_state(self, b0=0, nb=None, want_P=True):
        nb = self.B - b0 if nb is None else nb
        P = np.stack([self.P(b) for b in range(b0, b0 + nb)]) if want_P else None
        return self.x[b0:b0 + nb], P, np.full(nb, self.n_max, dtype=np.int32)

    def download_flags(self):
        return (np.arange(self.B * self.N) % 64).astype(np.uint8).reshape(self.B, self.N)

    def download_stats(self):
        from ekf_slam_b200._lib import STATS_FIELDS
        return {k: np.arange(self.B, dtype=np.int32) * (i + 1) for i, k in enumerate(STATS_FIELDS)}


@pytest.mark.parametrize("B,N", [(4096, 100), (3, 500)])
def test_dump_outputs_stays_in_budget(tmp_path, B, N):
    import bench
    bank = _HostBank(B, N)
    bench.dump_outputs(bank, str(tmp_path / "a"))
    bench.dump_outputs(bank, str(tmp_path / "b"))
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == sorted(n + ".npy" for n in ("filters", "x", "flags", "stats", "P_filters", "P_rows", "P"))
    d = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    assert sum((tmp_path / "a" / n).stat().st_size for n in names) <= 64e6
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    for n in names:                                           # the sample is fixed: the same files every time
        assert np.array_equal(d[n[:-4]], np.load(tmp_path / "b" / n))
    f = d["filters"].astype(int)
    assert np.array_equal(f, np.arange(B))                    # x / flags / stats of every filter fit at these sizes
    assert np.array_equal(d["x"], bank.x[f]) and np.array_equal(d["flags"], bank.download_flags()[f])
    assert np.array_equal(d["stats"][:, 1], 2.0 * f)
    pf, rows = d["P_filters"].astype(int), d["P_rows"].astype(int)
    for i, b in enumerate(pf):
        assert np.array_equal(d["P"][i], bank.P(b)[rows])
    if N == 100:
        assert len(pf) > 1 and np.array_equal(rows, np.arange(bank.n_max))
    else:                                                     # one covariance exceeds the budget: a sample of its rows
        assert len(pf) == 1 and 0 < len(rows) < bank.n_max


@pytest.mark.gpu
def test_dump_outputs_are_reproducible(tmp_path):
    """Same arguments, same inputs: two runs write identical outputs (the step is bit-deterministic)."""
    args = ["--steps", "3", "--warmup", "2", "--batch", "64", "--features", "20", "--no-e2e", "--no-extra",
            "--no-cpu-baseline"]
    for run in ("a", "b"):
        r = _run(args + ["--dump-outputs", str(tmp_path / run)])
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout)["steps"] == 3
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert "x.npy" in names and "P.npy" in names
    for n in names:
        a = np.load(tmp_path / "a" / n)
        assert np.array_equal(a, np.load(tmp_path / "b" / n)), n
    x = np.load(tmp_path / "a" / "x.npy")
    assert x.shape == (64, 13 + 6 * 20) and np.isfinite(x).all()
