"""-m gpu: bench.py --dump-outputs writes what the timed path returned in its last step; with the same arguments two
runs write the same arrays (fixed weights, inputs and noise seeds).  That exactly --steps steps are timed is checked on
the CPU (tests/test_host_logic.py)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out, *argv):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--no-cpu", "--no-also", "--dump-outputs", str(out)]
                       + list(argv), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_bench_dump_outputs_generate_repeatable(tmp_path):
    runs = [_bench(tmp_path / d, "--workload", "c1", "--steps", "4", "--warmup", "3") for d in ("a", "b")]
    for line in runs:
        assert line["steps"] == 4 and line["parity_check"] is True
    shapes = {"items": (64 * 5,), "z_mu": (64, 16), "resp": (64, 5)}
    assert sorted(os.listdir(tmp_path / "a")) == sorted(k + ".npy" for k in shapes)
    for k, shape in shapes.items():
        a, b = np.load(tmp_path / "a" / (k + ".npy")), np.load(tmp_path / "b" / (k + ".npy"))
        assert a.shape == shape and a.dtype == (np.float64 if k == "items" else np.float32)
        assert np.array_equal(a, b), k
    items = np.load(tmp_path / "a" / "items.npy")
    assert (items >= 0).all() and (items < 3707).all() and (items == np.round(items)).all()


def test_bench_dump_outputs_train(tmp_path):
    line = _bench(tmp_path, "--workload", "c3", "--mode", "train", "--batch", "256", "--steps", "2", "--warmup", "3")
    assert line["steps"] == 2
    names = os.listdir(tmp_path)
    for k in ("loss", "rec_loss", "kld"):
        v = np.load(tmp_path / (k + ".npy"))
        assert v.shape == () and np.isfinite(v)
    params = [n for n in names if n.startswith("param.")]
    assert "param.psm_1.weight.npy" in params and len(params) + 3 == len(names)
    assert all(np.isfinite(np.load(tmp_path / n)).all() for n in params)
