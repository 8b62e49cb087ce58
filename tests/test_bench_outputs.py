"""bench.py --dump-outputs and --steps: the item sample is fixed, bad arguments are refused without a GPU, and on the
GPU the dump holds the last timed step's outputs (float32 / float64, within 64 MiB)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*argv):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(argv), capture_output=True,
                          text=True, timeout=900, cwd=ROOT)


def test_item_sample_is_fixed_and_covers_the_hot_items():
    a, b = bench.sample_items(1000000, 8192), bench.sample_items(1000000, 8192)
    assert np.array_equal(a, b) and len(np.unique(a)) == 8192
    assert a.min() == 0 and a.max() < 1000000 and np.array_equal(a[:4096], np.arange(4096))
    assert np.array_equal(bench.sample_items(17, 8192), np.arange(17))


def test_saved_outputs_are_float():
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        bench.save_outputs(d, {"ids": np.arange(5, dtype=np.int32), "x": np.ones(3, dtype=np.float16)})
        assert np.load(os.path.join(d, "ids.npy")).dtype == np.float64
        assert np.load(os.path.join(d, "x.npy")).dtype == np.float32


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bad_arguments_are_refused(argv):
    r = _bench(*argv)
    assert r.returncode == 2 and "error" in r.stderr


@pytest.mark.gpu
def test_dump_holds_the_last_timed_step(tmp_path):
    r = _bench("--config", "cfg2_reddit_gru128", "--steps", "3", "--warmup", "3", "--no-cpu", "--no-sub",
               "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 3
    names = sorted(f[:-4] for f in os.listdir(tmp_path))
    assert names == ["U", "W_in_rows", "W_out_cols", "b", "loss", "sample_items"]
    arrays = {n: np.load(os.path.join(tmp_path, n + ".npy")) for n in names}
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(os.path.getsize(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)) <= 64 << 20
    assert float(arrays["loss"][0]) == line["final_loss"]
    n, H = 8192, 128
    assert np.array_equal(arrays["sample_items"], bench.sample_items(10000, n))
    assert arrays["W_in_rows"].shape == (n, 3 * H) and arrays["W_out_cols"].shape == (H, n)
    assert all(np.isfinite(a).all() for a in arrays.values())


@pytest.mark.gpu
def test_scoring_dump_holds_the_last_timed_step(tmp_path):
    r = _bench("--config", "cfg5_score_gru256_100k", "--steps", "1", "--warmup", "3", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 1
    names = sorted(f[:-4] for f in os.listdir(tmp_path))
    assert names == ["target_probs", "top_items", "top_probs"]
    a = {n: np.load(os.path.join(tmp_path, n + ".npy")) for n in names}
    V, T, B, k = 100000, 200, 4096, line["config"]["k"]
    assert a["top_items"].shape == a["top_probs"].shape == (B, k) and a["target_probs"].shape == (B, T)
    assert a["top_items"].dtype == np.float64 and a["top_probs"].dtype == a["target_probs"].dtype == np.float32
    ids = a["top_items"]
    assert np.array_equal(ids, np.round(ids)) and ids.min() >= 0 and ids.max() < V
    assert all(len(np.unique(row)) == k for row in ids[:64])
    for p in (a["top_probs"], a["target_probs"]):
        assert np.isfinite(p).all() and p.min() > 0 and p.max() <= 1
    assert (np.diff(a["top_probs"], axis=1) <= 0).all()
