"""The reference arm of bench.py (`--impl reference`: the oracle port timed on the host cores) runs without a GPU and
prints the contract's JSON line; under torchrun only rank 0 prints."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None):
    env = dict(os.environ, **(env_extra or {}))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config",
                        "cfg1_msnbc_gru100", "--steps", "2", "--warmup", "1"], capture_output=True, text=True, env=env,
                       timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_reference_arm_prints_contract_line():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "training sequences/sec" and d["unit"] == "sequences/sec"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["config"]["workload"] == "cfg1_msnbc_gru100"
    assert d["steps"] == 2 and d["cpu_baseline"]["timed_steps"] == [2]


def test_reference_timing_runs_exactly_the_requested_steps():
    """Both the full-batch timing and the two-batch fit (taken when the logits of the full batch are too large) time
    exactly `steps` steps at every batch size."""
    import torch
    import bench
    cfg = dict(cell="GRU", act="tanh", V=50, H=8, T=6, B=64)
    threads = torch.get_num_threads()                     # time_cpu takes every host core; later tests keep theirs
    try:
        for sample_b, want in ((64, [5]), (8, [5, 5])):
            assert bench.time_cpu(cfg, 5, 1, sample_b=sample_b)["timed_steps"] == want
    finally:
        torch.set_num_threads(threads)


def test_reference_arm_other_ranks_stay_silent():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []
