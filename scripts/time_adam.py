"""Cost of Keras Adam against Adagrad at cfg4 size (GRU-256, V = 1M, T = 50, B = 1024, id inputs), one process, one GPU.

  step     the whole captured training step (one CUDA-graph replay), Adagrad and Adam models alternated round by round,
           CUDA events around every step and the 126 MB L2 overwritten before it
  optim    the optimiser phase of the same steps launched eagerly with phase events (bench.py's per-phase timing: the
           norm passes and the update, halves serialised)
  kernels  seqrec_adam on the flat U | b | W_out buffer and seqrec_adam_table on the W_in table alone, L2 flushed before
           every launch; algorithmic bytes over event time against the HBM peak measured in DESIGN.md section 4

Algorithmic bytes: flat = n * 28 (read p, g, m, v; write p, m, v); table = F*GH * 24 (read and write p, m, v) + F * 4
(touched flags) + touched rows * GH * 8 (read the gradient row, write it back to zero).  The table kernel is timed with
the touched flags of one training batch set, so it reads the rows a step reads.  The GPU name and power limit are read
in the same run.  Usage: python scripts/time_adam.py [--steps K] [--rounds R] [--out profiles/adam_cfg4.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from seq_recommendations_b200 import synthetic  # noqa: E402
from seq_recommendations_b200._lib import call, ptr  # noqa: E402
from seq_recommendations_b200.engine import HotPath  # noqa: E402

V, H, T, B, CELL, ACT = 1000000, 256, 50, 1024, "GRU", "tanh"
HBM_PEAK_GBS = 6538.6                 # DESIGN.md section 4: measured copy bandwidth of a B200 at 1000 W


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl, clk = [s.strip() for s in out.split(",")]
        info.update(smi_name=name, power_limit=pl, max_sm_clock=clk)
    except Exception as e:                               # the numbers still stand; say what could not be read
        info["smi_error"] = repr(e)
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10, help="timed steps per model and round")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the two models")
    ap.add_argument("--out", default=os.path.join("profiles", "adam_cfg4.json"))
    a = ap.parse_args()
    torch.cuda.set_device(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # 256 MB > the 126 MB L2
    ws = synthetic.make_weights(CELL, V, H, seed=0)
    batches = [tuple(torch.from_numpy(x).cuda() for x in synthetic.make_batch(V, T, B, seed=i)) for i in range(4)]
    models = {}
    for kind in ("adagrad", "adam"):
        hot = HotPath(CELL, ACT, V, H, V, weights=ws, tc="x3")
        hot.set_optimizer(kind, lr=0.001 if kind == "adam" else 0.01, epsilon=1e-8, clipnorm=1.0)
        for s in range(3):                                # eager, capture, replay
            hot.train_batch(*batches[s % 4])
        models[kind] = hot
    torch.cuda.synchronize()

    def steps(hot, k):
        evs = []
        for s in range(k):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            hot.train_batch(*batches[s % 4])
            e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        return [x.elapsed_time(y) for x, y in evs]

    def optim_phase(hot, k):
        hot.use_graphs, hot.prof = False, []
        out = []
        for s in range(k):
            flush.zero_()
            hot.prof = []
            hot.train_batch(*batches[s % 4])
            torch.cuda.synchronize()
            out.append(hot.phase_times_ms()["optim"])
        hot.use_graphs, hot.prof = True, None
        return out

    step_ms = {k: [] for k in models}
    optim_ms = {k: [] for k in models}
    for _ in range(a.rounds):
        for kind, hot in models.items():
            step_ms[kind] += steps(hot, a.steps)
        for kind, hot in models.items():
            optim_ms[kind] += optim_phase(hot, a.steps)

    # ---- the two Adam kernels alone
    hot = models["adam"]
    o = hot.opt
    ids = batches[0][0].reshape(-1)
    rows = torch.unique(ids[ids >= 0])
    n_flat = hot.flat_p.numel()

    def flat():
        call("seqrec_adam", ptr(hot.flat_p), ptr(hot.flat_g), ptr(hot.flat_m), ptr(hot.flat_a), n_flat, o["lr"],
             o["beta_1"], o["beta_2"], o["eps"], o["decay"], o["clipnorm"], ptr(hot.sumsq), ptr(hot.n_valid_f),
             ptr(hot.iterations), hot.stream)

    def table():
        call("seqrec_adam_table", ptr(hot.W_in), ptr(hot.dW_in), ptr(hot.mW_in), ptr(hot.aW_in), ptr(hot.touched),
             hot.F, hot.GH, o["lr"], o["beta_1"], o["beta_2"], o["eps"], o["decay"], o["clipnorm"], ptr(hot.sumsq),
             ptr(hot.n_valid_f), ptr(hot.iterations), hot.stream)

    def kernel_ms(fn, prep=None, reps=20):
        fn()
        out = []
        for _ in range(reps):
            if prep:
                prep()
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            out.append(e0.elapsed_time(e1))
        return out

    def mark_rows():
        hot.touched[rows] = 1

    kernels = {}
    for name, fn, prep, nbytes in (
            ("seqrec_adam (flat U|b|W_out)", flat, None, n_flat * 28),
            ("seqrec_adam_table (W_in)", table, mark_rows,
             hot.F * hot.GH * 24 + hot.F * 4 + rows.numel() * hot.GH * 8)):
        ms = kernel_ms(fn, prep)
        med = statistics.median(ms)
        gbs = nbytes / (med * 1e-3) / 1e9
        kernels[name] = {"median_ms": round(med, 4), "min_ms": round(min(ms), 4), "max_ms": round(max(ms), 4),
                         "algorithmic_bytes": int(nbytes), "GB_per_s": round(gbs, 1),
                         "fraction_of_hbm_peak": round(gbs / HBM_PEAK_GBS, 3)}
    hot.touched.zero_()

    def summary(xs):
        return {"median_ms": round(statistics.median(xs), 3), "min_ms": round(min(xs), 3), "max_ms": round(max(xs), 3),
                "n": len(xs)}

    res = {
        "what": "Adam vs Adagrad at cfg4 (GRU-256, V=1M, T=50, B=1024, ids, x3 logits), one GPU",
        "gpu": gpu_info(),
        "timing": "CUDA events; 256 MiB memset before every timed step / launch (outside the events); models "
                  "alternated over %d rounds of %d steps" % (a.rounds, a.steps),
        "step_captured": {k: summary(v) for k, v in step_ms.items()},
        "optim_phase_eager": {k: summary(v) for k, v in optim_ms.items()},
        "kernels": kernels,
        "touched_rows_in_table_timing": int(rows.numel()),
        "hbm_peak_GB_per_s": HBM_PEAK_GBS,
    }
    res["adam_minus_adagrad_step_ms"] = round(res["step_captured"]["adam"]["median_ms"] -
                                              res["step_captured"]["adagrad"]["median_ms"], 3)
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
