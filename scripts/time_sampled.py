"""Sampled softmax against the full-catalog softmax at cfg4 size (GRU-256, V = 1M, T = 50, B = 1024, id inputs, x3), one
process, one GPU.

  step     the whole captured training step (one CUDA-graph replay) of the full-softmax model and of sampled models with
           S in {1024, 8192, 32768}, alternated round by round, CUDA events around every step and the 126 MB L2
           overwritten before it
  phases   the same steps launched eagerly with phase events (bench.py's per-phase timing, branches serialised):
           sample (draw, gather, operand staging), sampled_panels (target logit, the per-panel GEMMs and rows kernel),
           sampled_columns (target columns, scatter, loss), the recurrent backward and the optimiser
  kernels  each new kernel alone on the S = 8192 model's buffers, L2 overwritten before every launch; algorithmic bytes
           over event time against the HBM peak measured in DESIGN.md section 4

Algorithmic bytes: sample = S*4 (+ S*8 of alias table); gather = S*H*8 + S*12 (read the columns, write W_S, ids, bias,
log Q); rows = nb*S*8 (read and write one panel); target_columns = N*H*16 (hout, W_out column, dh read + write) + N*H*4
(dW_out column); scatter = S*H*12 (read dW_S, read-modify-write dW_out).  The GPU name and power limit are read in the
same run.  Usage: python scripts/time_sampled.py [--steps K] [--rounds R] [--out profiles/sampled_cfg4.json]"""
import argparse
import ctypes
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from seq_recommendations_b200 import synthetic  # noqa: E402
from seq_recommendations_b200._lib import call, ptr  # noqa: E402
from seq_recommendations_b200.engine import HotPath  # noqa: E402
from time_adam import HBM_PEAK_GBS, gpu_info  # noqa: E402

V, H, T, B, CELL, ACT = 1000000, 256, 50, 1024, "GRU", "tanh"
SIZES = (1024, 8192, 32768)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=6, help="timed steps per model and round")
    ap.add_argument("--rounds", type=int, default=5, help="alternations of the models")
    ap.add_argument("--out", default=os.path.join("profiles", "sampled_cfg4.json"))
    a = ap.parse_args()
    torch.cuda.set_device(0)
    gpu = gpu_info()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # 256 MB > the 126 MB L2
    ws = synthetic.make_weights(CELL, V, H, seed=0)
    batches = [tuple(torch.from_numpy(x).cuda() for x in synthetic.make_batch(V, T, B, seed=i)) for i in range(4)]
    models = {}
    for S in (None,) + SIZES:
        hot = HotPath(CELL, ACT, V, H, V, weights=ws, tc="x3")
        hot.set_optimizer("adagrad", lr=0.01, epsilon=1e-8, clipnorm=1.0)
        if S is not None:
            hot.set_loss("sampled_softmax", num_sampled=S)
        for s in range(3):                                # eager, capture, replay
            hot.train_batch(*batches[s % 4])
        models["full" if S is None else "S=%d" % S] = hot
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

    def phases(hot, k):
        hot.use_graphs = False
        out = []
        for s in range(k):
            flush.zero_()
            hot.prof = []
            hot.train_batch(*batches[s % 4])
            torch.cuda.synchronize()
            out.append(hot.phase_times_ms())
        hot.use_graphs, hot.prof = True, None
        return out

    step_ms = {k: [] for k in models}
    phase_ms = {k: [] for k in models}
    for _ in range(a.rounds):
        for name, hot in models.items():
            step_ms[name] += steps(hot, a.steps)
    for name, hot in models.items():
        phase_ms[name] = phases(hot, a.steps)

    # ---- the new kernels alone, on the S = 8192 model's buffers after its last step
    hot = models["S=8192"]
    sp = hot.sampled
    S = sp.S
    w = hot.work(B, T)
    N = w.N
    st = hot.stream
    b = w.sampled_bufs
    nb = b["z"].shape[0]
    parts = torch.zeros(1, dtype=torch.float32, device="cuda")
    kernels_fns = {
        "seqrec_sample_items": (lambda: call("seqrec_sample_items", ptr(sp.ids), S, None, None, V, 0,
                                             ptr(hot.sample_state), st), S * 4),
        "seqrec_gather_columns": (lambda: call("seqrec_gather_columns", ptr(hot.W_out), V, None, ptr(sp.logq),
                                               ptr(sp.ids), S, H, ptr(sp.W_S), ptr(sp.bias_S), st), S * H * 8 + S * 12),
        "seqrec_sampled_softmax_rows (one panel)": (
            lambda: call("seqrec_sampled_softmax_rows", ptr(b["z"]), S, ptr(sp.ids), ptr(w.zy), ptr(w.tgt), ptr(sp.logq),
                         ptr(w.mask), None, ptr(b["g"]), ptr(parts), nb, st), nb * S * 8),
        "seqrec_target_columns": (
            lambda: call("seqrec_target_columns", ptr(w.hout), None, ptr(hot.W_out), V, ptr(w.tgt), ptr(b["g"]),
                         ptr(w.dh), ptr(hot.dW_out), None, N, H, st), N * H * 20),
        "seqrec_scatter_add_columns": (
            lambda: call("seqrec_scatter_add_columns", ptr(sp.dW_S), None, ptr(sp.ids), S, H, ptr(hot.dW_out), V, None,
                         st), S * H * 12),
    }

    def kernel_ms(fn, reps=20):
        fn()
        out = []
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            out.append(e0.elapsed_time(e1))
        return out

    kernels = {}
    for name, (fn, nbytes) in kernels_fns.items():
        ms = kernel_ms(fn)
        med = statistics.median(ms)
        gbs = nbytes / (med * 1e-3) / 1e9
        kernels[name] = {"median_ms": round(med, 4), "min_ms": round(min(ms), 4), "max_ms": round(max(ms), 4),
                         "algorithmic_bytes": int(nbytes), "GB_per_s": round(gbs, 1),
                         "fraction_of_hbm_peak": round(gbs / HBM_PEAK_GBS, 3)}

    def summary(xs):
        return {"median_ms": round(statistics.median(xs), 3), "min_ms": round(min(xs), 3), "max_ms": round(max(xs), 3),
                "n": len(xs)}

    def phase_summary(runs):
        names = sorted({k for r in runs for k in r})
        return {k: round(statistics.median([r.get(k, 0.0) for r in runs]), 3) for k in names}

    res = {
        "what": "sampled softmax vs full softmax training step at cfg4 (GRU-256, V=1M, T=50, B=1024, ids, x3, Adagrad "
                "clipnorm 1), one GPU",
        "gpu": gpu,
        "timing": "CUDA events; 256 MiB memset before every timed step / launch (outside the events); models "
                  "alternated over %d rounds of %d steps; phases from %d eager steps per model with phase events" % (
                      a.rounds, a.steps, a.steps),
        "step_captured": {k: summary(v) for k, v in step_ms.items()},
        "phases_eager_median_ms": {k: phase_summary(v) for k, v in phase_ms.items()},
        "kernels_S8192": kernels,
        "panel_rows_S8192": nb,
        "hbm_peak_GB_per_s": HBM_PEAK_GBS,
    }
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
