"""Cost of re-scoring live sessions from a carried state at cfg5 size (V = 100k, T = 200, B = 4096; GRU-256, and
LSTM-256 alongside): seeded Zipf ids, whole calls timed with CUDA events and a synchronise after a warm-up, median of
--reps, the 126 MB L2 overwritten before every timed pass.

  (a) topk_batch(k=20, last_step_only=True) on the T = 200 windows   today's serving path: rescan the window
  (b) advance_state by one new event per session                     one recurrent step from the carried state
  (c) topk_from_state(k=20)                                          the last-step logits + top-k of the state rows
  (d) target_rank_from_state                                         rank of the true next item from the state

and (b)+(c) against (a).  The GPU name and power limit are read in the same run.
Usage: python scripts/time_state.py [--batch B] [--reps R] [--cells GRU,LSTM] [--out file.json]"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from seq_recommendations_b200 import synthetic  # noqa: E402
from seq_recommendations_b200.engine import HotPath  # noqa: E402
from time_rank import gpu_info  # noqa: E402

V, H, T = 100000, 256, 200


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cells", default="GRU,LSTM")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    B = a.batch
    torch.cuda.set_device(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # 256 MB > the 126 MB L2

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(a.reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        ms.sort()
        return {"ms_median": ms[len(ms) // 2], "ms_min": ms[0], "ms_max": ms[-1], "reps": a.reps}

    ids, _ = synthetic.make_batch(V, T + 1, B, seed=0)
    window = torch.from_numpy(ids[:, 1:]).cuda()                          # the last T events before the new one
    # one new event per session (never a pad) and the item that follows it
    new_ev = torch.from_numpy(synthetic.zipf_items(np.random.default_rng(1), V, (B, 1)).astype(np.int32)).cuda()
    tgt = torch.from_numpy(synthetic.zipf_items(np.random.default_rng(2), V, (B,)).astype(np.int32)).cuda()
    cells = {}
    for cell in a.cells.split(","):
        act = "tanh"
        hot = HotPath(cell, act, V, H, V, weights=synthetic.make_weights(cell, V, H, seed=0), tc="x3")
        st = hot.advance_state(window)
        res = {}
        res["a_topk20_last_step_T200"] = timed(lambda: hot.topk_batch(window, 20, last_step_only=True))
        res["b_advance_state_1_event"] = timed(lambda: hot.advance_state(new_ev, st))
        st1 = hot.advance_state(new_ev, st)
        res["c_topk20_from_state"] = timed(lambda: hot.topk_from_state(st1, 20))
        res["d_target_rank_from_state"] = timed(lambda: hot.target_rank_from_state(st1, tgt))
        bc = res["b_advance_state_1_event"]["ms_median"] + res["c_topk20_from_state"]["ms_median"]
        cells["%s-%d" % (cell, H)] = dict(results=res, b_plus_c_ms=bc,
                                          speedup_a_over_b_plus_c=res["a_topk20_last_step_T200"]["ms_median"] / bc,
                                          tensor_core_scan=bool(hot.rnn_tc))
        del hot
        torch.cuda.empty_cache()
    out = {
        "workload": dict(H=H, V=V, T=T, B=B, k=20, tc="x3", seed=0, ids="synthetic.make_batch Zipf(1.1)"),
        "gpu": gpu_info(),
        "note": ("CUDA-event medians of whole calls (host call overhead, staging, scan, logits, top-k), L2 overwritten "
                 "before each pass.  (a) rescans the T = 200 window; (b) continues the carried state by one event; "
                 "(c) / (d) score the state rows with the kernels of last_step_only."),
        "cells": cells,
    }
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
