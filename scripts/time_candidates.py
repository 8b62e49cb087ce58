"""Cost of scoring a given candidate list per session from a carried state at cfg5 size (GRU-256, V = 100k, B = 4096,
x3): seeded Zipf ids, whole calls timed with CUDA events and a synchronise, the 126 MB L2 overwritten before every timed
pass, the calls alternated in every round and the median over --reps rounds reported.

  (a) candidates_from_state, C = 100, logits, k = 100      the candidate kernels only: no catalog-wide pass
  (b) the same with probs=True                             plus one last-step statistics pass for (m, s)
  (c) candidate_rank_from_state, C = 100                   rank of the true next item among the candidates
  (d) topk_from_state(k=20)                                a catalog-wide logits pass + top-k
  (e) target_rank_from_state                               a catalog-wide logits pass with the rank count
  (f) the item-major copy W_out^T alone                    once per weight version

seqrec_candidate_logits is also timed alone: its algorithmic bytes (n*C*H*4 of W_out^T rows, the hidden rows, the ids
and the logits) over its time, against the HBM peak measured on the B200 (6538.6 GB/s).  Before timing, a list made of
(d)'s 20 ids per session is scored, and the candidate order must equal (d)'s wherever neighbouring logits are separated
by more than the x3 band.  The GPU name and power limit are read in the same run.
Usage: python scripts/time_candidates.py [--batch B] [--reps R] [--out profiles/candidates_cfg5.json]"""
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

V, H, T, C = 100000, 256, 200, 100
HBM_PEAK_GBS = 6538.6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    B = a.batch
    torch.cuda.set_device(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # 256 MB > the 126 MB L2
    hot = HotPath("GRU", "tanh", V, H, V, weights=synthetic.make_weights("GRU", V, H, seed=0), tc="x3")
    ids, _ = synthetic.make_batch(V, T, B, seed=0)
    st = hot.advance_state(torch.from_numpy(ids).cuda())
    rng = np.random.default_rng(1)
    tgt = torch.from_numpy(synthetic.zipf_items(rng, V, (B,)).astype(np.int32)).cuda()
    cand = torch.from_numpy(synthetic.zipf_items(rng, V, (B, C)).astype(np.int32)).cuda()
    cand[:, 0] = tgt                                           # the usual "target plus its negatives" list

    # ---- the candidate order of (d)'s own ids equals (d)'s order outside the band
    top_i, _ = hot.topk_from_state(st, 20)
    ci, cz = hot.candidates_from_state(st, top_i)
    h = st.h.double()
    band = (1e-4 * h.abs().sum(1) * hot.W_out.double().abs().max())[:, None]
    sep = torch.ones_like(ci, dtype=torch.bool)
    gap = (cz[:, :-1].double() - cz[:, 1:].double()) > band
    sep[:, 1:] &= gap
    sep[:, :-1] &= gap
    mismatches = int(((ci != top_i) & sep).sum())
    order_check = dict(rows=B, k=20, separated_positions=int(sep.sum()), mismatches=mismatches)
    if mismatches:
        print(json.dumps(order_check))
        raise SystemExit("candidate order differs from topk_from_state outside the band")

    rows = st.h.contiguous()

    def stage():
        hot._wt_version = -1                                  # as after a weight update (the bf16 operands are kept)
        hot._stage_item_major()

    calls = {
        "a_candidates_logits_C100_k100": lambda: hot.candidates_from_state(st, cand),
        "b_candidates_probs_C100_k100": lambda: hot.candidates_from_state(st, cand, probs=True),
        "c_candidate_rank_C100": lambda: hot.candidate_rank_from_state(st, tgt, cand),
        "d_topk20_from_state": lambda: hot.topk_from_state(st, 20),
        "e_target_rank_from_state": lambda: hot.target_rank_from_state(st, tgt),
        "f_item_major_copy": stage,
        "kernel_candidate_logits": lambda: hot._candidate_logits(rows, cand, 0),
    }
    for fn in calls.values():                                 # warm every shape
        fn()
    torch.cuda.synchronize()
    ms = {n: [] for n in calls}
    for _ in range(a.reps):
        for n, fn in calls.items():
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms[n].append(e0.elapsed_time(e1))
    res = {}
    for n, v in ms.items():
        v.sort()
        res[n] = {"ms_median": v[len(v) // 2], "ms_min": v[0], "ms_max": v[-1], "reps": a.reps}
    kb = B * C * H * 4 + B * H * 4 + B * C * 8                # W_out^T rows + hidden rows + ids + logits
    kt = res["kernel_candidate_logits"]["ms_median"] * 1e-3
    out = {
        "workload": dict(cell="GRU", H=H, V=V, T=T, B=B, C=C, tc="x3", seed=0, ids="synthetic.make_batch Zipf(1.1)"),
        "gpu": gpu_info(),
        "note": ("CUDA-event medians of whole calls (host overhead, validation, staging, kernels) from a state advanced "
                 "over T = 200 events, L2 overwritten before each pass, calls alternated within each round.  The "
                 "candidate logits kernel reads W_out^T (0.1 GB), which the L2 may partly serve within one call."),
        "results": res,
        "candidate_logits_kernel": dict(algorithmic_bytes=kb, GBps=kb / kt / 1e9,
                                        fraction_of_hbm_peak=kb / kt / 1e9 / HBM_PEAK_GBS,
                                        hbm_peak_GBps=HBM_PEAK_GBS),
        "order_check": order_check,
    }
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
