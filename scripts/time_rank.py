"""Cost of the target rank at cfg5 size (GRU-256, V = 100k, T = 200, B = 4096): one seeded workload, three scoring calls
timed with CUDA events after a warm-up, the 126 MB L2 overwritten before every timed pass.

  (a) target_prob_batch                        p(true next item), every step (the statistics pass)
  (b) target_rank_batch                        rank of the true next item, every step -- the same pass with the count,
                                               which also leaves p(target)'s statistics
  (c) topk_batch(k=20, last_step_only=False)   the only route to Recall@20 before (b)
  (b) and (c) also for the last step only; and the two logits kernels alone (seqrec_ce_tc_forward vs
  seqrec_ce_tc_forward_rank) on the staged operands, alternated.

Per call: ms per batch, tokens/s, and 2*H*V algorithmic flops per scored token over the time against the bf16 dense
GEMM rate measured in the same run (x3 issues three times those flops on the tensor cores).  The GPU name and power
limit are read in the same run.  Usage: python scripts/time_rank.py [--batch B] [--reps R] [--out file.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from seq_recommendations_b200 import synthetic  # noqa: E402
from seq_recommendations_b200._lib import call, ptr  # noqa: E402
from seq_recommendations_b200.engine import HotPath  # noqa: E402

V, H, T, CELL, ACT = 100000, 256, 200, "GRU", "tanh"


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
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    B = a.batch
    torch.cuda.set_device(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # 256 MB > the 126 MB L2

    def timed(fn, reps=a.reps):
        fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        ms.sort()
        return {"ms_median": ms[len(ms) // 2], "ms_min": ms[0], "ms_max": ms[-1], "reps": reps}

    # sustained bf16 dense GEMM rate (cuBLAS 8192^3, ~1 s of back-to-back products): the yardstick of the flop shares
    x = torch.randn(8192, 8192, device="cuda", dtype=torch.bfloat16)
    y = torch.randn(8192, 8192, device="cuda", dtype=torch.bfloat16)
    for _ in range(5):
        torch.matmul(x, y)
    torch.cuda.synchronize()
    n_mm, t0 = 0, time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    while time.perf_counter() - t0 < 1.0:
        for _ in range(20):
            torch.matmul(x, y)
        n_mm += 20
        torch.cuda.synchronize()
    e1.record()
    torch.cuda.synchronize()
    peak = 2.0 * 8192 ** 3 * n_mm / (e0.elapsed_time(e1) * 1e-3)
    del x, y

    hot = HotPath(CELL, ACT, V, H, V, weights=synthetic.make_weights(CELL, V, H, seed=0), tc="x3")
    ids, tgt = synthetic.make_batch(V, T, B, seed=0)
    di, dt = torch.from_numpy(ids).cuda(), torch.from_numpy(tgt).cuda()
    n_tok = B * T
    n_valid = int((dt >= 0).sum())
    flop_tok = 2.0 * H * V

    def entry(r, tokens):
        s = r["ms_median"] * 1e-3
        r.update(tokens_per_s=tokens / s, algo_flops_per_s=tokens * flop_tok / s,
                 algo_share_of_bf16_peak=tokens * flop_tok / s / peak)
        return r

    res = {}
    res["hidden_only"] = timed(lambda: hot.hidden_batch(di))
    res["a_target_prob_all_steps"] = entry(timed(lambda: hot.target_prob_batch(di, dt)), n_tok)
    res["b_target_rank_all_steps"] = entry(timed(lambda: hot.target_rank_batch(di, dt)), n_tok)
    res["c_topk20_all_steps"] = entry(timed(lambda: hot.topk_batch(di, 20, last_step_only=False)), n_tok)
    res["b_target_rank_last_step"] = entry(timed(lambda: hot.target_rank_batch(di, dt, last_step_only=True)), B)
    res["c_topk20_last_step"] = entry(timed(lambda: hot.topk_batch(di, 20, last_step_only=True)), B)

    # the two logits kernels alone on the operands (b) staged, alternated in one loop
    hot.target_rank_batch(di, dt)
    w = hot.work(B, T)
    rank = torch.zeros(w.N, dtype=torch.int32, device="cuda")
    st = hot.stream

    def k_stats():
        call("seqrec_ce_tc_forward", ptr(w.A_hi), ptr(w.A_lo), ptr(hot.Bt_hi), ptr(hot.Bt_lo), None, ptr(w.ws_m),
             ptr(w.ws_s), w.N, hot.Hk, V, 0, V, 1, st)

    def k_rank():
        call("seqrec_ce_tc_forward_rank", ptr(w.A_hi), ptr(w.A_lo), ptr(hot.Bt_hi), ptr(hot.Bt_lo), None, ptr(w.ws_m),
             ptr(w.ws_s), ptr(w.zy), ptr(w.tgt), 0, ptr(rank), w.N, hot.Hk, V, 0, V, 1, st)

    ks, kr = [], []
    for i in range(2 * a.reps):
        for fn, acc in ((k_stats, ks), (k_rank, kr)) if i % 2 == 0 else ((k_rank, kr), (k_stats, ks)):
            acc.append(timed(fn, reps=1)["ms_median"])
    ks.sort()
    kr.sort()
    res["kernel_stats_x3"] = entry({"ms_median": ks[len(ks) // 2], "ms_min": ks[0], "ms_max": ks[-1],
                                    "reps": len(ks)}, n_tok)
    res["kernel_rank_x3"] = entry({"ms_median": kr[len(kr) // 2], "ms_min": kr[0], "ms_max": kr[-1],
                                   "reps": len(kr)}, n_tok)

    out = {
        "workload": dict(cell=CELL, H=H, V=V, T=T, B=B, tokens=n_tok, valid_tokens=n_valid, tc="x3", seed=0),
        "gpu": gpu_info(),
        "bf16_dense_gemm_measured_flops_per_s": peak,
        "algo_flops_per_token": flop_tok,
        "note": ("algo flops = 2*H*V per scored token (all B*T rows are scored, pads included); the x3 mode issues 3x "
                 "that on the tensor cores.  Times are CUDA-event medians of whole calls (staging + recurrent scan + "
                 "logits), L2 overwritten before each pass; hidden_only is the staging + scan part alone."),
        "ratio_b_over_a_call": res["b_target_rank_all_steps"]["ms_median"] / res["a_target_prob_all_steps"]["ms_median"],
        "ratio_b_over_c_call": res["b_target_rank_all_steps"]["ms_median"] / res["c_topk20_all_steps"]["ms_median"],
        "ratio_rank_over_stats_kernel": res["kernel_rank_x3"]["ms_median"] / res["kernel_stats_x3"]["ms_median"],
        "results": res,
    }
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
