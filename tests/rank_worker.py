"""Worker of tests/test_gpu_ranking.py::test_two_gpu_ranks_equal_single_gpu: run under torchrun (one process per GPU,
NCCL).  A vocabulary-parallel model (W_out column shards, per-shard counts with global ids, summed) and a data-parallel
model (replicated weights, purely local) must give every process the ranks a single-GPU model computes for its rows."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from seq_recommendations_b200 import dist, synthetic  # noqa: E402
from seq_recommendations_b200.engine import HotPath  # noqa: E402


def main():
    comm = dist.init_from_env("nccl")
    ok = True
    solo = dist.Comm.__new__(dist.Comm)
    solo.enabled, solo.group, solo.rank, solo.world = False, None, 0, 1
    # tensor-core pass (shards of 5000 items, not a multiple of the 128-item tile) and the SIMT kernel (tc off)
    for V, H, T, B, cell, tc in ((10000, 128, 12, 64, "GRU", "x3"), (998, 32, 6, 40, "LSTM", "off")):
        act = "tanh" if cell == "GRU" else "relu"
        ws = synthetic.make_weights(cell, V, H, seed=3)
        ids, tgt = synthetic.make_batch(V, T, B, seed=4, min_len=1)
        lo, hi = dist.shard_rows(B, comm.rank, comm.world)
        ref = HotPath(cell, act, V, H, V, weights=ws, comm=solo, tc=tc)
        want = ref.target_rank_batch(ids[lo:hi], tgt[lo:hi]).cpu()
        want_last = ref.target_rank_batch(ids[lo:hi], tgt[lo:hi], last_step_only=True).cpu()
        for vp in (True, False):
            hot = HotPath(cell, act, V, H, V, weights=ws, comm=comm, tc=tc, vocab_parallel=vp)
            got = hot.target_rank_batch(ids[lo:hi], tgt[lo:hi]).cpu()
            got_last = hot.target_rank_batch(ids[lo:hi], tgt[lo:hi], last_step_only=True).cpu()
            same = torch.equal(got, want) and torch.equal(got_last, want_last)
            if not same:
                print("rank %d: %d of %d ranks differ" % (comm.rank, int((got != want).sum()), got.numel()))
            print("rank %d: ranks V=%d tc=%s vocab_parallel=%s -> %s" % (comm.rank, V, tc, vp,
                                                                         "OK" if same else "MISMATCH"), flush=True)
            ok = ok and same
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
