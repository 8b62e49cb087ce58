"""Worker of tests/test_gpu_state.py::test_two_gpu_states_equal_single_gpu: run under torchrun (one process per GPU,
NCCL).  Every process holds the states of its own sessions; with a vocabulary-parallel model (W_out column shards) and
with a data-parallel one, the states and the scores from them must equal what a single-GPU model computes."""
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
    for V, H, T, B, cell, tc in ((10000, 128, 12, 300, "GRU", "x3"), (998, 32, 6, 40, "LSTM", "off")):
        act = "tanh" if cell == "GRU" else "relu"
        ws = synthetic.make_weights(cell, V, H, seed=3)
        ids, tgt = synthetic.make_batch(V, T, B, seed=4, min_len=1)
        lo, hi = dist.shard_rows(B, comm.rank, comm.world)
        i, t = ids[lo:hi], tgt[lo:hi, -1]
        ref = HotPath(cell, act, V, H, V, weights=ws, comm=solo, tc=tc)
        rs = ref.advance_state(i[:, 4:], ref.advance_state(i[:, :4]))
        want = (rs.h.cpu(), ref.topk_from_state(rs, 10), ref.target_rank_from_state(rs, t).cpu(),
                ref.target_prob_from_state(rs, t).cpu().numpy())
        for vp in (True, False):
            hot = HotPath(cell, act, V, H, V, weights=ws, comm=comm, tc=tc, vocab_parallel=vp)
            st = hot.advance_state(i[:, 4:], hot.advance_state(i[:, :4]))
            ti, tp = hot.topk_from_state(st, 10)
            same = (torch.equal(st.h.cpu(), want[0]) and torch.equal(ti.cpu(), want[1][0].cpu())
                    and torch.allclose(tp.cpu(), want[1][1].cpu(), rtol=1e-6, atol=0)
                    and torch.equal(hot.target_rank_from_state(st, t).cpu(), want[2])
                    and np.allclose(hot.target_prob_from_state(st, t).cpu().numpy(), want[3], rtol=1e-6, atol=0))
            print("rank %d: states V=%d tc=%s vocab_parallel=%s -> %s" % (comm.rank, V, tc, vp,
                                                                          "OK" if same else "MISMATCH"), flush=True)
            ok = ok and same
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
