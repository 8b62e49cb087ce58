"""Worker of tests/test_gpu_sampled.py::test_two_gpu_sampled_step_equals_single_gpu_step: run under torchrun (one process
per GPU, NCCL).  Every rank trains its shard of a global batch with the sampled softmax; the ranks must draw the same
ids, and rank 0 also trains a single-GPU replica on the WHOLE batch, which must end with the same losses and weights."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from seq_recommendations_b200 import dist, synthetic  # noqa: E402
from seq_recommendations_b200.engine import HotPath  # noqa: E402


def rel(a, b):
    return float(np.linalg.norm(a.astype(np.float64) - b) / max(np.linalg.norm(b), 1e-30))


def main():
    import faulthandler
    comm = dist.init_from_env("nccl")
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    ok = True
    # (V, H, T, B_global, tc, S): the dense dW_in exchange with the SIMT GEMMs, the row exchange on the tensor cores
    for V, H, T, B, tc, S in ((100, 32, 6, 32, "off", 64), (20000, 128, 8, 128, "x3", 2048)):
        faulthandler.dump_traceback_later(150, exit=True)
        ws = synthetic.make_weights("GRU", V, H, seed=3, out_bias=True)
        steps = [synthetic.make_batch(V, T, B, seed=30 + s, min_len=1) for s in range(3)]
        hot = HotPath("GRU", "tanh", V, H, V, out_bias=True, weights=ws, comm=comm, device=dev, tc=tc, seed=5)
        hot.set_optimizer("adagrad", lr=0.05, epsilon=1e-8, clipnorm=1.0)
        hot.set_loss("sampled_softmax", num_sampled=S)
        lo, hi = dist.shard_rows(B, comm.rank, comm.world)
        losses, draws = [], []
        for i, t in steps:
            losses.append(float(hot.train_batch(i[lo:hi], t[lo:hi]).item()))
            draws.append(torch.from_numpy(hot.last_samples()).to(dev))
        mine = hot.get_weights()
        for d in draws:                                        # every rank drew rank 0's ids
            d0 = d.clone()
            torch.distributed.broadcast(d0, 0)
            ok = ok and bool(torch.equal(d, d0))
        if comm.rank == 0:
            solo = dist.Comm.__new__(dist.Comm)
            solo.enabled, solo.group, solo.rank, solo.world = False, None, 0, 1
            ref = HotPath("GRU", "tanh", V, H, V, out_bias=True, weights=ws, comm=solo, device=dev, tc=tc, seed=5)
            ref.set_optimizer("adagrad", lr=0.05, epsilon=1e-8, clipnorm=1.0)
            ref.set_loss("sampled_softmax", num_sampled=S)
            for k, (i, t) in enumerate(steps):
                want = float(ref.train_batch(i, t).item())
                same_ids = np.array_equal(ref.last_samples(), draws[k].cpu().numpy())
                good = same_ids and abs(losses[k] - want) <= 1e-5 * abs(want)
                ok = ok and good
            errs = [rel(a, b) for a, b in zip(mine, ref.get_weights())]
            good = max(errs) <= (1e-4 if tc == "off" else 5e-4)
            ok = ok and good
            print("sampled DP V=%d tc=%s S=%d: weight errs %s -> %s" % (V, tc, S, ["%.1e" % e for e in errs],
                                                                        "OK" if good else "MISMATCH"), flush=True)
    faulthandler.dump_traceback_later(60, exit=True)
    flag = torch.tensor([1 if ok else 0], device=dev)
    torch.distributed.all_reduce(flag, op=torch.distributed.ReduceOp.MIN)
    code = 0 if int(flag.item()) == 1 else 1
    comm.barrier()
    torch.cuda.synchronize()
    print("rank %d: done (%s)" % (comm.rank, "OK" if code == 0 else "MISMATCH"), flush=True)
    # leave without the communicator teardown (see tests/dp_worker.py)
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(code)


if __name__ == "__main__":
    main()
