"""Vocabulary-parallel scoring and training on ONE device: two ranks of a world of 2 run as two Python threads on cuda:0,
joined by an in-process stand-in for dist.Comm (the engine reaches torch.distributed only through Comm).  Every rank's
results are compared with a single-GPU HotPath on that rank's own rows, with the bounds of tests/rank_worker.py,
state_worker.py and dp_worker.py, so the vocabulary-parallel paths are covered without a second GPU.

The ranks run ONE AT A TIME: a lock is handed between the threads only inside a collective, so the library is never
entered from two threads at once.  Both ranks use the default stream, so the copies a collective issues are ordered with
the kernels around it.  With two ranks a sum is one addition, which is commutative: the stand-in's sums have the bits
NCCL's have.

Also here: scorer results own their storage -- with T == 1 or B == 1 a second call of the same shape must not change what
the first call returned."""
import threading

import numpy as np
import pytest
import torch

from seq_recommendations_b200 import dist, synthetic
from seq_recommendations_b200.engine import HotPath

pytestmark = pytest.mark.gpu

WORLD = 2
TIMEOUT_S = 30.0
# (V, H, T, B, cell, tc): shards of 5000 items on the tensor-core pass (not a multiple of the 128-item tile), and the
# SIMT kernels (tc off)
CASES = [(10000, 128, 12, 64, "GRU", "x3"), (998, 32, 6, 40, "LSTM", "off")]


class _Group:
    """What the ranks of one world share: a slot per rank, a barrier (waited at twice per collective) and the lock
    that the running rank holds."""

    def __init__(self):
        self.slots = [None] * WORLD
        self.barrier = threading.Barrier(WORLD, timeout=TIMEOUT_S)
        self.run = threading.Lock()


class ThreadComm:
    """dist.Comm for one rank of an in-process world of 2 (only the calls the engine's vocabulary-parallel paths make).

    A collective puts this rank's tensor in its slot, waits at the barrier, issues the reading copies on the stream and
    waits at the barrier again: no rank can enqueue a write to its slot before every other rank's read of it is
    enqueued."""

    def __init__(self, group, rank):
        self.enabled, self.group, self.rank, self.world = True, group, rank, WORLD

    def _wait(self):
        g = self.group
        g.run.release()                          # the other rank runs while this one waits
        try:
            g.barrier.wait()
        finally:
            g.run.acquire()

    def _exchange(self, t, read):
        """read(slots) -> this rank's result, issued between the two barriers."""
        self.group.slots[self.rank] = t
        self._wait()
        out = read(self.group.slots)
        self._wait()
        return out

    def all_gather_cat(self, t):
        return self._exchange(t.contiguous(), lambda slots: torch.cat(slots))

    def all_reduce_sum(self, t, async_op=False):
        if async_op:
            raise NotImplementedError("ThreadComm runs synchronous collectives only")
        t.copy_(self._exchange(t, lambda slots: slots[0] + slots[1]))

    def reduce_scatter_sum(self, out, inp):
        n = out.shape[0]
        lo = self.rank * n
        out.copy_(self._exchange(inp.contiguous(), lambda slots: slots[0][lo:lo + n] + slots[1][lo:lo + n]))

    def all_to_all_rows(self, inp):
        n = inp.shape[0] // WORLD
        lo = self.rank * n
        return self._exchange(inp.contiguous(), lambda slots: torch.cat([s[lo:lo + n] for s in slots]))

    def broadcast(self, t, src=0):
        t.copy_(self._exchange(t, lambda slots: slots[src].clone()))
        return t

    def barrier(self):
        self._wait()


def run_ranks(fn):
    """fn(comm) on every rank of a world of 2, one thread per rank; returns the per-rank results.  An error in one rank
    breaks the barrier (so the other rank stops waiting) and is raised here."""
    group = _Group()
    results, errors = [None] * WORLD, []

    def body(rank):
        torch.cuda.set_device(0)
        group.run.acquire()
        try:
            results[rank] = fn(ThreadComm(group, rank))
        except BaseException as e:          # noqa: BLE001 -- re-raised in the calling thread
            errors.append(e)
            group.barrier.abort()
        finally:
            torch.cuda.current_stream().synchronize()
            group.run.release()

    threads = [threading.Thread(target=body, args=(r,)) for r in range(WORLD)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        # the rank that failed first, not the one whose barrier it broke
        errors.sort(key=lambda e: isinstance(e, threading.BrokenBarrierError))
        raise errors[0]
    return results


def _solo():
    c = dist.Comm.__new__(dist.Comm)
    c.enabled, c.group, c.rank, c.world = False, None, 0, 1
    return c


def _case(V, H, T, B, cell, tc):
    act = "tanh" if cell == "GRU" else "relu"
    ws = synthetic.make_weights(cell, V, H, seed=3)
    ids, tgt = synthetic.make_batch(V, T, B, seed=4, min_len=1)
    return act, ws, ids, tgt


def _max_rel(got, want):
    got, want = got.detach().cpu().double(), want.detach().cpu().double()
    assert got.shape == want.shape, (got.shape, want.shape)
    return float(((got - want).abs() / want.abs()).max())


def _rel_ok(got, want, rtol):
    return _max_rel(got, want) <= rtol


def _rows(rank, B):
    return slice(*dist.shard_rows(B, rank, WORLD))


def _scores(hot, ids, tgt, T, k=10, state=None):
    """Every window scorer on a (rows, T) batch, as host tensors; `state` continues the chunk ids[:, T//2:]."""
    if state is not None:
        ids, tgt = ids[:, T // 2:], tgt[:, T // 2:]
    kw = dict(initial_state=state)
    out = dict(rank=hot.target_rank_batch(ids, tgt, **kw),
               rank_last=hot.target_rank_batch(ids, tgt, last_step_only=True, **kw),
               topk=hot.topk_batch(ids, k, last_step_only=False, **kw),
               topk_last=hot.topk_batch(ids, k, last_step_only=True, **kw),
               prob=hot.target_prob_batch(ids, tgt, **kw))
    if state is None:
        out["loss"] = hot.loss_batch(ids, tgt)[0]
    return {n: tuple(x.cpu() for x in v) if isinstance(v, tuple) else v.cpu() for n, v in out.items()}


def _check_scores(got, want, what):
    for n in ("rank", "rank_last"):
        assert torch.equal(got[n], want[n]), (what, n, int((got[n] != want[n]).sum()))
    for n in ("topk", "topk_last"):
        assert _rel_ok(got[n][1], want[n][1], 1e-6), (what, n, _max_rel(got[n][1], want[n][1]))
        bad = _untied_id_diffs(got[n][0], want[n][0], want[n][1], 1e-6)
        assert not bad.any(), (what, n, bad.nonzero().tolist())
    assert _rel_ok(got["prob"], want["prob"], 1e-6), (what, "prob", _max_rel(got["prob"], want["prob"]))


def _untied_id_diffs(got_i, want_i, want_p, rtol):
    """Positions where the top-k ids differ although the single-GPU probability there does not tie.  Items whose
    probabilities agree to rtol may come out in either order: on the tensor-core pass the single-GPU list can hold two
    probabilities 1 ulp apart that the merged vocabulary-parallel statistics make exactly equal, and equal ones are
    ordered by item id.  A position ties when its probability is within rtol of a neighbour's; the last position may tie
    with the item after it, which the list does not hold."""
    p = want_p.double()
    close = (p[..., 1:] - p[..., :-1]).abs() <= rtol * p[..., 1:]
    tied = torch.zeros_like(p, dtype=torch.bool)
    tied[..., 1:] |= close
    tied[..., :-1] |= close
    tied[..., -1] = True
    return (got_i != want_i) & ~tied


@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s%d-V%d-%s" % (c[4], c[1], c[0], c[5]))
def test_vocab_parallel_scorers_equal_single_gpu(case):
    V, H, T, B, cell, tc = case
    act, ws, ids, tgt = _case(*case)
    ref = HotPath(cell, act, V, H, V, weights=ws, comm=_solo(), tc=tc)
    want, want_state, want_loss = [], [], 0.0
    for r in range(WORLD):
        i, t = ids[_rows(r, B)], tgt[_rows(r, B)]
        want.append(_scores(ref, i, t, T))
        want_state.append(_scores(ref, i, t, T, state=ref.advance_state(i[:, :T // 2])))
        want_loss += float(want[-1]["loss"].double())

    def rank_fn(comm):
        hot = HotPath(cell, act, V, H, V, weights=ws, comm=comm, tc=tc, vocab_parallel=True)
        assert hot.vocab_parallel and hot.V == V // WORLD
        i, t = ids[_rows(comm.rank, B)], tgt[_rows(comm.rank, B)]
        return (_scores(hot, i, t, T), _scores(hot, i, t, T, state=hot.advance_state(i[:, :T // 2])))

    got = run_ranks(rank_fn)
    for r in range(WORLD):
        _check_scores(got[r][0], want[r], "rank %d" % r)
        _check_scores(got[r][1], want_state[r], "rank %d, initial_state" % r)
    # loss_batch reports each rank's share of the loss sum; the shares add up to the single-GPU sums of the shards
    got_loss = sum(float(g[0]["loss"].double()) for g in got)
    assert abs(got_loss - want_loss) <= 1e-5 * abs(want_loss), (got_loss, want_loss)


@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s%d-V%d-%s" % (c[4], c[1], c[0], c[5]))
def test_vocab_parallel_state_scorers_equal_single_gpu(case):
    V, H, T, B, cell, tc = case
    act, ws, ids, tgt = _case(*case)
    ref = HotPath(cell, act, V, H, V, weights=ws, comm=_solo(), tc=tc)

    def score(hot, r):
        i, t = ids[_rows(r, B)], tgt[_rows(r, B), -1]
        st = hot.advance_state(i[:, 4:], hot.advance_state(i[:, :4]))
        ti, tp = hot.topk_from_state(st, 10)
        return (st.h.cpu(), ti.cpu(), tp.cpu(), hot.target_rank_from_state(st, t).cpu(),
                hot.target_prob_from_state(st, t).cpu())

    want = [score(ref, r) for r in range(WORLD)]
    got = run_ranks(lambda comm: score(HotPath(cell, act, V, H, V, weights=ws, comm=comm, tc=tc, vocab_parallel=True),
                                       comm.rank))
    for r in range(WORLD):
        g, w = got[r], want[r]
        assert torch.equal(g[0], w[0]) and torch.equal(g[1], w[1]) and torch.equal(g[3], w[3]), r
        assert _rel_ok(g[2], w[2], 1e-6) and _rel_ok(g[4], w[4], 1e-6), (r, _max_rel(g[2], w[2]), _max_rel(g[4], w[4]))


def _rel_err(a, b):
    return float(np.linalg.norm(a.astype(np.float64) - b) / max(np.linalg.norm(b), 1e-30))


@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s%d-V%d-%s" % (c[4], c[1], c[0], c[5]))
def test_vocab_parallel_train_step_equals_single_gpu(case):
    """One eager step (a captured graph would not replay the in-process collectives), bounds of tests/dp_worker.py."""
    V, H, T, B, cell, tc = case
    act, ws, ids, tgt = _case(*case)
    ref = HotPath(cell, act, V, H, V, weights=ws, comm=_solo(), tc=tc)
    ref.set_optimizer("adagrad", lr=0.05, epsilon=1e-8, clipnorm=1.0)
    want_loss = float(ref.train_batch(ids, tgt).item())
    want_ws = ref.get_weights()

    def rank_fn(comm):
        hot = HotPath(cell, act, V, H, V, weights=ws, comm=comm, tc=tc, vocab_parallel=True)
        hot.use_graphs = False
        hot.set_optimizer("adagrad", lr=0.05, epsilon=1e-8, clipnorm=1.0)
        r = _rows(comm.rank, B)
        loss = float(hot.train_batch(ids[r], tgt[r]).item())
        return loss, hot.get_weights()

    for loss, mine in run_ranks(rank_fn):
        assert abs(loss - want_loss) <= 1e-5 * abs(want_loss), (loss, want_loss)
        errs = [_rel_err(a, b) for a, b in zip(mine, want_ws)]
        assert max(errs) < (2e-5 if tc == "off" else 1e-4), errs


@pytest.mark.parametrize("B,T", [(40, 1), (1, 12)])
def test_scorer_results_own_their_storage(B, T):
    """With T == 1 or B == 1 the time-major work buffers already have the per-session layout; the results must still be
    copies: a second call of the same shape leaves the first call's results unchanged."""
    V, H = 998, 32
    hot = HotPath("GRU", "tanh", V, H, V, weights=synthetic.make_weights("GRU", V, H, seed=3), comm=_solo(), tc="off")
    (i1, t1), (i2, t2) = (synthetic.make_batch(V, T, B, seed=s, min_len=1) for s in (5, 6))
    p = hot.target_prob_batch(i1, t1)
    h = hot.hidden_batch(i1)
    p0, h0 = p.clone(), h.clone()
    hot.target_prob_batch(i2, t2)
    hot.hidden_batch(i2)
    assert torch.equal(p, p0)
    assert torch.equal(h, h0)
