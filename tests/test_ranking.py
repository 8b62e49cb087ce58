"""The ranking contract on the CPU: the numpy oracle of the rank (oracle/ranking.py) against the top-k oracle's stable
argsort, hand-computed Recall / MRR / NDCG, the cutoff check of seq_recommendations_b200.ranking, and the
vocabulary-sharded count (per-shard counts with global ids) against the unsharded rank."""
import numpy as np
import pytest
import torch

from oracle import keras_semantics as ks
from oracle import ranking as orank
from seq_recommendations_b200 import ranking


def _tied_logits(rng, n, V):
    """Random logits on a coarse grid (many exact ties) with whole duplicated columns."""
    z = rng.integers(-6, 7, size=(n, V)).astype(np.float64) / 4.0
    for _ in range(3):
        a, b = rng.integers(0, V, size=2)
        z[:, b] = z[:, a]
    return z


def test_rank_is_the_position_in_the_stable_topk_order():
    rng = np.random.default_rng(0)
    n, V = 400, 37
    z = _tied_logits(rng, n, V)
    y = rng.integers(0, V, size=n)
    y[::17] = -1
    r = orank.target_rank(z, y)
    order = ks.topk_items(torch.from_numpy(z), V)           # stable argsort of -z: ties to the lower item id
    for i in range(n):
        if y[i] < 0:
            assert r[i] == 0
        else:
            assert r[i] == 1 + int(np.flatnonzero(order[i] == y[i])[0])
    lo, hi = orank.rank_band(z, y, 0.0)
    valid = y >= 0
    assert np.all(lo[valid] <= r[valid]) and np.all(r[valid] <= hi[valid])


def test_metrics_by_hand():
    # ranks of 6 steps in 2 left-padded sequences; 0 = pad
    rank = np.array([[0, 0, 1, 3, 12, 2],
                     [0, 5, 1, 25, 2, 7]])
    scored = [1, 3, 12, 2, 5, 1, 25, 2, 7]
    n = len(scored)
    m = orank.ranking_metrics(rank, ks=(1, 2, 5, 10))
    assert m["n"] == n
    assert m["recall@1"] == pytest.approx(2 / n)
    assert m["recall@2"] == pytest.approx(4 / n)
    assert m["recall@5"] == pytest.approx(6 / n)
    assert m["recall@10"] == pytest.approx(7 / n)
    assert m["mrr@1"] == pytest.approx(2 / n)
    assert m["mrr@2"] == pytest.approx((1 + 1 + 0.5 + 0.5) / n)
    assert m["mrr@5"] == pytest.approx((1 + 1 + 0.5 + 0.5 + 1 / 3 + 1 / 5) / n)
    assert m["mrr@10"] == pytest.approx((1 + 1 + 0.5 + 0.5 + 1 / 3 + 1 / 5 + 1 / 7) / n)
    assert m["mrr"] == pytest.approx(sum(1.0 / r for r in scored) / n)
    g = lambda r: 1.0 / np.log2(r + 1.0)
    assert m["ndcg@1"] == pytest.approx(2 / n)
    assert m["ndcg@2"] == pytest.approx((2 + 2 * g(2)) / n)
    assert m["ndcg@5"] == pytest.approx((2 + 2 * g(2) + g(3) + g(5)) / n)
    assert m["ndcg@10"] == pytest.approx((2 + 2 * g(2) + g(3) + g(5) + g(7)) / n)
    # last step only: column T-1 of each row
    last = orank.ranking_metrics(orank.last_step(rank), ks=(1, 5))
    assert last["n"] == 2
    assert last["recall@1"] == 0.0 and last["recall@5"] == pytest.approx(0.5)
    assert last["mrr@5"] == pytest.approx(0.5 / 2) and last["mrr"] == pytest.approx((1 / 2 + 1 / 7) / 2)
    # the sums the device returns give the same dict
    sums = []
    for k in (1, 2, 5, 10):
        hit = [r for r in scored if r <= k]
        sums += [len(hit), sum(1.0 / r for r in hit), sum(g(r) for r in hit)]
    sums += [n, sum(1.0 / r for r in scored), sum(g(r) for r in scored)]
    dev = ranking.metrics_from_sums(sums, (1, 2, 5, 10))
    for key, v in m.items():
        assert dev[key] == pytest.approx(v, rel=1e-15, abs=0), key


@pytest.mark.parametrize("bad", [0, -3, 2.5, (5, 0), (), True])
def test_bad_cutoffs_raise(bad):
    with pytest.raises(ValueError):
        ranking.ranking_metrics(np.array([1, 2, 3]), ks=bad)


def test_sharded_count_equals_unsharded_rank():
    """What a vocabulary shard [lo, hi) adds with global ids (id = lo + v) and the catalog-wide reference logit: summed
    over the shards, plus one, it is the unsharded rank -- ties across shard borders included."""
    rng = np.random.default_rng(3)
    n, V = 300, 60
    z = _tied_logits(rng, n, V)
    y = rng.integers(0, V, size=n)
    y[::11] = -1
    zy = z[np.arange(n), np.where(y >= 0, y, 0)]
    for world in (2, 3, 4, 5):
        bounds = np.linspace(0, V, world + 1).astype(int)
        total = np.zeros(n, dtype=np.int64)
        for lo, hi in zip(bounds[:-1], bounds[1:]):
            zs = z[:, lo:hi]                                 # the shard's logits, local columns v
            gid = lo + np.arange(hi - lo)                    # id_offset + v
            cnt = ((zs > zy[:, None]) | ((zs == zy[:, None]) & (gid < y[:, None]))) & (gid != y[:, None])
            total += np.where(y >= 0, cnt.sum(axis=1), 0)
        rank = total + (y >= 0)
        assert np.array_equal(rank, orank.target_rank(z, y)), world
