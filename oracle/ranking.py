"""numpy restatement of the next-item ranking contract (seq_recommendations_b200/ranking.py, the rank kernels of
include/seqrec_b200.h).  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

    rank[n] = 1 + #{v != y : z_v > z_y} + #{v < y : z_v == z_y}         (0 for pads, y < 0)

the 1-based position of y in the stable descending order of the logits, ties to the lower item id -- the order of
keras_semantics.topk_items."""
import numpy as np


def _gather(z, y):
    yc = np.where(y >= 0, y, 0)
    return np.take_along_axis(z, yc[..., None], axis=-1)[..., 0]


def target_rank(logits, targets):
    """logits (..., V), targets (...) int (pad < 0) -> int64 ranks by the definition."""
    z = np.asarray(logits, dtype=np.float64)
    y = np.asarray(targets).astype(np.int64)
    zy = _gather(z, y)[..., None]
    v = np.arange(z.shape[-1])
    yy = y[..., None]
    before = ((z > zy) | ((z == zy) & (v < yy))) & (v != yy)
    rank = 1 + before.sum(axis=-1)
    return np.where(y >= 0, rank, 0).astype(np.int64)


def rank_band(logits, targets, delta, exact_ties=False):
    """(rank_lo, rank_hi) of a rank computed from logits with an absolute error up to delta (per token, broadcast):
    rank_lo = 1 + #{v != y : z_v > z_y + delta}, rank_hi = 1 + #{v != y : z_v >= z_y - delta}; 0 for pads.
    exact_ties: items whose logit equals z_y exactly (duplicated weight columns, computed with the same arithmetic) are
    decided by the tie rule instead of the band -- the lower ids count, the higher ones do not."""
    z = np.asarray(logits, dtype=np.float64)
    y = np.asarray(targets).astype(np.int64)
    zy = _gather(z, y)[..., None]
    d = np.asarray(delta, dtype=np.float64)[..., None] if np.ndim(delta) else np.float64(delta)
    v = np.arange(z.shape[-1])
    yy = y[..., None]
    other = v != yy
    lo = 1 + ((z > zy + d) & other).sum(axis=-1)
    hi = 1 + ((z >= zy - d) & other).sum(axis=-1)
    if exact_ties:
        lo = lo + ((z == zy) & (v < yy)).sum(axis=-1)
        hi = hi - ((z == zy) & (v > yy)).sum(axis=-1)
    valid = y >= 0
    return np.where(valid, lo, 0).astype(np.int64), np.where(valid, hi, 0).astype(np.int64)


def ranking_metrics(rank, ks=(1, 5, 10, 20)):
    """Recall@k, MRR@k, NDCG@k, the uncut MRR and n over the entries with rank > 0."""
    r = np.asarray(rank).reshape(-1).astype(np.int64)
    r = r[r > 0]
    n = r.size
    out = {}
    with np.errstate(divide="ignore", invalid="ignore"):
        for k in ks:
            hit = r <= k
            out["recall@%d" % k] = np.float64(hit.sum()) / n
            out["mrr@%d" % k] = np.sum(1.0 / r[hit]) / n
            out["ndcg@%d" % k] = np.sum(1.0 / np.log2(r[hit] + 1.0)) / n
        out["mrr"] = np.sum(1.0 / r) / n
    out["n"] = int(n)
    return out


def last_step(rank_bt):
    """The scored entries of `last_step_only`: column T-1 of each (left-padded) row."""
    return np.asarray(rank_bt)[:, -1]
