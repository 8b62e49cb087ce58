"""numpy restatement of candidate scoring (the candidate entry points of include/seqrec_b200.h, HotPath.candidates_batch /
candidate_rank_batch).  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

    z_c   = hs . W_out[:, c] + b_out[c]                                    (0 for a pad, c < 0)
    order = valid entries first: score descending, then lower item id, then lower list position; pads as (-1, 0)
    rank  = 1 + #{j : c_j >= 0, c_j != y, z_j > z_y or (z_j == z_y and c_j < y)}        (0 for y < 0)"""
import numpy as np


def candidate_logits(hs, W_out, b_out, cand):
    """hs (..., H), W_out (H, V), b_out (V,) or None, cand (..., C) int -> float64 (..., C) logits, 0 on pads."""
    h = np.asarray(hs, dtype=np.float64)
    W = np.asarray(W_out, dtype=np.float64)
    c = np.asarray(cand).astype(np.int64)
    cc = np.where(c >= 0, c, 0)
    z = np.einsum("...h,...ch->...c", h, W.T[cc])
    if b_out is not None:
        z = z + np.asarray(b_out, dtype=np.float64)[cc]
    return np.where(c >= 0, z, 0.0)


def candidate_order(z, cand, k=None, m=None, s=None):
    """z, cand (..., C) -> (ids int64, scores float64) (..., k).  Scores are z, or exp(z - m) / s with the row's
    softmax statistics m, s (...)."""
    z = np.asarray(z, dtype=np.float64)
    c = np.asarray(cand).astype(np.int64)
    C = c.shape[-1]
    k = C if k is None else k
    lead = c.shape[:-1]
    zf, cf = z.reshape(-1, C), c.reshape(-1, C)
    ids = np.empty((zf.shape[0], k), dtype=np.int64)
    sc = np.empty((zf.shape[0], k), dtype=np.float64)
    mf = None if m is None else np.asarray(m, dtype=np.float64).reshape(-1)
    sf = None if s is None else np.asarray(s, dtype=np.float64).reshape(-1)
    pos = np.arange(C)
    for r in range(zf.shape[0]):
        valid = cf[r] >= 0
        # lexsort: the last key is the primary one
        order = np.lexsort((pos, cf[r], -np.where(valid, zf[r], 0.0), ~valid))[:k]
        ids[r] = np.where(valid[order], cf[r][order], -1)
        v = zf[r][order] if mf is None else np.exp(zf[r][order] - mf[r]) / sf[r]
        sc[r] = np.where(valid[order], v, 0.0)
    return ids.reshape(lead + (k,)), sc.reshape(lead + (k,))


def candidate_rank(z, cand, zy, y):
    """z, cand (..., C); zy, y (...) -> int64 rank of y among the candidates by the definition (0 where y < 0)."""
    z = np.asarray(z, dtype=np.float64)
    c = np.asarray(cand).astype(np.int64)
    zt = np.asarray(zy, dtype=np.float64)[..., None]
    yy = np.asarray(y).astype(np.int64)[..., None]
    other = (c >= 0) & (c != yy)
    before = other & ((z > zt) | ((z == zt) & (c < yy)))
    return np.where(yy[..., 0] >= 0, 1 + before.sum(-1), 0).astype(np.int64)


def candidate_rank_band(z, cand, zy, y, delta, exact_ties=False):
    """(rank_lo, rank_hi) of a rank computed from logits with an absolute error up to delta (per row, broadcast), like
    oracle.ranking.rank_band: lo counts the candidates above z_y + delta, hi those at or above z_y - delta.
    exact_ties: candidates whose logit equals z_y exactly (the same item, or a duplicated W_out column, computed with the
    same arithmetic) are decided by the tie rule instead of the band."""
    z = np.asarray(z, dtype=np.float64)
    c = np.asarray(cand).astype(np.int64)
    zt = np.asarray(zy, dtype=np.float64)[..., None]
    yy = np.asarray(y).astype(np.int64)[..., None]
    d = np.asarray(delta, dtype=np.float64)[..., None] if np.ndim(delta) else np.float64(delta)
    other = (c >= 0) & (c != yy)
    lo = 1 + ((z > zt + d) & other).sum(-1)
    hi = 1 + ((z >= zt - d) & other).sum(-1)
    if exact_ties:
        lo = lo + ((z == zt) & other & (c < yy)).sum(-1)
        hi = hi - ((z == zt) & other & (c > yy)).sum(-1)
    valid = yy[..., 0] >= 0
    return np.where(valid, lo, 0).astype(np.int64), np.where(valid, hi, 0).astype(np.int64)
