"""Next-item ranking metrics on the device (csrc/likelihood.cu): Recall@k, MRR@k, NDCG@k and the uncut MRR from the
per-token rank of the true next item (`target_rank_batch`, `_Net.predict_target_rank`).

    recall@k = |{rank <= k}| / |S|      mrr@k = sum_{rank <= k} 1/rank / |S|      ndcg@k = sum_{rank <= k} 1/log2(rank+1) / |S|
    mrr      = sum 1/rank / |S|         n     = |S|

S = the scored tokens: every entry with rank > 0 (rank 0 marks a pad).  With one target per step Recall@k is the hit
rate.  `rank` is a numpy array or -- without a host round trip -- the device tensor the scoring kernels produce.  The
sums are reduced in double on the device and divided on the host, as in likelihood.py."""
import ctypes

import numpy as np
import torch

from ._lib import call, ptr


def check_ks(ks):
    """-> tuple of int cutoffs; every k must be an integer >= 1."""
    out = []
    for k in (ks if isinstance(ks, (list, tuple, np.ndarray)) else (ks,)):
        if isinstance(k, (bool, np.bool_)) or int(k) != k or int(k) < 1:
            raise ValueError("ranking cutoffs must be integers >= 1, got %r" % (k,))
        out.append(int(k))
    if not out:
        raise ValueError("at least one ranking cutoff is needed")
    return tuple(out)


def rank_sums(rank, ks):
    """(3 len(ks) + 3) float64 device tensor of seqrec_rank_metrics: per k {hits, sum 1/rank, sum 1/log2(rank+1)}, then
    the same sums without a cutoff ({n scored, sum 1/rank, ...}).  Sums, so that shards of the data can be added."""
    ks = check_ks(ks)
    dev = torch.device("cuda:%d" % torch.cuda.current_device())
    if isinstance(rank, torch.Tensor):
        r = rank.to(dev, dtype=torch.int32).contiguous().view(-1)
    else:
        r = torch.from_numpy(np.ascontiguousarray(np.asarray(rank).reshape(-1), dtype=np.int32)).to(dev)
    out = torch.zeros(3 * len(ks) + 3, dtype=torch.float64, device=r.device)
    if r.numel() == 0:
        return out
    kt = torch.tensor(ks, dtype=torch.int32, device=r.device)
    st = ctypes.c_void_p(torch.cuda.current_stream(r.device).cuda_stream)
    call("seqrec_rank_metrics", ptr(r), r.numel(), ptr(kt), len(ks), ptr(out), st)
    return out


def metrics_from_sums(sums, ks):
    """The metric dict from the sums of rank_sums (host list or tensor)."""
    ks = check_ks(ks)
    s = [float(v) for v in (sums.cpu().tolist() if isinstance(sums, torch.Tensor) else sums)]
    n = s[3 * len(ks)]
    res = {}
    with np.errstate(divide="ignore", invalid="ignore"):
        for q, k in enumerate(ks):
            res["recall@%d" % k] = np.float64(s[3 * q]) / np.float64(n)
            res["mrr@%d" % k] = np.float64(s[3 * q + 1]) / np.float64(n)
            res["ndcg@%d" % k] = np.float64(s[3 * q + 2]) / np.float64(n)
        res["mrr"] = np.float64(s[3 * len(ks) + 1]) / np.float64(n)
    res["n"] = int(n)
    return res


def ranking_metrics(rank, ks=(1, 5, 10, 20)):
    """{'recall@k', 'mrr@k', 'ndcg@k' for every k, 'mrr', 'n'} over the entries of `rank` that are > 0."""
    ks = check_ks(ks)
    return metrics_from_sums(rank_sums(rank, ks), ks)
