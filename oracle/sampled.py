"""Sampled softmax with log-Q correction (seq_recommendations_b200/losses.py) restated in float64 on top of
oracle/keras_semantics.Model, with autograd gradients, one train step for Adagrad and Adam (oracle/adam.py), and a numpy
restatement of the device draw.  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

For a valid token with target y, logits o (bias included) and the step's samples s_1..s_S:
    l_0 = o_y - log Q(y),   l_j = o_{s_j} - log Q(s_j)  (-inf where s_j == y),   loss = -l_0 + log sum_{j=0..S} exp(l_j)
with log Q(v) = log(S q(v)); duplicates count once per occurrence, no probability clip; the step loss is the masked mean.

The draw: r_i = splitmix64(splitmix64(seed) ^ (offset + i)) in uint64 arithmetic; column c = ((r >> 32) * V) >> 32;
with an alias table the draw is c if (r mod 2^32) < thr[c], else alias[c]."""
import numpy as np
import torch

from . import adam as oa
from . import keras_semantics as ks

_U = np.uint64


def splitmix64(x):
    """splitmix64 of a uint64 array (wrapping arithmetic)."""
    x = np.asarray(x, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = x + _U(0x9E3779B97F4A7C15)
        x = (x ^ (x >> _U(30))) * _U(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> _U(27))) * _U(0x94D049BB133111EB)
    return x ^ (x >> _U(31))


def draw(S, V, seed, offset, thr=None, alias=None):
    """The S ids the device sampler draws at stream position `offset` (int64 numpy)."""
    key = splitmix64(np.array([seed], dtype=np.uint64))[0]
    with np.errstate(over="ignore"):
        r = splitmix64(key ^ (_U(offset) + np.arange(S, dtype=np.uint64)))
        col = ((r >> _U(32)) * _U(V)) >> _U(32)
    col = col.astype(np.int64)
    if thr is None:
        return col
    low = (r & _U(0xFFFFFFFF)).astype(np.int64)
    keep = low < np.asarray(thr, dtype=np.uint32).astype(np.int64)[col]
    return np.where(keep, col, np.asarray(alias, dtype=np.int64)[col])


def log_q(S, q):
    """log(S q(v)) in float64; q (V,) float64."""
    return np.log(S * np.asarray(q, dtype=np.float64))


def sampled_ce(z, targets, samples, logq):
    """Per-token sampled loss: z (..., V) logits, targets (...) >= 0, samples (S,) int64, logq (V,) tensors."""
    y = targets.clamp(min=0)
    l0 = torch.gather(z, -1, y.unsqueeze(-1)).squeeze(-1) - logq[y]
    ls = z[..., samples] - logq[samples]
    ls = torch.where(samples == y.unsqueeze(-1), torch.full_like(ls, -float("inf")), ls)
    return -l0 + torch.logsumexp(torch.cat([l0.unsqueeze(-1), ls], dim=-1), dim=-1)


class Model(oa.Model):
    """oa.Model whose training loss is the sampled softmax: q (V,) float64 (uniform when None) and the number of draws
    S fix log Q; the step's samples are passed to loss / grads / train_step as `samples`."""

    def __init__(self, cell, act_name, weights, S, q=None, dtype=torch.float64):
        oa.Model.__init__(self, cell, act_name, weights, dtype=dtype)
        V = np.asarray(weights[3]).shape[1]
        q = np.full(V, 1.0 / V) if q is None else np.asarray(q, dtype=np.float64)
        self.logq = torch.tensor(log_q(S, q), dtype=dtype)

    def loss(self, ids, targets, mask, x_dense=None, out_scale=None, in_scale=None, rec_masks=None, samples=None):
        Hout, mask = self.hidden(ids=ids, mask=mask, x_dense=x_dense, in_scale=in_scale, rec_masks=rec_masks)
        if out_scale is not None:
            Hout = Hout * out_scale
        z = ks.logits(Hout, self.W_out, self.b_out)
        mf = mask.to(z.dtype)
        ce = sampled_ce(z, targets, torch.as_tensor(samples, dtype=torch.int64), self.logq) * mf
        return ce.sum() / mf.sum(), ce, None
