"""Sampled softmax without a GPU: the float64 oracle's loss against hand-computed cases, the alias table against q, the
numpy restatement of the device draw, and the argument checks of losses.SampledSoftmax / losses.check_sampled."""
import math

import numpy as np
import pytest
import torch

from oracle import sampled as osm
from seq_recommendations_b200 import losses


def test_oracle_loss_hand_computed_with_accidental_hit_and_duplicate():
    """V = 3, S = 2, q = (0.5, 0.25, 0.25): log Q = log(2 q) = (0, -log 2, -log 2).
    Token a: y = 0, samples (0, 2) -- column 1 is an accidental hit and is dropped.
    Token b: y = 1, samples (2, 2) -- the duplicate counts twice.  Token c is a pad."""
    q = np.array([0.5, 0.25, 0.25])
    logq = torch.tensor(osm.log_q(2, q))
    z = torch.tensor([[1.0, 2.0, 0.5], [1.0, 2.0, 0.5], [9.0, 9.0, 9.0]], dtype=torch.float64)
    ln2 = math.log(2.0)
    l2 = 0.5 + ln2                                              # o_2 - log Q(2)
    want_a = -1.0 + math.log(math.exp(1.0) + math.exp(l2))
    ce_a = osm.sampled_ce(z[:1], torch.tensor([0]), torch.tensor([0, 2]), logq)
    assert math.isclose(float(ce_a[0]), want_a, rel_tol=1e-14)
    l0_b = 2.0 + ln2
    want_b = -l0_b + math.log(math.exp(l0_b) + 2.0 * math.exp(l2))
    ce_b = osm.sampled_ce(z[1:2], torch.tensor([1]), torch.tensor([2, 2]), logq)
    assert math.isclose(float(ce_b[0]), want_b, rel_tol=1e-14)
    # the masked mean of the model's loss over a, b (samples (0, 2) for both) and a pad
    samples = torch.tensor([0, 2])
    ce = osm.sampled_ce(z, torch.tensor([0, 1, -1]), samples, logq) * torch.tensor([1.0, 1.0, 0.0], dtype=torch.float64)
    want_b2 = -l0_b + math.log(math.exp(l0_b) + math.exp(1.0 - 0.0) + math.exp(l2))
    assert math.isclose(float(ce.sum() / 2), (want_a + want_b2) / 2, rel_tol=1e-14)


def _enumerated(thr, alias):
    """p(v) = (thr_v / 2^32 + sum_{u: alias_u = v} (1 - thr_u / 2^32)) / V."""
    V = thr.shape[0]
    t = thr.astype(np.float64) / 4294967296.0
    p = t.copy()
    np.add.at(p, alias.astype(np.int64), 1.0 - t)
    return p / V


@pytest.mark.parametrize("kind", ["uniform", "zipf", "spiky"])
def test_alias_table_reproduces_q(kind):
    V = 5003
    rng = np.random.default_rng(1)
    w = {"uniform": np.ones(V), "zipf": 1.0 / np.arange(1, V + 1) ** 1.1,
         "spiky": np.where(rng.random(V) < 0.01, 1e6, 1.0)}[kind]
    _, q = losses.check_sampled(64, w, V)
    thr, alias = losses.alias_table(q)
    assert thr.dtype == np.uint32 and alias.dtype == np.int32
    assert alias.min() >= 0 and alias.max() < V
    assert np.abs(_enumerated(thr, alias) - q).max() <= 1e-7


def _draw_python(S, V, seed, offset, thr=None, alias=None):
    """The draw in Python integers (mod 2^64), independent of numpy's uint64 arithmetic."""
    M = (1 << 64) - 1

    def sm(x):
        x = (x + 0x9E3779B97F4A7C15) & M
        x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & M
        x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & M
        return x ^ (x >> 31)

    key = sm(seed)
    out = []
    for i in range(S):
        r = sm(key ^ ((offset + i) & M))
        c = ((r >> 32) * V) >> 32
        out.append(c if thr is None or (r & 0xFFFFFFFF) < int(thr[c]) else int(alias[c]))
    return np.array(out)


def test_numpy_draw_equals_integer_restatement():
    V = 70001
    w = np.random.default_rng(2).random(V) + 0.01
    thr, alias = losses.alias_table(w / w.sum())
    for seed, offset in ((0, 0), (7, 123456789), (2 ** 63 + 5, 2 ** 64 - 10)):
        assert np.array_equal(osm.draw(300, V, seed, offset), _draw_python(300, V, seed, offset))
        assert np.array_equal(osm.draw(300, V, seed, offset, thr, alias),
                              _draw_python(300, V, seed, offset, thr, alias))


def test_log_q_tables():
    V, S = 1000, 128
    assert np.allclose(losses.log_q(S, None, V), np.log(S / V))
    w = np.arange(1, V + 1, dtype=np.float64)
    _, q = losses.check_sampled(S, w, V)
    lq = losses.log_q(S, q, V)
    assert lq.dtype == np.float32 and np.allclose(lq, np.log(S * w / w.sum()), rtol=1e-6)


def test_sampled_softmax_argument_checks():
    assert losses.SampledSoftmax(5).num_sampled == 5
    assert losses.SampledSoftmax(losses.MAX_SAMPLED).num_sampled == losses.MAX_SAMPLED
    for bad in (0, -3, losses.MAX_SAMPLED + 1, 2.0, True, "8"):
        with pytest.raises(ValueError):
            losses.SampledSoftmax(bad)
    for bad in ([1.0, 0.0, 2.0], [1.0, -1.0], [1.0, np.nan], [1.0, np.inf], np.ones((2, 2)), []):
        with pytest.raises(ValueError):
            losses.SampledSoftmax(2, weights=bad)
    with pytest.raises(ValueError, match="catalog"):
        losses.check_sampled(11, None, 10)
    with pytest.raises(ValueError, match="shape"):
        losses.check_sampled(2, np.ones(9), 10)
    S, q = losses.check_sampled(2, np.array([1.0, 3.0]), 2)
    assert S == 2 and np.allclose(q, [0.25, 0.75])
    assert losses.check_sampled(3, None, 10) == (3, None)
