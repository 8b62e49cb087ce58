"""Carried recurrent state without a GPU: the float64 oracle's chunking invariance and a hand-computed step from a
non-zero state, RecurrentState's take / put / save / load and its mismatch errors, and the C-ABI declarations."""
import os
import re

import numpy as np
import pytest
import torch

from oracle import keras_semantics as ks
from oracle import state as ost
from seq_recommendations_b200 import _lib
from seq_recommendations_b200.state import RecurrentState

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = {"simpleRNN": 1, "LSTM": 4, "GRU": 3}


def _inputs(cell, B, T, H, seed):
    rng = np.random.default_rng(seed)
    xp = torch.tensor(rng.standard_normal((B, T, G[cell] * H)) * 0.5)
    U = torch.tensor(rng.standard_normal((H, G[cell] * H)) / np.sqrt(H))
    L = rng.integers(0, T + 1, size=B)
    L[0] = 0                                                   # an all-pad row
    mask = torch.tensor(np.arange(T)[None, :] >= (T - L)[:, None])
    h0 = torch.tensor(rng.standard_normal((B, H)) * 0.5)
    c0 = torch.tensor(rng.standard_normal((B, H)) * 0.5) if cell == "LSTM" else None
    return xp, U, mask, h0, c0


@pytest.mark.parametrize("cell,act", [("simpleRNN", "tanh"), ("LSTM", "relu"), ("GRU", "tanh")])
def test_oracle_chunking_does_not_matter(cell, act):
    B, T, H = 9, 11, 5
    xp, U, mask, h0, c0 = _inputs(cell, B, T, H, 3)
    whole, h_w, c_w = ost.rnn_forward_state(xp, U, mask, cell, act, h0, c0)
    rng = np.random.default_rng(4)
    splits = [sorted(rng.choice(np.arange(1, T), size=3, replace=False).tolist()), list(range(1, T))]
    for cuts in splits:
        h, c, outs = h0, c0, []
        for a, b in zip([0] + cuts, cuts + [T]):
            o, h, c = ost.rnn_forward_state(xp[:, a:b], U, mask[:, a:b], cell, act, h, c)
            outs.append(o)
        assert torch.allclose(torch.cat(outs, dim=1), whole, rtol=0, atol=1e-12)
        assert torch.allclose(h, h_w, rtol=0, atol=1e-12)
        if cell == "LSTM":
            assert torch.allclose(c, c_w, rtol=0, atol=1e-12)
    # an all-pad chunk holds the state exactly
    o, h, c = ost.rnn_forward_state(xp[:, :4], U, torch.zeros(B, 4, dtype=torch.bool), cell, act, h0, c0)
    assert torch.equal(h, h0) and torch.equal(o, h0.unsqueeze(1).expand(B, 4, H))
    if cell == "LSTM":
        assert torch.equal(c, c0)
    # the zero state is the whole-window scan
    assert torch.equal(ost.rnn_forward_state(xp, U, mask, cell, act)[0], ks.rnn_forward(xp, U, mask, cell, act))


def test_oracle_one_step_known_answer():
    """H = 1, one batch row, one unmasked step: every gate worked out by hand (hard_sigmoid(a) = clip(0.2a + 0.5))."""
    h0, c0 = torch.tensor([[0.5]], dtype=torch.float64), torch.tensor([[-1.0]], dtype=torch.float64)
    m = torch.ones(1, 1, dtype=torch.bool)
    # LSTM, U = [0.2, 0.4, 1.0, -0.6], x = [0.1, 0.3, 0.2, 0.5], linear activation
    xp = torch.tensor([[[0.1, 0.3, 0.2, 0.5]]], dtype=torch.float64)
    U = torch.tensor([[0.2, 0.4, 1.0, -0.6]], dtype=torch.float64)
    _, h, c = ost.rnn_forward_state(xp, U, m, "LSTM", "linear", h0, c0)
    i = 0.2 * (0.1 + 0.1) + 0.5            # 0.54
    f = 0.2 * (0.3 + 0.2) + 0.5            # 0.60
    g = 0.2 + 0.5                          # 0.70
    o = 0.2 * (0.5 - 0.3) + 0.5            # 0.54
    c_want = f * -1.0 + i * g              # -0.222
    assert abs(float(c) - c_want) < 1e-15 and abs(float(h) - o * c_want) < 1e-15
    # GRU, U = [1.0, -1.0, 2.0], x = [0.0, 0.5, 0.1], linear activation: the reset gate multiplies h0 BEFORE U_h
    xp = torch.tensor([[[0.0, 0.5, 0.1]]], dtype=torch.float64)
    U = torch.tensor([[1.0, -1.0, 2.0]], dtype=torch.float64)
    _, h, c = ost.rnn_forward_state(xp, U, m, "GRU", "linear", h0)
    z = 0.2 * 0.5 + 0.5                    # 0.6
    r = 0.2 * (0.5 - 0.5) + 0.5            # 0.5
    hh = 0.1 + r * 0.5 * 2.0               # 0.6
    assert c is None and abs(float(h) - (z * 0.5 + (1 - z) * hh)) < 1e-15
    # SimpleRNN, tanh
    _, h, _ = ost.rnn_forward_state(torch.tensor([[[0.25]]], dtype=torch.float64), torch.tensor([[0.5]],
                                   dtype=torch.float64), m, "simpleRNN", "tanh", h0)
    assert abs(float(h) - np.tanh(0.5)) < 1e-15


def _state(n, cell="LSTM", H=4, seed=0):
    g = torch.Generator().manual_seed(seed)
    return RecurrentState(torch.randn(n, H, generator=g), torch.randn(n, H, generator=g) if cell == "LSTM" else None,
                          cell, H)


@pytest.mark.parametrize("cell", ["LSTM", "GRU"])
def test_take_put_round_trip(cell):
    pool = _state(10, cell)
    before = pool.h.clone()
    idx = [7, 2, 5]
    sub = pool.take(idx)
    assert len(sub) == 3 and torch.equal(sub.h, before[idx])
    sub.h.add_(1.0)                                            # a copy: the pool is untouched
    assert torch.equal(pool.h, before)
    pool.put(idx, sub)
    assert torch.equal(pool.h[idx], before[idx] + 1.0)
    rest = [i for i in range(10) if i not in idx]
    assert torch.equal(pool.h[rest], before[rest])
    pool.put(slice(0, 2), pool.take(slice(8, 10)))
    assert torch.equal(pool.h[0:2], pool.h[8:10])
    if cell == "LSTM":
        assert torch.equal(pool.c[0:2], pool.c[8:10])


def test_save_load_round_trip(tmp_path):
    for cell in ("LSTM", "GRU"):
        s = _state(6, cell, H=3, seed=1)
        p = str(tmp_path / ("s_%s.npz" % cell))
        s.save(p)
        t = RecurrentState.load(p)
        assert t.cell == cell and t.H == 3 and torch.equal(t.h, s.h)
        assert (t.c is None) == (cell != "LSTM")
        if t.c is not None:
            assert torch.equal(t.c, s.c)
    assert not [f for f in os.listdir(tmp_path) if ".tmp." in f]


def test_mismatch_errors():
    s = _state(5, "LSTM", H=4)
    with pytest.raises(ValueError):
        s.check("GRU", 4)
    with pytest.raises(ValueError):
        s.check("LSTM", 8)
    with pytest.raises(ValueError):
        s.check("LSTM", 4, n=6)
    s.check("LSTM", 4, n=5)
    with pytest.raises(ValueError):
        s.put([0, 1], _state(2, "GRU", H=4))
    with pytest.raises(ValueError):
        s.put([0, 1], _state(3, "LSTM", H=4))
    with pytest.raises(ValueError):
        RecurrentState(torch.zeros(2, 4), None, "LSTM", 4)     # an LSTM state needs c
    with pytest.raises(ValueError):
        RecurrentState(torch.zeros(2, 4), torch.zeros(2, 4), "GRU", 4)
    with pytest.raises(ValueError):
        RecurrentState(torch.zeros(2, 5), None, "GRU", 4)


def test_header_and_binding_declare_the_state_entry_points():
    text = open(os.path.join(ROOT, "include", "seqrec_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    for name, n_args in (("seqrec_rnn_forward_state", 13), ("seqrec_rnn_tc_forward_state", 14)):
        m = re.search(r"\bint\s+%s\s*\(([^)]*)\)" % name, text)
        assert m, name
        assert len(m.group(1).split(",")) == n_args == len(_lib.SIGNATURES[name])
