"""Keras `initial_state` restated on top of oracle/keras_semantics.py: the masked recurrence continued from a carried
state.  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py)."""
import torch

from .keras_semantics import GATES, activation, hard_sigmoid


def rnn_forward_state(xp, U, mask, cell, act_name, h0=None, c0=None):
    """`rnn_forward` continued from a carried state (Keras `initial_state`): h0 (B,H), and c0 (B,H) for LSTM; None
    stands for zeros.  A masked step holds h and c.  Returns (Hout (B,T,H), h_T, c_T) with c_T None unless LSTM.
    Chunking does not matter: advancing by a and then by b from (h_T, c_T) gives the state of a|b."""
    B, T, GH = xp.shape
    G = GATES[cell]
    H = GH // G
    act = activation(act_name)
    h = xp.new_zeros(B, H) if h0 is None else h0.to(xp.dtype).clone()
    c = xp.new_zeros(B, H) if c0 is None else c0.to(xp.dtype).clone()
    outs = []
    for t in range(T):
        m = mask[:, t].unsqueeze(1)
        x = xp[:, t]
        if cell == "simpleRNN":
            h_new = act(x + h @ U)
        elif cell == "LSTM":
            i = hard_sigmoid(x[:, 0:H] + h @ U[:, 0:H])
            f = hard_sigmoid(x[:, H:2 * H] + h @ U[:, H:2 * H])
            g = act(x[:, 2 * H:3 * H] + h @ U[:, 2 * H:3 * H])
            o = hard_sigmoid(x[:, 3 * H:4 * H] + h @ U[:, 3 * H:4 * H])
            c_new = f * c + i * g
            h_new = o * act(c_new)
            c = torch.where(m, c_new, c)
        elif cell == "GRU":
            z = hard_sigmoid(x[:, 0:H] + h @ U[:, 0:H])
            r = hard_sigmoid(x[:, H:2 * H] + h @ U[:, H:2 * H])
            hh = act(x[:, 2 * H:3 * H] + (r * h) @ U[:, 2 * H:3 * H])
            h_new = z * h + (1.0 - z) * hh
        else:
            raise ValueError(cell)
        h = torch.where(m, h_new, h)
        outs.append(h)
    Hout = torch.stack(outs, dim=1) if outs else xp.new_zeros(B, 0, H)
    return Hout, h, (c if cell == "LSTM" else None)
