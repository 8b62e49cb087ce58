"""Keras Adam without a GPU: the oracle's update against hand-computed steps, the oracle models' optimizer choice, and
the optimizer spec objects."""
import math

import numpy as np
import pytest
import torch

from oracle import adam as oa
from oracle import keras_semantics as ks
from seq_recommendations_b200 import optimizers as opt
from seq_recommendations_b200 import synthetic


def _t(x):
    return torch.tensor([x], dtype=torch.float64)


def test_adam_update_known_answers():
    """p = 1, lr = 0.1, default betas and epsilon: g = 0.5, then g = 0 (p still moves), then g = -0.25 with decay 0.5."""
    p, m, v = _t(1.0), _t(0.0), _t(0.0)
    p, m, v = oa.adam_update(p, _t(0.5), m, v, 0, lr=0.1)
    # step 1: lr_t = 0.1 * sqrt(0.001) / 0.1; m = 0.05; v = 0.00025; the move is lr * g / (|g| + eps / sqrt(1 - beta_2))
    assert math.isclose(float(m), 0.05, rel_tol=1e-14) and math.isclose(float(v), 0.00025, rel_tol=1e-14)
    assert math.isclose(float(p), 1.0 - 0.1 * 0.5 / (0.5 + 1e-8 / math.sqrt(0.001)), rel_tol=1e-14)
    assert math.isclose(float(p), 0.9000000632455132, rel_tol=1e-14)
    # step 2, zero gradient: m and v decay and p moves by lr_t * m / (sqrt(v) + eps), lr_t = 0.1 * sqrt(1 - 0.999^2) / 0.19
    p, m, v = oa.adam_update(p, _t(0.0), m, v, 1, lr=0.1)
    assert math.isclose(float(m), 0.045, rel_tol=1e-14) and math.isclose(float(v), 0.00024975, rel_tol=1e-14)
    assert math.isclose(float(p), 0.8329942802312424, rel_tol=1e-14)
    # step 3 with decay: lr_e = 0.1 / (1 + 0.5 * 2)
    p, m, v = oa.adam_update(p, _t(-0.25), m, v, 2, lr=0.1, decay=0.5)
    assert math.isclose(float(m), 0.0155, rel_tol=1e-12) and math.isclose(float(v), 0.00031200025, rel_tol=1e-12)
    assert math.isclose(float(p), 0.8241309253449605, rel_tol=1e-14)


def test_adam_update_leaves_untouched_coordinates_bit_for_bit():
    p = torch.tensor([0.3, -1.25, 7.0], dtype=torch.float64)
    z = torch.zeros(3, dtype=torch.float64)
    for k in range(5):
        p2, m2, v2 = oa.adam_update(p, z, z, z, k, lr=0.1, decay=0.1)
        assert torch.equal(p2, p) and not m2.any() and not v2.any()


def test_oracle_models_take_the_optimizer_choice():
    """Adagrad stays the default of the Adam-capable oracle models; Adam counts every step and skips frozen weights."""
    V, H, T, B = 20, 6, 5, 4
    ws = synthetic.make_weights("GRU", V, H, seed=1)
    ids, tgt = synthetic.make_batch(V, T, B, seed=2, min_len=1)
    i, t = torch.tensor(ids.astype(np.int64)), torch.tensor(tgt.astype(np.int64))
    a, b = ks.Model("GRU", "tanh", ws, dtype=torch.float64), oa.Model("GRU", "tanh", ws, dtype=torch.float64)
    a.train_step(i, t, i >= 0, lr=0.05)
    b.train_step(i, t, i >= 0, lr=0.05)
    for x, y in zip(a.params(), b.params()):
        assert torch.equal(x, y)
    c = oa.Model("GRU", "tanh", ws, dtype=torch.float64)
    for _ in range(2):
        c.train_step(i, t, i >= 0, lr=0.01, optimizer="adam", trainable=[True, True, True, False])
    assert c.iterations == 2
    assert np.array_equal(c.W_out.numpy(), ws[3].astype(np.float64))
    assert not c.moment[3].any() and not c.accum[3].any()
    never = np.setdiff1d(np.arange(V), ids[ids >= 0])           # W_in rows no batch touched: bit for bit
    assert len(never) and np.array_equal(c.W_in.numpy()[never], ws[0].astype(np.float64)[never])


def test_adam_spec_objects():
    o = opt.Adam()
    assert (o.kind, o.lr, o.beta_1, o.beta_2, o.epsilon, o.decay, o.clipnorm) == ("adam", 0.001, 0.9, 0.999, 1e-8, 0.0,
                                                                                   None)
    assert opt.resolve(o) is o
    o = opt.Adam(lr=0.01, beta_1=0.8, beta_2=0.99, epsilon=1e-7, decay=0.1, clipnorm=1.0)
    assert (o.lr, o.beta_1, o.beta_2, o.epsilon, o.decay, o.clipnorm) == (0.01, 0.8, 0.99, 1e-7, 0.1, 1.0)
    assert opt.resolve(o) is o
    assert opt.resolve("adam") == "adam"                         # the string keeps its compile-only meaning
    with pytest.raises(NotImplementedError):
        opt.Adam(clipvalue=0.5)

    class KerasLikeAdam(object):                                 # a foreign object of kind adam
        kind = "adam"
        lr, beta_1, beta_2, epsilon, decay, clipnorm = 0.002, 0.9, 0.999, 1e-8, 0.0, None
    k = KerasLikeAdam()
    assert opt.resolve(k) is k

    class Adam(object):                                          # e.g. a real keras.optimizers.Adam (by type name)
        lr, beta_1, beta_2, epsilon, decay = 0.002, 0.9, 0.999, 1e-8, 0.0
    k = Adam()
    assert opt.resolve(k) is k
