"""Keras-2.0.x Adam (`Adam.get_updates`) restated on top of oracle/keras_semantics.py, and the two oracle models with an
optimizer choice in `train_step` (Adagrad stays the default).  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

    g     = clip_norm(grads, clipnorm)             global norm over the trainable weights
    lr_e  = lr / (1 + decay * iterations)          iterations = updates applied before this one
    t     = iterations + 1
    lr_t  = lr_e * sqrt(1 - beta_2**t) / (1 - beta_1**t)
    m     = beta_1 * m + (1 - beta_1) * g
    v     = beta_2 * v + (1 - beta_2) * g**2
    p     = p - lr_t * m / (sqrt(v) + epsilon)
    iterations += 1                                once per step, whatever was frozen

The update is dense: a coordinate whose gradient is zero still moves by lr_t * m / (sqrt(v) + epsilon)."""
import math

import torch

from . import keras_semantics as ks


def adam_update(p, g, m, v, iterations, lr=0.001, beta_1=0.9, beta_2=0.999, epsilon=1e-8, decay=0.0):
    """One Adam update of one weight; iterations = updates applied before this one.  Returns (p, m, v)."""
    lr_e = lr / (1.0 + decay * iterations)
    t = iterations + 1
    lr_t = lr_e * math.sqrt(1.0 - beta_2 ** t) / (1.0 - beta_1 ** t)
    m2 = beta_1 * m + (1.0 - beta_1) * g
    v2 = beta_2 * v + (1.0 - beta_2) * g * g
    p2 = p - lr_t * m2 / (v2 ** 0.5 + epsilon)
    return p2, m2, v2


class Model(ks.Model):
    """ks.Model with Adam: self.moment holds m, self.accum v (as the device keeps v in the accumulator storage)."""

    def __init__(self, *args, **kw):
        ks.Model.__init__(self, *args, **kw)
        self.moment = None
        self.iterations = 0

    def train_step(self, ids, targets, mask, lr=0.01, epsilon=1e-8, clipnorm=1.0, trainable=None, optimizer="adagrad",
                   beta_1=0.9, beta_2=0.999, decay=0.0, **kw):
        """Returns (loss, clipped grads, norm) like ks.Model.train_step."""
        if optimizer != "adam":
            return ks.Model.train_step(self, ids, targets, mask, lr=lr, epsilon=epsilon, clipnorm=clipnorm,
                                       trainable=trainable, **kw)
        loss, gs = self.grads(ids, targets, mask, **kw)
        ps = self.params()
        if trainable is None:
            trainable = [True] * len(ps)
        gs_c, norm = ks.clip_by_global_norm([g for g, t in zip(gs, trainable) if t], clipnorm)
        it = iter(gs_c)
        gs_full = [next(it) if t else torch.zeros_like(p) for p, t in zip(ps, trainable)]
        if self.accum is None:
            self.accum = [torch.zeros_like(p) for p in ps]
            self.moment = [torch.zeros_like(p) for p in ps]
        new_ps = []
        for i, (p, g, t) in enumerate(zip(ps, gs_full, trainable)):
            if t:
                p, self.moment[i], self.accum[i] = adam_update(p, g, self.moment[i], self.accum[i], self.iterations,
                                                               lr, beta_1, beta_2, epsilon, decay)
            new_ps.append(p)
        self.set_params(new_ps)
        self.iterations += 1
        return loss, gs_full, norm


class SkipModel(ks.SkipModel):
    """ks.SkipModel with Adam; the kernel constraint applies to the updated weights, as with Adagrad."""

    def __init__(self, *args, **kw):
        ks.SkipModel.__init__(self, *args, **kw)
        self.moment = None
        self.iterations = 0

    def train_step(self, ids, x, targets, lr=0.01, epsilon=1e-8, clipnorm=1.0, frozen=(), optimizer="adagrad",
                   beta_1=0.9, beta_2=0.999, decay=0.0, **kw):
        if optimizer != "adam":
            return ks.SkipModel.train_step(self, ids, x, targets, lr=lr, epsilon=epsilon, clipnorm=clipnorm,
                                           frozen=frozen, **kw)
        loss, g = self.grads(ids, x, targets, **kw)
        names = [n for n in self.NAMES if n in self.p and n not in frozen]
        gs, norm = ks.clip_by_global_norm([g[n] for n in names], clipnorm)
        if self.accum is None:
            self.accum = {n: torch.zeros_like(v) for n, v in self.p.items()}
            self.moment = {n: torch.zeros_like(v) for n, v in self.p.items()}
        for n, gc in zip(names, gs):
            self.p[n], self.moment[n], self.accum[n] = adam_update(self.p[n], gc, self.moment[n], self.accum[n],
                                                                   self.iterations, lr, beta_1, beta_2, epsilon, decay)
        self.constrain()
        self.iterations += 1
        return loss, norm
