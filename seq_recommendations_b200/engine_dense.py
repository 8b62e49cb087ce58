"""Device-side orchestration of the HISTORY-FEATURE / SKIP-BRANCH models: RNNFullModel with any of x_to_z / x_to_y /
y_to_y (/root/reference/model.py:354-358, :376-392) and NoRecurrenceModel (model.py:264-319).

    logits  z = [hs ; x] . W_toy (+ b_out)  +  A[y_{t-1}] (+ a_bias)          hs = dropout(z_to_z_output)
    xp      = W_in[y_{t-1}]  +  x . W_in[V:]  + b                             (the RNN sees concatenate([y, x]))

These models carry per-(token, item) logit terms (a (V,V) transition kernel, history counts per item), and the reference
runs them on small catalogs (MSNBC: V = 17), so here the (N,V) logits ARE materialised -- unlike the y_to_z-only hot
path of engine.py, whose fused kernels never hold them.  The recurrent scan, the row gather / scatter-add, the clip +
Adagrad kernels are the ones of the hot path; the dense products run on the tcgen05 GEMM (csrc/gemm_tc.cu, 3-pass split
= fp32-grade) when they are large enough to fill tiles, else on the fp32 SIMT GEMMs.  Single process (the reference's
experiment scripts for these variants drive one device).

Same public methods as engine.HotPath (train_batch / loss_batch / grad_batch / predict_batch / target_prob_batch /
target_rank_batch / topk_batch / hidden_batch, get_weight / set_weight, trainable, set_optimizer), so model._Net drives
either.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import ACT, CELL, call, ptr
from .dist import Comm
from .engine import GATES, _align, _optimizer_spec
from .gemm import gemm

NAMES = ["W_in", "U", "b", "W_toy", "b_out", "A", "a_bias"]


class DensePath:
    def __init__(self, cell, act, y_dim, x_dim, hidden, weights, y_to_z=True, x_to_z=False, x_to_y=False, y_to_y=False,
                 diag_b=True, device=None, seed=0, tc="x3"):
        if not torch.cuda.is_available():
            raise _lib.SeqrecError("seq_recommendations_b200 needs a CUDA device (sm_100a); there is no CPU path")
        _lib.load()
        if cell is not None and cell not in CELL:
            raise ValueError("rnn_type must be one of %s" % sorted(CELL))
        if cell is not None and not (y_to_z or x_to_z):
            raise ValueError("ERROR: the model needs an input into z's! either x or y should be added.")
        if cell is None and not (x_to_y or y_to_y):
            raise ValueError("ERROR: the model needs an input! either x or y should be added.")
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.cell, self.act = cell, act
        self.G = GATES[cell] if cell else 0
        self.V, self.Fx, self.H = int(y_dim), int(x_dim or 0), int(hidden) if cell else 0
        self.GH = self.G * self.H
        self.y_to_z, self.x_to_z = bool(y_to_z) and cell is not None, bool(x_to_z) and cell is not None
        self.x_to_y, self.y_to_y, self.diag_b = bool(x_to_y), bool(y_to_y), bool(diag_b)
        if self.x_to_y and self.diag_b and self.Fx != self.V:
            raise ValueError("the diagonal constraint of the x -> y kernel needs x_dim == y_dim (model.py:57)")
        self.uses_y = self.y_to_z or self.y_to_y
        self.uses_x = self.x_to_z or self.x_to_y
        self.F = (self.V if self.y_to_z else 0) + (self.Fx if self.x_to_z else 0)     # rows of W_in
        self.Ft = self.H + (self.Fx if self.x_to_y else 0)                            # rows of W_toy
        self.comm = Comm()
        self.vocab_parallel = False
        self.V_total = self.V
        self.dropout_in = self.dropout_out = self.dropout_rec = 0.0
        self.seed = int(seed)
        self.rng_state = torch.zeros(2, dtype=torch.int64, device=self.device)
        self.tc_mode = tc
        self.tc_x3 = tc == "x3"
        self.opt = None
        self.prof = None
        f32 = torch.float32
        dev = self.device
        shapes = {}
        if cell is not None:
            shapes.update(W_in=(self.F, self.GH), U=(self.H, self.GH), b=(self.GH,))
        if self.Ft > 0:
            shapes.update(W_toy=(self.Ft, self.V), b_out=(self.V,))
        if self.y_to_y:
            shapes.update(A=(self.V, self.V), a_bias=(self.V,))
        self.present = {n: n in weights and weights[n] is not None for n in shapes}
        self._seg, o = {}, 0
        for n in NAMES:
            if n in shapes and self.present[n]:
                size = int(np.prod(shapes[n]))
                self._seg[n] = (o, size, shapes[n])
                o += _align(size)
        # one flat parameter / gradient / accumulator buffer: ONE norm pass and ONE Adagrad launch; the step floats
        # [n_valid, loss_sum] and the integer scalars sit around the gradients so that one fill clears them together
        self.flat_p = torch.zeros(o, dtype=f32, device=dev)
        self.flat_a = torch.zeros(o, dtype=f32, device=dev)
        self._gbuf = torch.zeros(64 + o + 4, dtype=f32, device=dev)
        self.stepf = self._gbuf[:64]
        self.flat_g = self._gbuf[64:64 + o]
        self.scal = self._gbuf[64 + o:].view(torch.int32)
        self.n_valid_f, self.step_loss_sum = self.stepf[0:1], self.stepf[1:2]
        self.sumsq = self.scal[2:4].view(torch.float64)
        for n, (off, size, shp) in self._seg.items():
            setattr(self, n, self.flat_p[off:off + size].view(shp))
            setattr(self, "d" + n, self.flat_g[off:off + size].view(shp))
            setattr(self, "a" + n, self.flat_a[off:off + size].view(shp))
        for n in NAMES:
            if n not in self._seg:
                setattr(self, n, None)
                setattr(self, "d" + n, None)
        self.trainable = {n: True for n in self._seg}
        self.flat_m = None                        # Adam's first moments (m* views), allocated when Adam is selected
        self.iterations = torch.zeros(1, dtype=torch.int64, device=dev)
        self.Ut = torch.empty((self.GH, self.H), dtype=f32, device=dev) if cell else None
        # scratch of the row scatter-adds (dense destinations: the flags are cleared after every use)
        nrow = max(self.V, 1)
        self.touched = torch.zeros(nrow, dtype=torch.int32, device=dev)
        self.rows = torch.empty(nrow, dtype=torch.int32, device=dev)
        self.n_rows = torch.zeros(1, dtype=torch.int32, device=dev)
        self.err_flag = torch.zeros(1, dtype=torch.int32, device=dev)
        self._work = {}
        self._w_version = 0
        for n in self._seg:
            self.set_weight(n, weights[n])

    # ------------------------------------------------------------------------------------------------ plumbing
    @property
    def stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def weight_names(self):
        return [n for n in NAMES if n in self._seg]

    def get_weight(self, name, prefix=""):
        return getattr(self, prefix + name).detach().cpu().numpy().copy()

    def set_weight(self, name, value, sync=True, prefix=""):
        t = getattr(self, prefix + name)
        v = np.asarray(value, dtype=np.float32)
        if tuple(v.shape) != tuple(t.shape):
            raise ValueError("weight %s: shape %s does not match %s" % (name, v.shape, tuple(t.shape)))
        t.copy_(torch.from_numpy(np.ascontiguousarray(v)))
        self._w_version += 1

    def get_accumulator(self, name):
        return self.get_weight(name, prefix="a")

    def set_accumulator(self, name, value):
        self.set_weight(name, value, prefix="a")

    def get_moments(self, name):
        return self.get_weight(name, prefix="m"), self.get_weight(name, prefix="a")

    def set_moments(self, name, m, v):
        self.set_weight(name, m, prefix="m")
        self.set_weight(name, v, prefix="a")

    def get_iterations(self):
        return int(self.iterations.item())

    def set_iterations(self, k):
        self.iterations.fill_(int(k))

    def get_weights(self):
        return [self.get_weight(n) for n in self.weight_names()]

    def set_weights(self, weights):
        names = self.weight_names()
        if len(weights) != len(names):
            raise ValueError("expected %d weight arrays, got %d" % (len(names), len(weights)))
        for n, w in zip(names, weights):
            self.set_weight(n, w)

    def reset_optimizer_state(self):
        self.flat_a.zero_()
        if self.flat_m is not None:
            self.flat_m.zero_()
        self.iterations.zero_()

    def set_optimizer(self, kind="adagrad", lr=0.01, epsilon=1e-8, clipnorm=0.0, decay=0.0, beta_1=0.9, beta_2=0.999):
        """Adagrad (the reference's optimizer, experiments_methods.py:41) or Keras Adam; resets the optimizer state."""
        self.opt = _optimizer_spec(kind, lr, epsilon, clipnorm, decay, beta_1, beta_2)
        if kind == "adam" and self.flat_m is None:
            self.flat_m = torch.zeros_like(self.flat_a)
            for n, (off, size, shp) in self._seg.items():
                setattr(self, "m" + n, self.flat_m[off:off + size].view(shp))
        self.reset_optimizer_state()

    def check_errors(self):
        bits = int(self.err_flag.item())
        if bits:
            self.err_flag.zero_()
            raise ValueError("batch holds an item id or a target outside [0, %d)" % self.V)

    def _check_host_ids(self, ids, tgt):
        for a in (ids, tgt):
            if a is not None and not isinstance(a, torch.Tensor):
                a = np.asarray(a)
                if a.size and int(a.max()) >= self.V:
                    raise ValueError("id %d is outside the catalog (%d items)" % (int(a.max()), self.V))

    def _dropout(self, shape, rate):
        t = torch.empty(shape, dtype=torch.float32, device=self.device)
        call("seqrec_dropout_mask_dev", ptr(t), t.numel(), float(rate), self.seed, ptr(self.rng_state), self.stream)
        return t

    # ------------------------------------------------------------------------------------------------ products
    def _gemm(self, A, Bm, C, form, bias=None, accumulate=False):
        gemm(self, A, Bm, C, form, bias=bias, accumulate=accumulate)

    # ------------------------------------------------------------------------------------------------ staging
    def work(self, B, T):
        key = (B, T)
        w = self._work.get(key)
        if w is None:
            if len(self._work) > 4:
                self._work.clear()
            w = self._work[key] = _DenseWork(self, B, T)
        return w

    def _stage(self, w, ids, tgt, x):
        """ids (B,T) int (pad < 0) or None; x (B,T,Fx) float or None; tgt (B,T) int or None.  Builds the time-major
        buffers and the masks: m_y = ids >= 0, m_x = any(x != 0) (Masking(0.0), model.py:335, :340), the scan mask =
        AND of the masks of the inputs into z (concatenate), the loss mask = AND over everything `add` / `concatenate`
        merged in front of the softmax (SURVEY 8(c) item 1)."""
        self._check_host_ids(ids, tgt)
        dev = self.device
        i32 = torch.int32
        self._gbuf.zero_()
        if self.uses_y:
            if ids is None:
                raise ValueError("this model needs the y (item) input")
            src = ids if isinstance(ids, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(ids, dtype=np.int32))
            w.ids_bt.copy_(src.to(dev, dtype=i32))
        else:
            w.ids_bt.zero_()
        have_t = tgt is not None
        if have_t:
            src = tgt if isinstance(tgt, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(tgt, dtype=np.int32))
            w.tgt_bt.copy_(src.to(dev, dtype=i32))
        else:
            w.tgt_bt.zero_()
        w.scal_tmp.zero_()
        fmt_t = have_t and self.uses_y        # (an x-only model has no y pads for the formatter to pair targets with)
        call("seqrec_format_batch", ptr(w.ids_bt), ptr(w.tgt_bt) if fmt_t else None, ptr(w.ids),
             ptr(w.tgt) if fmt_t else None, ptr(w.mask_y), ptr(w.scal_tmp), w.B, w.T, self.V, self.V,
             ptr(self.err_flag), self.stream)
        m_y = w.mask_y.bool() if self.uses_y else None
        m_x = None
        if self.uses_x:
            if x is None:
                raise ValueError("this model needs the x (history feature) input")
            xd = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
            xd = xd.to(dev, dtype=torch.float32)
            if tuple(xd.shape) != (w.B, w.T, self.Fx):
                raise ValueError("x input has shape %s, expected %s" % (tuple(xd.shape), (w.B, w.T, self.Fx)))
            w.x.copy_(xd.permute(1, 0, 2))
            m_x = (w.x != 0).any(dim=-1)
        if not self.uses_y:
            w.ids.fill_(-1)
        zm = [m for m, used in ((m_y, self.y_to_z), (m_x, self.x_to_z)) if used]
        om = list(zm) if self.cell else []
        om += [m for m, used in ((m_x, self.x_to_y), (m_y, self.y_to_y and self.cell is None)) if used]
        if self.cell:
            w.mask_z.copy_(zm[0] if len(zm) == 1 else zm[0] & zm[1])
        mo = om[0]
        for m in om[1:]:
            mo = mo & m
        w.mask_o.copy_(mo)
        if have_t:
            w.tgt.copy_(torch.where(mo, w.tgt_bt.t(), torch.full_like(w.tgt, -1)))
        self.scal[0:1].copy_(mo.sum().to(i32))
        return have_t

    # ------------------------------------------------------------------------------------------------ forward
    def _forward_logits(self, w, training):
        st = self.stream
        N = w.N
        w.in_scale = w.x_drop = w.hscale = w.rec_mask = None
        x_in = w.x.view(N, self.Fx) if self.uses_x else None
        if self.cell:
            # ---- xp = [y ; x] . W_in + b: row gather for the one-hot half (K1), GEMM for the dense half (K2)
            Vy = self.V if self.y_to_z else 0
            if training and self.dropout_in > 0:
                # Dropout on the concatenated RNN input (model.py:356-357): one factor per element; the one-hot half
                # only ever sees the factor at its hot position
                if self.y_to_z:
                    w.in_scale = self._dropout((N,), self.dropout_in)
                if self.x_to_z:
                    w.x_drop = x_in * self._dropout((N, self.Fx), self.dropout_in)
            if self.y_to_z:
                call("seqrec_gather_rows", ptr(self.W_in), ptr(self.b), ptr(w.ids), ptr(w.mask_y), ptr(w.in_scale),
                     ptr(w.xg), N, self.V, self.GH, st)
            if self.x_to_z:
                xz = w.x_drop if w.x_drop is not None else x_in
                self._gemm(xz, self.W_in[Vy:], w.xg.view(N, self.GH), "nn", bias=None if self.y_to_z else self.b,
                           accumulate=self.y_to_z)
            if training and self.dropout_rec > 0:
                w.rec_mask = self._dropout((self.G, w.B, self.H), self.dropout_rec)
                call("seqrec_rnn_forward_rd", CELL[self.cell], ACT[self.act], ptr(w.xg), ptr(self.U), ptr(w.rec_mask),
                     ptr(w.mask_z), ptr(w.hout), ptr(w.cst), w.T, w.B, self.H, st)
            else:
                call("seqrec_rnn_forward", CELL[self.cell], ACT[self.act], ptr(w.xg), ptr(self.U), ptr(w.mask_z),
                     ptr(w.hout), ptr(w.cst), w.T, w.B, self.H, st)
            hs = w.hout.view(N, self.H)
            if training and self.dropout_out > 0:
                w.hscale = self._dropout((N, self.H), self.dropout_out)
                hs = hs * w.hscale
            w.hs = hs
            # ---- logits: [hs ; x] . W_toy + b_out
            self._gemm(hs, self.W_toy[:self.H], w.Z, "nn", bias=self.b_out)
            if self.x_to_y:
                self._gemm(x_in, self.W_toy[self.H:], w.Z, "nn", accumulate=True)
        else:
            if self.x_to_y:
                self._gemm(x_in, self.W_toy, w.Z, "nn", bias=self.b_out)
            else:
                w.Z.zero_()
        if self.y_to_y:
            # one-hot(y_{t-1}) . A == row lookup of A; pads are all-zero rows (bias only)
            call("seqrec_add_rows", ptr(w.Z), ptr(self.A), ptr(self.a_bias), ptr(w.ids), N, self.V, st)

    def _stats(self, w, train):
        st = self.stream
        call("seqrec_softmax_rows_stats", ptr(w.Z), ptr(w.tgt), ptr(w.m), ptr(w.s), ptr(w.zy), w.N, self.V, st)
        if train:
            call("seqrec_ce_finalize_mean", ptr(w.m), ptr(w.s), ptr(w.zy), ptr(w.mask_o), ptr(w.m), ptr(w.s), ptr(w.ce),
                 ptr(w.py), ptr(w.coef), ptr(self.step_loss_sum), ptr(self.scal[0:1]), ptr(self.n_valid_f),
                 ptr(w.loss_mean), w.N, 1, None, st)
        else:
            call("seqrec_ce_finalize", ptr(w.m), ptr(w.s), ptr(w.zy), ptr(w.mask_o), ptr(w.m), ptr(w.s), ptr(w.ce),
                 ptr(w.py), ptr(w.coef), ptr(w.loss_sum), w.N, 1, st)

    # ------------------------------------------------------------------------------------------------ backward
    def _backward(self, w):
        """Un-normalised gradients of every present weight into flat_g (the optimiser divides by n_valid)."""
        st = self.stream
        N = w.N
        x_in = w.x.view(N, self.Fx) if self.uses_x else None
        call("seqrec_softmax_rows_dlogit", ptr(w.Z), ptr(w.tgt), ptr(w.m), ptr(w.s), ptr(w.coef), N, self.V, st)
        dZ = w.Z
        if self.db_out is not None:
            call("seqrec_colsum", ptr(dZ), ptr(self.db_out), N, self.V, self.V, st)
        if self.y_to_y:
            if self.da_bias is not None:
                call("seqrec_colsum", ptr(dZ), ptr(self.da_bias), N, self.V, self.V, st)
            self._scatter_rows(dZ, w.ids, w.mask_y, None, self.dA, self.V)
        if self.cell:
            self._gemm(w.hs, dZ, self.dW_toy[:self.H], "tn")
            if self.x_to_y:
                self._gemm(x_in, dZ, self.dW_toy[self.H:], "tn")
            self._gemm(dZ, self.W_toy[:self.H], w.dh.view(N, self.H), "nt")
            if w.hscale is not None:
                w.dh.view(N, self.H).mul_(w.hscale)
            call("seqrec_transpose", ptr(self.U), ptr(self.Ut), self.H, self.GH, st)
            if w.rec_mask is not None:
                call("seqrec_rnn_backward_rd", CELL[self.cell], ACT[self.act], ptr(w.xg), ptr(self.Ut), ptr(w.rec_mask),
                     ptr(w.mask_z), ptr(w.hout), ptr(w.cst), ptr(w.dh), w.T, w.B, self.H, st)
                call("seqrec_rnn_weight_grad_rd", CELL[self.cell], ptr(w.xg), ptr(w.hout), ptr(w.cst), ptr(w.rec_mask),
                     ptr(w.scratch), ptr(self.dU), ptr(self.db if self.db is not None else w.db_tmp), w.T, w.B, self.H,
                     st)
            else:
                call("seqrec_rnn_backward", CELL[self.cell], ACT[self.act], ptr(w.xg), ptr(self.U), ptr(self.Ut),
                     ptr(w.mask_z), ptr(w.hout), ptr(w.cst), ptr(w.dh), w.T, w.B, self.H, st)
                call("seqrec_rnn_weight_grad", CELL[self.cell], ptr(w.xg), ptr(w.hout), ptr(w.cst), ptr(self.dU),
                     ptr(self.db if self.db is not None else w.db_tmp), w.T, w.B, self.H, st)
            dxp = w.xg.view(N, self.GH)
            Vy = self.V if self.y_to_z else 0
            if self.y_to_z:
                self._scatter_rows(dxp, w.ids, w.mask_y, w.in_scale, self.dW_in, self.GH)
            if self.x_to_z:
                xz = w.x_drop if w.x_drop is not None else x_in
                self._gemm(xz, dxp, self.dW_in[Vy:], "tn")
        elif self.x_to_y:
            self._gemm(x_in, dZ, self.dW_toy, "tn")

    def _scatter_rows(self, src, ids, mask, scale, dst, width):
        """dst[ids[n], :] += scale[n] * src[n, :] into a DENSE (zeroed) destination; the touched-row bookkeeping of the
        kernel is scratch here and is cleared again."""
        self.n_rows.zero_()
        call("seqrec_scatter_add_rows", ptr(src), ptr(ids), ptr(mask), ptr(scale), ptr(dst), ptr(self.touched),
             ptr(self.rows), ptr(self.n_rows), src.shape[0], self.V, width, self.stream)
        self.touched.zero_()

    def _apply_update(self):
        st = self.stream
        o = self.opt
        den = ptr(self.n_valid_f)
        segs = [(n,) + self._seg[n][:2] for n in self.weight_names()]
        all_on = all(self.trainable[n] for n, _, _ in segs)
        self.sumsq.zero_()
        if o["clipnorm"] > 0:
            if all_on:
                call("seqrec_sumsq", ptr(self.flat_g), self.flat_g.numel(), ptr(self.sumsq), st)
            else:
                for n, off, sz in segs:
                    if self.trainable[n]:
                        call("seqrec_sumsq", ptr(self.flat_g[off:off + sz]), sz, ptr(self.sumsq), st)
        if o["kind"] == "adam":
            for off, sz in ([(0, self.flat_p.numel())] if all_on else
                            [(off, sz) for n, off, sz in segs if self.trainable[n]]):
                call("seqrec_adam", ptr(self.flat_p[off:off + sz]), ptr(self.flat_g[off:off + sz]),
                     ptr(self.flat_m[off:off + sz]), ptr(self.flat_a[off:off + sz]), sz, o["lr"], o["beta_1"],
                     o["beta_2"], o["eps"], o["decay"], o["clipnorm"], ptr(self.sumsq), den, ptr(self.iterations), st)
        elif all_on:
            call("seqrec_adagrad", ptr(self.flat_p), ptr(self.flat_g), ptr(self.flat_a), self.flat_p.numel(), o["lr"],
                 o["eps"], o["clipnorm"], ptr(self.sumsq), den, st)
        else:
            for n, off, sz in segs:
                if self.trainable[n]:
                    call("seqrec_adagrad", ptr(self.flat_p[off:off + sz]), ptr(self.flat_g[off:off + sz]),
                         ptr(self.flat_a[off:off + sz]), sz, o["lr"], o["eps"], o["clipnorm"], ptr(self.sumsq), den, st)
        if self.x_to_y and self.diag_b and self.trainable.get("W_toy", False):
            # Keras applies the kernel constraint to the UPDATED weights (model.py:379, :300-301)
            call("seqrec_diag_constraint", ptr(self.W_toy), self.H, self.V, st)
        if o["kind"] == "adam":
            self.iterations.add_(1)
        self._w_version += 1

    # ------------------------------------------------------------------------------------------------ public steps
    def _shape(self, ids, x):
        return tuple(int(v) for v in (ids.shape[:2] if ids is not None else x.shape[:2]))

    def train_batch(self, ids, tgt, x_dense=None):
        if self.opt is None:
            raise _lib.SeqrecError("compile_model / set_optimizer must be called before training")
        w = self.work(*self._shape(ids, x_dense))
        self._stage(w, ids, tgt, x_dense)
        self._forward_logits(w, training=True)
        self._stats(w, train=True)
        self._backward(w)
        self._apply_update()
        return w.loss_mean.clone()

    def grad_batch(self, ids, tgt, x_dense=None):
        """fwd + bwd without the update: loss and a dict of normalised gradients (parity tests)."""
        w = self.work(*self._shape(ids, x_dense))
        self._stage(w, ids, tgt, x_dense)
        self._forward_logits(w, training=True)
        self._stats(w, train=True)
        self._backward(w)
        self.check_errors()
        nv = float(self.n_valid_f.item())
        grads = {n: (getattr(self, "d" + n).double() / nv).float().cpu().numpy() for n in self.weight_names()}
        return float(self.step_loss_sum.item()) / nv, grads, {}

    def loss_batch(self, ids, tgt, x_dense=None):
        w = self.work(*self._shape(ids, x_dense))
        self._stage(w, ids, tgt, x_dense)
        self._forward_logits(w, training=False)
        self._stats(w, train=False)
        return w.loss_sum.clone(), self.scal[0:1].to(torch.float32)

    def predict_batch(self, ids, x_dense=None):
        w = self.work(*self._shape(ids, x_dense))
        self._stage(w, ids, None, x_dense)
        self._forward_logits(w, training=False)
        self._stats(w, train=False)
        probs = torch.empty((w.B, w.T, self.V), dtype=torch.float32, device=self.device)
        call("seqrec_softmax_rows_probs", ptr(w.Z), ptr(w.m), ptr(w.s), ptr(probs), w.T, w.B, self.V, self.stream)
        return probs

    def target_prob_batch(self, ids, tgt, x_dense=None):
        w = self.work(*self._shape(ids, x_dense))
        self._stage(w, ids, tgt, x_dense)
        self._forward_logits(w, training=False)
        self._stats(w, train=False)
        return w.py.view(w.T, w.B).t().contiguous()

    def target_rank_batch(self, ids, tgt, x_dense=None, last_step_only=False):
        """Rank of the true next item in the materialised logits (stable descending order, ties to the lower item id;
        pads 0): (B,T) int32 device tensor, or (B,) for the last step only."""
        w = self.work(*self._shape(ids, x_dense))
        self._stage(w, ids, tgt, x_dense)
        self._forward_logits(w, training=False)
        rank = torch.empty(w.N, dtype=torch.int32, device=self.device)
        call("seqrec_rows_rank", ptr(w.Z), ptr(w.tgt), ptr(rank), w.N, self.V, self.stream)
        rank = rank.view(w.T, w.B)
        return rank[w.T - 1].contiguous() if last_step_only else rank.t().contiguous()

    def topk_batch(self, ids, k, last_step_only=True, x_dense=None):
        """Top-k next items from the materialised probabilities: stable descending order, ties to the lower item id."""
        probs = self.predict_batch(ids, x_dense)
        if last_step_only:
            probs = probs[:, -1]
        order = torch.sort(probs, dim=-1, descending=True, stable=True)
        return order.indices[..., :k].to(torch.int32).contiguous(), order.values[..., :k].contiguous()

    def hidden_batch(self, ids, x_dense=None):
        if not self.cell:
            raise NotImplementedError("NoRecurrenceModel has no recurrent layer")
        w = self.work(*self._shape(ids, x_dense))
        self._stage(w, ids, None, x_dense)
        self._forward_logits(w, training=False)
        return w.hout.permute(1, 0, 2).contiguous()


class _DenseWork:
    def __init__(self, hp, B, T):
        dev = hp.device
        N = B * T
        f32, i32 = torch.float32, torch.int32
        self.B, self.T, self.N = B, T, N
        self.ids_bt = torch.empty((B, T), dtype=i32, device=dev)
        self.tgt_bt = torch.empty((B, T), dtype=i32, device=dev)
        self.ids = torch.empty((T, B), dtype=i32, device=dev)
        self.tgt = torch.empty((T, B), dtype=i32, device=dev)
        self.mask_y = torch.empty((T, B), dtype=torch.uint8, device=dev)
        self.mask_z = torch.empty((T, B), dtype=torch.uint8, device=dev)
        self.mask_o = torch.empty((T, B), dtype=torch.uint8, device=dev)
        self.scal_tmp = torch.zeros(1, dtype=i32, device=dev)
        self.x = torch.zeros((T, B, max(hp.Fx, 1)), dtype=f32, device=dev) if hp.uses_x else None
        if hp.cell:
            self.xg = torch.empty((T, B, hp.GH), dtype=f32, device=dev)
            self.hout = torch.empty((T, B, hp.H), dtype=f32, device=dev)
            self.cst = torch.empty((T, B, hp.H), dtype=f32, device=dev)
            self.dh = torch.empty((T, B, hp.H), dtype=f32, device=dev)
            self.scratch = torch.empty((T, B, hp.H), dtype=f32, device=dev)
            self.db_tmp = torch.zeros(hp.GH, dtype=f32, device=dev)
        self.Z = torch.empty((N, hp.V), dtype=f32, device=dev)
        self.m, self.s, self.zy, self.ce, self.py, self.coef = (torch.zeros(N, dtype=f32, device=dev) for _ in range(6))
        self.loss_sum = torch.zeros(1, dtype=f32, device=dev)
        self.loss_mean = torch.zeros(1, dtype=f32, device=dev)
        self.in_scale = self.x_drop = self.hscale = self.rec_mask = self.hs = None
