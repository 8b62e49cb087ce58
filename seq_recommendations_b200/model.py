"""Drop-in mirror of the reference's model.py surface for the recurrent next-item models, backed by the B200 kernels.

Same class names, constructor kwargs, method signatures and return conventions as /root/reference/model.py:170-403
(`BaseRNNModel`, `RNNBaseline`, `RNNFullModel`, `ModelResults`, `ValLossHistoryCut`), so the reference's drivers
(experiments_methods.py:19-50, :188-249) run against this module unchanged.  `self.model` plays the role of the Keras
`Model` the reference reaches into (`fit`, `evaluate`, `predict`, `get_weights`, `get_layer`, `load_weights`, ...).

Scope (SURVEY §8): RNNFullModel -- the `y_to_z`-only form ("ytoz", experiments_server.py:106-114) on the fused hot path
(engine.HotPath), the x_to_z / x_to_y / y_to_y history-feature and skip branches on engine_dense.DensePath --
RNNBaseline and NoRecurrenceModel; cells simpleRNN / LSTM (the reference's) and GRU (north-star).

Additive (not in the reference): id-format batches ((N,T) / (N,T,1) integer arrays, pad < 0), `predict_target_prob`,
`predict_topk`, `predict_target_rank` / `evaluate_ranking` (rank of the true next item; Recall@k, MRR@k, NDCG@k) and the
`RankingMetrics` callback.
"""
import os

import numpy as np
import torch

from . import callbacks as cb
from . import optimizers
from .engine import GATES, HotPath
from .engine_dense import DensePath
from .state import RecurrentState, write_npz
from .likelihood import compute_likelihood, compute_likelihood_cut  # noqa: F401  (utils.py:145-178, on the device)
from .preprocessor import is_one_hot, to_id_batch
from .ranking import check_ks, metrics_from_sums, rank_sums



class ModelResults():
    def __init__(self, train_loss=None, val_loss=None, epoch=None):
        self.val_loss = val_loss
        self.train_loss = train_loss
        self.epoch = epoch


class ValLossHistoryCut(cb.Callback):
    """model.py:94-117: per-epoch p(true next item) on the validation set and its within-sequence cut NLL.  Uses the
    fused on-device target-probability scoring instead of materialising predict()'s (N,T,V) output."""

    def __init__(self, val_data, orig_seqs_lengths):
        cb.Callback.__init__(self)
        self.val_data = val_data
        self.orig_seqs_lengths = orig_seqs_lengths

    def on_train_begin(self, logs=None):
        self.val_lossses = []
        if logs is not None and "my_loss" not in logs:
            logs["my_loss"] = 0.0

    def on_epoch_end(self, epoch, logs=None):
        p = self.model.predict_target_prob(self.val_data[0], self.val_data[1], device=True)   # stays in HBM
        _, val_neg_ll = compute_likelihood_cut(p, 0.7, orig_lengths=self.orig_seqs_lengths)
        self.val_lossses.append(val_neg_ll)
        if logs is not None:
            logs["my_loss"] = val_neg_ll


class RankingMetrics(cb.Callback):
    """Additive: per-epoch ranking metrics of the true next item on the validation set, written into `logs` as
    val_recall@k, val_mrr@k and val_ndcg@k -- placed before them in the callback list, EarlyStopping(monitor='val_mrr@20',
    mode='max') and ModelCheckpoint see them.  The ranks come from the fused on-device scoring pass."""

    def __init__(self, val_data, ks=(20,), last_step_only=False):
        cb.Callback.__init__(self)
        self.val_data = val_data
        self.ks = check_ks(ks)
        self.last_step_only = bool(last_step_only)
        self.history = []

    def on_epoch_end(self, epoch, logs=None):
        res = self.model.evaluate_ranking(self.val_data[0], self.val_data[1], ks=self.ks,
                                          last_step_only=self.last_step_only)
        self.history.append(res)
        if logs is not None:
            for k in self.ks:
                for name in ("recall", "mrr", "ndcg"):
                    logs["val_%s@%d" % (name, k)] = float(res["%s@%d" % (name, k)])


class BaseModel():
    def __init__(self, n_classes, model_name="test_model"):
        self.n_classes = n_classes
        self.model_name = model_name
        self.model = None


# ---------------------------------------------------------------------------------------------------------------------
class _Layer(object):
    """What `model.get_layer(name)` hands back: get_weights / set_weights / trainable."""

    def __init__(self, net, name, weight_names):
        self._net = net
        self.name = name
        self._weight_names = weight_names

    def get_weights(self):
        return [self._net._get(n) for n in self._weight_names]

    def set_weights(self, weights):
        if len(weights) != len(self._weight_names):
            raise ValueError("layer %s expects %d weight arrays" % (self.name, len(self._weight_names)))
        for n, w in zip(self._weight_names, weights):
            self._net._set(n, w)

    @property
    def trainable(self):
        return all(self._net.hot.trainable[n] for n in self._weight_names) if self._weight_names else True

    @trainable.setter
    def trainable(self, value):
        for n in self._weight_names:
            self._net.hot.trainable[n] = bool(value)


class _Net(object):
    """The object behind `BaseRNNModel.model`: the Keras-`Model` methods the reference calls, on top of HotPath."""

    def __init__(self, hot, layers, rnn_bias=True, seed=None, inputs=("y",)):
        self.hot = hot
        self.layers = layers
        self.rnn_bias = rnn_bias
        self.input_spec = tuple(inputs)           # which arrays the reference passes: ("y",), ("y", "x") or ("x",)
        self.stop_training = False
        self.metrics_names = ["loss"]
        self.optimizer = None
        self.loss = None
        if not rnn_bias and "b" in hot.trainable:
            hot.trainable["b"] = False
        for l in layers:
            l._net = self

    # ---- weights -------------------------------------------------------------------------------------------------
    def _names(self):
        """Weight names in `get_weights()` order = the layers' weights in layer order."""
        return [n for l in self.layers for n in l._weight_names]

    def _get(self, name):
        """Full-width array (the column shards of a vocabulary-parallel model are gathered by HotPath)."""
        return self.hot.get_weight(name)

    def _set(self, name, value):
        self.hot.set_weight(name, value)

    def get_weights(self):
        return [self._get(n) for n in self._names()]

    def set_weights(self, weights):
        names = self._names()
        if len(weights) != len(names):
            raise ValueError("expected %d weight arrays, got %d" % (len(names), len(weights)))
        for n, w in zip(names, weights):
            self._set(n, w)

    @property
    def trainable_weights(self):
        return [n for n in self._names() if self.hot.trainable[n]]

    @property
    def non_trainable_weights(self):
        return [n for n in self._names() if not self.hot.trainable[n]]

    def get_layer(self, name=None, index=None):
        if index is not None:
            return self.layers[index]
        for l in self.layers:
            if l.name == name:
                return l
        raise ValueError("No such layer: " + str(name))

    @staticmethod
    def _npz_path(filepath):
        """Checkpoints are .npz archives (h5py is absent from this image): a path that claims to be HDF5 gets '.npz'
        appended, so no file ever carries zip bytes under an .h5 / .hdf5 name."""
        return filepath + ".npz" if filepath.lower().endswith((".h5", ".hdf5")) else filepath

    def _write_npz(self, filepath, arrays):
        """Rank 0 writes (temp file + rename: a reader never sees a torn archive), everybody waits."""
        comm = self.hot.comm
        if comm.rank == 0:
            write_npz(filepath, arrays)
        comm.barrier()

    def save_weights(self, filepath, overwrite=True):
        """Weights-only checkpoint in `get_weights()` order, the flat `weight{i}` layout of model.py:201-208 as an .npz
        archive (collective in a multi-process run: shards are gathered, rank 0 writes)."""
        ws = self.get_weights()
        self._write_npz(self._npz_path(filepath), {"weight%d" % i: w for i, w in enumerate(ws)})

    @staticmethod
    def _open_npz(filepath):
        if not os.path.exists(filepath) and os.path.exists(_Net._npz_path(filepath)):
            filepath = _Net._npz_path(filepath)
        with open(filepath, "rb") as f:
            magic = f.read(8)
        if magic.startswith(b"\x89HDF"):
            raise IOError("%s is an HDF5 file (a Keras / reference checkpoint).  h5py is not available in this image; "
                          "convert it with `h5py` to an .npz archive holding weight0..weightN in get_weights() order "
                          "(model.py:201-208) and load that." % filepath)
        return np.load(filepath)

    def load_weights(self, filepath, by_name=False):
        with self._open_npz(filepath) as z:
            n = len([k for k in z.files if k.startswith("weight")])
            self.set_weights([z["weight%d" % i] for i in range(n)])

    def save_state(self, filepath, epoch=0):
        """Resumable checkpoint (not in the reference, whose checkpoints restart Adagrad): weights, the optimizer state
        of every weight, the optimizer hyper-parameters and the epoch counter.  Adagrad: `accum{i}` and
        opt = [lr, epsilon, clipnorm].  Adam: opt_kind = 'adam', opt = [lr, beta_1, beta_2, epsilon, clipnorm, decay],
        `iterations` and the moments `m{i}`, `v{i}` (i in get_weights() order)."""
        arrays = {"weight%d" % i: w for i, w in enumerate(self.get_weights())}
        o = self.hot.opt or {}
        arrays["epoch"] = np.asarray(int(epoch))
        if o.get("kind") == "adam":
            for i, n in enumerate(self._names()):
                arrays["m%d" % i], arrays["v%d" % i] = self.hot.get_moments(n)
            arrays["opt_kind"] = np.asarray("adam")
            arrays["opt"] = np.asarray([o["lr"], o["beta_1"], o["beta_2"], o["eps"], o["clipnorm"], o["decay"]],
                                       dtype=np.float64)
            arrays["iterations"] = np.asarray(self.hot.get_iterations(), dtype=np.int64)
        else:
            for i, n in enumerate(self._names()):
                arrays["accum%d" % i] = self.hot.get_accumulator(n)
            arrays["opt"] = np.asarray([o.get("lr", 0.0), o.get("eps", 0.0), o.get("clipnorm", 0.0)], dtype=np.float64)
        self._write_npz(self._npz_path(filepath), arrays)

    def load_state(self, filepath):
        """Inverse of save_state; returns the stored epoch.  compile() first (it resets the optimizer state), with the
        optimizer the checkpoint was written with: a different one raises ValueError.  An archive without `opt_kind`
        is an Adagrad checkpoint."""
        with self._open_npz(filepath) as z:
            kind = str(z["opt_kind"]) if "opt_kind" in z.files else "adagrad"
            compiled = (self.hot.opt or {}).get("kind", "adagrad")
            if kind != compiled:
                raise ValueError("%s holds %s optimizer state but the model is compiled with %s: compile it with the "
                                 "checkpoint's optimizer first" % (filepath, kind, compiled))
            names = self._names()
            self.set_weights([z["weight%d" % i] for i in range(len(names))])
            for i, n in enumerate(names):
                if kind == "adam":
                    self.hot.set_moments(n, z["m%d" % i], z["v%d" % i])
                else:
                    self.hot.set_accumulator(n, z["accum%d" % i])
            if kind == "adam":
                self.hot.set_iterations(int(z["iterations"]))
            return int(z["epoch"])

    # ---- compile -------------------------------------------------------------------------------------------------
    def compile(self, loss="categorical_crossentropy", optimizer="adam", metrics=None):
        if loss != "categorical_crossentropy":
            raise NotImplementedError("only categorical_crossentropy (experiments_methods.py:42) is built")
        self.loss = loss
        self.optimizer = optimizers.resolve(optimizer)
        self.metrics_names = ["loss"] + [m for m in (metrics or []) if isinstance(m, str)]
        if not isinstance(self.optimizer, str):
            o = self.optimizer
            if optimizers.kind_of(o) == "adam":
                self.hot.set_optimizer("adam", lr=o.lr, epsilon=o.epsilon, clipnorm=getattr(o, "clipnorm", None) or 0.0,
                                       decay=getattr(o, "decay", 0.0), beta_1=o.beta_1, beta_2=o.beta_2)
            else:
                self.hot.set_optimizer("adagrad", lr=o.lr, epsilon=o.epsilon,
                                       clipnorm=getattr(o, "clipnorm", None) or 0.0, decay=getattr(o, "decay", 0.0))

    # ---- batches -------------------------------------------------------------------------------------------------
    def _inputs(self, x):
        """Reference inputs are an ndarray or a list (experiments_methods.py:209-216: `[x]` for ytoz, `[x, xs]` when a
        history-feature branch is on, `xs` alone for the x-only NoRecurrenceModel).  Returns (ids, dense features)."""
        spec = self.input_spec
        if isinstance(x, (list, tuple)):
            if len(x) != len(spec):
                raise ValueError("this model takes %d input array(s) %s, got %d" % (len(spec), spec, len(x)))
            arrs = list(x)
        else:
            if len(spec) != 1:
                raise ValueError("this model takes a list of %d input arrays %s" % (len(spec), spec))
            arrs = [x]
        ids = xd = None
        for kind, a in zip(spec, arrs):
            if kind == "x" and isinstance(a, torch.Tensor):
                xd = a.to(dtype=torch.float32)             # history features built on the device (datasets.py) stay there
                continue
            a = np.asarray(a)
            if kind == "x":
                xd = np.ascontiguousarray(a, dtype=np.float32)
            elif (isinstance(self.hot, HotPath) and a.ndim == 3 and a.shape[2] > 1
                  and not (a.shape[2] == self.hot.F and is_one_hot(a))):
                if a.shape[2] != self.hot.F:
                    raise ValueError("input feature width %d does not match the model's %d" % (a.shape[2], self.hot.F))
                xd = np.ascontiguousarray(a, dtype=np.float32)         # dense-feature path of RNNBaseline (K2)
            else:
                ids = to_id_batch(a)                                   # gather path (K1)
        return ids, xd

    def _slice(self, ids, xd, idx):
        if isinstance(xd, torch.Tensor) and not isinstance(idx, slice):
            return (ids[idx] if ids is not None else None), xd.index_select(0, torch.as_tensor(idx, device=xd.device))
        return (ids[idx] if ids is not None else None), (xd[idx] if xd is not None else None)

    def _epoch_eval(self, ids, xd, tgt, batch_size):
        """Keras test_loop: batch-size-weighted mean of per-batch masked-mean losses (SURVEY a11).  The per-batch
        means stay on the device; one read-back per call."""
        n = len(tgt)
        per_batch, sizes = [], []
        for lo in range(0, n, batch_size):
            hi = min(n, lo + batch_size)
            i, d = self._slice(ids, xd, slice(lo, hi))
            ls, nv = self.hot.loss_batch(i, tgt[lo:hi], d)
            if self.hot.comm.enabled:
                self.hot.comm.all_reduce_sum(ls)
                self.hot.comm.all_reduce_sum(nv)
            per_batch.append(ls / nv)
            sizes.append(hi - lo)
        w = torch.tensor(sizes, dtype=torch.float64, device=self.hot.device)
        total = (torch.cat(per_batch).double() * w).sum()
        self.hot.check_errors()
        return float(total.item()) / n

    def _resident(self, a):
        """A whole id array in HBM (int32), when it is small enough to keep there for the epochs of a fit call."""
        if a is None or a.nbytes > (2 << 30):
            return None
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(self.hot.device)

    # ---- Keras Model methods ------------------------------------------------------------------------------------
    def fit(self, x, y, validation_data=None, epochs=10, batch_size=100, verbose=1, callbacks=None, shuffle=True):
        if isinstance(self.optimizer, str) or self.optimizer is None:
            raise NotImplementedError("training needs an optimizer object: optimizers.Adagrad(...) (experiments_methods.py:41) "
                                      "or optimizers.Adam(...); got %r" % (self.optimizer,))
        ids, xd = self._inputs(x)
        tgt = to_id_batch(y)
        self.hot._check_host_ids(ids, tgt)
        n = len(tgt)
        val = None
        if validation_data is not None:
            vi, vd = self._inputs(validation_data[0])
            val = (vi, vd, to_id_batch(validation_data[1]))
        # Keras 2.0.x order: user callbacks first, History last -- History records what the callbacks put into `logs`
        # (ValLossHistoryCut's `my_loss`, model.py:114)
        history = cb.History()
        cbs = list(callbacks or []) + [history]
        for c in cbs:
            c.set_model(self)
            c.set_params({"epochs": epochs, "batch_size": batch_size, "samples": n, "verbose": verbose})
        self.stop_training = False
        logs0 = {}
        for c in cbs:
            c.on_train_begin(logs0)
        # id batches: the training set goes to HBM once; an epoch then costs one H2D copy of the shuffled index and
        # two on-device row gathers per batch (no per-batch numpy fancy indexing, no pinned staging copy)
        dev_ids = dev_tgt = None
        if xd is None:
            dev_ids, dev_tgt = self._resident(ids), self._resident(tgt)
            if dev_ids is None or dev_tgt is None:
                dev_ids = dev_tgt = None
        n_batches = (n + batch_size - 1) // batch_size
        sizes = torch.tensor([min(batch_size, n - b * batch_size) for b in range(n_batches)], dtype=torch.float64,
                             device=self.hot.device)
        losses = torch.zeros(n_batches, dtype=torch.float32, device=self.hot.device)
        index = np.arange(n)
        for epoch in range(epochs):
            for c in cbs:
                c.on_epoch_begin(epoch)
            if shuffle:
                np.random.shuffle(index)
            dev_index = torch.from_numpy(index).to(self.hot.device) if dev_ids is not None else None
            for b, lo in enumerate(range(0, n, batch_size)):
                if dev_ids is not None:
                    sel = dev_index[lo:lo + batch_size]
                    loss = self.hot.train_batch(dev_ids.index_select(0, sel), dev_tgt.index_select(0, sel))
                else:
                    sel = index[lo:lo + batch_size]
                    i, d = self._slice(ids, xd, sel)
                    loss = self.hot.train_batch(i, tgt[sel], d)
                losses[b:b + 1].copy_(loss)
            logs = {"loss": float((losses.double() * sizes).sum().item()) / n}
            self.hot.check_errors()
            for m in self.metrics_names[1:]:
                logs[m] = logs["loss"]
            if val is not None:
                logs["val_loss"] = self._epoch_eval(val[0], val[1], val[2], batch_size)
                for m in self.metrics_names[1:]:
                    logs["val_" + m] = logs["val_loss"]
            for c in cbs:
                c.on_epoch_end(epoch, logs)
            if verbose:
                print("Epoch %d/%d - " % (epoch + 1, epochs) + " - ".join("%s: %.4f" % kv for kv in sorted(logs.items())))
            if self.stop_training:
                break
        for c in cbs:
            c.on_train_end()
        return history

    def fit_generator(self, generator, steps_per_epoch, epochs=1, verbose=1, callbacks=None, validation_data=None,
                      validation_steps=None):
        history = cb.History()
        cbs = list(callbacks or []) + [history]
        for c in cbs:
            c.set_model(self)
            c.set_params({"epochs": epochs, "steps": steps_per_epoch, "verbose": verbose})
        self.stop_training = False
        for c in cbs:
            c.on_train_begin({})
        for epoch in range(epochs):
            for c in cbs:
                c.on_epoch_begin(epoch)
            acc, cnt = 0.0, 0
            for _ in range(steps_per_epoch):
                x, y = next(generator)
                ids, xd = self._inputs(x)
                tgt = to_id_batch(y)
                loss = self.hot.train_batch(ids, tgt, xd)
                acc += float(loss.item()) * len(tgt)
                cnt += len(tgt)
            logs = {"loss": acc / max(cnt, 1)}
            if validation_data is not None:
                vacc, vcnt = 0.0, 0
                for _ in range(validation_steps or 1):
                    vx, vy = next(validation_data) if hasattr(validation_data, "__next__") else validation_data
                    vi, vd = self._inputs(vx)
                    vt = to_id_batch(vy)
                    vacc += self._epoch_eval(vi, vd, vt, len(vt)) * len(vt)
                    vcnt += len(vt)
                logs["val_loss"] = vacc / max(vcnt, 1)
            for c in cbs:
                c.on_epoch_end(epoch, logs)
            if self.stop_training:
                break
        for c in cbs:
            c.on_train_end()
        return history

    def train_on_batch(self, x, y):
        """Keras `Model.train_on_batch`: one optimisation step on one host batch; returns the scalar loss (host)."""
        ids, xd = self._inputs(x)
        return float(self.hot.train_batch(ids, to_id_batch(y), xd).item())

    def evaluate(self, x, y, batch_size=32, verbose=0):
        ids, xd = self._inputs(x)
        tgt = to_id_batch(y)
        loss = self._epoch_eval(ids, xd, tgt, batch_size)
        # the loss is registered again as a metric (model.py:177), so it comes back once per metrics_names entry
        return [loss] * len(self.metrics_names) if len(self.metrics_names) > 1 else loss

    def predict(self, x, batch_size=32, verbose=0):
        ids, xd = self._inputs(x)
        n = len(ids) if ids is not None else len(xd)
        out = []
        for lo in range(0, n, batch_size):
            i, d = self._slice(ids, xd, slice(lo, min(n, lo + batch_size)))
            out.append(self.hot.predict_batch(i, d).cpu().numpy())
        return np.concatenate(out, axis=0)

    # ---- additive scoring API --------------------------------------------------------------------------------------
    def predict_target_prob(self, x, y, batch_size=1024, device=False, initial_state=None):
        """(N,T) p(true next item), clipped to [1e-7, 1-1e-7]; pads give 1e-7 (model.py:108-110 semantics).
        device=True returns the device tensor (the likelihood metrics reduce it in HBM).  initial_state: the
        RecurrentState of the N sessions that x continues (None = zeros, the whole-window semantics)."""
        ids, xd = self._inputs(x)
        tgt = to_id_batch(y)
        self._check_state(initial_state, len(tgt))
        out = []
        for lo in range(0, len(tgt), batch_size):
            hi = min(len(tgt), lo + batch_size)
            i, d = self._slice(ids, xd, slice(lo, hi))
            out.append(self.hot.target_prob_batch(i, tgt[lo:hi], d, **self._state_kw(initial_state, lo, hi)).clone())
        out = torch.cat(out, dim=0)
        self.hot.check_errors()
        return out if device else out.cpu().numpy()

    def predict_topk(self, x, k=20, last_step_only=True, batch_size=1024, initial_state=None):
        """Top-k next-item ids (int32) and probabilities; ties broken by the lower item id.  initial_state: the
        RecurrentState of the sessions that x continues (None = zeros)."""
        ids, xd = self._inputs(x)
        n = len(ids) if ids is not None else len(xd)
        self._check_state(initial_state, n)
        oi, op = [], []
        for lo in range(0, n, batch_size):
            hi = min(n, lo + batch_size)
            i, d = self._slice(ids, xd, slice(lo, hi))
            a, b = self.hot.topk_batch(i, k, last_step_only=last_step_only, x_dense=d,
                                       **self._state_kw(initial_state, lo, hi))
            oi.append(a.cpu().numpy())
            op.append(b.cpu().numpy())
        return np.concatenate(oi, axis=0), np.concatenate(op, axis=0)

    def _target_ranks(self, x, y, batch_size, last_step_only, initial_state=None):
        ids, xd = self._inputs(x)
        tgt = to_id_batch(y)
        self._check_state(initial_state, len(tgt))
        out = []
        for lo in range(0, len(tgt), batch_size):
            hi = min(len(tgt), lo + batch_size)
            i, d = self._slice(ids, xd, slice(lo, hi))
            out.append(self.hot.target_rank_batch(i, tgt[lo:hi], d, last_step_only=last_step_only,
                                                  **self._state_kw(initial_state, lo, hi)).clone())
        out = torch.cat(out, dim=0)
        self.hot.check_errors()
        return out

    def predict_target_rank(self, x, y, batch_size=1024, device=False, initial_state=None):
        """(N,T) int32 rank of the true next item among all items: 1 + the items with a higher logit + the lower-id
        items with an equal one (so rank <= k <=> predict_topk holds it at index rank-1); pads give 0.
        device=True returns the device tensor (ranking.ranking_metrics reduces it in HBM).  initial_state: the
        RecurrentState of the sessions that x continues (None = zeros)."""
        out = self._target_ranks(x, y, batch_size, False, initial_state)
        return out if device else out.cpu().numpy()

    # ---- carried recurrent state (inference) ---------------------------------------------------------------------
    def _need_state_support(self):
        if not isinstance(self.hot, HotPath):
            raise NotImplementedError(
                "carried state is built for the recurrent hot path (ytoz RNNFullModel, RNNBaseline): the x_to_z / "
                "x_to_y / y_to_y branches and NoRecurrenceModel also read history features and the previous item, "
                "which a recurrent state does not carry")

    def _check_state(self, state, n):
        if state is not None:
            self._need_state_support()
            state.check(self.hot.cell, self.hot.H, n)

    @staticmethod
    def _state_kw(state, lo, hi):
        return {} if state is None else {"initial_state": state.take(slice(lo, hi))}

    def initial_state(self, n):
        """The zero state of n sessions (what scoring a whole window starts from)."""
        self._need_state_support()
        return self.hot.initial_state(n)

    def advance_state(self, x, state=None, batch_size=1024):
        """The state of each session after the new events x (any input `predict` takes: ids (n,T'), one-hot, or
        RNNBaseline's dense input), continuing `state` (None = zeros).  Pads hold the state."""
        self._need_state_support()
        ids, xd = self._inputs(x)
        n = len(ids) if ids is not None else len(xd)
        self._check_state(state, n)
        hs, cs = [], []
        for lo in range(0, n, batch_size):
            hi = min(n, lo + batch_size)
            i, d = self._slice(ids, xd, slice(lo, hi))
            st = self.hot.advance_state(i, None if state is None else state.take(slice(lo, hi)), d)
            hs.append(st.h)
            cs.append(st.c)
        self.hot.check_errors()
        return RecurrentState(torch.cat(hs), None if cs[0] is None else torch.cat(cs), self.hot.cell, self.hot.H)

    def _from_state(self, state, batch_size, fn):
        self._need_state_support()
        self._check_state(state, len(state))
        out = [fn(state.take(slice(lo, min(len(state), lo + batch_size))), lo, min(len(state), lo + batch_size))
               for lo in range(0, len(state), batch_size)]
        self.hot.check_errors()
        return out

    @staticmethod
    def _next_ids(y, n):
        t = y if isinstance(y, torch.Tensor) else torch.from_numpy(np.asarray(y, dtype=np.int64))
        if t.dim() != 1 or t.numel() != n:
            raise ValueError("y must be the (%d,) next-item ids of the sessions" % n)
        return t

    def predict_topk_from_state(self, state, k=20, batch_size=1024):
        """Top-k next items after each session's state: (n,k) int32 ids and probabilities, equal to predict_topk on
        the events the state has seen (for histories of at most T events)."""
        out = self._from_state(state, batch_size, lambda s, lo, hi: self.hot.topk_from_state(s, k))
        return (np.concatenate([a.cpu().numpy() for a, _ in out]), np.concatenate([b.cpu().numpy() for _, b in out]))

    def predict_target_prob_from_state(self, state, y, batch_size=1024, device=False):
        """(n,) p(y[i] is the next item of session i); y < 0 is a pad (1e-7)."""
        t = self._next_ids(y, len(state))
        out = torch.cat(self._from_state(state, batch_size,
                                         lambda s, lo, hi: self.hot.target_prob_from_state(s, t[lo:hi])))
        return out if device else out.cpu().numpy()

    def predict_target_rank_from_state(self, state, y, batch_size=1024, device=False):
        """(n,) int32 rank of y[i] after session i's state (the rank of predict_target_rank); y < 0 gives 0."""
        t = self._next_ids(y, len(state))
        out = torch.cat(self._from_state(state, batch_size,
                                         lambda s, lo, hi: self.hot.target_rank_from_state(s, t[lo:hi])))
        return out if device else out.cpu().numpy()

    def evaluate_ranking(self, x, y, ks=(1, 5, 10, 20), last_step_only=False, batch_size=1024):
        """Recall@k, MRR@k, NDCG@k for every k, the uncut MRR and n over the scored steps: every valid step, or with
        last_step_only the last step of each non-empty sequence.  Data-parallel processes each score their own rows;
        the sums are added over the processes."""
        ks = check_ks(ks)
        sums = rank_sums(self._target_ranks(x, y, batch_size, last_step_only), ks)
        if self.hot.comm.enabled:
            self.hot.comm.all_reduce_sum(sums)
        return metrics_from_sums(sums, ks)

    # ---- candidate scoring (a given list of items per session) -------------------------------------------------------
    def predict_candidates(self, x, candidates, k=None, probs=False, last_step_only=True, batch_size=1024,
                           initial_state=None):
        """How the model orders a given list of items per session: candidates (N, C) (last step) or (N, T, C) (every
        step), a numpy array or a device tensor, ids < 0 pads.  Returns (ids int32, scores float32) numpy arrays of the
        first k (default C) entries: score descending, then lower item id, then lower list position, pads last as
        (-1, 0).  Scores are logits, or with probs=True the catalog softmax probabilities of predict_topk."""
        ids, xd = self._inputs(x)
        n = len(ids) if ids is not None else len(xd)
        self._check_state(initial_state, n)
        oi, os_ = [], []
        for lo in range(0, n, batch_size):
            hi = min(n, lo + batch_size)
            i, d = self._slice(ids, xd, slice(lo, hi))
            a, b = self.hot.candidates_batch(i, candidates[lo:hi], k=k, probs=probs, last_step_only=last_step_only,
                                             x_dense=d, **self._state_kw(initial_state, lo, hi))
            oi.append(a.cpu().numpy())
            os_.append(b.cpu().numpy())
        return np.concatenate(oi, axis=0), np.concatenate(os_, axis=0)

    def _candidate_ranks(self, x, y, candidates, batch_size, last_step_only, initial_state=None):
        ids, xd = self._inputs(x)
        tgt = to_id_batch(y)
        self._check_state(initial_state, len(tgt))
        out = []
        for lo in range(0, len(tgt), batch_size):
            hi = min(len(tgt), lo + batch_size)
            i, d = self._slice(ids, xd, slice(lo, hi))
            out.append(self.hot.candidate_rank_batch(i, tgt[lo:hi], candidates[lo:hi], last_step_only=last_step_only,
                                                     x_dense=d, **self._state_kw(initial_state, lo, hi)))
        out = torch.cat(out, dim=0)
        self.hot.check_errors()
        return out

    def predict_candidate_rank(self, x, y, candidates, last_step_only=False, batch_size=1024, device=False,
                               initial_state=None):
        """(N,T) int32 rank of the true next item among each step's candidates (N, T, C), or (N,) with last_step_only
        (candidates (N, C)): 1 + the other candidates with a higher logit or an equal one and a lower id; y < 0 gives 0.
        A list may or may not hold the target."""
        out = self._candidate_ranks(x, y, candidates, batch_size, last_step_only, initial_state)
        return out if device else out.cpu().numpy()

    def predict_candidates_from_state(self, state, candidates, k=None, probs=False, batch_size=1024):
        """predict_candidates after each session's state: candidates (n, C)."""
        out = self._from_state(state, batch_size, lambda s, lo, hi: self.hot.candidates_from_state(
            s, candidates[lo:hi], k=k, probs=probs))
        return (np.concatenate([a.cpu().numpy() for a, _ in out]), np.concatenate([b.cpu().numpy() for _, b in out]))

    def predict_candidate_rank_from_state(self, state, y, candidates, batch_size=1024, device=False):
        """(n,) int32 rank of y[i] among candidates[i] after session i's state; y < 0 gives 0."""
        t = self._next_ids(y, len(state))
        out = torch.cat(self._from_state(state, batch_size, lambda s, lo, hi: self.hot.candidate_rank_from_state(
            s, t[lo:hi], candidates[lo:hi])))
        return out if device else out.cpu().numpy()

    def evaluate_candidate_ranking(self, x, y, candidates, ks=(1, 5, 10, 20), last_step_only=False, batch_size=1024):
        """evaluate_ranking over the ranks among the candidates (predict_candidate_rank)."""
        ks = check_ks(ks)
        sums = rank_sums(self._candidate_ranks(x, y, candidates, batch_size, last_step_only), ks)
        if self.hot.comm.enabled:
            self.hot.comm.all_reduce_sum(sums)
        return metrics_from_sums(sums, ks)

    def hidden_states(self, x, batch_size=1024):
        ids, xd = self._inputs(x)
        n = len(ids) if ids is not None else len(xd)
        out = []
        for lo in range(0, n, batch_size):
            i, d = self._slice(ids, xd, slice(lo, min(n, lo + batch_size)))
            out.append(self.hot.hidden_batch(i, d).cpu().numpy())
        return np.concatenate(out, axis=0)


# ---------------------------------------------------------------------------------------------------------------------
class BaseRNNModel(BaseModel):
    """model.py:170-238."""

    def __init__(self, n_classes, model_name="test_model", rnn_type='simpleRNN'):
        BaseModel.__init__(self, n_classes, model_name)
        self.rnn_type = rnn_type

    def compile_model(self, loss='categorical_crossentropy', metrics=[], optimizer='adam'):
        self.model.compile(loss=loss, optimizer=optimizer, metrics=[loss] + metrics)

    def fit_model(self, x_train, y_train, validation_data=None, n_epochs=10, batch_size=100, verbose=1,
                  callbacks=None):
        return self.model.fit(x_train, y_train, validation_data=validation_data, epochs=n_epochs,
                              batch_size=batch_size, verbose=verbose, callbacks=callbacks)

    def fit_generator(self, train_gen, steps_per_epoch, validation_steps, epochs, verbose, callbacks,
                      validation_data):
        return self.model.fit_generator(train_gen, validation_data=validation_data, callbacks=callbacks,
                                        steps_per_epoch=steps_per_epoch, validation_steps=validation_steps,
                                        epochs=epochs, verbose=verbose)

    def predict(self, x_test, batch_size=10, verbose=1):
        return self.model.predict(x_test, batch_size=batch_size, verbose=verbose)

    def evaluate(self, x_test, y_test, batch_size=10, verbose=0):
        scores = self.model.evaluate(x_test, y_test, verbose=verbose, batch_size=batch_size)
        return self.model.metrics_names, scores

    def save_model_weights(self, directory):
        if not os.path.exists(directory):
            os.makedirs(directory)
        self.model.save_weights(directory + self.model_name + ".npz")

    def load_model_weights(self, filepath):
        self.model.load_weights(filepath, by_name=False)

    def get_layer_weights(self, layer):
        if isinstance(layer, str):
            return self.model.get_layer(layer).get_weights()
        else:
            return self.model.layers[layer].get_weights()

    def set_layer_weights_trainable(self, name, trainable=True):
        self.model.get_layer(name).trainable = trainable

    def set_layer_weights(self, name, weights):
        self.model.get_layer(name).set_weights(weights)

    def get_model_weights(self):
        return self.model.trainable_weights, self.model.non_trainable_weights

    def get_activations(self, layer, inputs, input_layers):
        """Inference-phase output of a named layer (model.py:235-238).  Built for the recurrent layer (hidden states)
        and the final softmax; `inputs` is the list the reference passes (one array per input layer)."""
        rnn_names = [l.name for l in self.model.layers if l._weight_names[:1] == ["W_in"]]
        if layer in rnn_names:
            return self.model.hidden_states(inputs)
        if layer == self.model.layers[-1].name:
            return self.model.predict(inputs)
        raise NotImplementedError("get_activations is built for the recurrent layer and the output layer only")

    # additive
    def predict_target_prob(self, x_test, y_test, batch_size=1024, initial_state=None):
        return self.model.predict_target_prob(x_test, y_test, batch_size=batch_size, initial_state=initial_state)

    def predict_topk(self, x_test, k=20, last_step_only=True, batch_size=1024, initial_state=None):
        return self.model.predict_topk(x_test, k=k, last_step_only=last_step_only, batch_size=batch_size,
                                       initial_state=initial_state)

    def predict_target_rank(self, x_test, y_test, batch_size=1024, initial_state=None):
        return self.model.predict_target_rank(x_test, y_test, batch_size=batch_size, initial_state=initial_state)

    def initial_state(self, n):
        return self.model.initial_state(n)

    def advance_state(self, x, state=None, batch_size=1024):
        return self.model.advance_state(x, state=state, batch_size=batch_size)

    def predict_topk_from_state(self, state, k=20, batch_size=1024):
        return self.model.predict_topk_from_state(state, k=k, batch_size=batch_size)

    def predict_target_prob_from_state(self, state, y, batch_size=1024):
        return self.model.predict_target_prob_from_state(state, y, batch_size=batch_size)

    def predict_target_rank_from_state(self, state, y, batch_size=1024):
        return self.model.predict_target_rank_from_state(state, y, batch_size=batch_size)

    def evaluate_ranking(self, x_test, y_test, ks=(1, 5, 10, 20), last_step_only=False, batch_size=1024):
        return self.model.evaluate_ranking(x_test, y_test, ks=ks, last_step_only=last_step_only, batch_size=batch_size)

    def predict_candidates(self, x_test, candidates, k=None, probs=False, last_step_only=True, batch_size=1024,
                           initial_state=None):
        return self.model.predict_candidates(x_test, candidates, k=k, probs=probs, last_step_only=last_step_only,
                                             batch_size=batch_size, initial_state=initial_state)

    def predict_candidates_from_state(self, state, candidates, k=None, probs=False, batch_size=1024):
        return self.model.predict_candidates_from_state(state, candidates, k=k, probs=probs, batch_size=batch_size)

    def predict_candidate_rank(self, x_test, y_test, candidates, last_step_only=False, batch_size=1024,
                               initial_state=None):
        return self.model.predict_candidate_rank(x_test, y_test, candidates, last_step_only=last_step_only,
                                                 batch_size=batch_size, initial_state=initial_state)

    def predict_candidate_rank_from_state(self, state, y, candidates, batch_size=1024):
        return self.model.predict_candidate_rank_from_state(state, y, candidates, batch_size=batch_size)

    def evaluate_candidate_ranking(self, x_test, y_test, candidates, ks=(1, 5, 10, 20), last_step_only=False,
                                   batch_size=1024):
        return self.model.evaluate_candidate_ranking(x_test, y_test, candidates, ks=ks, last_step_only=last_step_only,
                                                     batch_size=batch_size)


def _glorot_uniform(rng, shape):
    limit = np.sqrt(6.0 / (shape[0] + shape[1]))
    return rng.uniform(-limit, limit, size=shape).astype(np.float32)


def _glorot_normal(rng, shape):
    return (rng.standard_normal(size=shape) * np.sqrt(2.0 / (shape[0] + shape[1]))).astype(np.float32)


def _orthogonal(rng, n):
    q, r = np.linalg.qr(rng.standard_normal(size=(n, n)))
    return (q * np.sign(np.diag(r))).astype(np.float32)


def _init_weights(cell, F, H, V, out_bias, kernel_init="glorot_uniform", seed=None):
    """Keras-2.0.x defaults: glorot_uniform kernels (glorot_normal for the ytoz LSTM, model.py:351), orthogonal
    recurrent kernel per gate block, zero biases with unit_forget_bias."""
    rng = np.random.default_rng(seed)
    G = GATES[cell]
    kin = _glorot_normal if kernel_init == "glorot_normal" else _glorot_uniform
    W_in = kin(rng, (F, G * H))
    U = np.concatenate([_orthogonal(rng, H) for _ in range(G)], axis=1)
    b = np.zeros(G * H, dtype=np.float32)
    if cell == "LSTM":
        b[H:2 * H] = 1.0
    ws = [W_in, U, b, _glorot_uniform(rng, (H, V))]
    if out_bias:
        ws.append(np.zeros(V, dtype=np.float32))
    return ws


class RNNBaseline(BaseRNNModel):
    """model.py:241-258: Input(T,F) -> Masking -> SimpleRNN/LSTM(z_dim) -> Dropout -> TimeDistributed(Dense(V, softmax,
    WITH bias))."""

    def __init__(self, timesteps, features, n_classes, model_name="baseline_model", rnn_type='simpleRNN',
                 out_activation="softmax", z_activation="relu", z_dim=20, z_to_y_drop=0.0, seed=None, comm=None):
        BaseRNNModel.__init__(self, n_classes, model_name=model_name, rnn_type=rnn_type)
        if out_activation != "softmax":
            raise NotImplementedError("only the softmax output of the reference's experiments is built")
        self.timesteps = timesteps
        hot = HotPath(rnn_type, z_activation, features, z_dim, n_classes, out_bias=True, comm=comm,
                      weights=_init_weights(rnn_type, features, z_dim, n_classes, True, seed=seed),
                      seed=0 if seed is None else seed)
        hot.dropout_out = float(z_to_y_drop)
        rnn_name = "rnn" if rnn_type == "simpleRNN" else ("lstm" if rnn_type == "LSTM" else "gru")
        layers = [_Layer(None, "myinput", []), _Layer(None, "mask", []), _Layer(None, rnn_name, ["W_in", "U", "b"]),
                  _Layer(None, "dropout_1", []), _Layer(None, "output", ["W_out", "b_out"])]
        self.model = _Net(hot, layers)


class ArrayInitializer(object):
    """model.py:32-45: an initializer that returns a given array (the Markov log-transition matrix of
    experiments_server.py:60-68 for the y -> y kernel)."""

    def __init__(self, values=0):
        self.values = values

    def __call__(self, shape, dtype=None):
        return self.values

    def get_config(self):
        return {"value": self.values}


class OnlyNonZeroDiagonal(object):
    """model.py:48-66 (spec object; the arithmetic is seqrec_diag_constraint, applied to the updated kernel)."""

    def __init__(self, input_dim, skip_cols):
        self.input_dim = input_dim
        self.skip_cols = skip_cols

    def get_config(self):
        return {"input_dim": self.input_dim, "skip_cols": self.skip_cols}


only_non_zero_diag = OnlyNonZeroDiagonal


def gauss_prior(means, var):
    raise NotImplementedError("GaussPriorRegularizer (model.py:74-91): every driver of the reference passes "
                              "y_to_y_regularizer=None / toy_regularizer=None, so kernel regularisers are not built")


def _init_kernel(init, rng, shape, default="glorot_uniform"):
    """Keras-2.0.x kernel initialisers as the reference passes them: a name, an ArrayInitializer-like callable
    (experiments_server.py:66), or an object with minval/maxval or mean/stddev attributes (tune_params.py:80, :91)."""
    if init is None:
        init = default
    if isinstance(init, str):
        if init == "glorot_uniform":
            return _glorot_uniform(rng, shape)
        if init == "glorot_normal":
            return _glorot_normal(rng, shape)
        if init == "random_uniform":
            return rng.uniform(-0.05, 0.05, size=shape).astype(np.float32)
        if init == "zeros":
            return np.zeros(shape, dtype=np.float32)
        raise NotImplementedError("initializer %r" % (init,))
    if hasattr(init, "minval") and hasattr(init, "maxval"):
        return rng.uniform(init.minval, init.maxval, size=shape).astype(np.float32)
    if hasattr(init, "stddev"):
        return (getattr(init, "mean", 0.0) + init.stddev * rng.standard_normal(size=shape)).astype(np.float32)
    if callable(init):
        v = np.asarray(init(shape), dtype=np.float32)
        if tuple(v.shape) != tuple(shape):
            raise ValueError("initializer returned shape %s, the kernel has %s" % (v.shape, tuple(shape)))
        return v.copy()
    raise NotImplementedError("initializer %r" % (init,))


class NoRecurrenceModel(BaseRNNModel):
    """model.py:264-319: softmax(f(B x_t) + g(A y_{t-1} + c)) without recurrence -- `y_output` = Dense(A) on the masked
    one-hot y input (a row lookup of A), `x_to_y_output` = Dense(B) on the history features with the diagonal
    constraint.  Runs on engine_dense.DensePath (materialised logits: these are small-catalog models)."""

    def __init__(self, timesteps, x_dim, y_dim, model_name="y_to_y_model",
                 y_to_y_activation="linear", x_to_y_activation="linear", y_to_y_w_initializer=None,
                 out_activation="softmax", mask_value=0.0,
                 y_bias=False, xy_bias=False, y_to_y_regularizer=None, z_dim=10, z_bias=True, connect_x=True,
                 connect_y=True, embed_y=False, diag_b=True, seed=None):
        BaseRNNModel.__init__(self, y_dim, model_name=model_name, rnn_type=None)
        if not (connect_x or connect_y):
            raise ValueError("ERROR: the model needs an input! either x or y should be added.")
        if out_activation != "softmax" or y_to_y_activation != "linear" or x_to_y_activation != "linear":
            raise NotImplementedError("only linear -> softmax outputs (every driver of the reference) are built")
        if y_to_y_regularizer is not None:
            raise NotImplementedError("y_to_y_regularizer is None in every driver of the reference")
        if embed_y:
            raise NotImplementedError("embed_y=True is never used by the reference's drivers (run_model_no_recurrence "
                                      "leaves it False)")
        if mask_value != 0.0:
            raise NotImplementedError("mask_value other than 0.0 is never used by the reference")
        self.timesteps = timesteps
        rng = np.random.default_rng(seed)
        ws, layers, inputs = {}, [], []
        if connect_y:
            ws["A"] = _init_kernel(y_to_y_w_initializer, rng, (y_dim, y_dim), default="random_uniform")
            if y_bias:
                ws["a_bias"] = np.zeros(y_dim, dtype=np.float32)
            inputs.append("y")
            layers += [_Layer(None, "y_input", []), _Layer(None, "mask1", []),
                       _Layer(None, "y_output", ["A"] + (["a_bias"] if y_bias else []))]
        if connect_x:
            ws["W_toy"] = _glorot_uniform(rng, (x_dim, y_dim))
            if xy_bias:
                ws["b_out"] = np.zeros(y_dim, dtype=np.float32)
            inputs.append("x")
            layers += [_Layer(None, "x_input", []), _Layer(None, "mask2", []),
                       _Layer(None, "x_to_y_output", ["W_toy"] + (["b_out"] if xy_bias else []))]
        layers.append(_Layer(None, "activation_1", []))
        hot = DensePath(None, "linear", y_dim, x_dim, 0, ws, x_to_y=connect_x, y_to_y=connect_y, diag_b=diag_b,
                        seed=0 if seed is None else seed)
        self.model = _Net(hot, layers, inputs=inputs)


class RNNFullModel(BaseRNNModel):
    """model.py:322-403.  Input(T,V) one-hot y [and Input(T,x_dim) history features x] -> Masking -> [concatenate] ->
    Dropout(y_to_z_dropout) -> SimpleRNN/LSTM/GRU(z_dim, activation=z_to_z_activation, recurrent_dropout=z_to_z_dropout)
    -> Dropout(z_to_y_dropout) -> [concatenate with x] -> TimeDistributed(Dense(V, linear, use_bias=toy_bias)) [+
    TimeDistributed(Dense(V))(y_input)] -> softmax.

    The `y_to_z`-only variant ("ytoz", experiments_server.py:106-114) is the hot path: engine.HotPath, fused kernels that
    never materialise the logits, data / vocabulary parallel.  Any other branch combination (x_to_z, x_to_y, y_to_y: the
    other six recurrent variants of experiments_server.py:116-191) runs on engine_dense.DensePath."""

    def __init__(self, timesteps, x_dim, y_dim, z_dim=20, model_name="y_to_y_model", rnn_type='simpleRNN',
                 z_to_z_activation="relu",
                 y_to_y_activation="linear", xz_to_y_activation="linear", y_to_y_w_initializer=None,
                 out_activation="softmax",
                 ytoy_bias=False, toy_bias=False, z_bias=True, y_to_y_regularizer=None, toy_regularizer=None,
                 y_to_z=True,
                 y_to_z_initializer="glorot_normal",
                 y_to_y=True, x_to_y=True, x_to_z=False, z_to_y_dropout=0.0, diag_b=True, y_to_z_dropout=0.0,
                 z_to_z_dropout=0.0, seed=None, comm=None, vocab_parallel=False):
        BaseRNNModel.__init__(self, y_dim, model_name=model_name, rnn_type=rnn_type)
        if not (x_to_z or y_to_z):
            raise ValueError("ERROR: the model needs an input into z's! either x or y should be added.")
        if out_activation != "softmax" or xz_to_y_activation != "linear" or y_to_y_activation != "linear":
            raise NotImplementedError("only linear -> softmax outputs (the reference's experiments) are built")
        if toy_regularizer is not None or y_to_y_regularizer is not None:
            raise NotImplementedError("kernel regularisers are None in every driver of the reference "
                                      "(experiments_server.py, tune_params*.py)")
        self.timesteps = timesteps
        rnn_w = ["W_in", "U"] + (["b"] if z_bias else [])
        kinit = y_to_z_initializer if rnn_type == "LSTM" else "glorot_uniform"
        if y_to_z and not (y_to_y or x_to_y or x_to_z):
            # ---- the hot path
            ws = _init_weights(rnn_type, y_dim, z_dim, y_dim, bool(toy_bias), kernel_init=kinit, seed=seed)
            hot = HotPath(rnn_type, z_to_z_activation, y_dim, z_dim, y_dim, out_bias=bool(toy_bias), weights=ws,
                          comm=comm, seed=0 if seed is None else seed, vocab_parallel=vocab_parallel)
            out_w = ["W_out"] + (["b_out"] if toy_bias else [])
            layers = [_Layer(None, "y_input", []), _Layer(None, "mask1", []), _Layer(None, "dropout_1", []),
                      _Layer(None, "z_to_z_output", rnn_w), _Layer(None, "dropout_2", []),
                      _Layer(None, "to_y_output", out_w), _Layer(None, "activation_1", [])]
            self.model = _Net(hot, layers, rnn_bias=bool(z_bias))
            if not z_bias:
                hot.b.zero_()
        else:
            # ---- history-feature / skip branches
            if comm is not None and comm.enabled:
                raise NotImplementedError("the history-feature variants run in one process (as in the reference)")
            rng = np.random.default_rng(seed)
            G = GATES[rnn_type]
            F_in = (y_dim if y_to_z else 0) + (x_dim if x_to_z else 0)
            ws = {"W_in": _init_kernel(kinit, rng, (F_in, G * z_dim)),
                  "U": np.concatenate([_orthogonal(rng, z_dim) for _ in range(G)], axis=1)}
            if z_bias:
                ws["b"] = np.zeros(G * z_dim, dtype=np.float32)
                if rnn_type == "LSTM":
                    ws["b"][z_dim:2 * z_dim] = 1.0
            ws["W_toy"] = _glorot_uniform(rng, (z_dim + (x_dim if x_to_y else 0), y_dim))
            if toy_bias:
                ws["b_out"] = np.zeros(y_dim, dtype=np.float32)
            if y_to_y:
                ws["A"] = _init_kernel(y_to_y_w_initializer, rng, (y_dim, y_dim), default="glorot_uniform")
                if ytoy_bias:
                    ws["a_bias"] = np.zeros(y_dim, dtype=np.float32)
            hot = DensePath(rnn_type, z_to_z_activation, y_dim, x_dim, z_dim, ws, y_to_z=y_to_z, x_to_z=x_to_z,
                            x_to_y=x_to_y, y_to_y=y_to_y, diag_b=diag_b, seed=0 if seed is None else seed)
            inputs = (["y"] if (y_to_y or y_to_z) else []) + (["x"] if (x_to_y or x_to_z) else [])
            layers = []
            if y_to_y or y_to_z:
                layers += [_Layer(None, "y_input", []), _Layer(None, "mask1", [])]
            if x_to_y or x_to_z:
                layers += [_Layer(None, "x_input", []), _Layer(None, "mask2", [])]
            layers += [_Layer(None, "dropout_1", []), _Layer(None, "z_to_z_output", rnn_w),
                       _Layer(None, "dropout_2", []),
                       _Layer(None, "to_y_output", ["W_toy"] + (["b_out"] if toy_bias else []))]
            if y_to_y:
                layers.append(_Layer(None, "y_to_y_output", ["A"] + (["a_bias"] if ytoy_bias else [])))
            layers.append(_Layer(None, "activation_1", []))
            self.model = _Net(hot, layers, rnn_bias=True, inputs=inputs)
        hot.dropout_in = float(y_to_z_dropout)
        hot.dropout_out = float(z_to_y_dropout)
        hot.dropout_rec = float(z_to_z_dropout)    # recurrent_dropout (model.py:346,351; tune_params.py:83)
