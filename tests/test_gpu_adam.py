"""Keras Adam on the device (csrc/optim.cu seqrec_adam / seqrec_adam_table) against the float64 oracle (oracle/adam.py),
through HotPath (single GPU, data parallel and vocabulary parallel on one device, eager and CUDA-graph replay),
DensePath and the reference-facing model surface.  Run with -m gpu on a B200.

Tolerances.  Adam's first update of a coordinate is lr * g / (|g| + eps / sqrt(1 - beta_2)): sign-like wherever
|g| >> 3e-7.  Where a gradient is a cancellation residue, the last-bit differences of a reordered or split-product sum
become a finite relative change of that coordinate's move (never more than the move itself).  So exact-fp32 (tc='off')
runs get norm-wise bounds, and runs whose gradient sums differ by more than rounding (x3 products, replays, other
reduction orders) the bound of test_state_checkpoint_resumes_with_adagrad_accumulators: few coordinates off, none by
more than the steps' displacement."""
import numpy as np
import pytest
import torch

from oracle import adam as oa
from seq_recommendations_b200 import synthetic
from seq_recommendations_b200 import model as M
from seq_recommendations_b200.engine import HotPath
from seq_recommendations_b200.engine_dense import DensePath
from seq_recommendations_b200.optimizers import Adagrad, Adam

from gpu_util import as_t, rel_err
from test_gpu_skip_models import VARIANTS, make_inputs
from test_gpu_skip_models import make_weights as skip_weights
from test_gpu_vocab_parallel_one_device import ThreadComm, _rows, _solo, run_ranks

pytestmark = pytest.mark.gpu
TOL = 1e-4
LR = 0.01
NAMES = ["W_in", "U", "b", "W_out", "b_out"]


def max_move(steps, lr=LR, beta_2=0.999):
    """A bound on the move of one coordinate over `steps` Adam steps: lr_t * |m| / sqrt(v) <= lr / sqrt(1 - beta_2)
    per step."""
    return steps * lr / np.sqrt(1 - beta_2)


def close_bulk(x, y, steps, lr=LR):
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    return np.mean(~np.isclose(x, y, rtol=1e-4, atol=1e-6)) < 0.01 and np.abs(x - y).max() <= 2 * max_move(steps, lr)


def make_pair(cell, act, V, H, seed, out_bias=False, tc="off", F=None):
    ws = synthetic.make_weights(cell, V, H, seed=seed, out_bias=out_bias, F=F)
    hot = HotPath(cell, act, F or V, H, V, out_bias=out_bias, weights=ws, tc=tc)
    return hot, oa.Model(cell, act, ws, dtype=torch.float64), ws


# (cell, act, V, H, T, B, out_bias, clipnorm, decay, tc): clip active / inactive, decay, output bias, every cell
CASES = [("GRU", "tanh", 300, 32, 12, 40, False, 1.0, 0.0, "off"),
         ("LSTM", "tanh", 1000, 64, 10, 160, True, 1.0, 0.05, "off"),
         ("simpleRNN", "relu", 80, 16, 6, 10, True, 1e3, 0.0, "off"),
         ("GRU", "tanh", 2000, 128, 10, 96, True, 0.5, 0.01, "x3")]


@pytest.mark.parametrize("cell,act,V,H,T,B,bias,clip,decay,tc", CASES)
def test_adam_steps_match_oracle(cell, act, V, H, T, B, bias, clip, decay, tc):
    hot, ora, _ = make_pair(cell, act, V, H, seed=10, out_bias=bias, tc=tc)
    hot.set_optimizer("adam", lr=LR, epsilon=1e-8, clipnorm=clip, decay=decay)
    steps = 4
    for step in range(steps):
        ids, tgt = synthetic.make_batch(V, T, B, seed=20 + step, min_len=1)
        loss = float(hot.train_batch(ids, tgt).item())
        rl, _, _ = ora.train_step(as_t(ids), as_t(tgt), as_t(ids) >= 0, lr=LR, epsilon=1e-8, clipnorm=clip,
                                  optimizer="adam", decay=decay)
        assert abs(loss - float(rl)) <= TOL * abs(float(rl)), (step, loss, float(rl))
        assert float(hot.dW_in.abs().max().item()) == 0.0 and int(hot.touched.abs().max().item()) == 0
    assert hot.get_iterations() == steps
    for name, w, r in zip(NAMES, hot.get_weights(), ora.numpy_weights()):
        if tc == "off":
            assert rel_err(w, r) <= 3e-4, (name, rel_err(w, r))
        else:
            assert close_bulk(w, r, steps), name
    m, v = hot.get_moments("U")
    assert rel_err(m, ora.moment[1].numpy()) <= 1e-3 and rel_err(v, ora.accum[1].numpy()) <= 1e-3


def test_adam_frozen_output_kernel_is_excluded_from_norm_and_update():
    V, H, T, B = 40, 8, 5, 6
    hot, ora, ws = make_pair("LSTM", "relu", V, H, seed=14)
    hot.set_optimizer("adam", lr=LR, epsilon=1e-8, clipnorm=0.05)
    hot.trainable["W_out"] = False
    for step in range(3):
        ids, tgt = synthetic.make_batch(V, T, B, seed=15 + step)
        hot.train_batch(ids, tgt)
        ora.train_step(as_t(ids), as_t(tgt), as_t(ids) >= 0, lr=LR, epsilon=1e-8, clipnorm=0.05,
                       trainable=[True, True, True, False], optimizer="adam")
    got = hot.get_weights()
    assert np.array_equal(got[3], ws[3])
    m, v = hot.get_moments("W_out")
    assert not m.any() and not v.any()
    assert hot.get_iterations() == 3                             # once per step, whatever was frozen
    for w, r in zip(got, ora.numpy_weights()):
        assert rel_err(w, r) <= 3e-4


def test_adam_dense_feature_inputs_match_oracle():
    """x_dense input path: W_in is a dense GEMM operand and takes the dense seqrec_adam."""
    V, F, H, T, B = 12, 24, 16, 6, 10
    rng = np.random.default_rng(23)
    ws = synthetic.make_weights("LSTM", V, H, seed=24, out_bias=True, F=F)
    hot = HotPath("LSTM", "relu", F, H, V, out_bias=True, weights=ws)
    ora = oa.Model("LSTM", "relu", ws, dtype=torch.float64)
    hot.set_optimizer("adam", lr=LR, epsilon=1e-8, clipnorm=1.0, decay=0.02)
    for step in range(3):
        x = (rng.random((B, T, F)) < 0.3).astype(np.float32) * rng.random((B, T, F)).astype(np.float32)
        x[:, :2] = 0.0
        tgt = rng.integers(0, V, size=(B, T)).astype(np.int32)
        mask = (x != 0).any(-1)
        tgt[~mask] = -1
        loss = float(hot.train_batch(None, tgt, x_dense=x).item())
        rl, _, _ = ora.train_step(None, as_t(tgt), torch.tensor(mask), lr=LR, epsilon=1e-8, clipnorm=1.0,
                                  optimizer="adam", decay=0.02, x_dense=torch.tensor(x, dtype=torch.float64))
        assert abs(loss - float(rl)) <= TOL * abs(float(rl))
        assert float(hot.dW_in.abs().max().item()) == 0.0
    for name, w, r in zip(NAMES, hot.get_weights(), ora.numpy_weights()):
        assert rel_err(w, r) <= 3e-4, (name, rel_err(w, r))


def test_adam_table_is_dense_and_keeps_untouched_rows():
    """A row touched at step 1 and absent from step 2 still moves at step 2 (g = 0, m and v decay) as the oracle says;
    a row never touched stays bit for bit with m = v = 0; dW_in and the touched flags are all zero after every step."""
    V, H, T, B = 200, 16, 6, 8
    hot, ora, ws = make_pair("GRU", "tanh", V, H, seed=31)
    hot.set_optimizer("adam", lr=LR, epsilon=1e-8, clipnorm=1.0)
    rng = np.random.default_rng(32)
    first, second = np.arange(0, 50), np.arange(50, 100)        # inputs of step 1 / step 2; rows >= 100 never touched
    snaps, inputs = [], []
    for items in (first, second):
        ids = rng.choice(items, size=(B, T)).astype(np.int32)
        tgt = rng.integers(0, V, size=(B, T)).astype(np.int32)
        hot.train_batch(ids, tgt)
        ora.train_step(as_t(ids), as_t(tgt), as_t(ids) >= 0, lr=LR, epsilon=1e-8, clipnorm=1.0, optimizer="adam")
        assert float(hot.dW_in.abs().max().item()) == 0.0 and int(hot.touched.abs().max().item()) == 0
        snaps.append(hot.get_weight("W_in"))
        inputs.append(np.unique(ids))
    W1, W2 = snaps
    seen1 = inputs[0]
    assert np.all(np.abs(W2[seen1] - W1[seen1]).max(axis=1) > 0)    # step-1 rows move at step 2 without a gradient
    ref = ora.W_in.numpy()
    assert rel_err(W2[:100], ref[:100]) <= 3e-4
    assert np.array_equal(W2[100:], ws[0][100:])
    m, v = hot.get_moments("W_in")
    assert not m[100:].any() and not v[100:].any()
    assert rel_err(m[:100], ora.moment[0].numpy()[:100]) <= 1e-3


def test_adam_graph_replay_equals_eager_and_recaptures_on_hyper_parameter_change():
    V, H, T, B = 3000, 64, 10, 64
    ws = synthetic.make_weights("GRU", V, H, seed=41)
    batches = [synthetic.make_batch(V, T, B, seed=42 + s, min_len=1) for s in range(8)]
    out = []
    for graphs in (True, False):
        hot = HotPath("GRU", "tanh", V, H, V, weights=ws, tc="x3")
        hot.use_graphs = graphs
        hot.set_optimizer("adam", lr=LR, epsilon=1e-8, clipnorm=1.0)
        losses = [float(hot.train_batch(i, t).item()) for i, t in batches[:5]]
        assert hot.get_iterations() == 5
        if graphs:
            assert hot.work(B, T).graph is not None
            key = hot.work(B, T).graph_key
        hot.set_optimizer("adam", lr=LR, epsilon=1e-8, clipnorm=1.0, decay=0.1, beta_1=0.8)
        losses += [float(hot.train_batch(i, t).item()) for i, t in batches[5:]]
        assert hot.get_iterations() == 3
        if graphs:
            assert hot.work(B, T).graph is not None and hot.work(B, T).graph_key != key
        out.append((losses, hot.get_weights()))
    (lg, wg), (le, we) = out
    assert np.allclose(lg, le, rtol=1e-5)
    for x, y in zip(wg, we):
        assert close_bulk(x, y, 3)


def test_adam_skip_branch_model_with_diagonal_constraint_and_frozen_transition_kernel():
    cell, act, y_to_z, x_to_z, x_to_y, y_to_y = VARIANTS[3]
    V, H, T, B = 17, 10, 7, 12
    ws = skip_weights(np.random.default_rng(8), cell, V, V, H, y_to_z, x_to_z, x_to_y, y_to_y, biases=False)
    for frozen in ((), ("A",)):
        hot = DensePath(cell, act, V, V, H, ws, y_to_z=y_to_z, x_to_z=x_to_z, x_to_y=x_to_y, y_to_y=y_to_y)
        ora = oa.SkipModel(cell, act, ws, y_to_z=y_to_z, x_to_z=x_to_z, x_to_y=x_to_y, y_to_y=y_to_y)
        hot.set_optimizer("adam", lr=LR, epsilon=1e-8, clipnorm=1.0, decay=0.01)
        for n in frozen:
            hot.trainable[n] = False
        for step in range(3):
            ids, tgt, x = make_inputs(V, T, B, seed=20 + step)
            loss = float(hot.train_batch(ids, tgt, x).item())
            rl, _ = ora.train_step(as_t(ids), torch.tensor(x, dtype=torch.float64), as_t(tgt), lr=LR, epsilon=1e-8,
                                   clipnorm=1.0, frozen=frozen, optimizer="adam", decay=0.01)
            assert abs(loss - float(rl)) <= TOL * abs(float(rl)), (step, loss, float(rl))
        assert hot.get_iterations() == 3
        for n in hot.weight_names():
            assert rel_err(hot.get_weight(n), ora.p[n].numpy()) <= 3e-4, (n, rel_err(hot.get_weight(n),
                                                                                    ora.p[n].numpy()))
        Wx = hot.get_weight("W_toy")[hot.H:]
        assert not (Wx - np.diag(np.diag(Wx))).any()
        if frozen:
            assert np.array_equal(hot.get_weight("A"), ws["A"])
            m, v = hot.get_moments("A")
            assert not m.any() and not v.any()


# ---- two ranks on one device (tests/test_gpu_vocab_parallel_one_device.py) ------------------------------------------
class _Done:
    def wait(self):
        pass


class AsyncThreadComm(ThreadComm):
    """ThreadComm with the asynchronous collectives of the data-parallel step, run synchronously."""

    def all_reduce_sum(self, t, async_op=False):
        ThreadComm.all_reduce_sum(self, t)
        return _Done() if async_op else None

    def all_gather_cat_async(self, t):
        return self.all_gather_cat(t), _Done()


# (V, H, T, B, cell, tc, vocab_parallel): vocabulary shards on the tensor-core and SIMT passes; data parallel with the
# dense dW_in exchange (V small against the global token count) and with the row exchange
TWO_RANK = [(10000, 128, 12, 64, "GRU", "x3", True), (998, 32, 6, 40, "LSTM", "off", True),
            (100, 32, 6, 30, "GRU", "off", False), (6000, 32, 4, 48, "LSTM", "off", False)]


@pytest.mark.parametrize("case", TWO_RANK, ids=lambda c: "%s%d-V%d-%s-%s" % (c[4], c[1], c[0], c[5],
                                                                            "vp" if c[6] else "dp"))
def test_adam_two_ranks_equal_single_gpu(case, monkeypatch):
    V, H, T, B, cell, tc, vp = case
    act = "tanh" if cell == "GRU" else "relu"
    ws = synthetic.make_weights(cell, V, H, seed=3)
    steps = [synthetic.make_batch(V, T, B, seed=50 + s, min_len=1) for s in range(2)]
    ref = HotPath(cell, act, V, H, V, weights=ws, comm=_solo(), tc=tc)
    ref.set_optimizer("adam", lr=LR, epsilon=1e-8, clipnorm=1.0, decay=0.01)
    want_losses = [float(ref.train_batch(i, t).item()) for i, t in steps]
    want_ws = ref.get_weights()

    def rank_fn(comm):
        hot = HotPath(cell, act, V, H, V, weights=ws, comm=comm, tc=tc, vocab_parallel=vp)
        hot.use_graphs = False                  # a captured graph would not replay the in-process collectives
        hot.set_optimizer("adam", lr=LR, epsilon=1e-8, clipnorm=1.0, decay=0.01)
        r = _rows(comm.rank, B)
        losses = [float(hot.train_batch(i[r], t[r]).item()) for i, t in steps]
        return losses, hot.get_weights(), hot.get_iterations()

    import test_gpu_vocab_parallel_one_device as vp1
    monkeypatch.setattr(vp1, "ThreadComm", AsyncThreadComm)    # run_ranks builds each rank's comm from this name
    for losses, mine, iters in run_ranks(rank_fn):
        assert iters == len(steps)
        for a, b in zip(losses, want_losses):
            assert abs(a - b) <= 1e-5 * abs(b), (a, b)
        for name, a, b in zip(NAMES, mine, want_ws):
            if tc == "off":
                assert rel_err(a, b) < 1e-4, (name, rel_err(a, b))
            else:
                assert close_bulk(a, b, len(steps)), name


# ---- model surface ---------------------------------------------------------------------------------------------------
def _learnable(V, T, n, seed):
    """Sessions that walk the catalog: the next item is (item + 1) mod V, so the loss can fall towards zero."""
    rng = np.random.default_rng(seed)
    start = rng.integers(0, V, size=(n, 1))
    seq = (start + np.arange(T + 1)) % V
    return seq[:, :T].astype(np.int32), seq[:, 1:].astype(np.int32)


def _model(V, T, H, optimizer, seed=5):
    m = M.RNNFullModel(T, V, V, z_dim=H, rnn_type="GRU", z_to_z_activation="tanh", y_to_y=False, x_to_y=False, seed=seed)
    m.compile_model(optimizer=optimizer)
    return m


def test_compile_model_with_adam_fits_and_the_loss_falls():
    V, T, H = 50, 8, 32
    ids, tgt = _learnable(V, T, 512, seed=1)
    m = _model(V, T, H, Adam(lr=0.03, clipnorm=1.0))
    np.random.seed(3)
    h = m.fit_model(ids, tgt, n_epochs=6, batch_size=64, verbose=0)
    loss = h.history["loss"]
    assert np.all(np.isfinite(loss)) and loss[-1] < 0.5 * loss[0], loss
    assert m.model.hot.get_iterations() == 6 * 8


def test_adam_state_checkpoint_resumes_and_refuses_another_optimizer(tmp_path):
    V, H, T, B = 400, 32, 8, 64
    ids, tgt = synthetic.make_batch(V, T, 4 * B, seed=3, min_len=1)
    adam = lambda: Adam(lr=LR, beta_1=0.85, epsilon=1e-8, decay=0.01, clipnorm=1.0)

    def steps(m, lo, hi):
        return [m.model.train_on_batch(ids[b * B:(b + 1) * B], tgt[b * B:(b + 1) * B]) for b in range(lo, hi)]

    a = _model(V, T, H, adam())
    steps(a, 0, 2)
    ck = str(tmp_path / "adam_state.npz")
    a.model.save_state(ck, epoch=7)
    wk = str(tmp_path / "weights_only")
    a.model.save_weights(wk)
    with np.load(ck) as z:
        assert str(z["opt_kind"]) == "adam" and int(z["iterations"]) == 2
        assert np.allclose(z["opt"], [LR, 0.85, 0.999, 1e-8, 1.0, 0.01])
        assert {"m%d" % i for i in range(4)} | {"v%d" % i for i in range(4)} <= set(z.files)
        assert not any(k.startswith("accum") for k in z.files)
    rest = steps(a, 2, 4)
    b = _model(V, T, H, adam())
    assert b.model.load_state(ck) == 7
    assert b.model.hot.get_iterations() == 2
    assert np.allclose(steps(b, 2, 4), rest, rtol=1e-5)
    for x, y in zip(a.model.get_weights(), b.model.get_weights()):
        assert close_bulk(x, y, 2)
    assert b.model.hot.get_iterations() == a.model.hot.get_iterations() == 4
    c = _model(V, T, H, adam())
    c.model.load_weights(wk)
    assert steps(c, 2, 4)[1] != rest[1]                         # moments and count restarted: another trajectory

    ag = str(tmp_path / "adagrad_state.npz")
    g = _model(V, T, H, Adagrad(lr=0.05, epsilon=1e-8, clipnorm=1.0))
    steps(g, 0, 1)
    g.model.save_state(ag)
    with pytest.raises(ValueError, match="adagrad"):
        _model(V, T, H, adam()).model.load_state(ag)
    with pytest.raises(ValueError, match="adam"):
        _model(V, T, H, Adagrad(lr=0.05, epsilon=1e-8, clipnorm=1.0)).model.load_state(ck)
