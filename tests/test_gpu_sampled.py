"""Sampled softmax training on the device (csrc/sampled.cu, HotPath.set_loss) against the float64 oracle
(oracle/sampled.py): the sampler bit for bit, one step's loss and gradients, training with Adagrad and Adam, graph replay,
the untouched default path, two data-parallel ranks on one device and the model surface.  Run with -m gpu on a B200.

Tolerances are the project's: 1e-4 relative (norm-wise) on loss and gradients in fp32 / x3 mode, 3e-2 in bf16 mode;
after updates, those of the Adagrad / Adam tests."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import sampled as osm
from seq_recommendations_b200 import _lib, losses, synthetic
from seq_recommendations_b200 import model as M
from seq_recommendations_b200.engine import HotPath
from seq_recommendations_b200.optimizers import Adagrad, Adam

from gpu_util import as_t, rel_err
from test_gpu_vocab_parallel_one_device import ThreadComm, _rows, _solo, run_ranks

pytestmark = pytest.mark.gpu
TOL = {"off": 1e-4, "x3": 1e-4, "bf16": 3e-2}
NAMES = ["W_in", "U", "b", "W_out", "b_out"]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _draw_device(S, V, seed, state, thr=None, alias=None):
    ids = torch.empty(S, dtype=torch.int32, device="cuda")
    _lib.call("seqrec_sample_items", _lib.ptr(ids), S, _lib.ptr(thr), _lib.ptr(alias), V, seed, _lib.ptr(state),
              ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    return ids.cpu().numpy().astype(np.int64)


# ---- 1. sampler ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("V", [1000, 70001])
@pytest.mark.parametrize("weighted", [False, True])
def test_sampler_equals_numpy_restatement_bit_for_bit(V, weighted):
    _lib.load()
    thr = alias = thr_np = alias_np = None
    if weighted:
        w = 1.0 / np.arange(1, V + 1) ** 0.9
        thr_np, alias_np = losses.alias_table(w / w.sum())
        thr = torch.from_numpy(thr_np.view(np.int32)).cuda()
        alias = torch.from_numpy(alias_np).cuda()
    S = 777
    for seed in (0, 3, 2 ** 40 + 11):
        for offset in (0, 5, 2 ** 33 + 1):
            state = torch.tensor([offset, 0], dtype=torch.int64, device="cuda")
            for call in range(3):                             # the state advances by S per call
                got = _draw_device(S, V, seed, state, thr, alias)
                want = osm.draw(S, V, seed, offset + call * S, thr_np, alias_np)
                assert np.array_equal(got, want), (seed, offset, call)
                assert state.tolist() == [offset + (call + 1) * S, 0]


def test_sampler_histogram_is_consistent_with_q():
    V, n = 50, 10 ** 7
    w = np.where(np.arange(V) % 7 == 0, 20.0, 1.0) * (1.0 + np.arange(V) / V)
    q = w / w.sum()
    thr_np, alias_np = losses.alias_table(q)
    state = torch.zeros(2, dtype=torch.int64, device="cuda")
    ids = _draw_device(n, V, 1234, state, torch.from_numpy(thr_np.view(np.int32)).cuda(),
                       torch.from_numpy(alias_np).cuda())
    counts = np.bincount(ids, minlength=V)
    expected = n * q
    chi2 = float(((counts - expected) ** 2 / expected).sum())
    assert chi2 < 3 * V, chi2                                  # V - 1 degrees of freedom: mean 49, sd 10


# ---- 2. one step against the oracle ----------------------------------------------------------------------------------
def _oracle_step(ora, ids, tgt, samples, out_scale=None):
    """Oracle loss, gradients and dL/dhout (the engine's dh) for the given samples."""
    mask = as_t(ids) >= 0
    loss, gs = ora.grads(as_t(ids), as_t(tgt), mask, out_scale=out_scale, samples=samples)
    Hout, _ = ora.hidden(ids=as_t(ids), mask=mask)
    Hout = Hout.detach().requires_grad_(True)
    hs = Hout * out_scale if out_scale is not None else Hout
    from oracle import keras_semantics as ks
    z = ks.logits(hs, ora.W_out, ora.b_out)
    mf = mask.to(z.dtype)
    ce = osm.sampled_ce(z, as_t(tgt), torch.as_tensor(samples, dtype=torch.int64), ora.logq) * mf
    dh, = torch.autograd.grad(ce.sum() / mf.sum(), Hout)
    return float(loss), [g.numpy() for g in gs], dh.numpy()


# (cell, act, V, H, T, B, tc, out_bias, S, weights): SIMT and tensor-core GEMMs, H above the fused kernels' 256, a tiny
# catalog where hits and duplicates are certain, weights concentrated on the batch's targets
CASES = [("GRU", "tanh", 3000, 64, 8, 40, "off", True, 512, None),
         ("LSTM", "relu", 3000, 128, 8, 40, "x3", False, 1024, "zipf"),
         ("simpleRNN", "tanh", 2000, 256, 6, 48, "x3", True, 384, None),
         ("GRU", "tanh", 2500, 320, 6, 40, "x3", True, 640, "zipf"),
         ("GRU", "tanh", 3000, 128, 8, 40, "bf16", True, 512, None),
         ("GRU", "tanh", 300, 64, 8, 40, "x3", True, 256, None),
         ("LSTM", "tanh", 300, 32, 8, 40, "off", False, 256, "zipf"),
         ("GRU", "tanh", 2000, 64, 8, 40, "x3", True, 512, "targets"),
         ("LSTM", "relu", 2000, 32, 6, 20, "off", True, 300, "targets")]


def _weights(kind, V, tgt):
    if kind is None:
        return None
    if kind == "zipf":
        return 1.0 / np.arange(1, V + 1) ** 0.8
    return 1.0 + 1e4 * np.isin(np.arange(V), tgt[tgt >= 0])


def _check_step(hot, ora, ids, tgt, tc, out_bias, frozen_w_out=False):
    out_scale = None
    loss, grads, extra = hot.grad_batch(ids, tgt)
    samples = hot.last_samples()
    B, T = ids.shape
    w = hot.work(B, T)
    if w.hscale is not None:
        out_scale = w.hscale.view(T, B, hot.H).permute(1, 0, 2).cpu().double()
    rl, rg, rdh = _oracle_step(ora, ids, tgt, samples, out_scale)
    tol = TOL[tc]
    assert abs(loss - rl) <= tol * abs(rl), (loss, rl)
    assert rel_err(extra["dh"].transpose(1, 0, 2), rdh) <= tol, rel_err(extra["dh"].transpose(1, 0, 2), rdh)
    for name, g, r in zip(NAMES, grads, rg):
        if name == "W_out" and frozen_w_out:
            assert not g.any()
            continue
        assert rel_err(g, r) <= tol, (name, rel_err(g, r))
    return samples


@pytest.mark.parametrize("cell,act,V,H,T,B,tc,bias,S,wk", CASES)
def test_one_step_matches_oracle(cell, act, V, H, T, B, tc, bias, S, wk):
    ws = synthetic.make_weights(cell, V, H, seed=5, out_bias=bias)
    if bias:
        ws[4] = np.random.default_rng(6).standard_normal(V).astype(np.float32) * 0.5
    ids, tgt = synthetic.make_batch(V, T, B, seed=7, min_len=1)
    weights = _weights(wk, V, tgt)
    hot = HotPath(cell, act, V, H, V, out_bias=bias, weights=ws, tc=tc)
    hot.set_loss("sampled_softmax", num_sampled=S, weights=weights)
    q = None if weights is None else weights / weights.sum()
    ora = osm.Model(cell, act, ws, S, q)
    samples = _check_step(hot, ora, ids, tgt, tc, bias)
    assert samples.shape == (S,) and samples.min() >= 0 and samples.max() < V
    if V == 300:                                              # duplicates and accidental hits are certain
        assert len(np.unique(samples)) < S and np.isin(tgt[tgt >= 0], samples).any()
    # a second step draws other ids
    _check_step(hot, ora, ids, tgt, tc, bias)
    assert not np.array_equal(hot.last_samples(), samples)


@pytest.mark.parametrize("tc", ["off", "x3"])
def test_one_step_with_output_dropout_and_frozen_output_kernel(tc):
    V, H, T, B, S = 2000, 64, 8, 40, 512
    ws = synthetic.make_weights("GRU", V, H, seed=8, out_bias=True)
    ids, tgt = synthetic.make_batch(V, T, B, seed=9, min_len=1)
    hot = HotPath("GRU", "tanh", V, H, V, out_bias=True, weights=ws, tc=tc)
    hot.dropout_out = 0.3
    hot.set_loss("sampled_softmax", num_sampled=S)
    _check_step(hot, osm.Model("GRU", "tanh", ws, S), ids, tgt, tc, True)
    assert hot.work(B, T).hscale is not None
    hot.trainable["W_out"] = False
    _check_step(hot, osm.Model("GRU", "tanh", ws, S), ids, tgt, tc, True, frozen_w_out=True)


# ---- 3. training -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("opt", ["adagrad", "adam"])
def test_training_steps_match_oracle(opt):
    V, H, T, B, S = 1500, 32, 8, 40, 300
    ws = synthetic.make_weights("GRU", V, H, seed=11, out_bias=True)
    w8 = 1.0 + np.arange(V) % 5
    hot = HotPath("GRU", "tanh", V, H, V, out_bias=True, weights=ws, tc="off")
    hot.set_optimizer(opt, lr=0.01, epsilon=1e-8, clipnorm=1.0)
    hot.set_loss("sampled_softmax", num_sampled=S, weights=w8)
    ora = osm.Model("GRU", "tanh", ws, S, w8 / w8.sum())
    for step in range(3):
        ids, tgt = synthetic.make_batch(V, T, B, seed=20 + step, min_len=1)
        loss = float(hot.train_batch(ids, tgt).item())
        rl, _, _ = ora.train_step(as_t(ids), as_t(tgt), as_t(ids) >= 0, lr=0.01, epsilon=1e-8, clipnorm=1.0,
                                  optimizer=opt, samples=hot.last_samples())
        assert abs(loss - float(rl)) <= 1e-4 * abs(float(rl)), (step, loss, float(rl))
        for name, a, b in zip(NAMES, hot.get_weights(), ora.numpy_weights()):
            assert rel_err(a, b) <= 3e-4, (step, name, rel_err(a, b))


# ---- 4. graph replay -------------------------------------------------------------------------------------------------
def test_graph_replay_draws_fresh_ids_and_equals_eager():
    V, H, T, B, S = 4000, 64, 10, 64, 1024
    ws = synthetic.make_weights("GRU", V, H, seed=41, out_bias=True)
    batches = [synthetic.make_batch(V, T, B, seed=42 + s, min_len=1) for s in range(6)]
    runs = []
    for graphs in (True, False):
        hot = HotPath("GRU", "tanh", V, H, V, out_bias=True, weights=ws, tc="x3", seed=3)
        hot.use_graphs = graphs
        hot.set_optimizer("adagrad", lr=0.05, epsilon=1e-8, clipnorm=1.0)
        hot.set_loss("sampled_softmax", num_sampled=S)
        losses_, ids_ = [], []
        for i, t in batches[:4]:
            losses_.append(float(hot.train_batch(i, t).item()))
            ids_.append(hot.last_samples())
        if graphs:
            w = hot.work(B, T)
            assert w.graph is not None
            key = w.graph_key
            hot.set_loss("sampled_softmax", num_sampled=512)     # another S re-captures
            hot.train_batch(*batches[4])
            hot.train_batch(*batches[5])
            assert w.graph is not None and w.graph_key != key and hot.last_samples().shape == (512,)
            key = w.graph_key
            hot.set_loss("categorical_crossentropy")             # so does switching the loss kind
            hot.train_batch(*batches[4])
            hot.train_batch(*batches[5])
            assert w.graph_key != key
        runs.append((losses_, ids_, hot))
    (lg, ig, _), (le, ie, _) = runs
    for a in range(len(ig)):
        assert np.array_equal(ig[a], ie[a])
        for b in range(a):
            assert not np.array_equal(ig[a], ig[b])
    assert np.allclose(lg, le, rtol=1e-5)


def test_graph_replay_weights_equal_eager():
    V, H, T, B, S = 3000, 32, 8, 48, 512
    ws = synthetic.make_weights("LSTM", V, H, seed=12)
    batches = [synthetic.make_batch(V, T, B, seed=60 + s, min_len=1) for s in range(4)]
    out = []
    for graphs in (True, False):
        hot = HotPath("LSTM", "relu", V, H, V, weights=ws, tc="off", seed=9)
        hot.use_graphs = graphs
        hot.set_optimizer("adagrad", lr=0.05, epsilon=1e-8, clipnorm=1.0)
        hot.set_loss("sampled_softmax", num_sampled=S)
        ls = [float(hot.train_batch(i, t).item()) for i, t in batches]
        out.append((ls, hot.get_weights()))
    (lg, wg), (le, we) = out
    assert np.allclose(lg, le, rtol=1e-5)
    for a, b in zip(wg, we):
        assert rel_err(a, b) <= 1e-5


# ---- 5. default path untouched ---------------------------------------------------------------------------------------
def test_categorical_after_sampled_equals_never_sampled():
    V, H, T, B = 3000, 64, 8, 64
    ws = synthetic.make_weights("GRU", V, H, seed=13)
    batches = [synthetic.make_batch(V, T, B, seed=70 + s, min_len=1) for s in range(3)]
    a = HotPath("GRU", "tanh", V, H, V, weights=ws, tc="x3")
    b = HotPath("GRU", "tanh", V, H, V, weights=ws, tc="x3")
    for h in (a, b):
        h.set_optimizer("adagrad", lr=0.05, epsilon=1e-8, clipnorm=1.0)
    a.set_loss("sampled_softmax", num_sampled=256)
    a.grad_batch(*batches[0])                                 # a sampled step without an update
    a.set_loss("categorical_crossentropy")
    assert a.last_samples() is None
    la, ga, _ = a.grad_batch(*batches[0])
    lb, gb, _ = b.grad_batch(*batches[0])
    assert la == lb
    for x, y in zip(ga, gb):
        assert rel_err(x, y) <= 1e-6
    for i, t in batches:
        assert float(a.train_batch(i, t).item()) == pytest.approx(float(b.train_batch(i, t).item()), rel=1e-6)
    for x, y in zip(a.get_weights(), b.get_weights()):
        assert rel_err(x, y) <= 1e-5


# ---- 6. two data-parallel ranks on one device ------------------------------------------------------------------------
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


@pytest.mark.parametrize("V", [100, 6000])                   # dense dW_in exchange, row exchange
def test_two_ranks_draw_the_same_ids_and_equal_single_gpu(V, monkeypatch):
    H, T, B, S = 32, 6, 48, 64
    ws = synthetic.make_weights("GRU", V, H, seed=3, out_bias=True)
    steps = [synthetic.make_batch(V, T, B, seed=50 + s, min_len=1) for s in range(2)]
    ref = HotPath("GRU", "tanh", V, H, V, out_bias=True, weights=ws, comm=_solo(), tc="off", seed=4)
    ref.set_optimizer("adagrad", lr=0.05, epsilon=1e-8, clipnorm=1.0)
    ref.set_loss("sampled_softmax", num_sampled=S)
    want = []
    for i, t in steps:
        want.append((float(ref.train_batch(i, t).item()), ref.last_samples()))
    want_ws = ref.get_weights()

    def rank_fn(comm):
        hot = HotPath("GRU", "tanh", V, H, V, out_bias=True, weights=ws, comm=comm, tc="off", seed=4)
        hot.use_graphs = False
        hot.set_optimizer("adagrad", lr=0.05, epsilon=1e-8, clipnorm=1.0)
        hot.set_loss("sampled_softmax", num_sampled=S)
        r = _rows(comm.rank, B)
        got = []
        for i, t in steps:
            got.append((float(hot.train_batch(i[r], t[r]).item()), hot.last_samples()))
        return got, hot.get_weights()

    import test_gpu_vocab_parallel_one_device as vp1
    monkeypatch.setattr(vp1, "ThreadComm", AsyncThreadComm)
    for got, mine in run_ranks(rank_fn):
        for (l, ids), (wl, wids) in zip(got, want):
            assert np.array_equal(ids, wids)
            assert abs(l - wl) <= 1e-5 * abs(wl), (l, wl)
        for name, a, b in zip(NAMES, mine, want_ws):
            assert rel_err(a, b) < 1e-4, (name, rel_err(a, b))


def test_vocab_parallel_refuses_sampled_softmax():
    V, H, T = 1000, 16, 4

    def rank_fn(comm):
        hot = HotPath("GRU", "tanh", V, H, V, comm=comm, vocab_parallel=True)
        with pytest.raises(NotImplementedError):
            hot.set_loss("sampled_softmax", num_sampled=64)
        m = M.RNNFullModel(T, V, V, z_dim=H, rnn_type="GRU", z_to_z_activation="tanh", y_to_y=False, x_to_y=False,
                           seed=1, comm=comm, vocab_parallel=True)
        with pytest.raises(NotImplementedError):
            m.compile_model(loss=losses.SampledSoftmax(64), optimizer=Adagrad(lr=0.05))
        return True

    assert all(run_ranks(rank_fn))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_two_gpu_sampled_step_equals_single_gpu_step():
    import socket
    sock = socket.socket()
    sock.bind(("127.0.0.1", 0))
    port = sock.getsockname()[1]
    sock.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "sampled_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    sys.stdout.write(r.stdout[-4000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "MISMATCH" not in r.stdout


# ---- 7. model surface ------------------------------------------------------------------------------------------------
def test_compile_model_with_sampled_softmax_fits_and_keeps_full_softmax_metrics():
    V, T, H = 20000, 10, 128
    ids, tgt = synthetic.make_batch(V, T, 2048, seed=1, min_len=2)
    # a learnable corpus: the next item is a fixed function of the current one
    tgt = np.where(ids >= 0, (ids * 7 + 3) % V, -1).astype(np.int32)
    vi, vt = ids[:256], tgt[:256]
    m = M.RNNFullModel(T, V, V, z_dim=H, rnn_type="GRU", z_to_z_activation="tanh", y_to_y=False, x_to_y=False, seed=2)
    m.compile_model(loss=losses.SampledSoftmax(2048), optimizer=Adagrad(lr=0.1, epsilon=1e-8, clipnorm=1.0))
    assert m.model.hot.sampled is not None and m.model.hot.sampled.S == 2048
    h = m.fit_model(ids[256:], tgt[256:], validation_data=(vi, vt), n_epochs=3, batch_size=256, verbose=0)
    vl = h.history["val_loss"]
    assert np.all(np.isfinite(h.history["loss"])) and vl[2] < vl[1] < vl[0], vl
    # evaluate is the full categorical cross-entropy: the same weights in a string-loss model give the same value
    _, got = m.evaluate(vi, vt, batch_size=64)
    ref = M.RNNFullModel(T, V, V, z_dim=H, rnn_type="GRU", z_to_z_activation="tanh", y_to_y=False, x_to_y=False, seed=2)
    ref.compile_model(optimizer=Adagrad(lr=0.1, epsilon=1e-8, clipnorm=1.0))
    assert ref.model.hot.sampled is None
    ref.model.set_weights(m.model.get_weights())
    _, want = ref.evaluate(vi, vt, batch_size=64)
    got, want = np.ravel(got)[0], np.ravel(want)[0]
    assert abs(got - want) <= 1e-5 * abs(want), (got, want)


def test_string_loss_models_unchanged_and_dense_models_refuse():
    V, T, H = 60, 6, 16
    m = M.RNNFullModel(T, V, V, z_dim=H, rnn_type="GRU", z_to_z_activation="tanh", y_to_y=False, x_to_y=False, seed=2)
    m.compile_model(optimizer=Adagrad(lr=0.1))
    assert m.model.hot.sampled is None
    m.compile_model(loss=losses.SampledSoftmax(16), optimizer=Adagrad(lr=0.1))
    m.compile_model(optimizer=Adagrad(lr=0.1))                # back to the full softmax
    assert m.model.hot.sampled is None
    skip = M.RNNFullModel(T, V, V, z_dim=H, rnn_type="GRU", z_to_z_activation="tanh", y_to_y=True, x_to_y=False, seed=2)
    with pytest.raises(NotImplementedError):
        skip.compile_model(loss=losses.SampledSoftmax(16), optimizer=Adagrad(lr=0.1))
    norec = M.NoRecurrenceModel(T, V, V, connect_x=False, seed=2)
    with pytest.raises(NotImplementedError):
        norec.compile_model(loss=losses.SampledSoftmax(16), optimizer=Adagrad(lr=0.1))
    with pytest.raises(ValueError):
        m.compile_model(loss=losses.SampledSoftmax(61), optimizer=Adagrad(lr=0.1))
