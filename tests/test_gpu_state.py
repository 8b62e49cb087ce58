"""Carried recurrent state on the B200: every forward scan family (generic fp32, register-resident, tcgen05 cluster)
started from a non-zero (h0, c0) against the float64 oracle; NULL pointers bit-identical to the existing entry points;
chunked scans bit-identical to one scan; the engine's *_from_state scorers equal to the last_step_only scorers; the
model surface and its state pool.

Tolerances: the scans are compared with the float64 oracle at 1e-4 relative, the fp32 bound of the existing scan tests.
Everything computed by the same kernels on the same problem shape is compared bitwise: a continued scan performs the
same per-step arithmetic as one longer scan, and the (n, 1) scoring problem of a state is the one last_step_only builds.
p(target) compared across different token counts is held to 1e-6 relative instead, because the tensor-core statistics
pass splits the vocabulary reduction by the token count (seqrec_ce_tc_partials(N, ...))."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import state as ost
from seq_recommendations_b200 import model as M
from seq_recommendations_b200 import synthetic
from seq_recommendations_b200._lib import ACT, CELL, SeqrecError, call, ptr
from seq_recommendations_b200.engine import HotPath
from seq_recommendations_b200.state import RecurrentState

from gpu_util import rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = {"simpleRNN": 1, "LSTM": 4, "GRU": 3}
B = 301          # not a multiple of 64 (tensor-core clusters) nor of the row blocks 2 / 4 / 8; > 148 so RB > 1

# (family, cell, act, H): generic = above the register scans' range; register = GRU / SimpleRNN H <= 128, LSTM <= 100
FAMILIES = [("generic", "simpleRNN", "tanh", 200), ("generic", "GRU", "tanh", 300), ("generic", "LSTM", "tanh", 160),
            ("register", "GRU", "tanh", 64), ("register", "GRU", "relu", 128), ("register", "simpleRNN", "tanh", 64),
            ("register", "simpleRNN", "tanh", 128), ("register", "LSTM", "tanh", 100),
            ("tc", "LSTM", "tanh", 128), ("tc", "LSTM", "relu", 256), ("tc", "GRU", "tanh", 128),
            ("tc", "GRU", "tanh", 256)]


@pytest.fixture(scope="module")
def dev():
    torch.cuda.set_device(0)
    return torch.device("cuda:0")


def _problem(cell, H, T, seed, dev):
    rng = np.random.default_rng(seed)
    GH = G[cell] * H
    xp = rng.standard_normal((T, B, GH)).astype(np.float32) * 0.5
    U = (rng.standard_normal((H, GH)) / np.sqrt(H)).astype(np.float32)
    L = rng.integers(0, T + 1, size=B)
    L[:3] = 0                                                  # all-pad rows
    L[3:6] = T
    mask = (np.arange(T)[:, None] >= (T - L)[None, :])         # (T, B) left-padded
    h0 = (rng.standard_normal((B, H)) * 0.5).astype(np.float32)
    c0 = (rng.standard_normal((B, H)) * 0.5).astype(np.float32) if cell == "LSTM" else None
    t = lambda a: None if a is None else torch.tensor(a, device=dev)
    return t(xp), t(U), t(mask.astype(np.uint8)), t(h0), t(c0)


def _scan(family, cell, act, xp, U, mask, h0, c0, state_api=True):
    """One forward scan through the C-ABI; returns (hout (T,B,H), cst (T,B,H), gates (T,B,GH))."""
    T, Bn, GH = xp.shape
    H = U.shape[0]
    xg = xp.clone()
    hout = torch.empty((T, Bn, H), dtype=torch.float32, device=xp.device)
    cst = torch.empty((T, Bn, H), dtype=torch.float32, device=xp.device)
    st = torch.cuda.current_stream().cuda_stream
    if family == "tc":
        Ut_hi = torch.empty((GH, H), dtype=torch.bfloat16, device=xp.device)
        Ut_lo = torch.empty_like(Ut_hi)
        call("seqrec_split_bf16", ptr(U), None, ptr(Ut_hi), ptr(Ut_lo), H, GH, H, 1, st)
        if state_api:
            call("seqrec_rnn_tc_forward_state", CELL[cell], ACT[act], ptr(xg), ptr(Ut_hi), ptr(Ut_lo), ptr(h0), ptr(c0),
                 ptr(mask), ptr(hout), ptr(cst), T, Bn, H, st)
        else:
            call("seqrec_rnn_tc_forward", CELL[cell], ACT[act], ptr(xg), ptr(Ut_hi), ptr(Ut_lo), ptr(mask), ptr(hout),
                 ptr(cst), T, Bn, H, st)
    elif state_api:
        call("seqrec_rnn_forward_state", CELL[cell], ACT[act], ptr(xg), ptr(U), ptr(h0), ptr(c0), ptr(mask), ptr(hout),
             ptr(cst), T, Bn, H, st)
    else:
        call("seqrec_rnn_forward", CELL[cell], ACT[act], ptr(xg), ptr(U), ptr(mask), ptr(hout), ptr(cst), T, Bn, H, st)
    torch.cuda.synchronize()
    return hout, cst, xg


def _final(cell, hout, cst):
    return hout[-1].clone(), (cst[-1].clone() if cell == "LSTM" else None)


# ------------------------------------------------------------------------------------------------ 1. against the oracle
@pytest.mark.parametrize("family,cell,act,H", FAMILIES)
@pytest.mark.parametrize("T", [1, 9])
def test_scan_from_state_matches_oracle(dev, family, cell, act, H, T):
    xp, U, mask, h0, c0 = _problem(cell, H, T, 11 + H + T, dev)
    hout, cst, _ = _scan(family, cell, act, xp, U, mask, h0, c0)
    d = lambda a: a.double().cpu()
    want, h_T, c_T = ost.rnn_forward_state(d(xp).permute(1, 0, 2), d(U), d(mask).bool().t(), cell, act, d(h0),
                                          None if c0 is None else d(c0))
    got = hout.permute(1, 0, 2).cpu().numpy()
    assert rel_err(got, want.numpy()) <= 1e-4, rel_err(got, want.numpy())
    assert rel_err(hout[-1].cpu().numpy(), h_T.numpy()) <= 1e-4
    if cell == "LSTM":
        assert rel_err(cst[-1].cpu().numpy(), c_T.numpy()) <= 1e-4
    # all-pad rows repeat the carried state bit for bit at every step
    assert torch.equal(hout[:, :3], h0[:3].unsqueeze(0).expand(T, 3, H))
    if cell == "LSTM":
        assert torch.equal(cst[:, :3], c0[:3].unsqueeze(0).expand(T, 3, H))


# ------------------------------------------------------------------------------------------------ 2. NULL = existing
@pytest.mark.parametrize("family,cell,act,H", FAMILIES)
def test_null_and_zero_state_are_the_existing_scan(dev, family, cell, act, H):
    T = 6
    xp, U, mask, _, _ = _problem(cell, H, T, 5, dev)
    ref = _scan(family, cell, act, xp, U, mask, None, None, state_api=False)
    null = _scan(family, cell, act, xp, U, mask, None, None)
    zeros = torch.zeros((B, H), dtype=torch.float32, device=dev)
    zero = _scan(family, cell, act, xp, U, mask, zeros, zeros if cell == "LSTM" else None)
    for a, b, c in zip(ref, null, zero):
        if cell != "LSTM" and a is ref[1]:
            continue                                           # cst is untouched scratch for GRU / SimpleRNN
        assert torch.equal(a, b) and torch.equal(a, c)


def test_c0_for_a_gru_is_an_argument_error(dev):
    xp, U, mask, h0, _ = _problem("GRU", 64, 2, 1, dev)
    with pytest.raises(SeqrecError):
        _scan("register", "GRU", "tanh", xp, U, mask, h0, h0)
    xp, U, mask, h0, _ = _problem("GRU", 128, 2, 1, dev)
    with pytest.raises(SeqrecError):
        _scan("tc", "GRU", "tanh", xp, U, mask, h0, h0)


# ------------------------------------------------------------------------------------------------ 3. chunking
@pytest.mark.parametrize("family,cell,act,H", FAMILIES)
def test_chunked_scan_is_bit_identical(dev, family, cell, act, H):
    T = 8
    xp, U, mask, h0, c0 = _problem(cell, H, T, 23, dev)
    whole = _scan(family, cell, act, xp, U, mask, h0, c0)
    h_w, c_w = _final(cell, whole[0], whole[1])
    for cuts in ([3], [1, 7], [5, 6], list(range(1, T))):
        h, c, outs = h0, c0, []
        for a, b in zip([0] + cuts, cuts + [T]):
            hout, cst, _ = _scan(family, cell, act, xp[a:b].contiguous(), U, mask[a:b].contiguous(), h, c)
            outs.append(hout)
            h, c = _final(cell, hout, cst)
        assert torch.equal(torch.cat(outs), whole[0]), cuts
        assert torch.equal(h, h_w), cuts
        if cell == "LSTM":
            assert torch.equal(c, c_w), cuts
    # an all-pad chunk keeps every row's state bitwise
    hout, cst, _ = _scan(family, cell, act, xp[:2].contiguous(), U, torch.zeros_like(mask[:2]), h_w, c_w)
    h, c = _final(cell, hout, cst)
    assert torch.equal(h, h_w) and (c is None or torch.equal(c, c_w))


# ------------------------------------------------------------------------------------------------ 4. engine
@pytest.mark.parametrize("cell,H", [("GRU", 128), ("LSTM", 256), ("LSTM", 100), ("GRU", 320)])
def test_engine_scores_from_state(dev, cell, H):
    V, T, n, k = 12000, 10, 300, 20
    act = "tanh"
    ws = synthetic.make_weights(cell, V, H, seed=2)
    hot = HotPath(cell, act, V, H, V, weights=ws)
    ids, tgt = synthetic.make_batch(V, T, n, seed=3, min_len=0)
    ids[:2] = -1
    tgt[:2] = -1                                               # all-pad sessions
    st = hot.advance_state(ids)
    assert isinstance(st, RecurrentState) and len(st) == n and st.h.data_ptr() != hot.work(n, T).hout.data_ptr()
    ti, tp = hot.topk_batch(ids, k, last_step_only=True)
    si, sp = hot.topk_from_state(st, k)
    assert torch.equal(si, ti) and torch.equal(sp, tp)
    # the last column of the whole-window scores: the rank bitwise, p(target) to 1e-6 (different token counts)
    r_whole = hot.target_rank_batch(ids, tgt)[:, -1]
    r_last = hot.target_rank_batch(ids, tgt, last_step_only=True)
    r_state = hot.target_rank_from_state(st, tgt[:, -1])
    assert torch.equal(r_state, r_last)
    if H <= 256:
        assert torch.equal(r_state, r_whole)
    p_whole = hot.target_prob_batch(ids, tgt)[:, -1].cpu().numpy()
    p_state = hot.target_prob_from_state(st, tgt[:, -1]).cpu().numpy()
    assert np.allclose(p_state, p_whole, rtol=1e-6, atol=0)
    # a chunk b scored as the continuation of a equals the b-columns of a|b
    s = 6
    st_a = hot.advance_state(ids[:, :s])
    h_ab = hot.hidden_batch(ids)
    assert torch.equal(hot.hidden_batch(ids[:, s:], initial_state=st_a), h_ab[:, s:])
    p_ab = hot.target_prob_batch(ids, tgt).cpu().numpy()
    p_b = hot.target_prob_batch(ids[:, s:], tgt[:, s:], initial_state=st_a).cpu().numpy()
    assert np.allclose(p_b, p_ab[:, s:], rtol=1e-6, atol=0)
    if H <= 256:
        rk_ab = hot.target_rank_batch(ids, tgt)
        assert torch.equal(hot.target_rank_batch(ids[:, s:], tgt[:, s:], initial_state=st_a), rk_ab[:, s:])
    bi, bp = hot.topk_batch(ids[:, s:], k, last_step_only=True, initial_state=st_a)
    assert torch.equal(bi, ti) and torch.equal(bp, tp)
    with pytest.raises(ValueError):
        hot.advance_state(ids[:10], st)                        # 300 states for 10 sessions


# ------------------------------------------------------------------------------------------------ 5. cfg5 widths
def test_cfg5_width_199_plus_1_equals_200(dev):
    """GRU-256, V = 100k, T = 200 (the cfg5 scoring shape) with the batch reduced 8x, to 512 sessions."""
    V, H, T, n = 100000, 256, 200, 512
    hot = HotPath("GRU", "tanh", V, H, V, weights=synthetic.make_weights("GRU", V, H, seed=5))
    assert hot.rnn_tc
    ids, _ = synthetic.make_batch(V, T, n, seed=6)
    whole = hot.advance_state(ids)
    st = hot.advance_state(ids[:, 199:], hot.advance_state(ids[:, :199]))
    assert torch.equal(st.h, whole.h)
    ti, tp = hot.topk_batch(ids, 20, last_step_only=True)
    si, sp = hot.topk_from_state(st, 20)
    assert torch.equal(si, ti) and torch.equal(sp, tp)


# ------------------------------------------------------------------------------------------------ 6. model surface
def _ytoz(cell, V, H):
    return M.RNNFullModel(timesteps=12, x_dim=V, y_dim=V, z_dim=H, model_name="ytoz", rnn_type=cell,
                          z_to_z_activation="tanh", y_to_z=True, y_to_y=False, x_to_y=False, x_to_z=False, seed=4)


@pytest.mark.parametrize("cell", ["LSTM", "GRU"])
def test_model_chunks_equal_predict_topk(dev, cell, tmp_path):
    V, T, n = 3000, 12, 150
    model = _ytoz(cell, V, 64)
    ids, tgt = synthetic.make_batch(V, T, n, seed=8, min_len=1)
    st = model.initial_state(n)
    for a, b in ((0, 5), (5, 6), (6, 12)):
        st = model.advance_state(ids[:, a:b], st, batch_size=64)
    want_i, want_p = model.predict_topk(ids, k=10, batch_size=64)
    got_i, got_p = model.predict_topk_from_state(st, k=10, batch_size=64)
    assert np.array_equal(got_i, want_i) and np.array_equal(got_p, want_p)
    # one batch of 150 rows: the whole-window and the state scorers both run the tensor-core logits pass (N >= 128)
    r = model.predict_target_rank_from_state(st, tgt[:, -1], batch_size=n)
    assert np.array_equal(r, model.model.predict_target_rank(ids, tgt, batch_size=n)[:, -1])
    p = model.predict_target_prob_from_state(st, tgt[:, -1], batch_size=n)
    assert np.allclose(p, model.predict_target_prob(ids, tgt, batch_size=n)[:, -1], rtol=1e-6, atol=0)
    # a serving pool: only the sessions with new events advance
    pool = model.initial_state(n)
    pool = model.advance_state(ids[:, :6], pool)
    idx = np.arange(0, n, 3)
    sub = model.advance_state(ids[idx, 6:], pool.take(idx))
    pool.put(idx, sub)
    path = str(tmp_path / "pool.npz")
    pool.save(path)
    back = RecurrentState.load(path, device=dev)
    assert torch.equal(back.h, pool.h) and (cell != "LSTM" or torch.equal(back.c, pool.c))
    # (other batch compositions than st's 64-row batches: equal to fp32 rounding, not necessarily bitwise)
    assert torch.allclose(back.h[idx], st.h[idx], rtol=1e-5, atol=1e-6)
    rest = np.setdiff1d(np.arange(n), idx)
    assert torch.allclose(back.h[rest], model.advance_state(ids[rest, :6], batch_size=64).h, rtol=1e-5, atol=1e-6)
    # continuation through the windowed scorers
    ci, cp = model.predict_topk(ids[:, 6:], k=10, batch_size=64,
                                initial_state=model.advance_state(ids[:, :6], batch_size=64))
    assert np.array_equal(ci, want_i) and np.array_equal(cp, want_p)
    with pytest.raises(ValueError):
        model.predict_topk_from_state(_ytoz("GRU" if cell == "LSTM" else "LSTM", V, 64).initial_state(n))
    with pytest.raises(ValueError):
        model.advance_state(ids[:10], st)


def test_baseline_dense_input_chunks(dev):
    rng = np.random.default_rng(9)
    n, T, F, V = 140, 8, 6, 40
    x = rng.standard_normal((n, T, F)).astype(np.float32)
    x[:, :2][rng.random((n, 2)) < 0.5] = 0.0                   # masked (all-zero) steps
    model = M.RNNBaseline(timesteps=T, features=F, n_classes=V, rnn_type="LSTM", z_dim=16, seed=3)
    st = model.advance_state(x[:, 5:], model.advance_state(x[:, :5]))
    want_i, want_p = model.predict_topk(x, k=5)
    got_i, got_p = model.predict_topk_from_state(st, k=5)
    assert np.array_equal(got_i, want_i) and np.array_equal(got_p, want_p)


def test_dense_path_models_refuse_state(dev):
    with pytest.raises(NotImplementedError):
        M.RNNFullModel(timesteps=5, x_dim=4, y_dim=4).initial_state(3)
    with pytest.raises(NotImplementedError):
        M.NoRecurrenceModel(5, 4, 4).advance_state(np.zeros((3, 5), dtype=np.int32))


# ------------------------------------------------------------------------------------------------ 7. two GPUs
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_two_gpu_states_equal_single_gpu():
    sock = socket.socket()
    sock.bind(("127.0.0.1", 0))
    port = sock.getsockname()[1]
    sock.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "state_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    sys.stdout.write(r.stdout[-4000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "MISMATCH" not in r.stdout and "OK" in r.stdout
