"""Rank of the true next item on the device (target_rank_batch, predict_target_rank, evaluate_ranking, RankingMetrics)
against the float64 oracle of oracle/ranking.py.  Run with -m gpu on a B200.

Exact paths (SIMT kernel, materialised logits) must give the oracle's ranks exactly.  The tensor-core pass compares
x3 / bf16 logits with the exact fp32 target logit, so its rank is exact only outside a band around z_y:
delta_n = c * sum_k |h_nk| * max|W_out| with c = 1e-4 (x3) / 1e-2 (bf16), and the kernel must satisfy
rank_lo <= rank <= rank_hi, rank == rank_lo where rank_lo == rank_hi (oracle.ranking.rank_band)."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import ranking as orank
from seq_recommendations_b200 import synthetic
from seq_recommendations_b200 import model as M
from seq_recommendations_b200.callbacks import EarlyStopping
from seq_recommendations_b200.engine import HotPath
from seq_recommendations_b200.engine_dense import DensePath
from seq_recommendations_b200.optimizers import Adagrad
from seq_recommendations_b200.ranking import ranking_metrics

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAND_C = {"x3": 1e-4, "bf16": 1e-2}


def band(hot, ids, tgt, c, chunk=1024):
    """(rank_lo, rank_hi) (B,T) from float64 logits of the model's own hidden states, on the GPU in token chunks."""
    h = hot.hidden_batch(ids).double()                                  # (B,T,H)
    W = hot.W_out.double()
    b = hot.b_out.double() if hot.b_out is not None else None
    wmax = float(W.abs().max())
    B, T, H = h.shape
    hf = h.reshape(-1, H)
    y = torch.as_tensor(np.asarray(tgt), dtype=torch.int64, device=h.device).reshape(-1)
    lo = torch.zeros_like(y)
    hi = torch.zeros_like(y)
    for n0 in range(0, hf.shape[0], chunk):
        z = hf[n0:n0 + chunk] @ W
        if b is not None:
            z = z + b
        yy = y[n0:n0 + chunk]
        zy = z.gather(1, yy.clamp(min=0)[:, None])
        d = c * hf[n0:n0 + chunk].abs().sum(1, keepdim=True) * wmax
        other = torch.arange(z.shape[1], device=z.device)[None, :] != yy[:, None]
        l = 1 + ((z > zy + d) & other).sum(1)
        u = 1 + ((z >= zy - d) & other).sum(1)
        lo[n0:n0 + chunk] = torch.where(yy >= 0, l, 0)
        hi[n0:n0 + chunk] = torch.where(yy >= 0, u, 0)
    return lo.view(B, T).cpu().numpy(), hi.view(B, T).cpu().numpy()


def check_band(rank, lo, hi, label):
    rank = np.asarray(rank)
    assert rank.dtype == np.int32
    assert np.all(lo <= rank) and np.all(rank <= hi), (label, int(np.sum((rank < lo) | (rank > hi))))
    sharp = (lo == hi)
    assert np.array_equal(rank[sharp], lo[sharp]), label
    valid = lo > 0
    print("%s: %.4f of %d tokens have an empty band" % (label, sharp[valid].mean(), int(valid.sum())))
    return sharp & valid


def check_simt_rank(hot, ids, tgt, rank, label):
    """The SIMT kernel ranks its own fp32 logits exactly.  Against float64 logits of the same hidden states that is:
    exact ties (duplicated W_out columns) decided by the tie rule, the rank exact wherever no other logit lies within the
    fp32 rounding of the H-term dot products (delta = 1e-5 * sum|h| * max|W_out| > H * 2^-24 * sum|h_k w_k| at H = 100),
    and within that band otherwise.  Returns (pinned, tied): the tokens whose rank the band pins exactly, and the
    tokens whose target logit some other item equals exactly."""
    h = hot.hidden_batch(ids).double().cpu().numpy()
    W = hot.W_out.double().cpu().numpy()
    z = h @ W
    if hot.b_out is not None:
        z = z + hot.b_out.double().cpu().numpy()
    d = 1e-5 * np.abs(h).sum(-1) * np.abs(W).max()
    lo, hi = orank.rank_band(z, tgt, d, exact_ties=True)
    pinned = check_band(rank, lo, hi, label)
    zy = np.take_along_axis(z, np.where(tgt >= 0, tgt, 0)[..., None], axis=-1)
    tied = (tgt >= 0) & ((z == zy).sum(-1) > 1)
    return pinned, tied


# ---------------------------------------------------------------------------------------------------- SIMT kernel
@pytest.mark.parametrize("dup", [False, True])
def test_simt_rank_is_exact_at_cfg1(dup):
    V, H, T, B = 17, 100, 20, 96
    ws = synthetic.make_weights("LSTM", V, H, seed=3)
    ids, tgt = synthetic.make_batch(V, T, B, seed=4, min_len=1)
    if dup:
        # duplicated W_out columns: exact ties in fp32 and float64, decided by the lower item id
        for a, b in ((2, 5), (2, 11), (7, 16)):
            ws[3][:, b] = ws[3][:, a]
        rng = np.random.default_rng(5)
        pick = (tgt >= 0) & (rng.random(tgt.shape) < 0.5)
        tgt = np.where(pick, rng.choice([2, 5, 11, 7, 16], size=tgt.shape), tgt).astype(tgt.dtype)
    hot = HotPath("LSTM", "relu", V, H, V, weights=ws, tc="off")
    rank = hot.target_rank_batch(ids, tgt).cpu().numpy()
    assert not hot.work(B, T).tc["fwd"]
    pinned, tied = check_simt_rank(hot, ids, tgt, rank, "SIMT cfg1 dup=%s" % dup)
    assert pinned.sum() >= 0.8 * int((tgt >= 0).sum())
    if dup:
        # exact ties between duplicated columns, decided by the lower item id, on tokens the band pins exactly
        assert (pinned & tied).sum() >= 100, int((pinned & tied).sum())
    last = hot.target_rank_batch(ids, tgt, last_step_only=True).cpu().numpy()
    assert np.array_equal(last, rank[:, -1])


# ---------------------------------------------------------------------------------------------- materialised logits
def _dense_inputs(V, T, B, seed):
    ids, tgt = synthetic.make_batch(V, T, B, seed=seed, min_len=1)
    x = np.zeros((B, T, V), dtype=np.float32)
    for b in range(B):
        cnt = np.zeros(V)
        for t in range(T):
            if ids[b, t] >= 0:
                cnt[ids[b, t]] += 1
                x[b, t] = np.log(cnt + 1)
    return ids, tgt, x


@pytest.mark.parametrize("cell", ["LSTM", None])
def test_materialised_rank_is_exact(cell):
    """DensePath: the x_to_y + y_to_y variant of RNNFullModel and NoRecurrenceModel (ytoy_xtoy), ranks from the path's
    own materialised logits; a duplicated column of every logit term gives exact ties."""
    V, H, T, B = 17, 12, 9, 40
    rng = np.random.default_rng(8)
    r = lambda *s: (rng.standard_normal(s) * 0.3).astype(np.float32)
    ws = dict(W_toy=r((H if cell else 0) + V, V), b_out=r(V), A=r(V, V), a_bias=r(V))
    if cell:
        ws.update(W_in=r(V, 4 * H), U=r(H, 4 * H), b=r(4 * H))
    for k in ("W_toy", "A"):
        ws[k][:, 9] = ws[k][:, 4]
    ws["b_out"][9] = ws["b_out"][4]
    ws["a_bias"][9] = ws["a_bias"][4]
    ws["W_toy"][(H if cell else 0) + 9, :] = 0.0                  # the x feature of item 9 no longer breaks the tie
    ws["W_toy"][(H if cell else 0) + 4, :] = 0.0
    ids, tgt, x = _dense_inputs(V, T, B, seed=9)
    tgt = np.where((tgt >= 0) & (rng.random(tgt.shape) < 0.3), 9, tgt).astype(tgt.dtype)
    hot = DensePath(cell, "relu", V, V, H, ws, y_to_z=cell is not None, x_to_z=False, x_to_y=True, y_to_y=True,
                    diag_b=False)
    rank = hot.target_rank_batch(ids, tgt, x).cpu().numpy()
    w = hot.work(B, T)
    Z = w.Z.double().cpu().numpy().reshape(T, B, V).transpose(1, 0, 2)
    y = w.tgt.cpu().numpy().T
    ref = orank.target_rank(Z, y)
    assert np.array_equal(rank, ref)
    assert np.any(ref[y == 9] > 0)
    assert np.array_equal(hot.target_rank_batch(ids, tgt, x, last_step_only=True).cpu().numpy(), rank[:, -1])


def test_panel_path_rank_is_exact():
    """H = 512: the tensor-core GEMM over token panels (hidden sizes above 256), ranks from the same materialised logits."""
    V, H, T, B = 700, 512, 5, 40
    ws = synthetic.make_weights("GRU", V, H, seed=11)
    ids, tgt = synthetic.make_batch(V, T, B, seed=12, min_len=1)
    hot = HotPath("GRU", "tanh", V, H, V, weights=ws, tc="x3")
    rank = hot.target_rank_batch(ids, tgt).cpu().numpy()
    w = hot.work(B, T)
    assert w.tc["panel"]
    Z, _, _ = hot._wide_logits(w.hout.view(w.N, H))
    Z = Z.double().cpu().numpy().reshape(T, B, V).transpose(1, 0, 2)
    assert np.array_equal(rank, orank.target_rank(Z, w.tgt.cpu().numpy().T))


# ------------------------------------------------------------------------------------------------ tensor-core pass
@pytest.mark.parametrize("mode", ["x3", "bf16"])
@pytest.mark.parametrize("V,bias", [(10000, False), (10007, False), (10000, True)])
def test_tc_rank_within_band(mode, V, bias):
    """cfg2 shape (GRU-128, V = 10k), a ragged catalog, and an output bias (RNNBaseline's layer)."""
    H, T, B = 128, 20, 64
    ws = synthetic.make_weights("GRU", V, H, seed=13, out_bias=bias)
    if bias:
        ws[4] = (np.random.default_rng(14).standard_normal(V) * 0.5).astype(np.float32)
    ids, tgt = synthetic.make_batch(V, T, B, seed=15, min_len=1)
    hot = HotPath("GRU", "tanh", V, H, V, out_bias=bias, weights=ws, tc=mode)
    rank = hot.target_rank_batch(ids, tgt).cpu().numpy()
    assert hot.work(B, T).tc["fwd"]
    lo, hi = band(hot, ids, tgt, BAND_C[mode])
    check_band(rank, lo, hi, "%s V=%d bias=%s" % (mode, V, bias))
    assert np.array_equal(rank == 0, tgt < 0)


def test_tc_rank_at_cfg5_widths():
    """GRU-256, V = 100k, T = 200 (cfg5) with the batch cut 128-fold (B = 32), all steps and the last step."""
    V, H, T, B = 100000, 256, 200, 32
    ws = synthetic.make_weights("GRU", V, H, seed=16)
    ids, tgt = synthetic.make_batch(V, T, B, seed=17, min_len=1)
    hot = HotPath("GRU", "tanh", V, H, V, weights=ws, tc="x3")
    rank = hot.target_rank_batch(ids, tgt).cpu().numpy()
    lo, hi = band(hot, ids, tgt, BAND_C["x3"])
    check_band(rank, lo, hi, "cfg5 widths")
    last = hot.target_rank_batch(ids, tgt, last_step_only=True).cpu().numpy()
    check_band(last[:, None], lo[:, -1:], hi[:, -1:], "cfg5 widths, last step")


def test_tc_rank_agrees_with_topk():
    V, H, T, B = 10000, 128, 20, 64
    ws = synthetic.make_weights("GRU", V, H, seed=18)
    ids, tgt = synthetic.make_batch(V, T, B, seed=19, min_len=1)
    hot = HotPath("GRU", "tanh", V, H, V, weights=ws, tc="x3")
    top, _ = hot.topk_batch(ids, 20, last_step_only=False)
    top = top.cpu().numpy()
    # half of the targets are items of the model's own top 25 (the top of a logit row is well separated, so most of
    # these ranks are pinned exactly by the band); the other half stay random (ranks far beyond 20)
    rng = np.random.default_rng(20)
    top25, _ = hot.topk_batch(ids, 25, last_step_only=False)
    pick = (tgt >= 0) & (rng.random(tgt.shape) < 0.5)
    mine = np.take_along_axis(top25.cpu().numpy(), rng.integers(0, 25, size=tgt.shape + (1,)), axis=-1)[..., 0]
    tgt = np.where(pick, mine, tgt).astype(tgt.dtype)
    rank = hot.target_rank_batch(ids, tgt).cpu().numpy()
    lo, hi = band(hot, ids, tgt, BAND_C["x3"])
    sharp = check_band(rank, lo, hi, "top-k agreement")
    n_hit = 0
    for b, t in zip(*np.nonzero(sharp)):
        r, y = rank[b, t], tgt[b, t]
        if r <= 20:
            assert top[b, t, r - 1] == y, (b, t, r)
            n_hit += 1
        else:
            assert y not in top[b, t], (b, t, r)
    print("top-k agreement: %d pinned ranks <= 20" % n_hit)
    assert n_hit >= 100


def test_tc_rank_pass_leaves_target_prob_and_is_deterministic():
    V, H, T, B = 10007, 128, 20, 64
    ws = synthetic.make_weights("GRU", V, H, seed=20)
    ids, tgt = synthetic.make_batch(V, T, B, seed=21, min_len=1)
    hot = HotPath("GRU", "tanh", V, H, V, weights=ws, tc="x3")
    r1 = hot.target_rank_batch(ids, tgt)
    w = hot.work(B, T)
    py_rank = w.py.view(T, B).t().clone()
    r2 = hot.target_rank_batch(ids, tgt)
    py = hot.target_prob_batch(ids, tgt)
    assert torch.equal(r1, r2)
    assert torch.equal(py_rank, py)


def test_tc_rank_with_extreme_logits():
    V, H, T, B = 1500, 128, 9, 40
    ws = synthetic.make_weights("GRU", V, H, seed=22)
    ws[3] = ws[3] * 4000.0
    ids, tgt = synthetic.make_batch(V, T, B, seed=23, min_len=1)
    hot = HotPath("GRU", "tanh", V, H, V, weights=ws, tc="x3")
    rank = hot.target_rank_batch(ids, tgt).cpu().numpy()
    valid = tgt >= 0
    assert np.all((rank[valid] >= 1) & (rank[valid] <= V)) and np.all(rank[~valid] == 0)
    lo, hi = band(hot, ids, tgt, BAND_C["x3"])
    check_band(rank, lo, hi, "W_out x 4000")


# ------------------------------------------------------------------------------------------------------- model API
def test_evaluate_ranking_and_callback():
    V, H, T, B = 3000, 64, 12, 96
    ids, tgt = synthetic.make_batch(V, T, B, seed=24, min_len=1)
    mdl = M.RNNFullModel(T, V, V, z_dim=H, rnn_type="GRU", z_to_z_activation="tanh", y_to_y=False, x_to_y=False, seed=5)
    mdl.compile_model(optimizer=Adagrad(lr=0.05, epsilon=1e-8, clipnorm=1.0))
    ks = (1, 5, 10, 20)
    for last in (False, True):
        rank = mdl.model._target_ranks(ids, tgt, 40, last).cpu().numpy()
        got = mdl.evaluate_ranking(ids, tgt, ks=ks, last_step_only=last, batch_size=40)
        want = orank.ranking_metrics(rank, ks)
        assert got.keys() == want.keys()
        for k in want:
            assert abs(got[k] - want[k]) <= 1e-12, (k, got[k], want[k])
        again = ranking_metrics(torch.from_numpy(rank).cuda(), ks)
        assert all(abs(again[k] - got[k]) <= 1e-12 for k in got)
    rank = mdl.predict_target_rank(ids, tgt, batch_size=40)
    assert np.array_equal(rank[:, -1], mdl.model._target_ranks(ids, tgt, 40, True).cpu().numpy())
    lo, hi = band(mdl.model.hot, ids, tgt, BAND_C["x3"])
    sharp = check_band(rank, lo, hi, "model surface")
    assert orank.ranking_metrics(rank[sharp], ks) == orank.ranking_metrics(lo[sharp], ks)
    with pytest.raises(ValueError):
        mdl.evaluate_ranking(ids, tgt, ks=(0,))
    # the callback feeds EarlyStopping: min_delta = 1 can never be met, so patience 0 stops after the second epoch
    cbk = M.RankingMetrics((ids[:48], tgt[:48]), ks=(20,))
    stop = EarlyStopping(monitor="val_mrr@20", mode="max", patience=0, min_delta=1.0)
    hist = mdl.model.fit(ids[48:], tgt[48:], epochs=5, batch_size=24, verbose=0, callbacks=[cbk, stop])
    assert len(hist.history["val_mrr@20"]) == 2 and stop.stopped_epoch == 1
    for key in ("val_recall@20", "val_mrr@20", "val_ndcg@20"):
        assert key in hist.history and 0.0 <= hist.history[key][-1] <= 1.0
    assert hist.history["val_mrr@20"][-1] == cbk.history[-1]["mrr@20"]


def test_model_classes_rank():
    """RNNBaseline (output bias, SIMT at this size), NoRecurrenceModel and a branch RNNFullModel through the surface."""
    V, T, B = 17, 9, 30
    ids, tgt, x = _dense_inputs(V, T, B, seed=25)
    onehot = np.zeros((B, T, V), dtype=np.float32)
    bb, tt = np.nonzero(ids >= 0)
    onehot[bb, tt, ids[bb, tt]] = 1.0
    base = M.RNNBaseline(timesteps=T, features=V, n_classes=V, rnn_type="LSTM", z_dim=8, seed=7)
    assert base.model.hot.out_bias
    r = base.predict_target_rank(onehot, tgt)
    check_simt_rank(base.model.hot, ids, tgt, r, "RNNBaseline")
    for mdl, xin in ((M.NoRecurrenceModel(T, V, V), [ids, x]),
                     (M.RNNFullModel(timesteps=T, x_dim=V, y_dim=V, z_dim=6, rnn_type="GRU"), [ids, x])):
        r = mdl.predict_target_rank(xin, tgt)
        w = mdl.model.hot.work(B, T)
        Z = w.Z.double().cpu().numpy().reshape(T, B, V).transpose(1, 0, 2)
        assert np.array_equal(r, orank.target_rank(Z, w.tgt.cpu().numpy().T))
        m = mdl.evaluate_ranking(xin, tgt, ks=(1, 5))
        assert m["n"] == int((r > 0).sum())


# --------------------------------------------------------------------------------------------------------- two GPUs
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_two_gpu_ranks_equal_single_gpu():
    sock = socket.socket()
    sock.bind(("127.0.0.1", 0))
    port = sock.getsockname()[1]
    sock.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "rank_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    sys.stdout.write(r.stdout[-4000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "MISMATCH" not in r.stdout and "OK" in r.stdout
