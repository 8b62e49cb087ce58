"""Candidate scoring on the device (csrc/candidates.cu, HotPath / DensePath candidates_batch and candidate_rank_batch,
the *_from_state scorers, the model surface) against the float64 oracle of oracle/candidates.py.  Run with -m gpu.

The candidate logits are exact fp32 dot products with the arithmetic of seqrec_target_logit: against float64 they lie
within delta = (H/32 + 6) * 2^-23 * sum|h| * max|W_out| (+ the bias rounding), and the logit of a candidate equal to the
target is seqrec_target_logit's zy bit for bit.  The order and the rank are exact functions of those fp32 logits."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import candidates as oc
from oracle import ranking as orank
from seq_recommendations_b200 import model as M
from seq_recommendations_b200 import synthetic
from seq_recommendations_b200._lib import call, ptr
from seq_recommendations_b200.engine import HotPath
from seq_recommendations_b200.engine_dense import DensePath
from seq_recommendations_b200.ranking import MAX_CANDIDATES, metrics_from_sums, rank_sums

from test_gpu_skip_models import VARIANTS, make_inputs
from test_gpu_skip_models import make_weights as skip_weights
from test_gpu_vocab_parallel_one_device import CASES, _rows, _solo, _untied_id_diffs, run_ranks

pytestmark = pytest.mark.gpu
U = 2.0 ** -23


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _delta(h, W, b=None):
    """fp32 band of the candidate logits of the rows h (n, H) (float64 tensors)."""
    H = h.shape[-1]
    d = (H / 32 + 6) * U * h.abs().sum(-1) * W.abs().max()
    if b is not None:
        d = d + U * b.abs().max()
    return d


def _make_lists(rng, lead, C, V, pad=0.1, extra=None):
    c = rng.integers(0, V, size=lead + (C,))
    if extra is not None:                               # the target at a random position of about half the lists
        put = rng.random(lead) < 0.5
        pos = rng.integers(0, C, size=lead)
        np.put_along_axis(c, pos[..., None], np.where(put, extra, np.take_along_axis(c, pos[..., None], -1)[..., 0])
                          [..., None], -1)
    c[rng.random(c.shape) < pad] = -1
    return c.astype(np.int32)


# ---------------------------------------------------------------------------------------------------- 1. logits kernel
@pytest.mark.parametrize("H", [32, 100, 128, 256, 500, 1000])
def test_candidate_logits_kernel(H):
    rng = np.random.default_rng(H)
    dev = torch.device("cuda")
    n, V, C, lo, vl = 37, 300, 50, 100, 150
    h = torch.tensor(rng.standard_normal((n, H)), dtype=torch.float32, device=dev)
    W = torch.tensor(rng.standard_normal((H, V)) * 0.2, dtype=torch.float32, device=dev)
    b = torch.tensor(rng.standard_normal(V), dtype=torch.float32, device=dev)
    cand = torch.tensor(_make_lists(rng, (n,), C, V), device=dev)
    st = _stream()
    # the whole catalog, then a shard [lo, lo + vl) with its slice of W_out
    Wt = W.t().contiguous()
    z = torch.empty((n, C), dtype=torch.float32, device=dev)
    call("seqrec_candidate_logits", ptr(h), ptr(Wt), ptr(b), ptr(cand), C, ptr(z), n, C, H, 0, V, st)
    Wts = W[:, lo:lo + vl].t().contiguous()
    zs = torch.empty_like(z)
    call("seqrec_candidate_logits", ptr(h), ptr(Wts), ptr(b[lo:lo + vl]), ptr(cand), C, ptr(zs), n, C, H,
         lo, vl, st)
    want = torch.tensor(oc.candidate_logits(h.double().cpu().numpy(), W.double().cpu().numpy(),
                                            b.double().cpu().numpy(), cand.cpu().numpy()), device=dev)
    d = _delta(h.double(), W.double(), b.double())[:, None]
    valid = cand >= 0
    assert bool(((z.double() - want).abs() <= d)[valid].all()), float(((z.double() - want).abs() - d).max())
    assert bool((z[~valid] == 0).all())
    mine = valid & (cand >= lo) & (cand < lo + vl)
    assert torch.equal(zs[mine], z[mine])                   # a shard computes its items' logits with the same bits
    assert bool((zs[~mine] == 0).all()) and int((zs[~mine].view(torch.int32) != 0).sum()) == 0
    # the logit of c == y is seqrec_target_logit's zy bit for bit
    for j in (0, 17, C - 1):
        y = cand[:, j].contiguous()
        zy = torch.zeros(n, dtype=torch.float32, device=dev)
        call("seqrec_target_logit", ptr(h), None, ptr(W), ptr(b), ptr(y), ptr(zy), n, H, V, None, None, st)
        ok = y >= 0
        assert torch.equal(zy[ok].view(torch.int32), z[ok, j].view(torch.int32)), j


# ----------------------------------------------------------------------------------------------------- 2. order kernel
@pytest.mark.parametrize("C", [1, 7, 100, 1024])
def test_candidate_order_kernel_is_exact(C):
    rng = np.random.default_rng(C)
    dev = torch.device("cuda")
    n = 61
    z = (rng.integers(-8, 9, size=(n, C)) / 4.0).astype(np.float32)          # a coarse grid: many exact ties
    cand = rng.integers(0, max(4, C // 3), size=(n, C)).astype(np.int32)     # many duplicates
    cand[rng.random((n, C)) < 0.15] = -1
    z[cand < 0] = 0.0
    y = rng.integers(-1, max(4, C // 3) + 2, size=n).astype(np.int32)
    zy = (rng.integers(-8, 9, size=n) / 4.0).astype(np.float32)
    m = rng.standard_normal(n).astype(np.float32)
    s = (rng.random(n) * 3 + 0.5).astype(np.float32)
    tz, tc, ty, tzy, tm, ts = (torch.tensor(a, device=dev) for a in (z, cand, y, zy, m, s))
    st = _stream()
    rank = torch.full((n,), -7, dtype=torch.int32, device=dev)
    call("seqrec_candidate_order", ptr(tz), ptr(tc), C, n, None, None, 0, None, None, ptr(tzy), ptr(ty), ptr(rank), st)
    assert np.array_equal(rank.cpu().numpy(), oc.candidate_rank(z, cand, zy, y))
    for k in sorted({1, (C + 1) // 2, C}):
        oi = torch.empty((n, k), dtype=torch.int32, device=dev)
        os_ = torch.empty((n, k), dtype=torch.float32, device=dev)
        call("seqrec_candidate_order", ptr(tz), ptr(tc), C, n, None, None, k, ptr(oi), ptr(os_), None, None, None, st)
        wi, ws = oc.candidate_order(z, cand, k)
        assert np.array_equal(oi.cpu().numpy(), wi) and np.array_equal(os_.cpu().numpy(), ws.astype(np.float32)), k
        call("seqrec_candidate_order", ptr(tz), ptr(tc), C, n, ptr(tm), ptr(ts), k, ptr(oi), ptr(os_), None, None,
             None, st)
        assert np.array_equal(oi.cpu().numpy(), wi), k
        zo = torch.tensor(np.where(wi >= 0, ws, 0.0).astype(np.float32), device=dev)
        p = torch.where(torch.tensor(wi >= 0, device=dev), torch.exp(zo - tm[:, None]) / ts[:, None], 0.0)
        assert torch.allclose(os_, p, rtol=3e-7, atol=0), float(((os_ - p).abs() / p.abs().clamp_min(1e-30)).max())


# ---------------------------------------------------------------------------------------------------- engine helpers
def _oracle_rows(hot, rows):
    """float64 logits of the model's own hidden rows (n, H) and their band."""
    h = rows.double()
    W = hot.W_out.double()
    b = hot.b_out.double() if hot.b_out is not None else None
    z = h @ W + (b if b is not None else 0.0)
    return z, _delta(h, W, b)


def _check_logit_order(hot, rows, cand, ids, scores):
    """(ids, scores) of a logits call: every valid entry's score within the band of its float64 logit, the scores
    non-increasing, ties by id, and the multiset of the list's valid ids."""
    z, d = _oracle_rows(hot, rows)
    ok = ids >= 0
    zi = z.gather(1, ids.clamp(min=0).long())
    assert bool(((scores.double() - zi).abs() <= d[:, None])[ok].all())
    sv = torch.where(ok, scores, torch.full_like(scores, -float("inf")))
    assert bool((sv[:, 1:] <= sv[:, :-1]).all())
    tie = (sv[:, 1:] == sv[:, :-1]) & ok[:, 1:]
    assert bool((ids[:, 1:] >= ids[:, :-1])[tie].all())
    assert torch.equal(ids.sort(1).values, torch.where(cand >= 0, cand, -1).int().sort(1).values)


# (cell, act, H, tc, V): register scan + x3 logits, tensor-core scan + bf16, tensor-core scan + SIMT logits, panel path
FAMILIES = [("GRU", "tanh", 128, "x3", 2000), ("LSTM", "tanh", 128, "bf16", 2000), ("GRU", "tanh", 256, "off", 2000),
            ("GRU", "tanh", 500, "x3", 2000)]


@pytest.mark.parametrize("cell,act,H,tc,V", FAMILIES, ids=lambda v: str(v))
def test_engine_candidates_every_family(cell, act, H, tc, V):
    B, T, C = 150, 8, 40
    rng = np.random.default_rng(H)
    ws = synthetic.make_weights(cell, V, H, seed=3, out_bias=True)
    ws[4] = (rng.standard_normal(V) * 0.1).astype(np.float32)
    hot = HotPath(cell, act, V, H, V, out_bias=True, weights=ws, tc=tc)
    ids, tgt = synthetic.make_batch(V, T, B, seed=4, min_len=1)
    dev = hot.device
    hs = hot.hidden_batch(ids)                                             # (B, T, H)
    last = _make_lists(rng, (B,), C, V, extra=tgt[:, -1])
    every = _make_lists(rng, (B, T), C, V, extra=tgt)
    # logits and order, last step and every step
    li, ls = hot.candidates_batch(ids, last)
    _check_logit_order(hot, hs[:, -1], torch.tensor(last, device=dev), li, ls)
    ei, es = hot.candidates_batch(ids, every, k=C, last_step_only=False)
    assert ei.shape == (B, T, C)
    _check_logit_order(hot, hs.reshape(B * T, H), torch.tensor(every.reshape(B * T, C), device=dev),
                       ei.reshape(B * T, C), es.reshape(B * T, C))
    # ranks inside the oracle band, every step
    r = hot.candidate_rank_batch(ids, tgt, every).cpu().numpy()
    z, d = _oracle_rows(hot, hs.reshape(B * T, H))
    zc = torch.where(torch.tensor(every.reshape(B * T, C), device=dev) >= 0,
                     z.gather(1, torch.tensor(every.reshape(B * T, C), device=dev).clamp(min=0).long()), 0.0)
    yy = torch.tensor(tgt.reshape(-1), device=dev)
    zy = z.gather(1, yy.clamp(min=0).long()[:, None])[:, 0]
    lo, hi = oc.candidate_rank_band(zc.cpu().numpy(), every.reshape(B * T, C), zy.cpu().numpy(), tgt.reshape(-1),
                                    2 * d.cpu().numpy(), exact_ties=True)
    r = r.reshape(-1)
    assert np.all(lo <= r) and np.all(r <= hi), int(np.sum((r < lo) | (r > hi)))
    assert np.array_equal(r[lo == hi], lo[lo == hi])
    # p(target) from a one-entry list [y]: clip(p) against target_prob_batch / target_prob_from_state
    pi, pp = hot.candidates_batch(ids, tgt[..., None], probs=True, last_step_only=False)
    clip = lambda p: p.clamp(1.0000000116860974e-07, 0.99999988079071045)
    valid = torch.tensor(tgt >= 0, device=dev)
    want = hot.target_prob_batch(ids, tgt)
    st = hot.advance_state(ids)
    si, sp = hot.candidates_from_state(st, tgt[:, -1:], probs=True)
    want_st = hot.target_prob_from_state(st, tgt[:, -1])
    fused = hot.work(B, T).tc["fwd"] and hot.work(B, 1).tc["fwd"]
    if fused:
        assert torch.equal(clip(pp[..., 0])[valid], want[valid])
        assert torch.equal(clip(sp[:, 0]), want_st)
    else:
        assert torch.allclose(clip(pp[..., 0])[valid], want[valid], rtol=1e-6, atol=0)
        assert torch.allclose(clip(sp[:, 0]), want_st, rtol=1e-6, atol=0)
    assert fused == (tc != "off" and H <= 256)


def test_dense_input_baseline_candidates():
    rng = np.random.default_rng(9)
    n, T, F, V, C = 140, 8, 6, 40, 12
    x = rng.standard_normal((n, T, F)).astype(np.float32)
    x[:, :2][rng.random((n, 2)) < 0.5] = 0.0
    model = M.RNNBaseline(timesteps=T, features=F, n_classes=V, rnn_type="LSTM", z_dim=16, seed=3)
    hot = model.model.hot
    cand = _make_lists(rng, (n,), C, V)
    ids, sc = model.predict_candidates(x, cand)
    rows = torch.tensor(model.model.hidden_states(x)[:, -1], device=hot.device)
    _check_logit_order(hot, rows, torch.tensor(cand, device=hot.device), torch.tensor(ids, device=hot.device),
                       torch.tensor(sc, device=hot.device))
    st = model.advance_state(x)
    si, ss = model.predict_candidates_from_state(st, cand, probs=True)
    pi, ps = model.predict_candidates(x, cand, probs=True)
    assert np.array_equal(si, ids) and np.array_equal(pi, ids) and np.array_equal(ss, ps)
    y = rng.integers(0, V, size=n)
    r = model.predict_candidate_rank_from_state(st, y, cand)
    assert r.shape == (n,) and np.all((r >= 1) & (r <= C + 1))


# ------------------------------------------------------------------------------------------- 3. exact ties by the rule
@pytest.mark.parametrize("tc", ["x3", "off"])
def test_duplicated_columns_tie_exactly(tc):
    V, H, B, T = 998, 64, 130, 5
    ws = synthetic.make_weights("GRU", V, H, seed=5)
    y = 500
    for c in (10, 900):
        ws[3][:, c] = ws[3][:, y]
    hot = HotPath("GRU", "tanh", V, H, V, weights=ws, tc=tc)
    ids, _ = synthetic.make_batch(V, T, B, seed=6, min_len=1)
    st = hot.advance_state(ids)
    rng = np.random.default_rng(7)
    cand = rng.integers(0, V, size=(B, 30)).astype(np.int32)
    cand[np.isin(cand, [10, y, 900])] = 0
    cand[:, [3, 11, 20]] = [900, y, 10]
    ci, cz = hot.candidates_from_state(st, cand)
    rank = hot.candidate_rank_from_state(st, np.full(B, y), cand).cpu().numpy()
    ci, cz = ci.cpu().numpy(), cz.cpu().numpy()
    for b in range(B):
        pos = [int(np.flatnonzero(ci[b] == c)[0]) for c in (10, y, 900)]
        assert pos == list(range(pos[0], pos[0] + 3)), (b, pos)             # 10, 500, 900 adjacent, in id order
        assert cz[b, pos[0]] == cz[b, pos[1]] == cz[b, pos[2]]
    # the rank from the list's own fp32 logits, with the tie rule
    z = np.zeros((B, 30), dtype=np.float64)
    for b in range(B):
        for j in range(30):
            z[b, j] = cz[b, int(np.flatnonzero(ci[b] == cand[b, j])[0])]
    zy = z[:, 11]
    assert np.array_equal(rank, oc.candidate_rank(z, cand, zy, np.full(B, y)))


# ------------------------------------------------------------------------------ 5. the whole catalog as the candidate list
def test_full_catalog_list_is_the_catalog_rank():
    V, H, T, B = 998, 64, 6, 40
    ws = synthetic.make_weights("GRU", V, H, seed=8)
    hot = HotPath("GRU", "tanh", V, H, V, weights=ws, tc="x3")
    ids, tgt = synthetic.make_batch(V, T, B, seed=9, min_len=1)
    full = np.broadcast_to(np.arange(V, dtype=np.int32), (B, T, V))
    r = hot.candidate_rank_batch(ids, tgt, full).cpu().numpy().reshape(-1)
    want = hot.target_rank_batch(ids, tgt).cpu().numpy().reshape(-1)
    hs = hot.hidden_batch(ids).reshape(B * T, H)
    z, _ = _oracle_rows(hot, hs)
    d = (1e-4 * hs.double().abs().sum(1) * hot.W_out.double().abs().max()).cpu().numpy()   # the x3 pass's band
    lo, hi = orank.rank_band(z.cpu().numpy(), tgt.reshape(-1), d, exact_ties=True)
    sharp = lo == hi
    assert sharp.mean() > 0.5
    assert np.array_equal(r[sharp], want[sharp])
    assert np.array_equal(r[sharp], lo[sharp])


@pytest.mark.parametrize("cell,act,y_to_z,x_to_z,x_to_y,y_to_y", VARIANTS)
def test_dense_path_full_catalog_list_equals_target_rank(cell, act, y_to_z, x_to_z, x_to_y, y_to_y):
    V, H, T, B = 17, 12, 9, 14
    rng = np.random.default_rng(5)
    ws = skip_weights(rng, cell, V, V, H, y_to_z, x_to_z, x_to_y, y_to_y)
    ids, tgt, x = make_inputs(V, T, B, seed=6)
    hot = DensePath(cell, act, V, V, H, ws, y_to_z=y_to_z, x_to_z=x_to_z, x_to_y=x_to_y, y_to_y=y_to_y)
    i, xx = (ids if hot.uses_y else None), (x if hot.uses_x else None)
    full = np.broadcast_to(np.arange(V, dtype=np.int32), (B, T, V))
    assert torch.equal(hot.candidate_rank_batch(i, tgt, full, x_dense=xx), hot.target_rank_batch(i, tgt, xx))
    assert torch.equal(hot.candidate_rank_batch(i, tgt, full[:, 0], last_step_only=True, x_dense=xx),
                       hot.target_rank_batch(i, tgt, xx, last_step_only=True))
    # the order of the whole catalog is topk's, and probs are the materialised probabilities
    ci, cp = hot.candidates_batch(i, full[:, 0], k=5, probs=True, x_dense=xx)
    ti, tp = hot.topk_batch(i, 5, last_step_only=True, x_dense=xx)
    assert not _untied_id_diffs(ci, ti, tp, 1e-6).any()
    assert torch.allclose(cp, tp, rtol=1e-6, atol=0)


# --------------------------------------------------------------------------------- 6. state, window and batch sizes
def _ytoz(cell, V, H):
    return M.RNNFullModel(timesteps=12, x_dim=V, y_dim=V, z_dim=H, model_name="ytoz", rnn_type=cell,
                          z_to_z_activation="tanh", y_to_z=True, y_to_y=False, x_to_y=False, x_to_z=False, seed=4)


@pytest.mark.parametrize("cell", ["LSTM", "GRU"])
def test_model_state_equals_window_and_batch_size_does_not_matter(cell):
    V, T, n, C = 3000, 12, 150, 64
    model = _ytoz(cell, V, 64)
    ids, tgt = synthetic.make_batch(V, T, n, seed=8, min_len=1)
    rng = np.random.default_rng(1)
    cand = _make_lists(rng, (n,), C, V, extra=tgt[:, -1])
    st = model.advance_state(ids, batch_size=64)
    for probs in (False, True):
        wi, wp = model.predict_candidates(ids, cand, k=20, probs=probs, batch_size=64)
        gi, gp = model.predict_candidates_from_state(st, cand, k=20, probs=probs, batch_size=64)
        assert np.array_equal(gi, wi) and np.array_equal(gp, wp), probs
    r = model.predict_candidate_rank_from_state(st, tgt[:, -1], cand, batch_size=64)
    assert np.array_equal(r, model.predict_candidate_rank(ids, tgt, cand, last_step_only=True, batch_size=64))
    dev_cand = torch.tensor(cand, device="cuda")
    assert np.array_equal(r, model.predict_candidate_rank_from_state(st, tgt[:, -1], dev_cand, batch_size=64))
    # logits and ranks do not depend on the batch size (the same scan kernel at 7 and 20 rows)
    small = _ytoz(cell, 500, 32)
    ids, tgt = synthetic.make_batch(500, T, 20, seed=9, min_len=1)
    cand = _make_lists(rng, (20, T), 16, 500, extra=tgt)
    a = small.predict_candidates(ids, cand, last_step_only=False, batch_size=7)
    b = small.predict_candidates(ids, cand, last_step_only=False, batch_size=1024)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert np.array_equal(small.predict_candidate_rank(ids, tgt, cand, batch_size=7),
                          small.predict_candidate_rank(ids, tgt, cand, batch_size=1024))


# ------------------------------------------------------------------------------- 7. vocabulary and data parallel
@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s%d-V%d-%s" % (c[4], c[1], c[0], c[5]))
def test_vocab_parallel_candidates_equal_single_gpu(case):
    V, H, T, B, cell, tc = case
    act = "tanh" if cell == "GRU" else "relu"
    ws = synthetic.make_weights(cell, V, H, seed=3)
    ids, tgt = synthetic.make_batch(V, T, B, seed=4, min_len=1)
    rng = np.random.default_rng(2)
    last = _make_lists(rng, (B,), 33, V, extra=tgt[:, -1])
    every = _make_lists(rng, (B, T), 9, V, extra=tgt)

    def score(hot, r):
        sl = _rows(r, B)
        i, t, cl, ce = ids[sl], tgt[sl], last[sl], every[sl]
        st = hot.advance_state(i)
        out = dict(last=hot.candidates_batch(i, cl, k=20), every=hot.candidates_batch(i, ce, last_step_only=False),
                   probs=hot.candidates_batch(i, cl, probs=True), rank=hot.candidate_rank_batch(i, t, ce),
                   rank_last=hot.candidate_rank_batch(i, t, cl, last_step_only=True),
                   state=hot.candidates_from_state(st, cl), state_rank=hot.candidate_rank_from_state(st, t[:, -1], cl))
        return {n: tuple(x.cpu() for x in v) if isinstance(v, tuple) else v.cpu() for n, v in out.items()}

    ref = HotPath(cell, act, V, H, V, weights=ws, comm=_solo(), tc=tc)
    want = [score(ref, r) for r in range(2)]
    got = run_ranks(lambda comm: score(HotPath(cell, act, V, H, V, weights=ws, comm=comm, tc=tc, vocab_parallel=True),
                                       comm.rank))
    for r in range(2):
        g, w = got[r], want[r]
        for n in ("last", "every", "state"):
            assert torch.equal(g[n][0], w[n][0]) and torch.equal(g[n][1], w[n][1]), (r, n)
        for n in ("rank", "rank_last", "state_rank"):
            assert torch.equal(g[n], w[n]), (r, n)
        assert torch.equal(g["probs"][0], w["probs"][0])
        assert torch.allclose(g["probs"][1], w["probs"][1], rtol=1e-6, atol=0), r


def test_data_parallel_candidate_ranking_equals_single_gpu():
    V, H, T, B, C = 998, 32, 12, 40, 25
    model = _ytoz("GRU", V, H)
    ws = model.model.hot.get_weights()
    ids, tgt = synthetic.make_batch(V, T, B, seed=4, min_len=1)
    cand = _make_lists(np.random.default_rng(3), (B, T), C, V, extra=tgt)
    want = model.evaluate_candidate_ranking(ids, tgt, cand, ks=(1, 5, 10))

    def rank_fn(comm):
        m = _ytoz("GRU", V, H)
        m.model.hot = HotPath("GRU", "tanh", V, H, V, weights=ws, comm=comm)
        sl = _rows(comm.rank, B)
        return m.evaluate_candidate_ranking(ids[sl], tgt[sl], cand[sl], ks=(1, 5, 10))

    for got in run_ranks(rank_fn):
        assert got["n"] == want["n"]
        for key in want:
            assert abs(got[key] - want[key]) <= 1e-12 * max(1.0, abs(want[key])), key
    # the metrics are those of the rank array
    r = model.model.predict_candidate_rank(ids, tgt, cand, device=True)
    again = metrics_from_sums(rank_sums(r, (1, 5, 10)), (1, 5, 10))
    assert all(abs(again[key] - want[key]) <= 1e-12 * max(1.0, abs(want[key])) for key in want)


# --------------------------------------------------------------------------------------------------------- 8. errors
def test_errors():
    V, T, n = 300, 12, 10
    model = _ytoz("GRU", V, 32)
    ids, tgt = synthetic.make_batch(V, T, n, seed=1, min_len=1)
    ok = np.zeros((n, 4), dtype=np.int32)
    st = model.advance_state(ids)
    bad_calls = [
        lambda: model.predict_candidates(ids, ok[:, None]),                          # (n, 1, C) for the last step
        lambda: model.predict_candidates(ids, ok, last_step_only=False),             # (n, C) for every step
        lambda: model.predict_candidates(ids, np.zeros((n, MAX_CANDIDATES + 1), dtype=np.int32)),
        lambda: model.predict_candidates(ids, ok, k=5),
        lambda: model.predict_candidates(ids, ok.astype(np.float32)),
        lambda: model.predict_candidates(ids, np.full((n, 4), V, dtype=np.int32)),
        lambda: model.predict_candidates(ids, torch.full((n, 4), V, dtype=torch.int32, device="cuda")),
        lambda: model.predict_candidate_rank(ids, tgt, np.full((n, T, 4), V + 5, dtype=np.int64)),
        lambda: model.predict_candidates_from_state(st, torch.full((n, 4), V, dtype=torch.int64, device="cuda")),
        lambda: model.predict_candidate_rank_from_state(st, tgt[:, -1], ok[:5]),
    ]
    for f in bad_calls:
        with pytest.raises(ValueError):
            f()
    dense = M.NoRecurrenceModel(5, 4, 4)
    with pytest.raises(NotImplementedError):
        dense.predict_candidates_from_state(model.initial_state(3), np.zeros((3, 2), dtype=np.int32))
    with pytest.raises(NotImplementedError):
        dense.predict_candidate_rank_from_state(model.initial_state(3), np.zeros(3), np.zeros((3, 2), dtype=np.int32))
