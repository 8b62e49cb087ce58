"""Candidate scoring on the CPU: hand-computed answers of the float64 oracle (oracle/candidates.py) -- ties decided by
the item id, then by the list position; duplicates counted once per occurrence; the target inside and outside the list;
pads; k < C; C = 1 -- and the input checks of seq_recommendations_b200.ranking.check_candidates."""
import numpy as np
import pytest
import torch

from oracle import candidates as oc
from oracle import ranking as orank
from seq_recommendations_b200 import ranking


def test_order_ties_go_to_the_lower_id_then_the_earlier_position():
    z = np.array([[1.0, 2.0, 2.0, 0.5, 2.0, 0.0]])
    c = np.array([[4, 9, 3, 7, 3, -1]])
    ids, sc = oc.candidate_order(z, c)
    # 2.0 ties: id 3 (positions 2 and 4, in that order) before id 9; then 1.0, 0.5; the pad last as (-1, 0)
    assert ids.tolist() == [[3, 3, 9, 4, 7, -1]]
    assert sc.tolist() == [[2.0, 2.0, 2.0, 1.0, 0.5, 0.0]]
    ids3, sc3 = oc.candidate_order(z, c, k=3)
    assert ids3.tolist() == [[3, 3, 9]] and sc3.tolist() == [[2.0, 2.0, 2.0]]


def test_order_probabilities_are_exp_z_minus_m_over_s():
    z = np.array([[0.0, 1.0, -1.0]])
    c = np.array([[2, 0, 1]])
    ids, p = oc.candidate_order(z, c, m=np.array([1.0]), s=np.array([2.0]))
    assert ids.tolist() == [[0, 2, 1]]
    assert np.allclose(p, [[0.5, np.exp(-1.0) / 2, np.exp(-2.0) / 2]], rtol=0, atol=1e-15)


def test_pads_and_a_single_candidate():
    ids, sc = oc.candidate_order(np.array([[3.0, 0.0, 0.0]]), np.array([[-1, -5, 6]]))
    assert ids.tolist() == [[6, -1, -1]] and sc.tolist() == [[0.0, 0.0, 0.0]]
    ids, sc = oc.candidate_order(np.array([[-2.5]]), np.array([[11]]))
    assert ids.tolist() == [[11]] and sc.tolist() == [[-2.5]]
    assert oc.candidate_rank(np.array([[-2.5]]), np.array([[11]]), np.array([-2.5]), np.array([11])).tolist() == [1]
    assert oc.candidate_rank(np.array([[-2.5]]), np.array([[11]]), np.array([0.0]), np.array([12])).tolist() == [1]
    assert oc.candidate_rank(np.array([[-2.5]]), np.array([[11]]), np.array([-3.0]), np.array([12])).tolist() == [2]


def test_rank_by_hand():
    z = np.array([[2.0, 1.0, 1.0, 1.0, 3.0, 0.0, 1.0]])
    c = np.array([[8, 5, 2, 2, 6, -1, 7]])
    # target 5 with z_y = 1: ahead are 8 (2.0), 6 (3.0) and both copies of 2 (tie, lower id); 7 ties with a higher id
    assert oc.candidate_rank(z, c, np.array([1.0]), np.array([5])).tolist() == [5]
    # the same target outside the list, same z_y: the same rank
    c_out = np.array([[8, 4, 2, 2, 6, -1, 7]])
    z_out = z.copy()
    z_out[0, 1] = -4.0
    assert oc.candidate_rank(z_out, c_out, np.array([1.0]), np.array([5])).tolist() == [5]
    # a pad target
    assert oc.candidate_rank(z, c, np.array([1.0]), np.array([-1])).tolist() == [0]
    # every entry ahead: C + 1
    assert oc.candidate_rank(np.full((1, 3), 9.0), np.array([[1, 2, 3]]), np.array([0.0]), np.array([4])).tolist() \
        == [4]


def test_rank_over_the_whole_catalog_is_the_catalog_rank():
    rng = np.random.default_rng(3)
    n, V = 200, 23
    z = rng.integers(-4, 5, size=(n, V)).astype(np.float64) / 2.0
    y = rng.integers(0, V, size=n)
    y[::11] = -1
    cand = np.broadcast_to(np.arange(V), (n, V))
    zy = np.take_along_axis(z, np.where(y >= 0, y, 0)[:, None], 1)[:, 0]
    assert np.array_equal(oc.candidate_rank(z, cand, zy, y), orank.target_rank(z, y))
    # and the order of the whole catalog is the stable descending argsort
    ids, _ = oc.candidate_order(z, cand)
    assert np.array_equal(ids, np.argsort(-z, axis=1, kind="stable"))
    lo, hi = oc.candidate_rank_band(z, cand, zy, y, 0.0, exact_ties=True)
    assert np.array_equal(lo, hi) and np.array_equal(lo, orank.target_rank(z, y))


def test_logits_oracle():
    rng = np.random.default_rng(1)
    hs = rng.standard_normal((3, 4, 5))
    W = rng.standard_normal((5, 9))
    b = rng.standard_normal(9)
    cand = rng.integers(-1, 9, size=(3, 4, 6))
    z = oc.candidate_logits(hs, W, b, cand)
    full = hs @ W + b
    want = np.where(cand >= 0, np.take_along_axis(full, np.where(cand >= 0, cand, 0), -1), 0.0)
    assert np.allclose(z, want, rtol=1e-13, atol=1e-13)


def test_rank_band_brackets_the_rank():
    rng = np.random.default_rng(2)
    z = rng.standard_normal((50, 30))
    c = rng.integers(-1, 40, size=(50, 30))
    y = rng.integers(-1, 40, size=50)
    zy = rng.standard_normal(50)
    r = oc.candidate_rank(z, c, zy, y)
    lo, hi = oc.candidate_rank_band(z, c, zy, y, 0.3)
    assert np.all(lo <= r) and np.all(r <= hi)
    assert np.array_equal(oc.candidate_rank_band(z, c, zy, y, 0.0, exact_ties=True)[0], r)


# ------------------------------------------------------------------------------------------------ check_candidates
@pytest.mark.parametrize("make", [np.asarray, torch.as_tensor])
def test_check_candidates_accepts(make):
    a = make(np.array([[1, -1, 3], [0, 2, 2]], dtype=np.int64))
    out, C, k = ranking.check_candidates(a, (2,), 4)
    assert C == 3 and k == 3 and out is a
    assert ranking.check_candidates(a, (2,), 4, k=1)[2] == 1
    b = make(np.zeros((2, 5, 1), dtype=np.int32))
    assert ranking.check_candidates(b, (2, 5), 1)[1:] == (1, 1)
    big = make(np.zeros((1, ranking.MAX_CANDIDATES), dtype=np.int16))
    assert ranking.check_candidates(big, (1,), 1)[1] == ranking.MAX_CANDIDATES


@pytest.mark.parametrize("make", [np.asarray, torch.as_tensor])
def test_check_candidates_refuses(make):
    ok = np.array([[1, -1, 3], [0, 2, 2]], dtype=np.int32)
    bad = [
        (ok, (3,), {}),                                               # rows
        (ok, (2, 3), {}),                                             # (n, T, C) expected
        (ok[0], (2,), {}),                                            # no C axis
        (ok.astype(np.float32), (2,), {}),                            # dtype
        (np.zeros((2, 0), dtype=np.int32), (2,), {}),                 # C = 0
        (np.zeros((1, ranking.MAX_CANDIDATES + 1), dtype=np.int32), (1,), {}),
        (ok, (2,), {"k": 4}),                                         # k > C
        (ok, (2,), {"k": 0}),
        (ok, (2,), {"k": 1.5}),
        (np.array([[1, 4, 0]], dtype=np.int32), (1,), {}),            # id == n_items
    ]
    for a, lead, kw in bad:
        with pytest.raises(ValueError):
            ranking.check_candidates(make(a), lead, 4, **kw)
    with pytest.raises(ValueError):
        ranking.check_candidates(make(ok.astype(bool)), (2,), 4)
