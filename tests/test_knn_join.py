"""CPU: the host logic of the k-nearest-neighbour join — `vector_db.mutual_best` (one-to-one correspondences from two kNN
lists) and `sharded.knn_plan` (the work of a row-sharded kNN join)."""
import numpy as np
import pytest

from revers_o_b200._lib import RvoError
from revers_o_b200.sharded import KnnItem, knn_plan, knn_sharded
from revers_o_b200.vector_db import mutual_best


def test_mutual_best_keeps_only_mutual_pairs_in_score_order():
    # A has 5 rows, B has 4.  k = 2 lists: only the first entry counts.
    rows_ab = np.array([[2, 0], [1, 3], [0, -1], [3, 2], [-1, -1]])
    scores_ab = np.array([[0.9, 0.5], [0.7, 0.6], [0.9, -np.inf], [0.7, 0.1], [-np.inf, -np.inf]], np.float32)
    counts_ab = np.array([2, 2, 1, 2, 0])
    rows_ba = np.array([[2, 1], [1, 0], [0, 3], [1, 3]])
    counts_ba = np.array([2, 2, 2, 1])
    pairs, scores = mutual_best(rows_ab, counts_ab, rows_ba, counts_ba, scores_ab)
    # a=0 -> b=2 -> a=0: mutual (0.9); a=2 -> b=0 -> a=2: mutual (0.9, tie: a=0 first); a=1 -> b=1 -> a=1: mutual (0.7);
    # a=3 -> b=3 -> a=1: one-sided; a=4 has no match (count 0)
    assert pairs.tolist() == [[0, 2], [2, 0], [1, 1]]
    assert scores.dtype == np.float32 and scores.tolist() == [np.float32(0.9), np.float32(0.9), np.float32(0.7)]


def test_mutual_best_ties_order_by_a_then_b_and_ignores_empty_lists():
    rows_ab = np.array([[1], [0], [2]])
    scores_ab = np.full((3, 1), 0.5, np.float32)
    counts_ab = np.array([1, 1, 1])
    rows_ba = np.array([[1], [0], [-1]])
    counts_ba = np.array([1, 1, 0])                 # b=2 has no match: a=2 -> b=2 is one-sided
    pairs, scores = mutual_best(rows_ab, counts_ab, rows_ba, counts_ba, scores_ab)
    assert pairs.tolist() == [[0, 1], [1, 0]] and scores.tolist() == [0.5, 0.5]
    # nothing on either side
    p, s = mutual_best(np.zeros((0, 1), np.int64), np.zeros(0, np.int32), np.zeros((0, 1), np.int64), np.zeros(0, np.int32),
                       np.zeros((0, 1), np.float32))
    assert p.shape == (0, 2) and s.shape == (0,) and p.dtype == np.int64 and s.dtype == np.float32
    p, s = mutual_best(rows_ab, np.zeros(3, np.int32), rows_ba, counts_ba, scores_ab)
    assert p.shape == (0, 2)


def test_mutual_best_agrees_with_a_brute_force():
    rs = np.random.RandomState(0)
    sc = rs.randint(0, 6, size=(40, 30)).astype(np.float32) / 5      # many ties
    best_ab = np.lexsort((np.tile(np.arange(30), (40, 1)), -sc), axis=1)[:, :1]
    best_ba = np.lexsort((np.tile(np.arange(40), (30, 1)), -sc.T), axis=1)[:, :1]
    pairs, scores = mutual_best(best_ab, np.ones(40), best_ba, np.ones(30), sc[np.arange(40)[:, None], best_ab])
    want = sorted(((-sc[a, b], a, b) for a in range(40) for b in range(30) if best_ab[a, 0] == b and best_ba[b, 0] == a))
    assert pairs.tolist() == [[a, b] for _, a, b in want]
    assert scores.tolist() == [-s for s, _, _ in want]


def test_knn_plan_covers_every_block_and_right_shard_once():
    left = [(0, 10_000), (1, 129), (0, 0), (2, 4096)]
    right = [(1, 500), (0, 7000), (1, 0), (2, 3)]
    plan = knn_plan(left, right, block=4096)
    assert sorted(plan) == [0, 1, 2]
    seen = []
    for dv, its in plan.items():
        for it in its:
            assert isinstance(it, KnnItem) and right[it.t_shard][0] == dv and right[it.t_shard][1] > 0
            assert it.q_lo % 4096 == 0 and 0 < it.q_hi - it.q_lo <= 4096 and it.q_hi <= left[it.q_shard][1]
            seen += [(it.q_shard, r, it.t_shard) for r in range(it.q_lo, it.q_hi)]
    want = [(a, r, b) for a, (_, na) in enumerate(left) for r in range(na) for b, (_, nb) in enumerate(right) if nb]
    assert sorted(seen) == sorted(want)                               # every (left row, right shard) exactly once
    for its in plan.values():                                         # block by block, in left row order
        keys = [(it.q_shard, it.q_lo) for it in its]
        assert keys == sorted(keys)


def test_query_blocks_must_be_whole_tiles():
    with pytest.raises(RvoError, match="multiple of 128"):
        knn_plan([(0, 1000)], [(0, 1000)], block=1000)
    with pytest.raises(RvoError, match="multiple of 128"):
        knn_sharded([], [], 64, 10, None, False, block=100)
