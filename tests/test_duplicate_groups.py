"""CPU: `group_labels`, which turns component labels into the groups `B200VectorDB.find_duplicate_groups` returns: members in
row order, the largest group first, groups of equal size by their smallest row, groups below `min_size` left out."""
import numpy as np

from revers_o_b200.vector_db import group_labels


def test_order_size_then_smallest_row():
    labels = [0, 1, 0, 3, 1, 0, 6, 3, 3, 9, 1]
    assert group_labels(labels) == [[0, 2, 5], [1, 4, 10], [3, 7, 8]]
    # equal sizes order by their smallest row, not by the label's value
    assert group_labels([5, 5, 0, 0, 2, 2]) == [[0, 1], [2, 3], [4, 5]]


def test_min_size_and_singletons():
    labels = [0, 1, 0, 3, 1, 0, 6, 3, 9]
    assert group_labels(labels, min_size=3) == [[0, 2, 5]]
    assert group_labels(labels, min_size=4) == []
    assert group_labels(labels, min_size=1) == [[0, 2, 5], [1, 4], [3, 7], [6], [8]]
    assert group_labels(labels, min_size=0) == group_labels(labels, min_size=1)
    assert group_labels(np.arange(5)) == []                       # all singletons
    assert group_labels([]) == [] and group_labels([7], min_size=1) == [[0]]


def test_rows_are_offset_and_labels_need_not_be_rows():
    labels = np.array([40, 12, 40, 12, 12], dtype=np.int64)
    assert group_labels(labels, row0=100) == [[101, 103, 104], [100, 102]]


def test_agrees_with_a_plain_restatement():
    rs = np.random.RandomState(0)
    for _ in range(20):
        n = int(rs.randint(1, 300))
        labels = rs.randint(0, max(1, n // 3), n)
        min_size = int(rs.randint(0, 5))
        groups: dict = {}
        for r, lab in enumerate(labels.tolist()):
            groups.setdefault(lab, []).append(r)
        want = sorted((g for g in groups.values() if len(g) >= max(min_size, 1)), key=lambda g: (-len(g), g[0]))
        assert group_labels(labels, min_size) == want
