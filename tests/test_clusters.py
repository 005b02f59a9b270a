"""CPU: the host logic of `B200VectorDB.cluster` — the cluster renumbering (`cluster_order`), the re-seeding choice
(`sharded.reseed_rows`) on hand-made scores with ties, and the argument checks that need no device."""
import numpy as np
import pytest
import torch

from revers_o_b200._lib import RvoError
from revers_o_b200.sharded import reseed_rows
from revers_o_b200.vector_db import check_cluster_args, cluster_order


def test_cluster_order_sizes_ties_and_empty_clusters():
    #            row: 0  1  2  3  4  5  6  7  8
    labels = np.array([3, 1, 3, 1, 4, 3, 4, 0, 1])
    new, order, sizes = cluster_order(labels, 6)
    # sizes: 0:1, 1:3, 2:0, 3:3, 4:2, 5:0.  1 and 3 tie at 3 members: 3's first row (0) precedes 1's (1)
    assert order.tolist() == [3, 1, 4, 0, 2, 5]
    assert sizes.tolist() == [3, 3, 2, 1, 0, 0]
    assert new.dtype == np.int32 and new.tolist() == [0, 1, 0, 1, 2, 0, 2, 3, 1]
    # the renumbering is a relabelling: same partition, and order maps new -> old
    assert np.array_equal(order[new], labels)
    assert sizes.dtype == np.int64 and sizes.sum() == labels.size


def test_cluster_order_random_consistency():
    rs = np.random.RandomState(0)
    C = 50
    labels = rs.randint(0, C - 7, size=1000)
    new, order, sizes = cluster_order(labels, C)
    assert np.array_equal(order[new], labels)
    assert np.array_equal(np.bincount(new, minlength=C), sizes)
    assert (np.diff(sizes) <= 0).all()
    firsts = [np.flatnonzero(new == j)[0] for j in range(C) if sizes[j]]
    for j in range(len(firsts) - 1):
        if sizes[j] == sizes[j + 1]:
            assert firsts[j] < firsts[j + 1]
    assert order[sizes == 0].tolist() == sorted(order[sizes == 0].tolist())   # empty clusters last, in index order


def test_reseed_rows_lowest_scores_ties_by_row():
    # two shards: global rows 0..4 and 5..9
    a = torch.tensor([0.5, 0.1, 0.3, 0.1, 0.9])
    b = torch.tensor([0.1, 0.2, -0.4, 0.1, 0.1])
    assert reseed_rows([a, b], [0, 5], 1) == [7]
    # 0.1 appears at rows 1, 3, 5, 8, 9: lower rows first, across the shards
    assert reseed_rows([a, b], [0, 5], 4) == [7, 1, 3, 5]
    assert reseed_rows([a, b], [0, 5], 6) == [7, 1, 3, 5, 8, 9]
    # one shard holding the same rows gives the same choice
    assert reseed_rows([torch.cat([a, b])], [0], 6) == [7, 1, 3, 5, 8, 9]
    # a shard with fewer rows than clusters to re-seed
    assert reseed_rows([torch.tensor([0.0]), b], [0, 1], 3) == [3, 0, 1]


def test_cluster_argument_checks():
    assert check_cluster_args(10, 4, 3, 0, None) is None
    init = check_cluster_args(10, 4, 2, 5, [[1, 0, 0, 0], [0, 2, 0, 0]])
    assert init.dtype == np.float32 and init.shape == (2, 4)
    with pytest.raises(RvoError, match="empty"):
        check_cluster_args(0, 4, 1, 5, None)
    for C in (0, -1, 11, 2.5, True):
        with pytest.raises(RvoError, match="n_clusters"):
            check_cluster_args(10, 4, C, 5, None)
    with pytest.raises(RvoError, match="n_clusters"):
        check_cluster_args(100_000, 4, 65537, 5, None)
    assert check_cluster_args(100_000, 4, 65536, 5, None) is None
    with pytest.raises(RvoError, match="max_iter"):
        check_cluster_args(10, 4, 2, -1, None)
    with pytest.raises(RvoError, match="2\\^31"):
        check_cluster_args(1 << 31, 4, 2, 5, None)
    with pytest.raises(RvoError, match="shape"):
        check_cluster_args(10, 4, 2, 5, np.ones((3, 4)))
    with pytest.raises(RvoError, match="shape"):
        check_cluster_args(10, 4, 2, 5, np.ones((2, 5)))
    with pytest.raises(RvoError, match="rows \\[1\\]"):
        check_cluster_args(10, 4, 2, 5, [[1, 0, 0, 0], [0, 0, 0, 0]])
    with pytest.raises(RvoError, match="rows \\[0\\]"):
        check_cluster_args(10, 4, 2, 5, [[np.nan, 0, 0, 1], [0, 1, 0, 0]])
    with pytest.raises(RvoError, match="rows \\[1\\]"):
        check_cluster_args(10, 4, 2, 5, [[1, 0, 0, 1], [0, np.inf, 0, 0]])
