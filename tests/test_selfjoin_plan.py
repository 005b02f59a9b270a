"""CPU: the work plan of the self-join of a row-sharded collection (`sharded.selfjoin_plan`).  Every unordered pair of rows is
examined by exactly one item (checked by enumeration with a small block size), only blocks of queries move, and the devices'
loads stay within 10 % of even unless one shard's own triangle, which cannot leave its device, is larger."""
import itertools

import numpy as np
import pytest

from revers_o_b200.sharded import JoinItem, selfjoin_plan

LAYOUTS = [[1024] * 2, [1024] * 3, [1024] * 4, [512] * 8, [1024, 1024, 952], [1024, 0, 640], [0, 768, 768],
           [2048, 256], [128, 1024, 512, 768], [300, 200, 100], [5000, 4096, 128, 77]]


def pairs_of(it: JoinItem) -> int:
    m = it.q_hi - it.q_lo
    if it.q_shard == it.t_shard:          # i in [q_lo, q_hi), i < j < t_hi
        return m * (it.t_hi - 1) - (it.q_lo + it.q_hi - 1) * m // 2
    return m * (it.t_hi - it.t_lo)


def loads(plan):
    return [sum(pairs_of(it) for it in items) for items in plan]


def least_max_load(sizes):
    """No plan can do better: the triangles of a set S of shards and the rectangles between them run on S's devices, so some
    device of S carries at least 1/|S| of that work."""
    live = [n for n in sizes if n]
    best = 0.0
    for k in range(1, len(live) + 1):
        for S in itertools.combinations(live, k):
            work = sum(n * (n - 1) // 2 for n in S) + sum(a * b for a, b in itertools.combinations(S, 2))
            best = max(best, work / k)
    return best


@pytest.mark.parametrize("sizes", LAYOUTS)
def test_every_pair_of_rows_is_examined_by_exactly_one_item(sizes):
    block = 128
    plan = selfjoin_plan(sizes, block)
    assert len(plan) == len(sizes)
    row0 = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    N = int(row0[-1])
    seen = np.zeros((N, N), np.int32)
    for g, items in enumerate(plan):
        for it in items:
            assert it.t_shard == g, "an item runs where its target rows live"
            assert 0 <= it.q_lo < it.q_hi <= sizes[it.q_shard] and 0 <= it.t_lo < it.t_hi <= sizes[g]
            assert it.q_hi - it.q_lo <= block and it.q_lo % block == 0 and it.t_lo % 128 == 0
            qi = np.arange(it.q_lo, it.q_hi) + row0[it.q_shard]
            tj = np.arange(it.t_lo, it.t_hi) + row0[g]
            a, b = np.meshgrid(qi, tj, indexing="ij")
            keep = (b > a) if it.q_shard == g else np.ones_like(a, bool)
            lo, hi = np.minimum(a, b)[keep], np.maximum(a, b)[keep]
            np.add.at(seen, (lo, hi), 1)
    upper = np.triu(np.ones((N, N), bool), 1)
    assert (seen[upper] == 1).all() and (seen[~upper] == 0).all()
    assert sum(loads(plan)) == N * (N - 1) // 2


@pytest.mark.parametrize("sizes", LAYOUTS + [[250_000] * 8, [500_000] * 4, [1_000_000] * 2, [2_000_000],
                                             [700_000, 700_000, 600_000], [1_000_000, 500_000, 250_000, 250_000],
                                             [4_194_304, 4_194_304, 1_000_000], [4_194_304] * 7 + [2_000]])
def test_device_loads_are_balanced(sizes):
    block = 128 if max(sizes) <= 8192 else 4096
    plan = selfjoin_plan(sizes, block)
    ld = loads(plan)
    live = [n for n in sizes if n]
    total = sum(ld)
    biggest_item = max(pairs_of(it) for items in plan for it in items)
    biggest_triangle = max(n * (n - 1) // 2 for n in live)
    # an empty shard holds no target rows, so no work can run on its device: the even share is over the shards with rows.
    # Where a few big shards and their rectangles outweigh their share (e.g. [1M, 500k, 250k, 250k]), no plan meets that
    # bound; the least possible largest load applies there.
    best = least_max_load(sizes)
    assert max(ld) <= max(1.10 * total / len(live), biggest_triangle, best) + biggest_item, (ld, total)
    assert max(ld) <= 1.01 * best + biggest_item, (ld, best)


def test_equal_shards_split_every_rectangle_in_half():
    sizes = [250_000] * 8
    ld = loads(selfjoin_plan(sizes, 4096))
    assert max(ld) / (sum(ld) / 8) < 1.01


def test_nothing_to_do_for_empty_or_single_row_layouts():
    assert selfjoin_plan([0, 0], 4096) == [[], []]
    plan = selfjoin_plan([1, 0, 1], 128)
    assert sum(pairs_of(it) for items in plan for it in items) == 1
    for sizes in itertools.product([0, 130], repeat=3):
        plan = selfjoin_plan(list(sizes), 128)
        n = sum(sizes)
        assert sum(loads(plan)) == n * (n - 1) // 2
