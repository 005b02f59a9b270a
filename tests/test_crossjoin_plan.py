"""CPU: the work plan of the join between two row-sharded collections (`sharded.crossjoin_plan`).  Every (left row, right row)
pair is examined by exactly one item (checked by enumeration with a small block size), every item runs on the device that holds
its target rows, only blocks of queries move, and the devices' loads stay within 10 % of even unless the layout itself forces
more work onto some devices."""
import itertools

import numpy as np
import pytest

from revers_o_b200.sharded import JoinItem, crossjoin_plan

# (left [(device, rows)], right [(device, rows)])
LAYOUTS = [
    ([(0, 1024), (1, 1024)], [(0, 768), (1, 768)]),                              # same devices on both sides
    ([(0, 640), (1, 640), (2, 512)], [(0, 1000), (1, 1000), (2, 1000)]),
    ([(0, 1024), (1, 1024)], [(2, 896), (3, 896)]),                              # disjoint device sets
    ([(0, 1024)], [(g, 384) for g in range(8)]),                                 # left on one device, right on 8
    ([(0, 1500)], [(g, 300) for g in range(1, 9)]),                              # left on one device, right on 8 others
    ([(0, 512), (0, 512)], [(0, 700), (0, 700), (0, 700)]),                      # virtual shards sharing a device
    ([(0, 512), (1, 512), (0, 512)], [(1, 640), (0, 640)]),
    ([(0, 1024), (1, 0), (2, 640)], [(0, 0), (1, 768), (2, 768)]),               # empty shards
    ([(0, 0), (1, 0)], [(0, 300), (1, 300)]),
    ([(0, 1)], [(1, 1)]),                                                        # one-row sides
    ([(0, 1)], [(0, 1), (1, 1)]),
    ([(0, 1), (1, 1)], [(0, 1000), (1, 1)]),
    ([(0, 2048), (1, 256)], [(0, 130), (1, 3000), (2, 77)]),                     # uneven sizes
    ([(3, 5000)], [(0, 4096), (1, 128), (2, 77)]),
]

BIG = [
    ([(0, 1_000_000)], [(0, 2_000_000)]),
    ([(g, 500_000) for g in range(2)], [(g, 1_000_000) for g in range(2)]),
    ([(g, 250_000) for g in range(4)], [(g, 500_000) for g in range(4)]),
    ([(g, 125_000) for g in range(8)], [(g, 250_000) for g in range(8)]),
    ([(0, 1_000_000)], [(g, 250_000) for g in range(8)]),
    ([(0, 1_000_000)], [(g, 250_000) for g in range(1, 9)]),
    ([(0, 700_000), (1, 300_000)], [(2, 2_000_000), (3, 50_000)]),
    ([(0, 4_194_304), (1, 4_194_304)], [(0, 1_000_000), (1, 9_000), (2, 2_000_000)]),
    ([(g % 2, 400_000) for g in range(4)], [(g % 2, 300_000) for g in range(4)]),
    ([(0, 3_000_000), (1, 10_000)], [(1, 3_000_000), (2, 10_000)]),
]


def device_of(left, right, shard):
    return (left + right)[shard][0]


def rows_of(left, right, shard):
    return (left + right)[shard][1]


def pairs_of(it: JoinItem) -> int:
    return (it.q_hi - it.q_lo) * (it.t_hi - it.t_lo)


def loads(plan):
    return {dv: sum(pairs_of(it) for it in its) for dv, its in plan.items()}


def least_max_load(left, right):
    """No plan can do better: the rectangles whose two shards both live on a device set S run on S, so some device of S
    carries at least 1/|S| of them."""
    devs = sorted({dv for dv, n in left + right if n})
    best = 0.0
    for k in range(1, len(devs) + 1):
        for S in itertools.combinations(devs, k):
            work = sum(na * nb for da, na in left for db, nb in right if da in S and db in S)
            best = max(best, work / k)
    return best


@pytest.mark.parametrize("left,right", LAYOUTS)
def test_every_pair_of_rows_is_examined_by_exactly_one_item(left, right):
    block = 128
    plan = crossjoin_plan(left, right, block)
    assert set(plan) == {dv for dv, _ in left + right}
    nl = len(left)
    lrow0 = np.concatenate([[0], np.cumsum([n for _, n in left])]).astype(np.int64)
    rrow0 = np.concatenate([[0], np.cumsum([n for _, n in right])]).astype(np.int64)
    NL, NR = int(lrow0[-1]), int(rrow0[-1])
    seen = np.zeros((NL, NR), np.int32)
    for dv, items in plan.items():
        for it in items:
            assert device_of(left, right, it.t_shard) == dv, "an item runs where its target rows live"
            assert (it.q_shard < nl) != (it.t_shard < nl), "an item pairs a left shard with a right shard"
            nq, nt = rows_of(left, right, it.q_shard), rows_of(left, right, it.t_shard)
            assert 0 <= it.q_lo < it.q_hi <= nq and 0 <= it.t_lo < it.t_hi <= nt
            assert it.q_hi - it.q_lo <= block and it.q_lo % block == 0 and it.t_lo % 128 == 0
            q = np.arange(it.q_lo, it.q_hi)
            t = np.arange(it.t_lo, it.t_hi)
            if it.q_shard < nl:
                a, b = np.meshgrid(q + lrow0[it.q_shard], t + rrow0[it.t_shard - nl], indexing="ij")
            else:
                b, a = np.meshgrid(q + rrow0[it.q_shard - nl], t + lrow0[it.t_shard], indexing="ij")
            np.add.at(seen, (a.ravel(), b.ravel()), 1)
    assert (seen == 1).all()
    assert sum(loads(plan).values()) == NL * NR


@pytest.mark.parametrize("left,right", LAYOUTS + BIG)
def test_device_loads_are_balanced(left, right):
    block = 128 if max(n for _, n in left + right) <= 8192 else 4096
    plan = crossjoin_plan(left, right, block)
    ld = loads(plan)
    total = sum(ld.values())
    holding = {dv for dv, n in left + right if n}
    if total == 0:
        return
    biggest_item = max(pairs_of(it) for items in plan.values() for it in items)
    best = least_max_load(left, right)
    assert max(ld.values()) <= max(1.10 * total / len(holding), best) + biggest_item, (ld, total, best)


@pytest.mark.parametrize("G", [2, 4, 8])
def test_equal_shards_over_the_same_devices_are_even(G):
    plan = crossjoin_plan([(g, 1_000_000 // G) for g in range(G)], [(g, 2_000_000 // G) for g in range(G)], 4096)
    ld = list(loads(plan).values())
    assert len(ld) == G and max(ld) / (sum(ld) / G) < 1.01


def test_one_device_on_both_sides_is_one_run_of_left_blocks():
    plan = crossjoin_plan([(0, 10_000)], [(0, 20_000)], 4096)
    assert list(plan) == [0]
    assert plan[0] == [JoinItem(0, lo, min(lo + 4096, 10_000), 1, 0, 20_000) for lo in range(0, 10_000, 4096)]


def test_nothing_to_do_when_a_side_is_empty():
    assert crossjoin_plan([(0, 0)], [(1, 500)], 128) == {0: [], 1: []}
    assert crossjoin_plan([(0, 500)], [], 128) == {0: []}
