"""GPU: the near-duplicate self-join (BASELINE config 4) of a row-sharded collection.  `find_near_duplicates` on a collection
loaded with `devices=[...]` returns the same id pairs with bit-identical scores as the single-device join, and matches the
oracle; `rvo_join_threshold` in rectangle mode equals a brute-force fp32 restatement and in triangle mode the existing join; a
static scene spread over the shards is joined exactly through the overflow protocol.  On a 1-GPU box the shards are virtual
(the same device listed twice or three times); with two or more GPUs the real devices are used as well."""
import numpy as np
import pytest
import torch

from oracle import reverso_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    return torch.device("cuda:0")


def device_sets():
    sets = [[0, 0], [0, 0, 0]]
    if torch.cuda.is_available() and torch.cuda.device_count() >= 2:
        sets.append(list(range(min(torch.cuda.device_count(), 8))))
    return sets


def _rows(n, d, dev, seed, dup_frac=0.05, cluster=0):
    from revers_o_b200 import ops, synth
    return ops.untile_rows(synth.make_selfjoin_db(n, d, dup_frac, dev, seed=seed, cluster=cluster), n, d).float().cpu().numpy()


def _ingest(db, rows):
    from revers_o_b200.vector_db import models
    db.recreate_collection("frames", vectors_config=models.VectorParams(size=rows.shape[1], distance=models.Distance.COSINE))
    for lo in range(0, len(rows), 5000):
        db.upsert_batch("frames", list(range(lo, min(len(rows), lo + 5000))), rows[lo: lo + 5000], assume_new=True)


def _by_pair(pairs, scores):
    got = {tuple(p): float(s) for p, s in zip(pairs, scores)}
    assert len(got) == len(pairs), "duplicate pairs emitted"
    return got


def _check_oracle(got, rows_f32, thr):
    rp, rs = O.selfjoin_threshold(rows_f32, thr, db_is_normalized=True)
    ref = {(int(a), int(b)): float(s) for (a, b), s in zip(rp, rs)}
    for key in set(got) ^ set(ref):   # may differ only within the tolerance of the threshold itself
        s = got.get(key, ref.get(key))
        assert abs(s - thr) <= 1e-3, (key, s)
    for key in set(got) & set(ref):
        assert abs(got[key] - ref[key]) <= 1e-3
    assert len(set(got) & set(ref)) >= 0.99 * len(ref) and len(ref) > 0


@pytest.mark.parametrize("devices", device_sets())
@pytest.mark.parametrize("n,d", [(20_000, 256), (9000, 1024)])
def test_sharded_join_equals_single_device_join(dev, tmp_path, n, d, devices):
    from revers_o_b200 import ops
    from revers_o_b200.vector_db import B200VectorDB
    thr, path = 0.95, str(tmp_path / "db")
    one = B200VectorDB(path=path, device=dev)
    _ingest(one, _rows(n, d, dev, seed=n))
    many = B200VectorDB(path=path, devices=devices)               # loaded from disk: split evenly, whole 128-row blocks
    cn = many._coll("frames")
    assert len([s for s in cn.shards if s.n]) == len(devices) and cn.n == n
    p1, s1 = one.find_near_duplicates("frames", thr)
    pn, sn = many.find_near_duplicates("frames", thr)
    assert sn.dtype == np.float32 and all(a < b for a, b in pn)   # ids are the rows here: the lower global row comes first
    single, sharded = _by_pair(p1, s1), _by_pair(pn, sn)
    assert sharded == single                                      # same pairs, bit-identical scores
    _check_oracle(sharded, ops.untile_rows(one._coll("frames").vectors, n, d).float().cpu().numpy(), thr)


def test_incrementally_ingested_shards_join_like_one_device(dev):
    """Uneven shards as incremental ingest leaves them ([4096, 4096, 808] rows), string ids."""
    from revers_o_b200.vector_db import B200VectorDB, models
    n, d, thr = 9000, 256, 0.95
    rows = _rows(n, d, dev, seed=4, dup_frac=0.2)
    dbs = [B200VectorDB(device=dev), B200VectorDB(devices=[0, 0, 0], shard_rows=4096)]
    for db in dbs:
        db.recreate_collection("frames", vectors_config=models.VectorParams(size=d, distance=models.Distance.COSINE))
        for lo in range(0, n, 1000):
            db.upsert_batch("frames", [f"f{i:05d}" for i in range(lo, min(n, lo + 1000))], rows[lo: lo + 1000])
    assert [s.n for s in dbs[1]._coll("frames").shards] == [4096, 4096, 808]
    (p1, s1), (p3, s3) = (db.find_near_duplicates("frames", thr) for db in dbs)
    assert len(p1) > 500 and _by_pair(p3, s3) == _by_pair(p1, s1)
    assert all(a < b for a, b in p3)                              # "f%05d" ids sort like their rows


def test_join_threshold_rectangle_triangle_and_append(dev):
    from revers_o_b200 import ops, synth
    n, d, thr = 12_000, 512, 0.95
    db = synth.make_selfjoin_db(n, d, 0.3, dev, seed=3)
    rows = ops.untile_rows(db, n, d).float()
    split = 4096                                                   # rows [0, 4096) x rows [4096, n)
    # rectangle, queries copied to a buffer of their own, target a block-aligned sub-range of the DB
    out = ops.join_out(1 << 16, dev)
    qbuf = db[: split // 128].clone()
    ops.join_threshold(qbuf, 0, split, 0, db[split // 128:], n - split, d, thr, split, 32768, out)
    torch.cuda.synchronize()
    m = int(out[2].item())
    assert int(out[3].item()) == 0 and 0 < m < (1 << 16)
    rect = _by_pair(out[0][:m].cpu().numpy(), out[1][:m].cpu().numpy())
    assert all(a < split <= b for a, b in rect)
    sc = rows[:split] @ rows[split:].T                             # brute force in fp32 on the GPU
    ij = torch.nonzero(sc >= thr)
    want = {(int(i), int(j) + split) for i, j in ij.tolist()}
    near = {(int(i), int(j) + split) for i, j in torch.nonzero((sc - thr).abs() <= 1e-4).tolist()}
    assert (set(rect) ^ want) <= near and len(want) > 100
    for (a, b), s in rect.items():
        assert abs(s - float(sc[a, b - split])) <= 1e-4
    # the other way round (queries = the later rows, read in place from the same DB) appends the same pairs, same scores
    ops.join_threshold(db[split // 128:], 0, n - split, split, db, split, d, thr, 0, 32768, out)
    torch.cuda.synchronize()
    assert int(out[2].item()) == 2 * m and int(out[3].item()) == 0
    assert _by_pair(out[0][m: 2 * m].cpu().numpy(), out[1][m: 2 * m].cpu().numpy()) == rect
    # triangle (qdb is db, equal offsets) == rvo_selfjoin_threshold_ex bit for bit, rows [1000, 7000) as queries
    tri = ops.join_out(1 << 16, dev)
    ops.join_threshold(db, 1000, 7000, 17, db, n, d, thr, 17, 32768, tri)
    ref = ops.selfjoin_threshold(db, n, d, thr, 1000, 7000, out_cap=1 << 16, id_offset=17)
    torch.cuda.synchronize()
    mt, mr = int(tri[2].item()), int(ref[2].item())
    assert mt == mr > 0 and int(tri[3].item()) == 0
    assert _by_pair(tri[0][:mt].cpu().numpy(), tri[1][:mt].cpu().numpy()) == \
        _by_pair(ref[0][:mr].cpu().numpy(), ref[1][:mr].cpu().numpy())
    # row sets that overlap are refused
    with pytest.raises(Exception):
        ops.join_threshold(db, 0, 4096, 0, db[16:], n - 2048, d, thr, 2048, 32768, out)


@pytest.mark.parametrize("devices", device_sets())
def test_static_scene_across_shards_falls_back_exactly(dev, devices):
    """3000 exact copies of row 0 spread over every shard: with 64 candidates per sub-list the fixed-capacity join overflows;
    the sharded join re-runs the affected devices with larger lists and returns every one of the 3001*3000/2 clique pairs —
    the same pairs and scores as the single-device exact join."""
    from revers_o_b200 import ops, synth
    from revers_o_b200.sharded import selfjoin_sharded, shard_bounds
    n, d, thr, cl = 60_000, 256, 0.95, 3000
    db = synth.make_selfjoin_db(n, d, 0.02, dev, seed=9, cluster=cl)
    G = len(devices)
    shards = []
    for g, dv in enumerate(devices):
        lo, hi = shard_bounds(n, G, g)
        shards.append((db[lo // 128: (hi + 127) // 128].clone().to(torch.device("cuda", dv)), hi - lo, lo))
    out = ops.join_out(1 << 22, dev)
    ops.join_threshold(shards[0][0], 0, shards[0][1], 0, shards[0][0], shards[0][1], d, thr, 0, 1024, out)
    torch.cuda.synchronize()
    assert int(out[3].item()) > 0                                  # the small capacity does overflow
    p, s = selfjoin_sharded(shards, d, thr, max_pairs=1 << 16, cand_cap=1024)
    rows = ops.untile_rows(db, n, d).float()
    clique = set((rows @ rows[0] > 0.99).nonzero().flatten().tolist())
    assert len(clique) == cl + 1
    assert sum(1 for a, b in p.tolist() if a in clique and b in clique) == (cl + 1) * cl // 2
    p1, s1 = ops.selfjoin_exact(db, n, d, thr)
    assert _by_pair(p, s) == _by_pair(p1, s1)
