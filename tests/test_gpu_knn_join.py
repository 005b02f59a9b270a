"""GPU: the k-nearest-neighbour join.  `rvo_knn_join` in self and cross mode against an fp64 brute force over the stored bf16
rows; the self exclusion on a row stored three times; a static scene through the overflow protocol; agreement with the
threshold joins at their threshold; row-sharded layouts against one device (virtual shards on a 1-GPU box, the real devices
as well with two or more); the public interface (`B200VectorDB.knn_join`, `SimpleReverso.find_best_matches`)."""
import numpy as np
import pytest
import torch

from test_gpu_crossjoin import FakeEncoder, Det, _db, _fill, device_sets, make_image, mixed_layouts, preprocess

pytestmark = pytest.mark.gpu
TOL = 1e-5


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    return torch.device("cuda:0")


def brute(q, t):
    """fp64 scores of the stored rows (bf16 values, exact in fp64 up to the sum)."""
    return q.double() @ t.double().T


def check_lists(got, sc, k, thr=None, t_off=0, self_cols=None):
    """got = (ids, scores, counts) against the brute-force scores sc [nq, nt]: counts as the threshold gives them (hits within
    TOL of it excused), scores equal to the brute force's best within TOL, every id's true score equal to its reported score,
    no id twice, order score descending with ties by lower id, padding -1 / -inf."""
    ids, scores, counts = (x.to(sc.device) for x in got)
    sc = sc.clone()
    nq = sc.shape[0]
    if self_cols is not None:
        sc[torch.arange(nq, device=sc.device), self_cols] = -float("inf")
    lo_thr = -float("inf") if thr is None else thr
    n_hi = (sc >= lo_thr + TOL).sum(1).clamp(max=k)
    n_lo = (sc >= lo_thr - TOL).sum(1).clamp(max=k)
    c = counts.long()
    assert bool(((c >= n_hi) & (c <= n_lo)).all()), "counts"
    best = sc.topk(k, dim=1).values
    col = torch.arange(k, device=sc.device).expand(nq, k)
    valid = col < c[:, None]
    assert bool(((scores.double() - best).abs()[valid] <= TOL).all()), "scores"
    true = sc.gather(1, (ids - t_off).clamp(min=0))
    assert bool(((true - scores.double()).abs()[valid] <= TOL).all()), "ids"
    assert bool((ids[~valid] == -1).all()) and bool(torch.isinf(scores[~valid]).all())
    s_ids = ids.masked_fill(~valid, -1).sort(1).values
    assert not bool(((s_ids[:, 1:] == s_ids[:, :-1]) & (s_ids[:, 1:] >= 0)).any()), "duplicate id"
    nxt = valid[:, 1:]
    desc = (scores[:, 1:] < scores[:, :-1]) | ((scores[:, 1:] == scores[:, :-1]) & (ids[:, 1:] > ids[:, :-1]))
    assert bool(desc[nxt].all()), "order"


@pytest.mark.parametrize("d,k", [(256, 1), (256, 511), (1024, 10), (1024, 100), (1280, 10), (1280, 512), (2304, 10)])
def test_knn_entry_against_brute_force(dev, d, k):
    from revers_o_b200 import ops, synth
    n = 9_000 if d > 2048 else 12_000
    db = synth.make_selfjoin_db(n, d, 0.3, dev, seed=d + k)
    rows = ops.untile_rows(db, n, d)
    off = 1000
    if k < 512:
        # self mode: ranges not aligned to 128 that span two query blocks (a 700-row and a 3-row last block), and a 3-row call
        for lo, hi in ((37, 37 + 8192 + 700), (37, 37 + 8192 + 3), (n - 3, n)):
            got = ops.knn_exact(db, lo, hi, off, db, n, d, k, None, off, True)
            check_lists(got, brute(rows[lo:hi], rows), k, None, off, torch.arange(lo, hi, device=dev))
    # cross mode: left rows from another buffer, overlapping ids, no exclusion (a row's own copy is a hit)
    nl = 3_001
    left = ops.tile_rows(rows[5_000:5_000 + nl].contiguous())
    kc = min(k, 512)
    got = ops.knn_exact(left, 0, nl, 0, db, n, d, kc, None, 7, False)
    sc = brute(rows[5_000:5_000 + nl], rows)
    check_lists(got, sc, kc, None, 7)
    assert bool((got[0][:, 0] - 7 == torch.arange(5_000, 5_000 + nl, device=dev)).float().mean() > 0.99)
    # a threshold exactly equal to a stored score: that hit is kept
    thr = float(got[1][10, min(3, kc - 1)])
    got_t = ops.knn_exact(left, 0, nl, 0, db, n, d, kc, thr, 7, False)
    assert int(got_t[2][10]) >= min(4, kc) and float(got_t[1][10, min(3, kc - 1)]) == thr
    check_lists(got_t, sc, kc, thr, 7)
    # arguments are refused with the library's message
    with pytest.raises(Exception, match="outside 1..511"):
        ops.knn_join(db, 0, 10, 0, db, n, d, 512, None, 0, True)


def test_fp32_routes_and_exclusion_entry(dev):
    """The SMALL and DENSE routes on a q_rows list equal the brute force, and `rvo_knn_exclude_self` on k + 1 lists equals the
    self mode."""
    from revers_o_b200 import _lib, ops, synth
    n, d, k = 140_000, 512, 20                      # above 131072 rows: the SMALL route samples, then filters
    db = synth.make_selfjoin_db(n, d, 0.3, dev, seed=5)
    rows = ops.untile_rows(db, n, d)
    q_rows = torch.tensor([5, 139_999, 70_001, 128], dtype=torch.int64, device=dev)
    for path in (_lib.RVO_PATH_SMALL, _lib.RVO_PATH_DENSE):
        got = ops.knn_join(db, 0, 4, 0, db, n, d, k, None, 0, True, q_rows, path)
        check_lists(got, brute(rows[q_rows], rows), k, None, 0, q_rows)
    full = ops.knn_join(db, 100, 400, 0, db, n, d, k + 1, None, 0, False)
    ex = ops.knn_exclude_self(*full, 100, 0)
    ref = ops.knn_join(db, 100, 400, 0, db, n, d, k, None, 0, True)
    for a, b in zip(ex, ref):
        assert torch.equal(a, b)
    with pytest.raises(Exception, match="q_rows list"):
        ops.knn_join(db, 0, 4, 0, db, n, d, k, None, 0, True, None, _lib.RVO_PATH_SMALL)


def test_self_exclusion_keeps_exact_copies(dev):
    from revers_o_b200 import ops, synth
    n, d, k = 10_000, 1024, 10
    rows = ops.untile_rows(synth.make_selfjoin_db(n, d, 0.2, dev, seed=11), n, d).clone()
    copies = [1234, 4321, 9000]
    rows[copies[1]] = rows[copies[0]]
    rows[copies[2]] = rows[copies[0]]
    db = ops.tile_rows(rows)
    ids, scores, counts = ops.knn_exact(db, 0, n, 0, db, n, d, k, None, 0, True)
    for c in copies:
        others = [x for x in copies if x != c]
        assert ids[c, :2].tolist() == others                         # the other two copies, lower row first
        assert c not in ids[c].tolist()
        assert float(scores[c, 0]) == float(scores[c, 1])
    assert not bool((ids == torch.arange(n, device=dev)[:, None]).any())
    check_lists((ids, scores, counts), brute(rows, rows), k, None, 0, torch.arange(n, device=dev))


def static_scene(dev, n=50_000, m=5001, d=256, seed=3):
    from revers_o_b200 import ops, synth
    rows = ops.untile_rows(synth.make_selfjoin_db(n, d, 0.0, dev, seed=seed), n, d).clone()
    g = torch.Generator(device=dev).manual_seed(seed)
    at = torch.randperm(n, generator=g, device=dev)[:m].sort().values
    rows[at] = rows[at[0]].clone()
    return rows, at


def test_static_scene_through_the_overflow_route(dev):
    from revers_o_b200 import ops
    n, k = 50_000, 10
    rows, at = static_scene(dev, n)
    d = rows.shape[1]
    db = ops.tile_rows(rows)
    fused = ops.knn_join(db, 0, n, 0, db, n, d, k, None, 0, True)
    assert int((fused[2] < 0).sum()) > 0                              # the fused path flagged rows
    ids, scores, counts = ops.knn_exact(db, 0, n, 0, db, n, d, k, None, 0, True)
    assert int(counts.min()) == k
    at_l = at.tolist()
    for i in at_l[:50] + at_l[-50:] + at_l[2000:2050]:
        assert ids[i].tolist() == [x for x in at_l[:k + 1] if x != i][:k]


def test_knn_agrees_with_the_threshold_joins(dev):
    from revers_o_b200 import ops, synth
    n, d, thr = 20_000, 256, 0.95
    rows = ops.untile_rows(synth.make_selfjoin_db(n, d, 0.05, dev, seed=21), n, d).float().cpu().numpy()
    one = _fill(_db([0], n), "all", rows)
    pairs, ps = one.find_near_duplicates("all", thr)
    pairs = np.asarray(pairs, np.int64)
    deg = np.bincount(pairs.ravel(), minlength=n)
    k = int(deg.max()) + 2
    assert len(pairs) > 200 and k <= 511
    r, s, c = one.knn_join("all", k, thr)
    got = {(i, int(j)): float(x) for i in range(n) for j, x in zip(r[i, :c[i]], s[i, :c[i]])}
    want = {}
    for (a, b), x in zip(pairs.tolist(), ps.tolist()):
        want[a, b] = want[b, a] = x
    for key in set(got) ^ set(want):
        assert abs(got.get(key, want.get(key)) - thr) <= TOL, key
    for key in set(got) & set(want):
        assert abs(got[key] - want[key]) <= TOL
    # cross mode against join_collections
    nl = 12_000
    two = _fill(_fill(_db([0], n), "left", rows[:nl]), "right", rows[nl:])
    jp, js = two.join_collections("left", "right", thr)
    r, s, c = two.knn_join("left", 64, thr, other_collection_name="right")
    assert int(c.max()) < 64
    got = {(i, int(j)): float(x) for i in range(nl) for j, x in zip(r[i, :c[i]], s[i, :c[i]])}
    want = {(int(a), int(b)): float(x) for (a, b), x in zip(jp, js)}
    assert len(want) > 50
    for key in set(got) ^ set(want):
        assert abs(got.get(key, want.get(key)) - thr) <= TOL, key
    for key in set(got) & set(want):
        assert abs(got[key] - want[key]) <= TOL


def assert_same_lists(a, b):
    assert np.array_equal(a[2], b[2]) and np.array_equal(a[0], b[0])
    assert np.allclose(a[1], b[1], atol=1e-6, rtol=0)


@pytest.fixture(scope="module")
def mixed(dev):
    from revers_o_b200 import ops, synth
    n, d = 21_000, 256
    return ops.untile_rows(synth.make_selfjoin_db(n, d, 0.2, dev, seed=31), n, d).float().cpu().numpy()


@pytest.mark.parametrize("layout", mixed_layouts())
def test_sharded_equals_single_device(dev, mixed, layout):
    ld, rd = layout
    nl = 12_000
    one = _fill(_fill(_db([0], len(mixed)), "left", mixed[:nl]), "right", mixed[nl:])
    a = _fill(_db(ld, nl), "left", mixed[:nl])
    b = _fill(_db(rd, len(mixed) - nl), "right", mixed[nl:])
    assert len([s for s in a._coll("left").shards if s.n]) == len(ld)
    for k, thr in ((10, None), (100, 0.3)):
        assert_same_lists(a.knn_join("left", k, thr, "right", other=b), one.knn_join("left", k, thr, "right"))
        assert_same_lists(a.knn_join("left", k, thr), one.knn_join("left", k, thr))


@pytest.mark.parametrize("devices", device_sets())
def test_static_scene_across_shards(dev, devices):
    rows, at = static_scene(dev, 30_000, 5001, 256, seed=8)
    rows = rows.float().cpu().numpy()
    one = _fill(_db([0], len(rows)), "s", rows)
    sh = _fill(_db(devices, len(rows)), "s", rows)
    assert len([s for s in sh._coll("s").shards if s.n]) == len(devices)
    ref = one.knn_join("s", 10)
    got = sh.knn_join("s", 10)
    assert_same_lists(got, ref)
    at_l = at.tolist()
    for i in at_l[:20] + at_l[-20:]:
        assert got[0][i].tolist() == [x for x in at_l[:11] if x != i][:10]


def test_knn_join_interface(dev, tmp_path, mixed):
    from revers_o_b200._lib import RvoError
    from revers_o_b200.vector_db import B200VectorDB, models
    nl = 12_000
    a = _fill(B200VectorDB(path=str(tmp_path / "a"), device=dev), "frames", mixed[:nl], [f"a{i}" for i in range(nl)])
    _fill(B200VectorDB(path=str(tmp_path / "b"), device=dev), "frames", mixed[nl:], [f"b{i}" for i in range(len(mixed) - nl)]).close()
    b = B200VectorDB(path=str(tmp_path / "b"), devices=[0, 0])
    r, s, c = a.knn_join("frames", 5, other_collection_name="frames", other=b)
    assert r.shape == (nl, 5) and r.dtype == np.int64 and s.dtype == np.float32 and c.dtype == np.int32
    sc = mixed[:nl].astype(np.float64) @ mixed[nl:].astype(np.float64).T
    assert np.allclose(s[:, 0], sc.max(1), atol=TOL)
    rs, ss, cs = a.knn_join("frames", 5)                              # self mode
    assert (c == 5).all() and (cs == 5).all() and not (rs == np.arange(nl)[:, None]).any()
    a.recreate_collection("small", vectors_config=models.VectorParams(size=128, distance=models.Distance.COSINE))
    a.upsert_batch("small", ["s0"], np.ones((1, 128), np.float32))
    with pytest.raises(RvoError, match="Wrong input: Vector dimension error: expected dim: 256, got 128"):
        a.knn_join("frames", 5, other_collection_name="small")
    with pytest.raises(RvoError, match="outside 1..511"):
        a.knn_join("frames", 512)
    with pytest.raises(RvoError, match="outside 1..512"):
        a.knn_join("frames", 513, other_collection_name="frames", other=b)
    with pytest.raises(RvoError, match="outside 1..511"):
        a.knn_join("frames", 0)
    assert a.knn_join("small", 3)[2].tolist() == [0]                 # one point: no other point to match
    a.recreate_collection("empty", vectors_config=models.VectorParams(size=256, distance=models.Distance.COSINE))
    r, s, c = a.knn_join("empty", 4, other_collection_name="frames")
    assert r.shape == (0, 4) and c.shape == (0,)
    r, s, c = a.knn_join("frames", 4, other_collection_name="empty")
    assert (c == 0).all() and (r == -1).all() and np.isneginf(s).all() and r.shape == (nl, 4)


def test_find_best_matches(dev, tmp_path):
    from revers_o_b200.core_system import SimpleReverso
    from revers_o_b200.vector_db import mutual_best

    def detector(pil, prompt):
        H, W = pil.height, pil.width
        m = np.zeros((3, H, W), bool)
        m[0, : H // 2, : W // 2] = True
        m[1, H // 4:, W // 3:] = True
        m[2, H // 2:, :] = True
        return Det(mask=m, confidence=np.array([0.9, 0.8, 0.7]), class_id=np.array([0, 0, 0]),
                   xyxy=np.array([[0, 0, W, H]] * 3))

    root = str(tmp_path / "simple_reverso_db")
    r = SimpleReverso(encoder=FakeEncoder(dev), preprocess=preprocess, detector=detector, parity_mode="pooled", db_root=root,
                      device=dev)
    assert r.find_best_matches("b")[0] == "❌ No database loaded. Please create or load a database first."
    fa, fb = tmp_path / "imgs_a", tmp_path / "imgs_b"
    fa.mkdir()
    fb.mkdir()
    for i in range(5):
        make_image(i).save(fa / f"img{i}.png")
    for i in range(3, 8):
        make_image(i).save(fb / f"img{i}.png")
    assert "ready for searching" in r.create_database(folder_path=str(fa), database_name="a", text_prompt="object .")
    assert "ready for searching" in r.create_database(folder_path=str(fb), database_name="b", text_prompt="object .")
    assert r.load_database("a").startswith("✅")
    assert r.find_best_matches("nope")[0].startswith("❌ Database not found")
    assert r.find_best_matches("a")[0].startswith("❌ a is the loaded database")
    assert r.find_best_matches("")[0] == "❌ Please provide a database name"
    text, items = r.find_best_matches("b", 0.0, 1000)
    assert text.startswith("🎯") and items
    # against mutual_best of an fp64 brute force over the stored rows
    from revers_o_b200 import ops
    from revers_o_b200.vector_db import B200VectorDB
    ca = r.vector_db._coll(r.current_database)
    other = B200VectorDB(path=f"{root}/b", device=dev)
    cb = other._coll(other.get_collections().collections[0].name)
    va = ops.untile_rows(ca.vectors, ca.n, ca.dim).double().cpu().numpy()
    vb = ops.untile_rows(cb.vectors, cb.n, cb.dim).double().cpu().numpy()
    sc = va @ vb.T
    ab, ba = sc.argmax(1)[:, None], sc.argmax(0)[:, None]
    pairs, _ = mutual_best(ab, np.ones(len(va)), ba, np.ones(len(vb)), sc.max(1)[:, None].astype(np.float32))
    row_a = {(p["filename"], tuple(p["bbox"])): i for i, p in enumerate(ca.payloads[i] for i in range(ca.n))}
    row_b = {(p["filename"], tuple(p["bbox"])): j for j, p in enumerate(cb.payloads[j] for j in range(cb.n))}
    got = [(row_a[it["filename"], tuple(it["bbox"])], row_b[it["other_filename"], tuple(it["other_bbox"])]) for it in items]
    for (i, j), it in zip(got, items):                                # each is the other's best match, up to TOL
        assert sc[i, j] >= sc[i].max() - TOL and sc[i, j] >= sc[:, j].max() - TOL and abs(it["score"] - sc[i, j]) <= TOL
    top2 = np.sort(sc, 1)[:, -2:], np.sort(sc, 0)[-2:]
    if min((top2[0][:, 1] - top2[0][:, 0]).min(), (top2[1][1] - top2[1][0]).min()) > 1e-4:   # no near ties: exactly the brute force
        assert sorted(got) == sorted(map(tuple, pairs.tolist()))
    # the images both folders hold match themselves, region for region
    shared = {(it["filename"], tuple(it["bbox"])) for it in items if it["filename"] == it["other_filename"]
              and it["bbox"] == it["other_bbox"]}
    assert len(shared) == 6
    other.close()
    assert r.find_best_matches("b", 0.0, 2)[1] == items[:2]
    assert r.find_best_matches("b", 1.01)[0].startswith("❌ No mutual best matches")


def test_block_pipeline_memory_does_not_grow_with_the_collection(dev):
    """The sharded pipeline merges every query block as it goes: small blocks with a tail, and chunked single-shard calls, give
    the one-call result, and the device memory a join takes beyond its reusable buffers does not scale with the left rows."""
    from revers_o_b200 import ops, synth
    from revers_o_b200.sharded import knn_sharded
    n, d, k = 100_000, 128, 200
    db = synth.make_selfjoin_db(n, d, 0.2, dev, seed=41)
    one = [(db, n, 0)]
    half = 50_048                                                      # a whole number of 128-row tiles
    two = [(db[: half // 128], half, 0), (db[half // 128:], n - half, half)]
    ref = knn_sharded(one, one, d, k, None, True, chunk=n)             # one rvo_knn_join call
    assert_same_lists(knn_sharded(one, one, d, k, None, True, chunk=7_000), ref)
    assert_same_lists(knn_sharded(two, two, d, k, None, True, block=1_024), ref)
    knn_sharded(two, two, d, k, None, True)                           # warm-up: workspace and allocator pools
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    assert_same_lists(knn_sharded(two, two, d, k, None, True), ref)
    peak = torch.cuda.max_memory_allocated(dev) - base
    # reusable buffers: ~160 MB at 8192-row blocks; lists for every left row per right shard would be 2 * 12 * n * (k + 1)
    # = 482 MB, plus as much again to merge them
    assert peak < 192 << 20, peak
    with pytest.raises(Exception, match="multiple of 128"):
        knn_sharded(two, two, d, k, None, True, block=1_000)
