"""GPU: spherical k-means.  `rvo_kmeans_update` / `rvo_kmeans_finalize` against a numpy int64 restatement, bit for bit; one
assignment against an fp64 brute force over the stored bf16 values; planted clusters recovered exactly, deterministically and
equal to a numpy restatement of the loop; bit-identical results on row-sharded layouts (virtual shards on a 1-GPU box, the real
devices as well with two or more); a static scene through tied centroids, empty clusters, re-seeding and the kNN overflow
route; the public interface (`B200VectorDB.cluster`, `SimpleReverso.find_visual_themes`)."""
import numpy as np
import pytest
import torch

from test_gpu_crossjoin import FakeEncoder, Det, _db, _fill, device_sets, make_image, preprocess
from test_gpu_knn_join import static_scene

pytestmark = pytest.mark.gpu
TOL = 1e-5


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    return torch.device("cuda:0")


def fixed(x):
    """bf16 values (any float array) -> the int64 fixed point of the update, rint(x * 2^31)."""
    return np.rint(np.asarray(x, np.float64) * 2.0 ** 31).astype(np.int64)


def within_one_ulp(got, ref):
    """Every bf16 value of `got` within one bf16 ulp (at the magnitude of the exact value) of the fp64 `ref`."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    e = np.floor(np.log2(np.maximum(np.abs(ref), 2.0 ** -126)))
    return bool((np.abs(got - ref) <= 2.0 ** (e - 7)).all())


def normalise_bf16(s):
    """fp64 normalisation of integer sums [C, d] rounded to bf16, as float64."""
    f = s.astype(np.float64)
    f = f / np.linalg.norm(f, axis=1, keepdims=True)
    return torch.from_numpy(f).to(torch.bfloat16).double().numpy()


def argmax_ok(labels, sc):
    """labels [n] against fp64 scores sc [n, C]: the first index of the maximum, except for rows whose best two scores lie
    within TOL (then any index within TOL of the maximum)."""
    best = sc.max(1)
    first = sc.argmax(1)
    near = (sc >= best[:, None] - TOL).sum(1) > 1
    ok = labels == first
    ok[near] = sc[np.flatnonzero(near), labels[near]] >= best[near] - TOL
    return bool(ok.all()), int(near.sum())


@pytest.mark.parametrize("d", [256, 1024, 1280, 2304])
@pytest.mark.parametrize("C", [1, 2, 1000])
def test_update_entry_against_numpy(dev, d, C):
    from revers_o_b200 import ops, synth
    n_all, lo = 3077, 77
    n = n_all - lo                                                    # 3000 rows starting inside a 128-row block
    db = synth.make_selfjoin_db(n_all, d, 0.1, dev, seed=d + C)
    X = ops.untile_rows(db, n_all, d).double().cpu().numpy()[lo:]
    rs = np.random.RandomState(C)
    lab = rs.randint(0, C, size=n)
    lab[rs.choice(n, 5, replace=False)] = -1                           # rows with no assignment add nothing
    off = 7
    ids = torch.from_numpy(np.where(lab >= 0, lab + off, -1)).to(dev)
    prev = torch.from_numpy(rs.randint(0, C, size=n).astype(np.int32)).to(dev)
    labels = torch.empty(n, dtype=torch.int32, device=dev)
    sums = torch.zeros((C, d), dtype=torch.int64, device=dev)
    counts = torch.zeros(C, dtype=torch.int64, device=dev)
    changed = torch.zeros(1, dtype=torch.int64, device=dev)
    ops.kmeans_update(db, lo, n_all, d, ids, C, prev, labels, sums, counts, changed, id_offset=off)
    want = np.zeros((C, d), np.int64)
    keep = lab >= 0
    np.add.at(want, lab[keep], fixed(X[keep]))
    assert np.array_equal(labels.cpu().numpy(), lab)
    assert np.array_equal(sums.cpu().numpy(), want)
    assert np.array_equal(counts.cpu().numpy(), np.bincount(lab[keep], minlength=C))
    assert int(changed.item()) == int((lab != prev.cpu().numpy()).sum())
    # the same rows in two calls (two shards) add up to the same sums, bit for bit
    s2, c2, ch2 = torch.zeros_like(sums), torch.zeros_like(counts), torch.zeros_like(changed)
    mid = 1500
    ops.kmeans_update(db, lo, lo + mid, d, ids[:mid], C, None, labels[:mid], s2, c2, ch2, id_offset=off)
    ops.kmeans_update(db, lo + mid, n_all, d, ids[mid:], C, None, labels[mid:], s2, c2, ch2, id_offset=off)
    assert torch.equal(s2, sums) and torch.equal(c2, counts) and int(ch2.item()) == n
    # finalisation: within one bf16 ulp of the fp64 normalised sums; empty clusters flagged
    cent = ops.db_alloc(C, d, dev)
    empty = torch.zeros(C, dtype=torch.int32, device=dev)
    n_empty = torch.zeros(1, dtype=torch.int64, device=dev)
    ops.kmeans_finalize(sums, counts, d, cent, empty, n_empty)
    got = ops.untile_rows(cent, C, d).double().cpu().numpy()
    cnt = np.bincount(lab[keep], minlength=C)
    live = cnt > 0
    f = want[live].astype(np.float64)
    assert within_one_ulp(got[live], f / np.linalg.norm(f, axis=1, keepdims=True))
    assert np.array_equal(empty.cpu().numpy(), (~live).astype(np.int32))
    assert int(n_empty.item()) == int((~live).sum()) and (not got[~live].any())
    if C == 1000:
        assert (~live).any()


@pytest.mark.parametrize("d", [256, 1024])
def test_one_assignment_against_brute_force(dev, d):
    from revers_o_b200 import ops, synth
    n, C = 20_003, 300
    db = synth.make_selfjoin_db(n, d, 0.05, dev, seed=5)
    X = ops.untile_rows(db, n, d)
    init = torch.randn((C, d), generator=torch.Generator(device=dev).manual_seed(2), device=dev)
    cent = ops.db_alloc(C, d, dev)
    ops.normalize_rows(init, db=cent, row0=0)
    r = ops.kmeans_exact(db, n, d, cent, C, max_iter=0)
    assert r.iterations == 0 and not r.converged
    assert torch.equal(ops.untile_rows(r.centroids, C, d), ops.untile_rows(cent, C, d))   # the initial centroids
    sc = (X.double() @ ops.untile_rows(cent, C, d).double().T).cpu().numpy()
    ok, _ = argmax_ok(r.labels.astype(np.int64), sc)
    assert ok
    assert np.abs(r.scores - sc.max(1)).max() <= TOL
    assert np.array_equal(r.sizes, np.bincount(r.labels, minlength=C))


def planted(dev, C=12, per=400, d=256, seed=0):
    """C random directions, `per` members each at cos ~0.8 from their direction, in shuffled row order.  Returns (stored rows
    as bf16 [n, d] on dev, planted label per row)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    dirs = torch.randn((C, d), generator=g, device=dev)
    dirs = dirs / dirs.norm(dim=1, keepdim=True)
    lab = torch.arange(C, device=dev).repeat_interleave(per)
    noise = torch.randn((C * per, d), generator=g, device=dev)
    noise = noise / noise.norm(dim=1, keepdim=True)
    x = 0.8 * dirs[lab] + 0.6 * noise
    x = x / x.norm(dim=1, keepdim=True)
    p = torch.randperm(C * per, generator=g, device=dev)
    return x[p].to(torch.bfloat16), lab[p].cpu().numpy()


def numpy_kmeans(X, init, max_iter):
    """The loop restated in numpy: fp64 argmax assignment, int64 fixed-point sums, fp64 normalisation rounded to bf16."""
    Xi = fixed(X)
    cent, prev, it = init, None, 0
    while True:
        sc = X @ cent.T
        lab = sc.argmax(1)
        if prev is not None and (lab == prev).all():
            return lab, cent, it, True
        if it == max_iter:
            return lab, cent, it, False
        sums = np.zeros((len(cent), X.shape[1]), np.int64)
        np.add.at(sums, lab, Xi)
        assert (np.bincount(lab, minlength=len(cent)) > 0).all()
        cent, prev, it = normalise_bf16(sums), lab, it + 1


def test_planted_clusters_converge_deterministically(dev):
    from revers_o_b200 import ops
    C, d = 12, 256
    x, truth = planted(dev, C, 400, d)
    n = len(truth)
    db = ops.tile_rows(x)
    X = ops.untile_rows(db, n, d).double().cpu().numpy()
    first = [int(np.flatnonzero(truth == c)[0]) for c in range(C)]     # one member of each planted cluster
    from revers_o_b200.sharded import gather_rows
    cent = gather_rows([(db, n, 0)], first, d, dev)
    r = ops.kmeans_exact(db, n, d, cent, C, max_iter=50)
    assert r.converged and r.iterations < 50
    # the planted partition, up to renumbering
    pairs = set(zip(r.labels.tolist(), truth.tolist()))
    assert len(pairs) == C and len({a for a, _ in pairs}) == C
    r2 = ops.kmeans_exact(db, n, d, cent, C, max_iter=50)
    assert np.array_equal(r.labels, r2.labels) and np.array_equal(r.scores.view(np.uint32), r2.scores.view(np.uint32))
    assert torch.equal(r.centroids, r2.centroids) and r.iterations == r2.iterations
    lab, ncent, it, conv = numpy_kmeans(X, ops.untile_rows(cent, C, d).double().cpu().numpy(), 50)
    assert np.array_equal(r.labels, lab) and it == r.iterations and conv
    assert within_one_ulp(ops.untile_rows(r.centroids, C, d).double().cpu().numpy(), ncent)
    assert np.array_equal(r.sizes, np.bincount(lab, minlength=C))


def assert_same_clusters(a, b):
    assert np.array_equal(a.labels, b.labels)
    assert np.array_equal(a.scores.view(np.uint32), b.scores.view(np.uint32))
    assert np.array_equal(a.centroids.view(np.uint32), b.centroids.view(np.uint32))
    assert np.array_equal(a.sizes, b.sizes)
    assert a.iterations == b.iterations and a.converged == b.converged


def layouts():
    """(devices, shard_rows or None for an even split): virtual shards, an uneven split, the real devices."""
    return [(s, None) for s in device_sets()] + [([0, 0, 0], 128 * 12)]


def _sharded_db(devices, n, shard_rows):
    from revers_o_b200.vector_db import B200VectorDB
    return _db(devices, n) if shard_rows is None else B200VectorDB(devices=devices, shard_rows=shard_rows)


@pytest.fixture(scope="module")
def mixed(dev):
    from revers_o_b200 import ops, synth
    n, d = 9_001, 256
    return ops.untile_rows(synth.make_selfjoin_db(n, d, 0.1, dev, seed=41), n, d).float().cpu().numpy()


@pytest.mark.parametrize("layout", layouts())
def test_layout_invariance(dev, mixed, layout):
    devices, shard_rows = layout
    one = _fill(_db([0], len(mixed)), "m", mixed)
    sh = _fill(_sharded_db(devices, len(mixed), shard_rows), "m", mixed)
    assert len([s for s in sh._coll("m").shards if s.n]) == len(devices)
    for C, it in ((64, 8), (7, 30)):
        ref = one.cluster("m", C, max_iter=it, seed=3)
        assert ref.iterations >= 2
        assert_same_clusters(sh.cluster("m", C, max_iter=it, seed=3), ref)


@pytest.fixture
def small_candidate_lists():
    """Candidate lists of 64 per sub-list (option "cand_cap"), so that a few hundred tied centroids overflow the fused path."""
    from revers_o_b200 import _lib
    _lib.set_option("cand_cap", 64)
    yield
    _lib.set_option("cand_cap", 32768)


def test_static_scene(dev, small_candidate_lists):
    """5001 exact copies of one row among 20k rows, and initial centroids that hold the static row 3000 times: the copies tie
    on 3000 centroids (with small candidate lists the kNN's fused path overflows on them and the rows take the exact fp32
    route), the higher-index copies lose every tie and are re-seeded."""
    from revers_o_b200 import ops
    n, m, C = 20_000, 5001, 4000
    rows, at = static_scene(dev, n, m, 256, seed=11)
    d = rows.shape[1]
    db = ops.tile_rows(rows)
    X = ops.untile_rows(db, n, d)
    init = X[torch.randperm(n, generator=torch.Generator(device=dev).manual_seed(1), device=dev)[:C]].float()
    idx = torch.arange(C, device=dev)
    init[idx[idx % 4 != 0]] = X[at[0]].float()                          # 3000 copies of the static row
    cent = ops.db_alloc(C, d, dev)
    ops.normalize_rows(init.contiguous(), db=cent, row0=0)
    fused = ops.knn_join(db, 0, n, 0, cent, C, d, 1, None, 0, False)
    n_flagged = int((fused[2] < 0).sum())
    r = ops.kmeans_exact(db, n, d, cent, C, max_iter=6)
    sc = (X.double() @ ops.untile_rows(r.centroids, C, d).double().T).cpu().numpy()
    ok, _ = argmax_ok(r.labels.astype(np.int64), sc)
    assert ok
    assert np.abs(r.scores - sc.max(1)).max() <= TOL
    assert np.array_equal(r.sizes, np.bincount(r.labels, minlength=C))
    lab_at = np.unique(r.labels[at.cpu().numpy()])
    assert len(lab_at) == 1                                            # every copy in one cluster: the lowest tied index
    tied = np.flatnonzero(sc[int(at[0])] >= sc[int(at[0])].max() - TOL)
    assert lab_at[0] == tied[0]
    print(f"static scene: {n_flagged} rows flagged by the fused path, {r.iterations} iterations, "
          f"{int((r.sizes == 0).sum())} empty clusters at the end")
    # the public result on sharded layouts equals one device, in cluster_order's numbering
    rows_np = X.float().cpu().numpy()
    ref = _fill(_db([0], n), "s", rows_np).cluster("s", C, max_iter=4)
    assert (np.diff(ref.sizes) <= 0).all() and np.array_equal(ref.sizes, np.bincount(ref.labels, minlength=C))
    for devices in device_sets():
        assert_same_clusters(_fill(_db(devices, n), "s", rows_np).cluster("s", C, max_iter=4), ref)
    assert n_flagged > 0


def test_cluster_interface(dev, mixed):
    from revers_o_b200._lib import RvoError
    from revers_o_b200.vector_db import models
    db = _fill(_db([0], len(mixed)), "m", mixed)
    c = db._coll("m")
    X = ops_rows(c)
    for kw, msg in ((dict(n_clusters=0), "n_clusters"), (dict(n_clusters=len(mixed) + 1), "n_clusters"),
                    (dict(n_clusters=4, max_iter=-1), "max_iter"), (dict(n_clusters=4, init=np.ones((3, 256))), "shape"),
                    (dict(n_clusters=2, init=np.zeros((2, 256))), "zero")):
        with pytest.raises(RvoError, match=msg):
            db.cluster("m", **kw)
    with pytest.raises(RvoError, match="not found"):
        db.cluster("nope", 3)
    db.recreate_collection("empty", vectors_config=models.VectorParams(size=256, distance=models.Distance.COSINE))
    with pytest.raises(RvoError, match="empty"):
        db.cluster("empty", 1)
    # max_iter = 0: the assignment to the given init, renumbered
    init = np.random.RandomState(0).randn(16, 256).astype(np.float32)
    r = db.cluster("m", 16, max_iter=0, init=init)
    assert r.iterations == 0 and not r.converged
    assert r.labels.dtype == np.int32 and r.scores.dtype == np.float32 and r.centroids.dtype == np.float32
    assert r.sizes.dtype == np.int64 and r.centroids.shape == (16, 256)
    sc = X @ r.centroids.astype(np.float64).T
    assert np.abs(r.scores - sc.max(1)).max() <= TOL
    assert (sc[np.arange(len(X)), r.labels] >= sc.max(1) - TOL).all()
    assert np.array_equal(r.sizes, np.bincount(r.labels, minlength=16)) and (np.diff(r.sizes) <= 0).all()
    # the default initialisation: the rows numpy's default_rng(seed) picks, bit for bit
    r0 = db.cluster("m", 5, max_iter=0, seed=9)
    pick = X[np.random.default_rng(9).choice(len(X), 5, replace=False)]
    assert sorted(map(tuple, r0.centroids.tolist())) == sorted(map(tuple, pick.astype(np.float32).tolist()))
    full = db.cluster("m", 5, seed=9)
    assert full.iterations >= 1 and (full.converged or full.iterations == 50)


def ops_rows(c):
    from revers_o_b200 import ops
    return ops.untile_rows(c.vectors, c.n, c.dim).double().cpu().numpy()


def test_find_visual_themes(dev, tmp_path):
    from revers_o_b200.core_system import SimpleReverso

    def detector(pil, prompt):
        H, W = pil.height, pil.width
        m = np.zeros((3, H, W), bool)
        m[0, : H // 2, : W // 2] = True
        m[1, H // 4:, W // 3:] = True
        m[2, H // 2:, :] = True
        return Det(mask=m, confidence=np.array([0.9, 0.8, 0.7]), class_id=np.array([0, 0, 0]),
                   xyxy=np.array([[0, 0, W, H]] * 3))

    r = SimpleReverso(encoder=FakeEncoder(dev), preprocess=preprocess, detector=detector, parity_mode="pooled",
                      db_root=str(tmp_path / "simple_reverso_db"), device=dev)
    assert r.find_visual_themes()[0] == "❌ No database loaded. Please create or load a database first."
    folder = tmp_path / "imgs"
    folder.mkdir()
    for i in range(6):
        make_image(i).save(folder / f"img{i}.png")
    assert "ready for searching" in r.create_database(folder_path=str(folder), database_name="a", text_prompt="object .")
    assert r.load_database("a").startswith("✅")
    text, items = r.find_visual_themes(n_themes=4, max_themes=3, examples=2)
    assert text.startswith("🎯") and 1 <= len(items) <= 3
    assert all(x["size"] >= y["size"] for x, y in zip(items, items[1:]))
    for it in items:
        assert it["images"] == sorted(set(it["images"])) and 1 <= len(it["examples"]) <= 2
        assert all(e["filename"] in it["images"] for e in it["examples"])
        assert all(x["score"] >= y["score"] for x, y in zip(it["examples"], it["examples"][1:]))
    _, all_items = r.find_visual_themes(n_themes=100, max_themes=100, examples=100)   # more themes than regions: one each
    assert sum(it["size"] for it in all_items) == 18 and len(all_items) <= 18
