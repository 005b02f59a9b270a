"""GPU: duplicate groups — the connected components of the self-join's pairs, unioned on the device while the join runs.
The labels equal the components of `find_near_duplicates`'s pairs exactly, on several shapes, on long chains whose hooks race,
on a static scene through the candidate-overflow retry, when disjoint query ranges are folded together with
`rvo_components_merge`, and on row-sharded collections; the public interface (`B200VectorDB.find_duplicate_groups`,
`SimpleReverso.find_recurring_regions`).  On a 1-GPU box the shards are virtual (the same device listed twice or three
times); with two or more GPUs the real devices are used as well."""
import uuid

import numpy as np
import pytest
import torch
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from test_gpu_crossjoin import Det, FakeEncoder, device_sets, make_image, preprocess

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    return torch.device("cuda:0")


def scipy_labels(pairs, n):
    """Components of the graph on n rows with the given edges, each row labelled with its component's smallest row."""
    pairs = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    g = coo_matrix((np.ones(len(pairs), np.int8), (pairs[:, 0], pairs[:, 1])), shape=(n, n))
    _, comp = connected_components(g, directed=False)
    smallest = np.full(comp.max() + 1, n, np.int64)
    np.minimum.at(smallest, comp, np.arange(n))
    return smallest[comp]


@pytest.mark.parametrize("n,d", [(20_000, 256), (9000, 1024), (5000, 1280)])
def test_labels_are_the_components_of_the_pair_join(dev, n, d):
    from revers_o_b200 import ops, synth
    thr = 0.95
    db = synth.make_selfjoin_db(n, d, 0.2, dev, seed=n + d)
    pairs, _ = ops.selfjoin_exact(db, n, d, thr)
    labels, n_pairs = ops.components_exact(db, n, d, thr)
    assert labels.dtype == np.int64 and labels.shape == (n,)
    assert n_pairs == len(pairs) > 100
    ref = scipy_labels(pairs, n)
    assert np.array_equal(labels, ref)
    assert len(np.unique(labels)) < n - 100                        # many rows are grouped
    # ids = row + id_offset: the same components, labelled with the smallest id
    labels_off, m = ops.components_exact(db, n, d, thr, id_offset=1000)
    assert m == n_pairs and np.array_equal(labels_off, ref + 1000)


def _chain(rs, m, d, a):
    """Random walk r_{k+1} = a r_k + sqrt(1 - a^2) n_k, n_k a random unit vector orthogonal to r_k: neighbours at cos a, rows
    k apart near a^k, so at threshold 0.95 the chain is a path, not a clique."""
    r = rs.standard_normal(d)
    r /= np.linalg.norm(r)
    out = [r]
    for _ in range(m - 1):
        nk = rs.standard_normal(d)
        nk -= (nk @ r) * r
        nk /= np.linalg.norm(nk)
        r = a * r + np.sqrt(1 - a * a) * nk
        r /= np.linalg.norm(r)
        out.append(r)
    return np.stack(out)


def test_long_chains_in_shuffled_order(dev):
    """Two chains of 1200 and 1000 rows scattered among 3000 random rows: every hook of a chain races with the others, and the
    components must still be exactly the two chains."""
    from revers_o_b200 import ops
    d, thr = 512, 0.95
    rs = np.random.RandomState(7)
    c1, c2 = _chain(rs, 1200, d, 0.965), _chain(rs, 1000, d, 0.965)
    noise = rs.standard_normal((3000, d))
    noise /= np.linalg.norm(noise, axis=1, keepdims=True)
    x = np.concatenate([c1, c2, noise])
    n = len(x)
    perm = rs.permutation(n)                                       # stored row r holds x[perm[r]]
    db = ops.tile_rows(torch.from_numpy(x[perm]).float().to(dev).to(torch.bfloat16))
    rows = ops.untile_rows(db, n, d).float()
    sc = rows @ rows.T                                             # fp32 brute force over the stored bf16 rows
    sc.fill_diagonal_(-1.0)
    assert float((sc - thr).abs().min()) >= 1e-3                   # no score the two summation orders could split
    edges = torch.nonzero(torch.triu(sc >= thr, 1)).cpu().numpy()
    assert len(edges) == 1199 + 999                                # the chains' path edges, nothing else
    labels, n_pairs = ops.components_exact(db, n, d, thr)
    assert n_pairs == len(edges)
    assert np.array_equal(labels, scipy_labels(edges, n))
    where = np.argsort(perm)                                       # x row -> stored row
    groups = {}
    for r, lab in enumerate(labels):
        groups.setdefault(int(lab), []).append(r)
    big = sorted((g for g in groups.values() if len(g) > 1), key=len, reverse=True)
    assert [sorted(g) for g in big] == [sorted(where[:1200].tolist()), sorted(where[1200:2200].tolist())]


def test_static_scene_through_the_overflow_retry(dev):
    """Row 0 and 5000 exact copies: about 12.5M pairs, more than find_near_duplicates' default pair buffer.  With 1024
    candidates per query row the first join overflows and is re-run with larger lists, keeping the forest."""
    from revers_o_b200 import ops, synth
    n, d, thr, cl = 20_000, 256, 0.95, 5000
    db = synth.make_selfjoin_db(n, d, 0.05, dev, seed=11, cluster=cl)
    out = ops.components_out(n, dev)
    ops.join_components(db, 0, n, 0, db, n, d, thr, 0, 1024, out)
    torch.cuda.synchronize()
    assert int(out[2].item()) > 0                                  # the small capacity does overflow
    labels, n_pairs = ops.components_exact(db, n, d, thr, cand_cap=1024)
    pairs, _ = ops.selfjoin_exact(db, n, d, thr)
    assert len(pairs) > (1 << 22) and n_pairs == len(pairs)
    assert np.array_equal(labels, scipy_labels(pairs, n))
    rows = ops.untile_rows(db, n, d).float()
    scene = (rows @ rows[0] > 0.999).nonzero().flatten().cpu().numpy()
    assert len(scene) >= cl + 1 and np.all(labels[scene] == 0)


def test_merge_folds_forests_of_disjoint_query_ranges(dev):
    """The cross-device merge on one GPU: three disjoint query ranges of one collection into three forests, flattened and
    merged into the first; the labels are those of the full join, which none of the forests has alone."""
    from revers_o_b200 import ops, synth
    n, d, thr = 20_000, 256, 0.95
    db = synth.make_selfjoin_db(n, d, 0.3, dev, seed=21)
    full, n_pairs = ops.components_exact(db, n, d, thr)
    bounds = [0, 4096, 12_288, n]
    forests = []
    for lo, hi in zip(bounds, bounds[1:]):
        out = ops.components_out(n, dev)
        ops.join_components(db, lo, hi, 0, db, n, d, thr, 0, 32768, out)
        forests.append(out)
    torch.cuda.synchronize()
    assert sum(int(o[1].item()) for o in forests) == n_pairs and all(int(o[2].item()) == 0 for o in forests)
    for o in forests:
        assert not np.array_equal(ops.components_flatten(o[0]).cpu().numpy(), full)
    root = forests[0][0]
    for o in forests[1:]:
        ops.components_merge(root, ops.components_flatten(o[0]))
    assert np.array_equal(ops.components_flatten(root).cpu().numpy().astype(np.int64), full)


def _ingest(db, name, ids, rows, batch=5000):
    from revers_o_b200.vector_db import models
    db.recreate_collection(name, vectors_config=models.VectorParams(size=rows.shape[1], distance=models.Distance.COSINE))
    for lo in range(0, len(rows), batch):
        db.upsert_batch(name, list(ids[lo: lo + batch]), rows[lo: lo + batch], assume_new=True)


@pytest.mark.parametrize("devices", device_sets())
def test_sharded_groups_equal_single_device_groups(dev, tmp_path, devices):
    from revers_o_b200 import ops, synth
    from revers_o_b200.sharded import components_sharded, shard_bounds
    from revers_o_b200.vector_db import B200VectorDB
    n, d, thr = 20_000, 256, 0.95
    rows = ops.untile_rows(synth.make_selfjoin_db(n, d, 0.3, dev, seed=5), n, d).float().cpu().numpy()
    path = str(tmp_path / "db")
    one = B200VectorDB(path=path, device=dev)
    _ingest(one, "frames", range(n), rows)
    many = B200VectorDB(path=path, devices=devices)                # loaded from disk: split evenly, whole 128-row blocks
    assert len([s for s in many._coll("frames").shards if s.n]) == len(devices)
    g1 = one.find_duplicate_groups("frames", thr, min_size=1)
    gn = many.find_duplicate_groups("frames", thr, min_size=1)
    assert gn == g1 and sum(len(g) for g in g1) == n and len(g1[0]) > 2
    # a static scene spread over every shard, through the per-device overflow retry (the forests are kept across it)
    db = synth.make_selfjoin_db(60_000, d, 0.02, dev, seed=9, cluster=3000)
    shards = []
    for g, dv in enumerate(devices):
        lo, hi = shard_bounds(60_000, len(devices), g)
        shards.append((db[lo // 128: (hi + 127) // 128].clone().to(torch.device("cuda", dv)), hi - lo, lo))
    labels, n_pairs = components_sharded(shards, d, thr, cand_cap=1024)
    ref, m = ops.components_exact(db, 60_000, d, thr)
    assert n_pairs == m > 3001 * 3000 // 2 and np.array_equal(labels, ref)


def _group_rows(d, rs):
    """12 rows: rows {1, 5, 9} are one point, {2, 7} another, {3, 10} a third, the rest are unrelated."""
    x = rs.standard_normal((12, d)).astype(np.float32)
    x[5] = x[9] = x[1]
    x[7] = x[2]
    x[10] = x[3]
    return x


@pytest.mark.parametrize("kind", ["int", "uuid"])
def test_find_duplicate_groups(dev, kind):
    from revers_o_b200.vector_db import B200VectorDB, models
    d = 256
    rows = _group_rows(d, np.random.RandomState(3))
    ids = [1000 - 7 * i for i in range(12)] if kind == "int" else [str(uuid.UUID(int=(i * 7919) % 97)) for i in range(12)]
    db = B200VectorDB(device=dev)
    _ingest(db, "frames", ids, rows)
    want = [[1, 5, 9], [2, 7], [3, 10]]                            # largest first, equal sizes by their smallest row
    assert db.find_duplicate_groups("frames", 0.99) == [[ids[r] for r in g] for g in want]
    assert db.find_duplicate_groups("frames", 0.99, min_size=3) == [[ids[r] for r in want[0]]]
    singles = db.find_duplicate_groups("frames", 0.99, min_size=1)
    assert singles[:3] == [[ids[r] for r in g] for g in want]
    assert singles[3:] == [[ids[r]] for r in (0, 4, 6, 8, 11)]
    assert db.find_duplicate_groups("frames", 1.01) == []          # above every score: no pair, no group
    db.recreate_collection("empty", vectors_config=models.VectorParams(size=d, distance=models.Distance.COSINE))
    assert db.find_duplicate_groups("empty") == []
    db.upsert_batch("empty", [ids[0]], rows[:1])
    assert db.find_duplicate_groups("empty", min_size=1) == []     # a single row
    # the same rows first in a row-sharded collection (shards of 128 and 84 rows, as incremental ingest fills them)
    many = B200VectorDB(devices=[0, 0], shard_rows=128)
    more = np.random.RandomState(4).standard_normal((200, d)).astype(np.float32)
    _ingest(many, "frames", ids + [f"r{i}" for i in range(200)], np.concatenate([rows, more]), batch=64)
    assert len([s for s in many._coll("frames").shards if s.n]) == 2
    assert many.find_duplicate_groups("frames", 0.99) == [[ids[r] for r in g] for g in want]


def test_find_recurring_regions(dev, tmp_path):
    from revers_o_b200 import ops
    from revers_o_b200.core_system import SimpleReverso
    from revers_o_b200.vector_db import group_labels

    def detector(pil, prompt):                                       # three regions with distinct boxes
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
    assert r.find_recurring_regions() == ("❌ No database loaded. Please create or load a database first.", [])
    folder = tmp_path / "imgs"
    folder.mkdir()
    for i in range(4):
        make_image(i).save(folder / f"img{i}.png")
    make_image(2).save(folder / "img2_copy.png")                    # the same picture twice: its three regions recur
    assert "ready for searching" in r.create_database(folder_path=str(folder), database_name="a", text_prompt="object .")
    assert r.load_database("a").startswith("✅")
    thr = 0.999
    text, groups = r.find_recurring_regions(thr, max_groups=1000)
    assert text.startswith("🎯") and groups
    # the groups are the components of the pair join's edges, as (filename, bbox) of their regions in row order
    c = r.vector_db._coll(r.current_database)
    pairs, _ = ops.selfjoin_exact(c.vectors, c.n, c.dim, thr)
    pay = [c.payloads[i] or {} for i in range(c.n)]
    want = [[(pay[i]["filename"], tuple(pay[i]["bbox"])) for i in g] for g in group_labels(scipy_labels(pairs, c.n))]
    assert [[(m["filename"], tuple(m["bbox"])) for m in g["members"]] for g in groups] == want
    assert [g["size"] for g in groups] == [len(g) for g in want]
    # every region of the copied picture is in one group with its copy
    for g in want:
        regions = set(g)
        for f, box in g:
            if f == "img2.png":
                assert ("img2_copy.png", box) in regions
    assert sum(f == "img2.png" for g in want for f, _ in g) == 3
    assert r.find_recurring_regions(thr, max_groups=1)[1] == groups[:1]
    assert r.find_recurring_regions(1.01)[0].startswith("❌ No recurring regions found")
