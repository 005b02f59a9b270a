"""GPU: the threshold join between two collections.  `rvo_cross_join_threshold` in both orientations equals an fp32 brute force
with bit-identical scores either way; `join_collections` on two halves of one synthetic collection equals the self-join of all
its rows restricted to pairs that straddle the halves, on one device, on row-sharded layouts and with the two sides on
different device lists; a static scene spread over the shards is joined exactly through the overflow protocol; the public
interface (`join_collections`, `SimpleReverso.find_shared_regions`).  On a 1-GPU box the shards are virtual (the same device
listed twice or three times); with two or more GPUs the real devices are used as well."""
from types import SimpleNamespace as NS

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


class FakeEncoder:
    """Deterministic stand-in for pe.CLIP.encode_image: [1,3,H,W] -> [1, 1+24*24, 1024] tokens."""
    def __init__(self, dev):
        g = torch.Generator().manual_seed(0)
        self.w = torch.randn((3, 1024), generator=g).to(dev)

    def encode_image(self, x):
        p = torch.nn.functional.adaptive_avg_pool2d(x.float(), 24).flatten(2).transpose(1, 2)   # [1,576,3]
        t = torch.tanh(p @ self.w + torch.linspace(-1, 1, 1024, device=x.device))
        return torch.cat([t.mean(1, keepdim=True), t], 1)


def preprocess(pil):
    a = np.asarray(pil.resize((336, 336)), dtype=np.float32) / 255.0
    return torch.from_numpy(a).permute(2, 0, 1)


class Det(NS):
    def __len__(self):
        return len(self.mask)


def make_image(seed, size=(96, 80)):
    from PIL import Image
    rs = np.random.RandomState(seed)
    coarse = Image.fromarray((rs.rand(5, 6, 3) * 255).astype(np.uint8))
    img = np.asarray(coarse.resize(size, Image.BILINEAR), dtype=np.float32)
    img += rs.rand(size[1], size[0], 3) * 20
    return Image.fromarray(np.clip(img, 0, 255).astype(np.uint8))


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


def mixed_layouts():
    """(left devices, right devices): one device on both sides, each device set on both sides, and sides on different lists."""
    out = [([0], [0])] + [(s, s) for s in device_sets()] + [([0, 0, 0], [0, 0]), ([0], [0, 0, 0])]
    if torch.cuda.is_available() and torch.cuda.device_count() >= 2:
        g = list(range(min(torch.cuda.device_count(), 8)))
        out += [([0], g), (g[::-1], g), (g[: len(g) // 2], g[len(g) // 2:])]
    return out


def sorted_pairs(pairs, scores):
    """Pairs and scores in (left, right) order, checked free of duplicates: two results are equal iff these arrays are."""
    p = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    s = np.asarray(scores, dtype=np.float32)
    o = np.lexsort((p[:, 1], p[:, 0]))
    p, s = p[o], s[o]
    assert not (len(p) > 1 and ((p[1:] == p[:-1]).all(1)).any()), "duplicate pairs emitted"
    return p, s


def assert_same(a, b):
    (pa, sa), (pb, sb) = sorted_pairs(*a), sorted_pairs(*b)
    assert np.array_equal(pa, pb)
    assert np.array_equal(sa.view(np.uint32), sb.view(np.uint32))          # bit-identical scores


def _db(devices, n):
    from revers_o_b200.vector_db import B200VectorDB
    G = len(devices)
    return B200VectorDB(devices=devices, shard_rows=max(128, -(-n // G // 128) * 128))


def _fill(db, name, rows, ids=None):
    from revers_o_b200.vector_db import models
    db.recreate_collection(name, vectors_config=models.VectorParams(size=rows.shape[1], distance=models.Distance.COSINE))
    ids = list(range(len(rows))) if ids is None else ids
    for lo in range(0, len(rows), 4000):
        db.upsert_batch(name, ids[lo: lo + 4000], rows[lo: lo + 4000], assume_new=True)
    return db


def test_cross_join_entry_both_orientations(dev):
    from revers_o_b200 import ops, synth
    n, d, thr, nl = 12_000, 512, 0.95, 5120
    db = synth.make_selfjoin_db(n, d, 0.3, dev, seed=3)
    L, R = db[: nl // 128].clone(), db[nl // 128:].clone()
    nr = n - nl
    rows = ops.untile_rows(db, n, d).float()
    rl, rr = rows[:nl], rows[nl:]
    off_l, off_r = 0, 100                                            # overlapping id ranges [0, 5120) and [100, 6980)
    sc = rl @ rr.T                                                   # fp32 brute force on the GPU

    def check(got, sc, t0=0):
        want = {(int(i), int(j) + t0 + off_r) for i, j in torch.nonzero(sc >= thr).tolist()}
        near = {(int(i), int(j) + t0 + off_r) for i, j in torch.nonzero((sc - thr).abs() <= 1e-4).tolist()}
        keys = {(int(a), int(b)) for a, b in got[0]}
        assert (keys ^ want) <= near and len(want) > 100
        for (a, b), s in zip(got[0].tolist(), got[1].tolist()):
            assert abs(s - float(sc[a - off_l, b - off_r - t0])) <= 1e-4

    def result(out, lo=0):
        torch.cuda.synchronize()
        m = int(out[2].item())
        assert int(out[3].item()) == 0 and m <= out[0].shape[0]
        return out[0][lo:m].cpu().numpy(), out[1][lo:m].cpu().numpy()

    # left rows as queries, then right rows as queries appended to the same buffer: the same pairs as (left, right)
    out = ops.join_out(1 << 16, dev)
    ops.cross_join_threshold(L, 0, nl, off_l, R, nr, d, thr, off_r, False, 32768, out)
    left_q = result(out)
    m1 = len(left_q[0])
    check(left_q, sc)
    ops.cross_join_threshold(R, 0, nr, off_r, L, nl, d, thr, off_l, True, 32768, out)
    right_q = result(out, m1)
    assert int(out[2].item()) == 2 * m1
    assert np.array_equal(out[0][:m1].cpu().numpy(), left_q[0])     # the pairs already there are untouched
    assert_same(left_q, right_q)                                     # same pairs, bit-identical scores either way
    # a block-aligned target sub-range: right rows [2048, nr)
    sub = ops.join_out(1 << 16, dev)
    ops.cross_join_threshold(L, 0, nl, off_l, R[16:], nr - 2048, d, thr, off_r + 2048, False, 32768, sub)
    got = result(sub)
    check(got, sc[:, 2048:], 2048)
    keep = left_q[0][:, 1] >= off_r + 2048
    assert_same(got, (left_q[0][keep], left_q[1][keep]))
    # qdb == db: the full ordered join of the left rows with themselves, self pairs included
    full = ops.join_out(1 << 17, dev)
    ops.cross_join_threshold(L, 0, nl, 7, L, nl, d, thr, 7, False, 32768, full)
    p, s = result(full)
    got = {(int(a), int(b)): float(x) for (a, b), x in zip(p.tolist(), s.tolist())}
    assert len(got) == len(p) and all((i + 7, i + 7) in got for i in range(nl))
    assert all(got[b, a] == x for (a, b), x in got.items())         # symmetric, bit for bit
    ss = rl @ rl.T
    want = {(int(i) + 7, int(j) + 7) for i, j in torch.nonzero(ss >= thr).tolist()}
    near = {(int(i) + 7, int(j) + 7) for i, j in torch.nonzero((ss - thr).abs() <= 1e-4).tolist()}
    assert (set(got) ^ want) <= near
    # bad arguments are refused
    lib = ops._lib.load()
    ws = ops.workspace(dev, lib.rvo_join_workspace_bytes(d, 32768))
    rc = lib.rvo_cross_join_threshold(L.data_ptr(), 0, nl, 0, R.data_ptr(), nr, d, ops.d_pad_of(d), thr, 0, 2, 32768,
                                      out[0].data_ptr(), out[1].data_ptr(), out[0].shape[0], out[2].data_ptr(),
                                      out[3].data_ptr(), ws.data_ptr(), lib.rvo_join_workspace_bytes(d, 32768),
                                      torch.cuda.current_stream(dev).cuda_stream)
    assert rc != 0 and b"query_is_right" in lib.rvo_last_error()
    with pytest.raises(Exception):
        ops.cross_join_threshold(L, 0, nl, 0, R, nr, d + 64, thr, 0, False, 32768, out)


@pytest.fixture(scope="module")
def halves(dev):
    """21k rows of the configs[4] generator: rows [0, 12000) are the left collection, rows [12000, 21000) the right one, and
    `find_near_duplicates` on one device over all the rows, restricted to i < 12000 <= j, as (i, j - 12000)."""
    from revers_o_b200 import ops, synth
    n, nl, d, thr = 21_000, 12_000, 256, 0.95
    rows = ops.untile_rows(synth.make_selfjoin_db(n, d, 0.05, dev, seed=21), n, d).float().cpu().numpy()
    p, s = _fill(_db([0], n), "all", rows).find_near_duplicates("all", thr)
    p = np.asarray(p, dtype=np.int64)
    keep = (p[:, 0] < nl) & (p[:, 1] >= nl)
    ref = (p[keep] - np.array([0, nl]), s[keep])
    assert len(ref[0]) > 200
    return rows[:nl], rows[nl:], ref, thr


@pytest.mark.parametrize("layout", mixed_layouts())
def test_join_of_two_halves_equals_the_restricted_self_join(dev, halves, layout):
    left_rows, right_rows, ref, thr = halves
    ld, rd = layout
    a = _fill(_db(ld, len(left_rows)), "left", left_rows)
    b = _fill(_db(rd, len(right_rows)), "right", right_rows)
    assert len([s for s in a._coll("left").shards if s.n]) == len(ld)
    assert len([s for s in b._coll("right").shards if s.n]) == len(rd)
    pairs, scores = a.join_collections("left", "right", thr, other=b)
    assert scores.dtype == np.float32
    assert_same((pairs, scores), ref)
    # one B200VectorDB holding both collections gives the same answer
    one = _fill(_fill(_db([0], len(left_rows)), "left", left_rows), "right", right_rows)
    assert_same(one.join_collections("left", "right", thr), ref)
    # the oracle: fp32 dot of the stored rows on the host
    from revers_o_b200 import ops
    c1, c2 = one._coll("left"), one._coll("right")
    sc = ops.untile_rows(c1.vectors, c1.n, c1.dim).float().cpu().numpy() @ ops.untile_rows(c2.vectors, c2.n, c2.dim).float().cpu().numpy().T
    want = set(map(tuple, np.argwhere(sc >= thr).tolist()))
    got = {(int(i), int(j)): float(s) for (i, j), s in zip(pairs, scores)}
    for key in set(got) ^ want:
        assert abs(float(sc[key]) - thr) <= 1e-3, key
    for (i, j), s in got.items():
        assert abs(s - float(sc[i, j])) <= 1e-3


@pytest.mark.parametrize("devices", device_sets())
def test_static_scene_across_shards_is_joined_exactly(dev, devices):
    """1500 exact copies of one row on the left and 2000 on the right, spread over every shard: with 64 candidates per
    sub-list the fixed-capacity join overflows; the join re-runs the affected devices with larger lists and pair buffers and
    returns all 3,000,000 pairs, equal to the single-device result."""
    from revers_o_b200 import ops, synth
    from revers_o_b200.sharded import crossjoin_sharded
    nl, nr, d, thr = 20_000, 24_000, 256, 0.95
    rows = ops.untile_rows(synth.make_selfjoin_db(nl + nr, d, 0.02, dev, seed=9), nl + nr, d).float()
    g = torch.Generator(device=dev).manual_seed(1)
    v = torch.randn(d, generator=g, device=dev)
    v = v / v.norm()
    rows[torch.randperm(nl, generator=g, device=dev)[:1500]] = v
    rows[nl + torch.randperm(nr, generator=g, device=dev)[:2000]] = v
    a = _fill(_db(devices, nl), "left", rows[:nl])
    b = _fill(_db(devices, nr), "right", rows[nl:])
    left = [(s.vectors, s.n, s.row0) for s in a._coll("left").shards if s.n]
    right = [(s.vectors, s.n, s.row0) for s in b._coll("right").shards if s.n]
    assert len(left) == len(right) == len(devices)
    one_l = _fill(_db([0], nl), "left", rows[:nl])._coll("left")
    one_r = _fill(_db([0], nr), "right", rows[nl:])._coll("right")
    out = ops.join_out(1 << 22, dev)
    ops.cross_join_threshold(one_l.vectors, 0, nl, 0, one_r.vectors, nr, d, thr, 0, False, 1024, out)
    torch.cuda.synchronize()
    assert int(out[3].item()) > 0                                    # the small capacity does overflow
    single = crossjoin_sharded([(one_l.vectors, nl, 0)], [(one_r.vectors, nr, 0)], d, thr)
    sharded = crossjoin_sharded(left, right, d, thr, max_pairs=1 << 16, cand_cap=1024)
    pairs, scores = a.join_collections("left", "right", thr, max_pairs=1 << 16, other=b)
    stored = ops.untile_rows(one_l.vectors, nl, d).float() @ v.to(torch.bfloat16).float()
    cl_l = set((stored > 0.999).nonzero().flatten().tolist())
    stored = ops.untile_rows(one_r.vectors, nr, d).float() @ v.to(torch.bfloat16).float()
    cl_r = set((stored > 0.999).nonzero().flatten().tolist())
    assert len(cl_l) == 1500 and len(cl_r) == 2000
    p = single[0]
    assert int((np.isin(p[:, 0], list(cl_l)) & np.isin(p[:, 1], list(cl_r))).sum()) == 3_000_000
    assert_same(sharded, single)
    assert_same((pairs, scores), single)


def test_join_collections_interface(dev, tmp_path, halves):
    from revers_o_b200._lib import RvoError
    from revers_o_b200.vector_db import B200VectorDB, models
    left_rows, right_rows, ref, thr = halves
    a = _fill(B200VectorDB(path=str(tmp_path / "a"), device=dev), "frames", left_rows,
              [f"a{i:05d}" for i in range(len(left_rows))])
    _fill(B200VectorDB(path=str(tmp_path / "b"), device=dev), "frames", right_rows,
          [f"b{i:05d}" for i in range(len(right_rows))]).close()
    b = B200VectorDB(path=str(tmp_path / "b"), devices=[0, 0])   # another instance, loaded from a different path, sharded
    pairs, scores = a.join_collections("frames", "frames", thr, other=b)
    assert all(x.startswith("a") and y.startswith("b") for x, y in pairs)     # left id first
    assert_same(([(int(x[1:]), int(y[1:])) for x, y in pairs], scores), ref)
    pairs2, scores2 = b.join_collections("frames", "frames", thr, other=a)     # the other way round: (b id, a id)
    assert sorted((y, x) for x, y in pairs2) == sorted(pairs)
    # a dimension mismatch, and a collection joined with itself, raise
    a.recreate_collection("small", vectors_config=models.VectorParams(size=128, distance=models.Distance.COSINE))
    a.upsert_batch("small", ["s0"], np.ones((1, 128), np.float32))
    with pytest.raises(RvoError, match="Wrong input: Vector dimension error: expected dim: 256, got 128"):
        a.join_collections("frames", "small")
    with pytest.raises(RvoError, match="find_near_duplicates"):
        a.join_collections("frames", "frames")
    # an empty side
    a.recreate_collection("empty", vectors_config=models.VectorParams(size=256, distance=models.Distance.COSINE))
    for args in (("frames", "empty"), ("empty", "frames")):
        p, s = a.join_collections(*args, threshold=thr)
        assert p == [] and s.dtype == np.float32 and s.shape == (0,)


def test_find_shared_regions(dev, tmp_path):
    from revers_o_b200.core_system import SimpleReverso

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
    assert r.find_shared_regions("b")[0] == "❌ No database loaded. Please create or load a database first."
    folder = tmp_path / "imgs"
    folder.mkdir()
    for i in range(5):
        make_image(i).save(folder / f"img{i}.png")
    for name in ("a", "b"):
        assert "ready for searching" in r.create_database(folder_path=str(folder), database_name=name, text_prompt="object .")
    assert r.load_database("a").startswith("✅")
    assert r.find_shared_regions("nope")[0].startswith("❌ Database not found")
    text, items = r.find_shared_regions("b", 0.999, 1000)
    assert text.startswith("🎯") and items
    assert all(x["score"] >= y["score"] for x, y in zip(items, items[1:]))
    regions = {(p["filename"], tuple(p["bbox"])) for p in r.vector_db._coll(r.current_database).payloads}
    assert len(regions) == 15
    found = {(it["filename"], tuple(it["bbox"])) for it in items
             if (it["other_filename"], tuple(it["other_bbox"])) == (it["filename"], tuple(it["bbox"])) and it["score"] >= 0.999}
    assert found == regions                                          # every region is found in the other database
    top = r.find_shared_regions("b", 0.999, 3)[1]
    assert top == items[:3]
    assert r.find_shared_regions("b", 1.01)[0].startswith("❌ No shared regions")
