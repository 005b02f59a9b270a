"""The reference's OWN code through the boundary (VERDICT r1 item 2) — the strongest parity evidence this image allows.

  CPU (here, every round)
    * the committed trace (tests/golden/reference_trace.*) is what the UNMODIFIED /root/reference/core_system.py + ui.py produce
      today (re-run when the reference is present), and
    * the vectors the reference itself computed and upserted equal the oracle's restatement of core_system.py:345-349,363,
      398-408,447 — i.e. the oracle's embedding half is PINNED to outputs of the reference run here.
  GPU (-m gpu)
    * replay: every vector-DB call the reference made (recreate_collection / upsert / search, byte for byte the recorded
      arguments) goes to B200VectorDB; hits must equal what the reference got back (ids up to 1e-3 ties, scores within 1e-3);
    * drop-in: `revers_o_b200.core_system.SimpleReverso()` — the NO-ARGUMENT constructor ui.py:20 uses, encoder and detector
      loaded lazily through the reference's own imports — driven through the same scenario returns the same texts and hits;
    * the unmodified reference modules themselves (source here, `oracle/_ref/*.rvoc` bytecode on the GPU box) with
      `qdrant_client` -> B200VectorDB: build_database_ui -> load_selected_database_ui -> detect_and_extract_ui ->
      search_database_ui; every search equals QdrantLocalOracle fed the same points.
"""
import json
import os
import re
import sys
from types import SimpleNamespace as NS

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import reference_harness as H  # noqa: E402

from oracle import reverso_oracle as O  # noqa: E402

TOL = 1e-3   # north_star: scores within 1e-3 absolute, id sets identical except ties within 1e-3


@pytest.fixture(scope="module")
def trace():
    t = json.load(open(os.path.join(HERE, "golden", "reference_trace.json")))
    arrays = np.load(os.path.join(HERE, "golden", "reference_trace.npz"))
    for c in t["calls"]:
        for key in ("vectors", "query"):
            if key in c:
                c[key] = arrays[c[key]]
    return t


def hits_match(got, ref, tol=TOL, what=""):
    """got / ref: lists of (id, score, payload) in rank order.  Same length (up to boundary ties), scores position by position
    within tol, ids identical except among scores within tol of each other."""
    if len(got) != len(ref):
        m = min(len(got), len(ref))
        edge = [s for _, s, _ in (got[m:] or ref[m:])]
        assert abs(len(got) - len(ref)) <= 4 and max(edge) - min(edge) <= 2 * tol, f"{what}: {len(got)} hits vs {len(ref)}"
        got, ref = got[:m], ref[:m]
    for (gi, gs, gp), (ri, rs, rp) in zip(got, ref):
        assert abs(gs - rs) <= tol, f"{what}: score {gs} vs {rs}"
    gmap = {i: (s, p) for i, s, p in got}
    rmap = {i: (s, p) for i, s, p in ref}
    for i in set(gmap) & set(rmap):
        assert gmap[i][1] == rmap[i][1], f"{what}: payload of {i} differs"
    if set(gmap) != set(rmap):
        boundary = min(got[-1][1], ref[-1][1])
        for i in set(gmap) ^ set(rmap):
            s = (gmap.get(i) or rmap.get(i))[0]
            assert abs(s - boundary) <= tol, f"{what}: id {i} (score {s}) differs beyond the tie tolerance"


def mask_uuids(text):
    return re.sub(r"[0-9a-f]{8}-[0-9a-f]{4}-[0-9a-f]{4}-[0-9a-f]{4}-[0-9a-f]{12}", "<uuid>", text)


def items_match(got, ref, tol, what, threshold=None):
    """UI-level hit lists: (filename, score, bbox) in rank order; exact ties (the reference gives every region of an image the
    same embedding, core_system.py:406) may come back in any order."""
    if len(got) != len(ref):
        # only hits sitting on the score threshold may appear / disappear (a 0.9999 threshold against self-matches whose
        # score is 1 - O(1e-4) once the encoder runs in fp16 and the rows are stored as bf16)
        m = min(len(got), len(ref))
        extra = (got[m:] or ref[m:])
        assert threshold is not None and all(abs(it["score"] - threshold) <= tol for it in extra), \
            f"{what}: {len(got)} items vs {len(ref)}"
        got, ref = got[:m], ref[:m]
        if not got:
            return
    for g, r in zip(got, ref):
        assert abs(g["score"] - r["score"]) <= tol, f"{what}: {g} vs {r}"
    key = lambda it: (it["filename"], tuple(it["bbox"]))
    if sorted(map(key, got)) != sorted(map(key, ref)):
        boundary = min(got[-1]["score"], ref[-1]["score"])
        gk, rk = {key(i): i["score"] for i in got}, {key(i): i["score"] for i in ref}
        for kk in set(gk) ^ set(rk):
            assert abs((gk.get(kk) if kk in gk else rk[kk]) - boundary) <= tol, f"{what}: {kk} differs beyond the tie tolerance"


# ======================================================================================================================
# CPU
# ======================================================================================================================
def test_committed_trace_is_what_the_unmodified_reference_does_today(trace, tmp_path, monkeypatch):
    kind, where = H.reference_location()
    if kind != "source":
        pytest.skip("the reference sources are only present in the authoring container")
    rec = H.Recorder()
    saved = H.install_stubs(H.oracle_backend_factory(), rec)
    monkeypatch.chdir(tmp_path)
    try:
        ui = H.load_reference(kind, where)
        assert type(ui.reverso).__module__ == "core_system" and ui.reverso.pe_model.name == "PE-Core-L14-336"   # core_system.py:177
        out = H.run_scenario(ui)
    finally:
        H.restore_modules(saved)
    ref = trace["ui"]
    for k in ("load", "load_missing", "detect_text", "detect_choices", "detect_meta", "direct_text", "unlock", "delete"):
        assert out[k] == ref[k], k
    assert sorted(out["build_regions"].splitlines()) == sorted(ref["build_regions"].splitlines())     # os.listdir order is arbitrary
    for a, b in zip(out["searches"], ref["searches"]):
        assert a["text"].splitlines()[0] == b["text"].splitlines()[0]
        items_match(a["items"], b["items"], 1e-6, f"search thr={a['threshold']}")
    ops_now = [c["op"] for c in rec.calls]
    assert ops_now == [c["op"] for c in trace["calls"]]
    # the same points (by payload identity: filename + detection_index) with the same vectors
    def points(calls):
        d = {}
        for c in calls:
            if c["op"] == "upsert":
                for v, p in zip(c["vectors"], c["payloads"]):
                    d[(c["name"], p["filename"], p["detection_index"])] = v
        return d
    a, b = points(rec.calls), points(trace["calls"])
    assert a.keys() == b.keys() and all(np.allclose(a[k], b[k], atol=1e-6) for k in a)


def test_oracle_embedding_half_is_pinned_to_reference_outputs(trace, tmp_path):
    """The vectors the unmodified reference computed (core_system.py:341-349, 363, 398-408 / 442-447) and handed to
    `upsert` as python lists of floats (:608) == the oracle's restatement on the same encoder output and masks."""
    import torch
    enc, tf, det = H.FakePE("PE-Core-L14-336"), H.fake_transform(336), H.FakeGroundedSAM(H.FakeOntology({"object": "object"}))
    ups = [c for c in trace["calls"] if c["op"] == "upsert"]
    assert [c["vector_type"] for c in ups] == ["list", "list"] and [len(c["ids"]) for c in ups] == [24, 8]
    seen = 0
    for c in ups:
        for v, p in zip(c["vectors"], c["payloads"]):
            i = int(re.search(r"img(\d+)\.png", p["filename"]).group(1))
            pil = H.make_image(i)
            feats = enc.encode_image(tf(pil.convert("RGB")).unsqueeze(0)).numpy()
            if p["detected_class"] == "full_image":                        # process_image_direct_pe, core_system.py:431-455
                want = O.l2_normalize(O.global_embedding(feats)[0])
                assert p["bbox"] == [0, 0, pil.width, pil.height] and p["area_ratio"] == 1.0
            else:                                                          # extract_embeddings, core_system.py:320-429
                probe = str(tmp_path / "probe.jpg")
                pil.convert("RGB").save(probe)
                masks = det.predict(probe).mask
                embs = O.extract_embeddings_reference(feats, masks)
                kept = [j for j in range(len(masks)) if O.binarize_mask(masks[j]).sum() > 0]
                assert len(embs) == 3 and kept == [0, 1, 3]                # the empty mask is dropped, later regions shift up
                want = embs[kept.index(p["detection_index"])]
                ys, xs = np.where(masks[p["detection_index"]])
                assert p["bbox"] == [int(xs.min()), int(ys.min()), int(xs.max()), int(ys.max())]
            assert np.allclose(v, want, atol=2e-7), (p["filename"], float(np.abs(v - want).max()))
            assert abs(float(np.linalg.norm(v)) - 1) < 1e-6
            assert set(p) >= {"region_id", "original_region_id", "bbox", "area_ratio", "detection_index", "confidence",
                              "detected_class", "image_source", "filename"}                         # core_system.py:413-418,569-574
            seen += 1
    assert seen == 32


def test_recorded_hits_follow_the_restated_qdrant_semantics(trace):
    oc = O.QdrantLocalOracle()
    n_search = 0
    for c in trace["calls"]:
        if c["op"] == "recreate_collection":
            oc.recreate_collection(c["name"], size=c["size"])
        elif c["op"] == "upsert":
            oc.upsert(c["name"], [NS(id=i, vector=v, payload=p) for i, v, p in zip(c["ids"], c["vectors"], c["payloads"])])
        elif c["op"] == "search":
            hits = oc.search(c["name"], c["query"], limit=c["limit"], score_threshold=c["score_threshold"])
            hits_match([(h.id, h.score, h.payload) for h in hits], [(h["id"], h["score"], h["payload"]) for h in c["hits"]], 1e-6)
            assert all(h["score"] >= c["score_threshold"] for h in c["hits"]) and len(c["hits"]) <= c["limit"]
            n_search += 1
    assert n_search == 6


# ======================================================================================================================
# GPU
# ======================================================================================================================
def _gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    return torch.device("cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_replay_of_the_reference_calls_on_b200(trace, tmp_path, devices):
    """Every call the unmodified reference made to qdrant, replayed argument for argument against the CUDA library."""
    dev = _gpu()
    from revers_o_b200.vector_db import B200VectorDB, models
    clients = {}
    cur = None
    for c in trace["calls"]:
        if c["op"] == "open":
            path = str(tmp_path / c["path"].lstrip("./"))
            cur = clients[path] = B200VectorDB(path=path, device=dev, devices=devices, shard_rows=128)   # a NEW client per open,
        elif c["op"] == "get_collections":                                                               # like the reference
            assert [x.name for x in cur.get_collections().collections] == c["names"]                     # persisted implicitly
        elif c["op"] == "recreate_collection":
            cur.recreate_collection(collection_name=c["name"],
                                    vectors_config=models.VectorParams(size=c["size"], distance=models.Distance.COSINE))
        elif c["op"] == "upsert":
            cur.upsert(collection_name=c["name"],
                       points=[models.PointStruct(id=i, vector=v.tolist(), payload=p)                     # python lists of floats
                               for i, v, p in zip(c["ids"], c["vectors"], c["payloads"])])
        elif c["op"] == "search":
            hits = cur.search(collection_name=c["name"], query_vector=c["query"].tolist(), limit=c["limit"],
                              score_threshold=c["score_threshold"])
            hits_match([(h.id, h.score, h.payload) for h in hits], [(h["id"], h["score"], h["payload"]) for h in c["hits"]],
                       TOL, f"search limit={c['limit']} thr={c['score_threshold']}")
            assert [h.score for h in hits] == sorted((h.score for h in hits), reverse=True)


def _dropin_scenario(r):
    """The calls ui.py's callbacks make (ui.py:29-159, 200-214), on the drop-in class."""
    out = {}
    H.write_images("imgs")
    out["build_regions"] = r.create_database(folder_path="imgs", database_name="trace", text_prompt="object .", use_direct_pe=False,
                                             resume_from_checkpoint=False, include_subfolders=False,
                                             progress_callback=lambda m, p=None: None)
    out["build_direct"] = r.create_database(folder_path="imgs", database_name="direct", text_prompt="", use_direct_pe=True,
                                            resume_from_checkpoint=False, include_subfolders=False, progress_callback=None)
    out["list"] = r.list_databases()
    out["load_missing"] = r.load_database("nope")
    out["load"] = r.load_database("trace")
    out["n_devices"] = len(r.vector_db.devices)
    q = H.make_image(2)
    r.region_embeddings = []
    n = r.detect_regions(q, "object .")
    embs, meta = r.extract_embeddings(q)
    r.region_embeddings = embs
    out["detect_text"] = (f"✅ Found {n} regions\n🧠 Extracted {len(embs)} embeddings\n"
                          f"🎯 Select a region to search with (or uses first by default)")
    out["detect_choices"] = [f"Region {i + 1}: {m.get('detected_class', 'object')} (Conf: {m.get('confidence', 0.0):.2f})"
                             for i, m in enumerate(meta)]
    out["detect_meta"] = [{k: v for k, v in m.items() if k != "region_id"} for m in meta]
    searches = []
    for thr, k, sel in ((0.5, 5, None), (0.5, 5, 1), (0.0, 20, 2), (0.9999, 3, None), (1.01, 5, None)):
        keep = r.region_embeddings
        if sel is not None:
            r.region_embeddings = [keep[sel]]                              # ui.py:125-133
        text, items = r.search_similar(thr, k)
        r.region_embeddings = keep
        searches.append({"text": text, "items": [{"score": it["score"], "filename": it["filename"], "bbox": it["bbox"]} for it in items]})
    out["load_direct"] = r.load_database("direct")
    embs, meta = r.process_image_direct_pe(H.make_image(5))
    r.region_embeddings = embs
    text, items = r.search_similar(0.3, 10)
    searches.append({"text": text, "items": [{"score": it["score"], "filename": it["filename"], "bbox": it["bbox"]} for it in items]})
    out["searches"] = searches
    out["unlock"] = r.unlock_database("trace")
    out["delete"] = r.delete_database("direct")
    out["list_after"] = r.list_databases()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [None, "0,0"])
def test_dropin_no_arg_constructor_matches_the_reference_trace(trace, tmp_path, monkeypatch, devices):
    """`SimpleReverso()` exactly as ui.py:20 constructs it: device, PE encoder and GroundedSAM come up lazily through the
    reference's own imports (stand-ins here), fp16 tokens (`.half()` on CUDA, core_system.py:195-196) are consumed natively."""
    _gpu()
    rec = H.Recorder()
    saved = H.install_stubs(H.oracle_backend_factory(), rec)     # only the encoder / detector stand-ins are used by the drop-in
    monkeypatch.chdir(tmp_path)
    if devices:
        monkeypatch.setenv("RVO_DEVICES", devices)
    try:
        from revers_o_b200.core_system import SimpleReverso
        r = SimpleReverso()
        assert r.pe_model is None                                # nothing loaded yet
        out = _dropin_scenario(r)
        assert r.pe_model.name == "PE-Core-L14-336" and r.pe_model.is_half and r.pe_model.device.type == "cuda"
        assert H.FakeGroundedSAM.instances > 0 and r.grounded_sam.box_threshold == 0.35 and r.grounded_sam.text_threshold == 0.25
        assert out["n_devices"] == (2 if devices else 1)
    finally:
        H.restore_modules(saved)
    ref = trace["ui"]
    for k in ("load", "load_missing", "detect_text", "detect_choices", "direct_text", "unlock", "delete"):
        if k in out:
            assert out[k] == ref[k], k
    assert out["list"] == ["direct", "trace"] or sorted(out["list"]) == ["direct", "trace"]
    for a, b in zip(out["detect_meta"], ref["detect_meta"]):
        assert a == b
    want = set(ref["build_regions"].splitlines())
    got = set(out["build_regions"].splitlines())
    # not compared: the order images are visited in (os.listdir), the reference's dead checkpoint code (SURVEY.md F6: it logs
    # "Error saving checkpoint: name 'datetime' is not defined"), and the line ui.build_database_ui appends (ui.py:97-99)
    strip = lambda ls: {re.sub(r"Processing \d+/", "Processing N/", x) for x in ls
                        if "checkpoint" not in x.lower() and "Finalization complete" not in x}
    assert strip(got) == strip(want), strip(got) ^ strip(want)
    for a, b in zip(out["searches"], ref["searches"]):
        if len(a["items"]) == len(b["items"]):
            assert a["text"].splitlines()[0] == b["text"].splitlines()[0], (a["text"], b["text"])
        # fp16 encoder output on CUDA vs fp32 on the CPU run
        items_match(a["items"], b["items"], 2e-3, "drop-in search", threshold=b["threshold"])


@pytest.mark.gpu
def test_unmodified_reference_modules_run_on_b200vectordb(trace, tmp_path, monkeypatch):
    """core_system.py and ui.py of the reference, not a byte changed, with `qdrant_client` -> B200VectorDB."""
    dev = _gpu()
    kind, where = H.reference_location()
    if kind is None:
        pytest.skip("neither /root/reference nor oracle/_ref/*.rvoc (python oracle/build_ref.py) is present")
    rec = H.Recorder()
    saved = H.install_stubs(H.b200_backend_factory(device=dev), rec)
    monkeypatch.chdir(tmp_path)
    try:
        ui = H.load_reference(kind, where)
        assert type(ui.reverso).__module__ == "core_system" and "revers_o_b200" not in type(ui.reverso).__module__
        out = H.run_scenario(ui)
        from revers_o_b200.vector_db import B200VectorDB
        assert isinstance(ui.reverso.vector_db._b, B200VectorDB)
    finally:
        H.restore_modules(saved)
    ref = trace["ui"]
    for k in ("load", "load_missing", "detect_text", "detect_choices", "detect_meta", "direct_text", "unlock", "delete"):
        assert out[k] == ref[k], k
    assert sorted(out["build_regions"].splitlines()) == sorted(ref["build_regions"].splitlines())
    # every search the reference issued == QdrantLocalOracle fed the very same points (this run's upserts: fp16 encoder on CUDA)
    oc = O.QdrantLocalOracle()
    n_search = 0
    for c in rec.calls:
        if c["op"] == "recreate_collection":
            oc.recreate_collection(c["name"], size=c["size"])
        elif c["op"] == "upsert":
            oc.upsert(c["name"], [NS(id=i, vector=v, payload=p) for i, v, p in zip(c["ids"], c["vectors"], c["payloads"])])
        elif c["op"] == "search":
            want = oc.search(c["name"], c["query"], limit=c["limit"], score_threshold=c["score_threshold"])
            hits_match([(h["id"], h["score"], h["payload"]) for h in c["hits"]], [(h.id, h.score, h.payload) for h in want], TOL,
                       f"reference search limit={c['limit']} thr={c['score_threshold']}")
            n_search += 1
    assert n_search == 6
    for a, b in zip(out["searches"], ref["searches"]):
        if len(a["items"]) == len(b["items"]):
            assert a["text"].splitlines()[0] == b["text"].splitlines()[0]
        items_match(a["items"], b["items"], 2e-3, "reference-on-B200 search", threshold=b["threshold"])
