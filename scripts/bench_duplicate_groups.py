"""Duplicate groups against the pair join they are built from, through the public API and on one GPU.

Input 1, configs[4]: synth.make_selfjoin_db(2_000_000, 1024, 0.05, seed=5) as collection "frames" of a B200VectorDB (integer ids
= rows, persistence off), cos >= 0.95.  Three paths, alternated over --rounds rounds after one warm-up call of each:
  groups         B200VectorDB.find_duplicate_groups (edges unioned on the GPU while the join runs, no pair stored)
  pairs          B200VectorDB.find_near_duplicates (the flat pair list)
  pairs+scipy    find_near_duplicates, then scipy.sparse.csgraph.connected_components of the pairs on the host: what a user
                 had to do to get groups before find_duplicate_groups
Host-clock seconds of each synchronising call.  In the same run the labels of ops.components_exact must equal the scipy
components of the returned pairs (each row labelled with its component's smallest row), its pair count the pair list's
length, and find_duplicate_groups' groups those components' groups.

Input 2, a static scene: synth.make_selfjoin_db(--scene-rows, 1024, 0.05, seed=6, cluster=--scene) — row 0 and `scene` exact
copies of it, about scene^2 / 2 pairs.  At the ops level (the pair list is too long for Python tuples): ops.components_exact
against ops.selfjoin_exact, each once after a warm-up, with the peak device memory of each call: torch.cuda.max_memory_allocated
during the call minus what was allocated before it, with the library's cached join workspace dropped first so that each path
allocates its own.  The labels are checked against the scipy components of the pairs as above.

The GPU name and power limit are read in the same run.

  python scripts/bench_duplicate_groups.py [--n 2000000] [--rounds 3] [--scene 20000] [--scene-rows 200000] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from revers_o_b200 import ops, synth                                    # noqa: E402
from revers_o_b200.vector_db import B200VectorDB, group_labels, models  # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        lines = [x.strip() for x in r.stdout.strip().splitlines() if x.strip()]
    except (OSError, subprocess.SubprocessError):
        lines = []
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": lines or "unavailable", "device_count": torch.cuda.device_count()}


def scipy_labels(pairs, n):
    """Connected components of the pairs on n rows, each row labelled with its component's smallest row."""
    p = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    g = coo_matrix((np.ones(len(p), np.int8), (p[:, 0], p[:, 1])), shape=(n, n))
    _, comp = connected_components(g, directed=False)
    smallest = np.full(comp.max() + 1, n, np.int64)
    np.minimum.at(smallest, comp, np.arange(n))
    return smallest[comp]


def load(tiled, n, d):
    db = B200VectorDB(device=tiled.device)
    db.recreate_collection("frames", vectors_config=models.VectorParams(size=d, distance=models.Distance.COSINE))
    for a in range(0, n, 131072):
        b = min(n, a + 131072)
        rows = ops.untile_rows(tiled, n, d, rows=torch.arange(a, b, device=tiled.device)).float()
        db.upsert_batch("frames", range(a, b), rows, assume_new=True, persist=False)
    torch.cuda.synchronize()
    return db


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return time.perf_counter() - t0, out


def peak_of(fn):
    """(result, seconds, bytes allocated at the peak of the call above what was allocated before it)."""
    ops._workspaces.clear()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    sec, out = timed(fn)
    torch.cuda.synchronize()
    return out, sec, torch.cuda.max_memory_allocated() - base


def configs4(n, d, thr, rounds):
    dev = torch.device("cuda:0")
    tiled = synth.make_selfjoin_db(n, d, 0.05, dev, seed=5)
    db = load(tiled, n, d)
    del tiled
    torch.cuda.empty_cache()
    c = db._coll("frames")

    def pairs_scipy():
        p, _ = db.find_near_duplicates("frames", thr)
        return scipy_labels(p, n)

    paths = {"groups": lambda: db.find_duplicate_groups("frames", thr),
             "pairs": lambda: db.find_near_duplicates("frames", thr),
             "pairs+scipy": pairs_scipy}
    for fn in paths.values():                                        # warm-up
        fn()
    secs = {k: [] for k in paths}
    for _ in range(rounds):
        for k, fn in paths.items():
            sec, _ = timed(fn)
            secs[k].append(sec)
    rec = {"workload": f"configs[4]: {n} x {d}, cos >= {thr}, public API on one GPU",
           "seconds": secs, "median_seconds": {k: statistics.median(v) for k, v in secs.items()}}
    m = rec["median_seconds"]
    rec["groups_over_pairs"] = m["groups"] / m["pairs"]
    rec["groups_over_pairs_scipy"] = m["groups"] / m["pairs+scipy"]
    # peak device memory of one call of each (the collection itself is allocated before and not counted)
    for k in ("groups", "pairs"):
        _, _, peak = peak_of(paths[k])
        rec.setdefault("peak_device_bytes_over_baseline", {})[k] = peak
    # the check, in the same run
    p, _ = db.find_near_duplicates("frames", thr)
    p = np.asarray(p, dtype=np.int64).reshape(-1, 2)
    ref = scipy_labels(p, n)
    labels, n_pairs = ops.components_exact(c.vectors, n, d, thr)
    groups = db.find_duplicate_groups("frames", thr)
    rec.update({"pairs": len(p), "n_pairs_of_components": n_pairs, "groups": len(groups),
                "largest_group": len(groups[0]) if groups else 0,
                "labels_equal_scipy_components": bool(np.array_equal(labels, ref)),
                "groups_equal_scipy_groups": groups == group_labels(ref),
                "n_pairs_equal": n_pairs == len(p)})
    del db, c
    torch.cuda.empty_cache()
    return rec


def scene(n, d, thr, cluster):
    dev = torch.device("cuda:0")
    db = synth.make_selfjoin_db(n, d, 0.05, dev, seed=6, cluster=cluster)
    torch.cuda.synchronize()
    ops.components_exact(db, n, d, thr)                             # warm-up of both paths
    ops.selfjoin_exact(db, n, d, thr)
    (labels, n_pairs), sec_g, peak_g = peak_of(lambda: ops.components_exact(db, n, d, thr))
    (pairs, _), sec_p, peak_p = peak_of(lambda: ops.selfjoin_exact(db, n, d, thr))
    t0 = time.perf_counter()
    ref = scipy_labels(pairs, n)
    sec_scipy = time.perf_counter() - t0
    rec = {"workload": f"static scene: {n} x {d} with {cluster} exact copies of row 0, cos >= {thr}, ops level on one GPU",
           "seconds": {"components_exact": sec_g, "selfjoin_exact": sec_p, "scipy_connected_components_of_the_pairs": sec_scipy},
           "peak_device_bytes_over_baseline": {"components_exact": peak_g, "selfjoin_exact": peak_p},
           "pairs": len(pairs), "n_pairs_of_components": n_pairs, "n_pairs_equal": n_pairs == len(pairs),
           "host_bytes_of_the_pairs": int(pairs.nbytes), "labels_equal_scipy_components": bool(np.array_equal(labels, ref)),
           "group_of_row_0": int((labels == 0).sum())}
    del db
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=2_000_000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--scene", type=int, default=20_000)
    ap.add_argument("--scene-rows", type=int, default=200_000)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a GPU: there is no CPU path to measure")
    d, thr = 1024, 0.95
    summary = {"gpu": gpu_info()}
    print(json.dumps(summary), flush=True)
    summary["configs4"] = configs4(args.n, d, thr, args.rounds)
    print(json.dumps(summary["configs4"]), flush=True)
    if args.scene > 0:
        summary["static_scene"] = scene(args.scene_rows, d, thr, args.scene)
        print(json.dumps(summary["static_scene"]), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)


if __name__ == "__main__":
    main()
