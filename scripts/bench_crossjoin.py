"""The join between two collections through the public API: `B200VectorDB.join_collections(threshold=0.95)` of a left collection of
N_L frame embeddings and a right collection of N_R, 1024-d.  Both come from ONE seeded configs[4] input,
synth.make_selfjoin_db(N_L + N_R, 1024, 0.05, seed=5): rows [0, N_L) are the left collection, rows [N_L, N_L + N_R) the right
one (integer ids from 0 on each side, persistence off, one B200VectorDB per side as revers-o opens one per database), so the
planted near-copies of earlier rows give cross pairs, and the join must equal the self-join of all N_L + N_R rows restricted to
pairs (i, j) with i < N_L <= j, bit for bit.

Layouts: both sides on one GPU; both row-sharded over the same G GPUs (G in --gpus, above 1); the left side on one GPU and the
right side sharded over all GPUs present; --virtual G lists the SAME device G times on both sides (the sharded code path on one
GPU: copies, split rectangles, G pair buffers), a measure of its overhead and not of scaling.  Per layout: host-clock seconds of
the synchronising call after one warm-up call, pairs, TFLOP/s on 2 * N_L * N_R * D, each device's busy time from CUDA events (a
second, instrumented run of the same join) and the max/mean imbalance, and whether the pairs and scores equal the restricted
self-join, which is computed once in the same run (`find_near_duplicates` on one GPU over all rows).  With the one-GPU layout
the self-join is also timed (after a warm-up) and its TFLOP/s on N^2 * D reported: the rate of the same kernels on their
reference workload.  The GPU name and power limit are read in the same run.

  python scripts/bench_crossjoin.py [--nl 1000000] [--nr 2000000] [--gpus 1,2,4,8] [--virtual 2,4] [--out FILE]

GPU counts above the devices present are reported as not measured."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from revers_o_b200 import ops, synth                                    # noqa: E402
from revers_o_b200.sharded import crossjoin_sharded                     # noqa: E402
from revers_o_b200.vector_db import B200VectorDB, models                # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        lines = [x.strip() for x in r.stdout.strip().splitlines() if x.strip()]
    except (OSError, subprocess.SubprocessError):
        lines = []
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": lines or "unavailable", "device_count": torch.cuda.device_count()}


def load(tiled, lo, hi, d, devices, name):
    """Rows [lo, hi) of the tiled input as collection `name` (ids 0 ..) of a B200VectorDB row-sharded over `devices`."""
    n = hi - lo
    db = B200VectorDB(devices=devices, shard_rows=(n + len(devices) - 1) // len(devices) // 128 * 128 + 128)
    db.recreate_collection(name, vectors_config=models.VectorParams(size=d, distance=models.Distance.COSINE))
    for a in range(lo, hi, 131072):
        b = min(hi, a + 131072)
        rows = ops.untile_rows(tiled, hi, d, rows=torch.arange(a, b, device=tiled.device)).float()
        db.upsert_batch(name, range(a - lo, b - lo), rows, assume_new=True, persist=False)
    torch.cuda.synchronize()
    return db


def canonical(pairs, scores):
    p = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    s = np.asarray(scores, dtype=np.float32)
    o = np.lexsort((p[:, 1], p[:, 0]))
    return p[o], s[o]


def same(a, b):
    return bool(np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nl", type=int, default=1_000_000)
    ap.add_argument("--nr", type=int, default=2_000_000)
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--virtual", default="", help="shard counts to run on device 0 alone (overhead of the sharded path)")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a GPU: there is no CPU path to measure")
    nl, nr, d, thr = args.nl, args.nr, 1024, 0.95
    n = nl + nr
    info = gpu_info()
    ngpu = torch.cuda.device_count()
    dev0 = torch.device("cuda:0")
    tiled = synth.make_selfjoin_db(n, d, 0.05, dev0, seed=5)
    gpus = [int(g) for g in args.gpus.split(",") if g]
    layouts = [("one GPU", [0], [0])] if 1 in gpus else []
    layouts += [(f"both sharded over {g} GPUs", list(range(g)), list(range(g))) for g in gpus if g > 1]
    layouts += [(f"left on 1 GPU, right over {ngpu} GPUs", [0], list(range(ngpu)))] if ngpu > 1 else \
        [("left on 1 GPU, right over all GPUs", None, None)]
    layouts += [(f"virtual {g} shards on GPU 0", [0] * g, [0] * g) for g in (int(x) for x in args.virtual.split(",") if x)]

    # the restricted self-join, once: find_near_duplicates over all rows on one GPU, pairs (i, j) with i < nl <= j
    whole = load(tiled, 0, n, d, [0], "all")
    p, s = whole.find_near_duplicates("all", thr)
    p = np.asarray(p, dtype=np.int64).reshape(-1, 2)
    keep = (p[:, 0] < nl) & (p[:, 1] >= nl)
    ref = canonical(p[keep] - np.array([0, nl]), s[keep])
    selfjoin = {"pairs_all": len(p), "pairs_straddling": int(keep.sum())}
    if 1 in gpus:
        t0 = time.perf_counter()
        whole.find_near_duplicates("all", thr)                             # timed after the warm-up above
        sec = time.perf_counter() - t0
        selfjoin.update({"seconds": sec, "tflops_upper_triangle": float(n) * n * d / sec / 1e12})
    del whole
    torch.cuda.empty_cache()
    print(json.dumps({"restricted_selfjoin": selfjoin}), flush=True)

    results = []
    for name, ld, rd in layouts:
        rec = {"workload": f"join_collections, {nl} x {d} with {nr} x {d}, cos >= {thr}", "layout": name}
        need = 1 + max(ld + rd) if ld else 2
        if ld is None or need > ngpu:
            rec["status"] = f"not measured: needs {need} GPUs, {ngpu} present"
            results.append(rec)
            print(json.dumps(rec), flush=True)
            continue
        left = load(tiled, 0, nl, d, ld, "left")
        right = load(tiled, nl, n, d, rd, "right")
        a, b = left._coll("left"), right._coll("right")
        rec["left_shard_rows"] = {f"cuda:{s.device.index}": s.n for s in a.shards if s.n} if len(set(ld)) == len(ld) else \
            [s.n for s in a.shards]
        rec["right_shard_rows"] = {f"cuda:{s.device.index}": s.n for s in b.shards if s.n} if len(set(rd)) == len(rd) else \
            [s.n for s in b.shards]
        left.join_collections("left", "right", thr, other=right)                     # warm-up
        t0 = time.perf_counter()
        pairs, scores = left.join_collections("left", "right", thr, other=right)     # synchronises: returns host data
        sec = time.perf_counter() - t0
        ms = {}
        crossjoin_sharded([(s.vectors, s.n, s.row0) for s in a.shards if s.n], [(s.vectors, s.n, s.row0) for s in b.shards if s.n],
                          d, thr, device_ms=ms)
        busy = list(ms.values())
        rec.update({"seconds": sec, "pairs": len(pairs), "tflops_2_nl_nr_d": 2.0 * nl * nr * d / sec / 1e12,
                    "device_busy_ms": {f"cuda:{k}": v for k, v in ms.items()},
                    "imbalance_max_over_mean": max(busy) / (sum(busy) / len(busy)),
                    "verified": same(canonical(pairs, scores), ref)})
        if name == "one GPU" and "seconds" in selfjoin:
            rec["cross_over_selfjoin_tflops"] = rec["tflops_2_nl_nr_d"] / selfjoin["tflops_upper_triangle"]
        results.append(rec)
        print(json.dumps(rec), flush=True)
        del left, right, a, b
        torch.cuda.empty_cache()
    summary = {"gpu": info, "restricted_selfjoin": selfjoin, "results": results}
    if args.out:
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)
    print(json.dumps({"gpu": info}))


if __name__ == "__main__":
    main()
