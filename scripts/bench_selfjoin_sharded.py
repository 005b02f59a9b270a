"""BASELINE configs[4] through the public API on a row-sharded collection: N frame embeddings x 1024-d with 5 % planted
near-duplicates (synth.make_selfjoin_db(N, 1024, 0.05, seed=5)), loaded into a B200VectorDB collection row-sharded over G devices
of ONE process (integer ids, persistence off), then `find_near_duplicates(threshold=0.95)`.

Per G: host-clock seconds of the synchronising call after one warm-up call, pairs, TFLOP/s on N^2 * D (the upper triangle),
each device's busy time from CUDA events (a second, instrumented run of the same join) and the max/mean imbalance, and
whether the pair set and scores equal those of the G = 1 run of this process.  Beside it, the replicated-DB join of
scripts/bench_selfjoin.py at the same G (torchrun, one process per GPU) when that many GPUs are present; otherwise it is
reported as not run.  The GPU name and power limit are read in the same run.

  python scripts/bench_selfjoin_sharded.py [--n 2000000] [--gpus 1,2,4,8] [--virtual 2,4] [--no-replicated] [--out FILE]

--virtual G lists the SAME device G times: the sharded code path on one GPU (copies, rectangles, G pair buffers), a measure
of its overhead against G = 1 and not of scaling.  GPU counts above the devices present are reported as not measured."""
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
from revers_o_b200.sharded import selfjoin_sharded                      # noqa: E402
from revers_o_b200.vector_db import B200VectorDB, models                # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        lines = [x.strip() for x in r.stdout.strip().splitlines() if x.strip()]
    except (OSError, subprocess.SubprocessError):
        lines = []
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": lines or "unavailable", "device_count": torch.cuda.device_count()}


def load(tiled, n, d, devices):
    db = B200VectorDB(devices=devices, shard_rows=(n + len(devices) - 1) // len(devices) // 128 * 128 + 128)
    db.recreate_collection("frames", vectors_config=models.VectorParams(size=d, distance=models.Distance.COSINE))
    for lo in range(0, n, 131072):
        hi = min(n, lo + 131072)
        rows = ops.untile_rows(tiled, n, d, rows=torch.arange(lo, hi, device=tiled.device)).float()
        db.upsert_batch("frames", range(lo, hi), rows, assume_new=True, persist=False)
    torch.cuda.synchronize()
    return db


def replicated(n, g):
    """scripts/bench_selfjoin.py at g GPUs (torchrun for g > 1): its JSON line, or why it was not run."""
    if g > torch.cuda.device_count():
        return f"not run: needs {g} GPUs, {torch.cuda.device_count()} present"
    script = os.path.join(ROOT, "scripts", "bench_selfjoin.py")
    cmd = [sys.executable, script, str(n)] if g == 1 else \
        [sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc_per_node={g}", script, str(n)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1800)
    for line in reversed(r.stdout.strip().splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    return f"failed (exit {r.returncode}): {r.stderr.strip()[-400:]}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=2_000_000)
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--virtual", default="", help="shard counts to run on device 0 alone (overhead of the sharded path)")
    ap.add_argument("--no-replicated", action="store_true")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a GPU: there is no CPU path to measure")
    n, d, thr = args.n, 1024, 0.95
    info = gpu_info()
    dev0 = torch.device("cuda:0")
    tiled = synth.make_selfjoin_db(n, d, 0.05, dev0, seed=5)
    configs = [("real", int(g)) for g in args.gpus.split(",") if g] + [("virtual", int(g)) for g in args.virtual.split(",") if g]
    ref, results = None, []
    for kind, g in configs:
        rec = {"workload": f"configs[4]: find_near_duplicates, {n} x {d}, cos >= {thr}", "shards": g, "layout": kind}
        if kind == "real" and g > torch.cuda.device_count():
            rec["status"] = f"not measured: needs {g} GPUs, {torch.cuda.device_count()} present"
            results.append(rec)
            print(json.dumps(rec), flush=True)
            continue
        devices = list(range(g)) if kind == "real" else [0] * g
        db = load(tiled, n, d, devices)
        c = db._coll("frames")
        rec["shard_rows"] = [s.n for s in c.shards]
        db.find_near_duplicates("frames", thr)                                 # warm-up
        t0 = time.perf_counter()
        pairs, scores = db.find_near_duplicates("frames", thr)                 # synchronises: returns host data
        sec = time.perf_counter() - t0
        active = [s for s in c.shards if s.n]
        ms = {}
        if len(active) > 1:
            selfjoin_sharded([(s.vectors, s.n, s.row0) for s in active], d, thr, device_ms=ms)
        else:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ops.selfjoin_exact(active[0].vectors, active[0].n, d, thr)
            e1.record()
            torch.cuda.synchronize()
            ms[0] = e0.elapsed_time(e1)
        busy = list(ms.values())
        got = {tuple(p): float(s) for p, s in zip(pairs, scores)}
        rec.update({"seconds": sec, "pairs": len(pairs), "tflops_upper_triangle": float(n) * n * d / sec / 1e12,
                    "device_busy_ms": {f"cuda:{k}": v for k, v in ms.items()},
                    "imbalance_max_over_mean": max(busy) / (sum(busy) / len(busy))})
        if ref is None and kind == "real" and g == 1:
            ref = got
            rec["verified_against_1_gpu"] = "this is the reference"
        else:
            rec["verified_against_1_gpu"] = "not run: no G = 1 run in this process" if ref is None else (got == ref)
        if not args.no_replicated and kind == "real":
            rec["replicated_db"] = replicated(n, g)
        results.append(rec)
        print(json.dumps(rec), flush=True)
        del db, c, active
        torch.cuda.empty_cache()
    summary = {"gpu": info, "results": results}
    if args.out:
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)
    print(json.dumps({"gpu": info}))


if __name__ == "__main__":
    main()
