"""Spherical k-means (`B200VectorDB.cluster`) on configs[4]-shaped rows: synth.make_selfjoin_db(2_000_000, 1024, 0.05, seed=5).

For C = 256, 1024 and 4096 centroids (the stored rows numpy.random.default_rng(0) picks):
  assign     one `ops.knn_join` (k = 1) of every row against the C centroids: TFLOP/s on 2 * N * C * D;
  update     one `ops.kmeans_update` of that assignment: GB/s on the N * D * 2 bytes of rows it reads, and its share of the
             7.7 TB/s HBM bound of the data sheet;
  loop       `sharded.kmeans_sharded` with max_iter = 5 (iterations, seconds per iteration), on 1 shard and on 2 and 4 virtual
             shards on GPU 0 (views of one tiled buffer; bit-identical labels and centroids checked);
  cuBLAS     the yardstick: torch bf16 matmul of the untiled rows against the centroids plus argmax, in row chunks of 2^18, and
             the share of rows whose label agrees with the kNN assignment.
Each: median of 3 host-clock timings of synchronised work after one warm-up.  The GPU name and power limit are read in the
same run.

  python scripts/bench_clusters.py [--n 2000000] [--out profiles/clusters_n1.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from revers_o_b200 import ops, synth                                    # noqa: E402
from revers_o_b200.sharded import gather_rows, kmeans_sharded           # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        lines = [x.strip() for x in r.stdout.strip().splitlines() if x.strip()]
    except (OSError, subprocess.SubprocessError):
        lines = []
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": lines or "unavailable", "device_count": torch.cuda.device_count()}


def timed(fn, rounds=3):
    fn()                                                              # warm-up
    ts, out = [], None
    for _ in range(rounds):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts), ts, out


def virtual_shards(tiled, n, G):
    nblk = -(-n // 128)
    blk = -(-nblk // G)
    return [(tiled[g * blk: min((g + 1) * blk, nblk)], min(n, min((g + 1) * blk, nblk) * 128) - g * blk * 128, g * blk * 128)
            for g in range(G)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=2_000_000)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a GPU: there is no CPU path to measure")
    n, d = args.n, 1024
    info = gpu_info()
    dev = torch.device("cuda:0")
    results = []

    def emit(rec):
        results.append(rec)
        print(json.dumps(rec), flush=True)

    tiled = synth.make_selfjoin_db(n, d, 0.05, dev, seed=5)
    X = ops.untile_rows(tiled, n, d).contiguous()                      # row-major copy for the cuBLAS yardstick
    ids = torch.empty((n, 1), dtype=torch.int64, device=dev)
    sc = torch.empty((n, 1), dtype=torch.float32, device=dev)
    cnt = torch.empty((n,), dtype=torch.int32, device=dev)
    labels = torch.empty((n,), dtype=torch.int32, device=dev)
    for C in (256, 1024, 4096):
        cent = gather_rows([(tiled, n, 0)], np.random.default_rng(0).choice(n, C, replace=False), d, dev)
        flop = 2.0 * n * C * d
        sec, ts, _ = timed(lambda: ops.knn_join(tiled, 0, n, 0, cent, C, d, 1, None, 0, False, out=(ids, sc, cnt)))
        flagged = int((cnt < 0).sum())
        emit({"workload": f"assign: knn_join k = 1, {n} x {d} against C = {C}", "C": C, "seconds": sec, "rounds": ts,
              "tflops_2_n_c_d": flop / sec / 1e12, "rows_flagged": flagged})
        sums = torch.zeros((C, d), dtype=torch.int64, device=dev)
        counts = torch.zeros((C,), dtype=torch.int64, device=dev)
        changed = torch.zeros((1,), dtype=torch.int64, device=dev)

        def update():
            sums.zero_()
            counts.zero_()
            changed.zero_()
            ops.kmeans_update(tiled, 0, n, d, ids, C, None, labels, sums, counts, changed)
        sec, ts, _ = timed(update)
        emit({"workload": f"update: kmeans_update, {n} x {d} into C = {C}", "C": C, "seconds": sec, "rounds": ts,
              "gb_per_s_n_d_2": n * d * 2 / sec / 1e9, "share_of_hbm_7_7_tb_s": n * d * 2 / sec / HBM_BYTES_PER_S,
              "counts_sum": int(counts.sum())})

        def cublas():
            out = torch.empty(n, dtype=torch.int64, device=dev)
            cm = ops.untile_rows(cent, C, d)
            for a in range(0, n, 1 << 18):
                out[a: a + (1 << 18)] = (X[a: a + (1 << 18)] @ cm.T).argmax(1)
            return out
        sec, ts, lab = timed(cublas)
        emit({"workload": f"yardstick: cuBLAS bf16 matmul + argmax, {n} x {d} against C = {C}", "C": C, "seconds": sec,
              "rounds": ts, "tflops_2_n_c_d": flop / sec / 1e12,
              "label_agreement_with_knn": float((lab == ids.view(-1)).float().mean())})
        ref = None
        for G in (1, 2, 4):
            shards = virtual_shards(tiled, n, G)
            sec, ts, r = timed(lambda: kmeans_sharded(shards, d, cent, C, max_iter=5))
            if ref is None:
                ref = r
            same = (np.array_equal(r.labels, ref.labels) and torch.equal(r.centroids, ref.centroids)
                    and np.array_equal(r.scores.view(np.uint32), ref.scores.view(np.uint32)) and r.iterations == ref.iterations)
            emit({"workload": f"loop: kmeans_sharded max_iter = 5, {n} x {d}, C = {C}, {G} virtual shard(s) on GPU 0", "C": C,
                  "shards": G, "seconds": sec, "rounds": ts, "iterations": r.iterations, "converged": r.converged,
                  "seconds_per_assignment": sec / (r.iterations + 1), "bit_identical_to_one_shard": same})
        del cent, sums, counts
        torch.cuda.empty_cache()
    summary = {"gpu": info, "results": results}
    if args.out:
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)
    print(json.dumps({"gpu": info}))


if __name__ == "__main__":
    main()
