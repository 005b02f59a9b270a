"""The k-nearest-neighbour join (`rvo_knn_join`) on configs[4]-sized inputs, with `find_near_duplicates` on the same input as
the reference rate of the same kernels.

Workloads (1024-d, seeded):
  self kNN   synth.make_selfjoin_db(2_000_000, 1024, 0.05, seed=5), every row against every other, a row's own match left out,
             at k = 10 and k = 100 (`ops.knn_exact`, device result);
  cross kNN  the 1M x 2M rows of scripts/bench_crossjoin.py: rows [0, 1M) and [1M, 3M) of make_selfjoin_db(3_000_000, 1024,
             0.05, seed=5), the left rows' k = 10 best right rows;
  public     `B200VectorDB.knn_join(k=10)` on the self input, host arrays included;
  blocks     the self kNN at k = 10 with query blocks (option "knn_block") of 2048 to 16384 rows, with the workspace size;
  virtual    `sharded.knn_sharded` with the self input cut into G = 1, 2, 4 shards on GPU 0 (views of one tiled buffer): the
             sharded code path (per-shard lists, merge, exclusion) on one GPU, a measure of its overhead and not of scaling;
  reference  `B200VectorDB.find_near_duplicates(0.95)` on the self input.
Each: median of 3 host-clock timings of the synchronising call after one warm-up call; TFLOP/s on 2 * N_L * N_R * D for the
kNN joins (every pair is scored from both sides) and on N^2 * D for the self-join (its upper triangle).  Each kNN result is
checked in the same run: 256 sampled rows against an fp32 brute force over all the right rows (scores within 1e-5 of the brute
force's best, every returned row's true score within 1e-5 of its reported score, counts k).  The GPU name and power limit are
read in the same run.

  python scripts/bench_knn_join.py [--n 2000000] [--out profiles/knn_join_n1.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from revers_o_b200 import _lib, ops, synth                              # noqa: E402
from revers_o_b200.sharded import knn_sharded                          # noqa: E402
from revers_o_b200.vector_db import B200VectorDB, models                # noqa: E402


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


def check(ids, scores, counts, q_tiled, q_rows, t_tiled, n_t, d, k, exclude, t_off=0, sample=256):
    """Sampled rows against an fp32 brute force over every target row (chunked): returns (ok, worst score error)."""
    dev = t_tiled.device
    g = torch.Generator(device="cpu").manual_seed(1)
    rows = torch.randperm(q_rows, generator=g)[:sample].to(dev)
    q = ops.untile_rows(q_tiled, q_rows, d, rows=rows).float()
    best = []
    for a in range(0, n_t, 1 << 18):
        b = min(n_t, a + (1 << 18))
        sc = q @ ops.untile_rows(t_tiled, n_t, d, rows=torch.arange(a, b, device=dev)).float().T
        if exclude:
            hit = (rows >= a) & (rows < b)
            sc[hit.nonzero().flatten(), (rows[hit] - a)] = -float("inf")
        best.append(sc.topk(min(k, b - a), dim=1).values)
    best = torch.cat(best, 1).topk(k, dim=1).values
    gi, gs, gc = (torch.as_tensor(x).to(dev)[rows] for x in (ids, scores, counts))
    true = (ops.untile_rows(t_tiled, n_t, d, rows=(gi - t_off).clamp(min=0).flatten()).float().view(len(rows), k, d)
            * q[:, None, :]).sum(-1)
    err = max(float((gs - best).abs().max()), float((gs - true).abs().max()))
    self_listed = exclude and bool((gi - t_off == rows[:, None]).any())
    return bool((gc == k).all()) and err <= 1e-5 and not self_listed, err


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

    src = synth.make_selfjoin_db(n, d, 0.05, dev, seed=5)
    db = B200VectorDB(device=dev)
    db.recreate_collection("all", vectors_config=models.VectorParams(size=d, distance=models.Distance.COSINE))
    for a in range(0, n, 131072):
        b = min(n, a + 131072)
        db.upsert_batch("all", range(a, b), ops.untile_rows(src, n, d, rows=torch.arange(a, b, device=dev)).float(),
                        assume_new=True, persist=False)
    del src
    c = db._coll("all")
    tiled = c.vectors                                                # the stored rows: every workload reads these
    for k in (10, 100):
        sec, ts, out = timed(lambda: ops.knn_exact(tiled, 0, n, 0, tiled, n, d, k, None, 0, True))
        ok, err = check(*out, tiled, n, tiled, n, d, k, True)
        emit({"workload": f"self kNN, {n} x {d}, k = {k}", "seconds": sec, "rounds": ts,
              "tflops_2_n_n_d": 2.0 * n * n * d / sec / 1e12, "verified": ok, "max_score_err": err})
        del out
    sec, ts, out = timed(lambda: db.knn_join("all", 10))
    ok, err = check(*out, tiled, n, tiled, n, d, 10, True)
    emit({"workload": f"B200VectorDB.knn_join, {n} x {d}, k = 10 (host arrays)", "seconds": sec, "rounds": ts,
          "tflops_2_n_n_d": 2.0 * n * n * d / sec / 1e12, "verified": ok, "max_score_err": err})
    del out
    for blk in (2048, 4096, 8192, 16384):
        _lib.set_option("knn_block", blk)
        ws = _lib.load().rvo_knn_workspace_bytes(n, d, n, 10, 0)
        sec, ts, out = timed(lambda: ops.knn_exact(tiled, 0, n, 0, tiled, n, d, 10, None, 0, True))
        ok, err = check(*out, tiled, n, tiled, n, d, 10, True)
        emit({"workload": f"self kNN, {n} x {d}, k = 10, query blocks of {blk} rows", "knn_block": blk, "workspace_bytes": ws,
              "seconds": sec, "rounds": ts, "tflops_2_n_n_d": 2.0 * n * n * d / sec / 1e12, "verified": ok, "max_score_err": err})
        del out
    _lib.set_option("knn_block", 8192)                                # the default
    base = None
    for G in (1, 2, 4):
        nblk = -(-n // 128)
        blk = -(-nblk // G)
        shards = []
        for g in range(G):
            b0, b1 = g * blk, min((g + 1) * blk, nblk)
            shards.append((tiled[b0:b1], min(n, b1 * 128) - b0 * 128, b0 * 128))
        sec, ts, out = timed(lambda: knn_sharded(shards, shards, d, 10, None, True))
        ok, err = check(*out, tiled, n, tiled, n, d, 10, True)
        base = sec if G == 1 else base
        emit({"workload": f"knn_sharded self kNN, {n} x {d}, k = 10, {G} virtual shard(s) on GPU 0", "seconds": sec, "rounds": ts,
              "tflops_2_n_n_d": 2.0 * n * n * d / sec / 1e12, "over_one_shard": sec / base, "verified": ok, "max_score_err": err})
        del out
    sec, ts, out = timed(lambda: db.find_near_duplicates("all", 0.95))
    emit({"workload": f"find_near_duplicates, {n} x {d}, cos >= 0.95 (reference)", "seconds": sec, "rounds": ts,
          "pairs": len(out[0]), "tflops_n_n_d": float(n) * n * d / sec / 1e12})
    del db, c, tiled, out
    torch.cuda.empty_cache()

    nl, nr = n // 2, n
    both = synth.make_selfjoin_db(nl + nr, d, 0.05, dev, seed=5)
    left = both[: -(-nl // 128)]                                      # rows [0, nl): the tiles holding them
    right = ops.tile_rows(ops.untile_rows(both, nl + nr, d, rows=torch.arange(nl, nl + nr, device=dev)).contiguous())
    del both
    torch.cuda.empty_cache()
    sec, ts, out = timed(lambda: ops.knn_exact(left, 0, nl, 0, right, nr, d, 10, None, 0, False))
    ok, err = check(*out, left, nl, right, nr, d, 10, False)
    emit({"workload": f"cross kNN, {nl} x {d} against {nr} x {d}, k = 10", "seconds": sec, "rounds": ts,
          "tflops_2_nl_nr_d": 2.0 * nl * nr * d / sec / 1e12, "verified": ok, "max_score_err": err})
    summary = {"gpu": info, "results": results}
    if args.out:
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)
    print(json.dumps({"gpu": info}))


if __name__ == "__main__":
    main()
