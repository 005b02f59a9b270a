#!/usr/bin/env python
"""bench.py — the reference's headline metric on B200:  exact top-100 cosine queries/s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg1|...] [--exchange auto|push|nccl]

A "step" is one pass of the hot path (rvo_search_topk: normalise queries -> threshold seeding -> fused tcgen05
scan/select -> exact top-k -> fp32 re-score) over one synthetic query batch.

  N = 1   workload cfg1 = BASELINE.json configs[1]: 1M x 1024 bf16 DB, 256-query batch, top-100 (the metric's own
          100M x 1280 DB does not fit one GPU, so the largest single-GPU search configuration is used).
  N > 1   the SAME total DB row-sharded over the N ranks (strong scaling): every rank scans its shard, the per-shard
          lists are exchanged once (peer-memory push fused into the last K2 kernel when the box allows CUDA IPC, else ONE
          NCCL all-gather), K3 merge on every rank.  Launch with torchrun (one rank per GPU).

Printed JSON (rank 0, one line):
  value         queries/s with inputs resident in HBM (CUDA events, barrier + synchronize on both sides, max over ranks)
  e2e           the same through the public API with pinned HOST buffers (H2D of the queries and D2H of ids/scores/counts
                inside the timed region): B200VectorDB.search_batch at N = 1, ShardedIndex.search + copies at N > 1
  roofline      the dominant kernel (full-shard scan) timed alone by the library's own CUDA events on its stream, against
                MEASURED_PEAKS.json; `traffic` = DRAM bytes of that kernel from the committed ncu capture (profiles/traffic.json)
  verify        the TIMED result checked in-run against a plain fp32 restatement on the GPU (every rank scores a query sample
                against its shard, lists merged on the host): ids / scores, not just counts; verify_oracle (N = 1): the CPU
                oracle itself on the downloaded DB
  north_star    BASELINE.json's metric layout — 12.5M x 1280 rows PER GPU (N = 8 is configs[3], 100M x 1280), Q = 4096 / 64 / 16 —
                as a weak-scaling series; north_star_strong: the full 100M x 1280 DB over N = 2 / 4 ranks (N = 8: the weak point)
  mask_pool     the other half of the path (K1) on configs[2], one batch per GPU (replicas, no collective)
  selfjoin      configs[4]: 2M x 1024 near-duplicate self-join at cos >= 0.95 over the N ranks, with its tensor roofline
  cfg0          configs[0], the reference's own operating point (10k x 1024, ONE query, top-10): resident, e2e, the qdrant-shaped
                `search()` call on the host clock, and the CPU oracle at full size
  cpu_baseline  the CPU oracle (numpy port of the reference's qdrant-local search) timed on this box's host cores on a
                bounded query sample, plus a labelled "fair batched" figure (one sgemm + argpartition)
  clocks, gpu_launches, local_shard_ms_per_step (N > 1: K2 alone, max over ranks)
(--no-north-star: the primary workload only.)

--dump-outputs DIR writes what the last timed step returned (ids, scores, counts of the primary workload) as DIR/<name>.npy.
It is refused with --impl reference, whose steps search a query sample of their own: nothing there to compare output for output.

`--impl reference` times that CPU implementation alone (numpy-only process; the reference's own dependency
qdrant-client is not installable here, so kind="port").
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (rows, dim, queries, k, description)
    "cfg0": (10_000, 1024, 1, 10, "configs[0]: 10k x 1024, single query, top-10"),
    "cfg1": (1_000_000, 1024, 256, 100, "configs[1]: 1M x 1024 bf16 DB, 256-query batch, top-100, fp32 rescore"),
    "cfg3": (100_000_000, 1280, 4096, 100, "configs[3]: 100M x 1280 bf16 DB row-sharded over the ranks, 4096-query batch, top-100, NCCL top-k merge"),
    "cfg3q64": (100_000_000, 1280, 64, 100, "configs[3] DB, bandwidth regime: 100M x 1280 row-sharded, 64 queries"),
    "cfg3q16": (100_000_000, 1280, 16, 100, "configs[3] DB, bandwidth regime: 100M x 1280 row-sharded, 16 queries"),
    "cfg3shard": (12_500_000, 1280, 4096, 100, "configs[3] per-GPU shard: 12.5M x 1280 bf16, 4096-query batch, top-100"),
    "cfg3shardq16": (12_500_000, 1280, 16, 100, "configs[3] per-GPU shard, bandwidth regime: 12.5M x 1280, 16 queries"),
    "cfg3shardq64": (12_500_000, 1280, 64, 100, "configs[3] per-GPU shard, bandwidth regime: 12.5M x 1280, 64 queries"),
    "cfg3shardq1": (12_500_000, 1280, 1, 100, "configs[3] per-GPU shard, the reference's operating point: 12.5M x 1280, 1 query"),
    "cfg1shard8": (125_000, 1024, 256, 100, "configs[1] per-GPU shard at 8 GPUs: 125k x 1024, 256 queries (fixed-chain diagnostics)"),
    "cfg1q1": (1_000_000, 1024, 1, 10, "configs[1] DB, the reference's operating point: 1M x 1024, 1 query, top-10"),
}
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return d, "measured"
        except Exception:
            pass
    return dict(FALLBACK_PEAKS), "fallback"


# ------------------------------------------------------------------------------------------------------
# reference arm: the CPU implementation of the path (numpy-only process)
# ------------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        # torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm runs on rank 0 alone with all host threads
        for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
            os.environ[var] = str(os.cpu_count())
    import numpy as np
    from oracle import reverso_oracle as O
    n, d, nq, k, desc = WORKLOADS[args.workload]
    t0 = time.perf_counter()
    rng = np.random.default_rng(1000)
    db = np.empty((n, d), dtype=np.float32)
    step = 1 << 16
    for lo in range(0, n, step):
        blk = rng.standard_normal((min(step, n - lo), d), dtype=np.float32)
        blk /= np.linalg.norm(blk, axis=1, keepdims=True)
        db[lo: lo + len(blk)] = O.round_to_bf16_inplace(blk)          # the same bf16-valued DB the GPU searches
    gen_s = time.perf_counter() - t0
    # bounded sample: calibrate on one query, then size the per-step query sample so that the whole
    # --steps/--warmup run stays near `--cpu-budget` seconds of CPU work
    q1 = rng.standard_normal((1, d), dtype=np.float32)
    O.search_batch(db, q1, k, None, db_is_normalized=True)
    t = time.perf_counter()
    O.search_batch(db, q1, k, None, db_is_normalized=True)
    t_q = time.perf_counter() - t
    sample_q = int(args.cpu_budget / max(t_q * (args.steps + args.warmup), 1e-9))
    sample_q = max(1, min(nq, args.sample_queries, sample_q))
    q = rng.standard_normal((sample_q, d), dtype=np.float32)

    def one_step():
        # exactly how the reference issues queries: one search() per query (core_system.py:657-664)
        return O.search_batch(db, q, k, None, db_is_normalized=True)

    for _ in range(args.warmup):
        one_step()
    times = []
    for _ in range(args.steps):
        t = time.perf_counter()
        one_step()
        times.append(time.perf_counter() - t)
    total = sum(times)
    qps = sample_q * args.steps / total
    cores = os.cpu_count()
    # second, labelled CPU figure (BASELINE.md §4): the same answer computed the way a CPU would be used fairly — one sgemm
    # over a query batch + argpartition — instead of the reference's one gemv + full argsort per query
    fair = None
    try:
        fq = rng.standard_normal((min(nq, 64), d), dtype=np.float32)
        O.search_batch_fair(db, fq[:2], k)
        t = time.perf_counter()
        O.search_batch_fair(db, fq, k)
        fair = {"value": len(fq) / (time.perf_counter() - t), "unit": "queries/s", "cores": cores,
                "what": f"one sgemm over {len(fq)} queries + argpartition (not how the reference issues queries)"}
    except Exception as e:
        fair = {"value": None, "what": f"failed: {e}"}
    line = {
        "impl": "reference", "metric": "exact top-%d cosine queries/s" % k, "value": qps, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "rows": n, "dim": d, "queries": nq, "k": k},
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port",
                         "sample": f"{sample_q} of {nq} queries per step against the full {n}x{d} fp32 DB, one numpy "
                                   f"gemv + full argsort per query (qdrant-local semantics), median step "
                                   f"{1e3 * statistics.median(times):.1f} ms, DB generation {gen_s:.1f} s untimed"},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "cpu_fair_batched": fair,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------------
# clocks sampler (NVML), runs during the timed regions
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz, self.ok = [], set(), None, False
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                mhz = self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
                util = self.nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                self.samples.append((mhz, util))
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        if self.ok:
            self.t.start()

    def stop(self):
        self._stop.set()
        if self.ok:
            self.t.join(timeout=1)
        if not self.samples:
            return None
        loaded = [m for m, u in self.samples if u > 0] or [m for m, _ in self.samples]
        return {"sm_mhz": statistics.median(loaded), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------------
def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from revers_o_b200 import _lib, ops, synth
    from revers_o_b200.sharded import ShardedIndex, selfjoin_blocks, shard_bounds
    from revers_o_b200.vector_db import B200VectorDB, models

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 arm has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.gpus != world and rank == 0:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; launch N>1 with torchrun", file=sys.stderr)

    n, d, nq, k, desc = WORKLOADS[args.workload]
    lo, hi = shard_bounds(n, world, rank)
    n_local = hi - lo
    if n_local * d * 2 > 150e9:
        raise SystemExit(f"bench.py: workload {args.workload} needs {n_local * d * 2 / 1e9:.0f} GB per GPU at {world} GPU(s); "
                         "launch it on more ranks")
    lib = _lib.load()
    for kv in filter(None, os.environ.get("RVO_OPTS", "").split(",")):  # tuning sweeps only (scripts/gpu_sweep.sh)
        name, val = kv.split("=")
        _lib.set_option(name.strip(), int(val))
    peaks, peaks_kind = load_peaks()
    extras = args.workload == "cfg1" and not args.no_north_star
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        traffic = json.load(open(tp))
    except Exception:
        traffic = {}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def min_over_ranks(ms):
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return float(t.item())

    def timed(step_fn, steps, warm):
        """`warm` untimed + exactly `steps` timed calls, CUDA events on the launching stream, barrier + synchronize
        on both sides, max over ranks.  Returns (ms per step, library kernel launches, last result)."""
        for _ in range(warm):
            out = step_fn()
        barrier()
        l0 = _lib.kernel_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            out = step_fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps, _lib.kernel_launch_count() - l0, out

    def scan_rooflines(idx, q, kk, ms_step, reps, after_idle=False):
        """The dominant kernel (full-shard scan) timed alone with CUDA events recorded by the library around that one
        launch on its stream; algorithmic bytes = n_local*d*2 (DB read once), flops = 2*Q*n_local*d (DESIGN.md §4).
        `kernel_ms` is taken in back-to-back steps (the regime `value` is measured in; for sub-millisecond tensor-heavy steps
        that is the board's power-capped regime).  `after_idle` adds the same launch timed after a 10-step burst and 20 ms of idle GPU — the
        kernel by itself at full clocks, comparable with the BURST peaks of MEASURED_PEAKS.json."""
        _lib.set_option("time_scan", 1)
        scan_ms = []
        for _ in range(reps):
            idx.search_local(q, kk)
            scan_ms.append(float(lib.rvo_last_scan_ms()))
        idle_ms = []
        if after_idle:
            for _ in range(7):
                for _ in range(10):          # a burst first: the GPU holds full clocks only after sustained load ...
                    idx.search_local(q, kk)
                torch.cuda.synchronize()
                time.sleep(0.02)             # ... then 20 ms for the power limiter to relax (0.3-3 ms would catch the clock ramp instead:
                idx.search_local(q, kk)      # scripts/dev/scan_after_idle.py, profiles/r02_chain_timeline.md)
                idle_ms.append(float(lib.rvo_last_scan_ms()))
        _lib.set_option("time_scan", 0)
        torch.cuda.synchronize()
        scan_fastest = min_over_ranks(statistics.mean(scan_ms))     # the spread between the GPUs of one box under simultaneous load
        scan_avg = max_over_ranks(statistics.mean(scan_ms))
        nq_ = q.shape[0]
        alg_bytes = idx.n_local * idx.d * 2
        alg_flops = 2.0 * nq_ * idx.n_local * idx.d
        hbm_ach = alg_bytes / (scan_avg * 1e-3) / 1e9
        tf_ach = alg_flops / (scan_avg * 1e-3) / 1e12
        small_ = nq_ <= _lib.RVO_SMALL_Q
        hbm = {"bound": "hbm", "achieved": hbm_ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
               "frac": hbm_ach / peaks["hbm_gbs"], "traffic": None, "peak_kind": peaks_kind,
               "kernel": "scan_small_kernel (fp32, every row)" if small_ else "scan_tc2_kernel<FILTER> / scan_tc_kernel<FILTER> (full-shard level)",
               "kernel_ms": scan_avg, "kernel_ms_fastest_rank": scan_fastest, "algorithmic_bytes": alg_bytes,
               "share_of_step": scan_avg / ms_step}
        if idle_ms:
            alone = max_over_ranks(statistics.median(idle_ms))
            hbm["after_idle"] = {"kernel_ms": alone, "achieved": alg_bytes / (alone * 1e-3) / 1e9, "frac": alg_bytes / (alone * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                 "tflops": alg_flops / (alone * 1e-3) / 1e12, "frac_of_burst_bf16": alg_flops / (alone * 1e-3) / 1e12 / peaks["bf16_tflops"],
                                 "what": "the same launch after a 10-step burst + 20 ms of idle GPU (median of 7): the kernel by itself at full clocks, before the board's power limiter engages"}
        tensor = None if small_ else {
            "bound": "tensor", "achieved": tf_ach, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
            "frac": tf_ach / peaks["bf16_tflops"], "peak_kind": peaks_kind + " burst (kernel timed alone)",
            # the kernel is timed inside back-to-back steps, where the board's power cap (clocks.reasons: sw_power_cap) holds
            # cuBLAS itself to the sustained figure: that is the ceiling a tensor-bound kernel can reach in this regime
            "peak_sustained": peaks.get("bf16_tflops_sustained"),
            "frac_of_sustained": (tf_ach / peaks["bf16_tflops_sustained"]) if peaks.get("bf16_tflops_sustained") else None,
            "arithmetic_intensity_flop_per_byte": alg_flops / alg_bytes,
            "machine_balance_flop_per_byte": peaks["bf16_tflops"] * 1e12 / (peaks["hbm_gbs"] * 1e9),
            "kernel": "scan_tc2_kernel<FILTER> / scan_tc_kernel<FILTER> (full-shard level)", "kernel_ms": scan_avg,
            "kernel_ms_fastest_rank": scan_fastest, "algorithmic_flops": alg_flops, "share_of_step": scan_avg / ms_step}
        return hbm, tensor

    def verify(idx, q, out, kk, n_sample=8, tol=1e-3):
        """The TIMED result, checked in-run (not just `counts == k`): a plain fp32 restatement of the search on the GPU — every
        rank scores a sample of the queries against its own shard with torch fp32 matmuls (checker code, not the product), the
        per-rank lists are gathered and merged on the host by (score desc, id asc), and compared with what the step returned:
        scores within 1e-3, identical id sets except ties within 1e-3 (north_star)."""
        nq_ = q.shape[0]
        sel = sorted(set(np.linspace(0, nq_ - 1, min(n_sample, nq_)).astype(int).tolist()))
        qs = q[sel].float()
        qs = qs / qs.norm(dim=1, keepdim=True)
        best_s = torch.full((len(sel), kk), -float("inf"), device=dev)
        best_i = torch.full((len(sel), kk), -1, dtype=torch.int64, device=dev)
        nblk = (idx.n_local + 127) // 128
        step_blk = 4096                                              # 512k rows per matmul
        for b0 in range(0, nblk, step_blk):
            b1 = min(nblk, b0 + step_blk)
            rows = idx.db[b0:b1].permute(0, 2, 1, 3).reshape((b1 - b0) * 128, -1)[:, : idx.d].float()
            sc = qs @ rows.T
            valid = idx.n_local - b0 * 128
            if valid < sc.shape[1]:
                sc[:, valid:] = -float("inf")
            kk2 = min(kk, sc.shape[1])
            ts, ti = sc.topk(kk2, dim=1)
            cs = torch.cat([best_s, ts], 1)
            ci = torch.cat([best_i, ti + b0 * 128 + idx.id_offset], 1)
            o = cs.argsort(dim=1, descending=True, stable=True)[:, :kk]
            best_s, best_i = cs.gather(1, o), ci.gather(1, o)
            del rows, sc
        part = (best_s.cpu().numpy(), best_i.cpu().numpy())
        parts = [part]
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, part)
        got_i, got_s, got_c = (t[sel].cpu().numpy() for t in out)
        if rank != 0:
            return None
        bad_ids = 0
        max_diff = 0.0
        for j in range(len(sel)):
            cs = np.concatenate([p[0][j] for p in parts])
            ci = np.concatenate([p[1][j] for p in parts])
            keep = ci >= 0
            cs, ci = cs[keep], ci[keep]
            o = np.lexsort((ci, -cs.astype(np.float64)))[:kk]
            rs, ri = cs[o], ci[o]
            c = int(got_c[j])
            if c != len(ri):
                bad_ids += abs(c - len(ri))
                continue
            max_diff = max(max_diff, float(np.max(np.abs(got_s[j, :c] - rs))) if c else 0.0)
            boundary = min(got_s[j, c - 1], rs[-1]) if c else 0.0
            smap = dict(zip(got_i[j, :c].tolist(), got_s[j, :c].tolist()))
            rmap = dict(zip(ri.tolist(), rs.tolist()))
            for i_ in set(smap) ^ set(rmap):
                if abs(smap.get(i_, rmap.get(i_)) - boundary) > tol:
                    bad_ids += 1
        return {"checker": "fp32 restatement on the GPU (torch matmul per shard + host merge), compared with the timed step's result",
                "queries_checked": len(sel), "k": kk, "max_abs_score_diff": max_diff, "ids_differing_beyond_1e-3_ties": bad_ids,
                "ok": bool(bad_ids == 0 and max_diff <= tol)}

    # ---- primary workload: value with inputs resident in HBM ------------------------------------------------
    q_dev = synth.make_queries(nq, d, seed=7, device=dev)
    db = synth.make_db(n_local, d, q_dev, n_plant=max(1, 128 // world), seed=1000 + rank, device=dev)
    index = ShardedIndex(db, n_local, d, lo)
    exchange = "none"
    if world > 1:
        exchange = "peer-memory push fused into K2 (NVLink stores + epoch flags)" if (
            args.exchange != "nccl" and index.enable_peer_exchange(nq, k)) else "NCCL all_gather_into_tensor"
    sampler = ClockSampler(local)
    sampler.start()
    ms_serial, launches, out_serial = timed(lambda: index.search(q_dev, k), args.steps, max(3, args.warmup))
    serial_check = verify(index, q_dev, out_serial, k)
    out_serial = tuple(t.clone() for t in out_serial)

    # The same K steps through the pipelined public API (ShardedIndex.submit / collect, two batches in flight): the scan of step
    # i+1 is enqueued before the exchange + merge of step i, so a rank scans while it waits for the slowest peer's lists; on one
    # GPU the two batches run on two streams.  This is `value`; the synchronous call is reported next to it as `serial`.
    def pipe_block(steps):
        prev, res = None, None
        for _ in range(steps):
            t = index.submit(q_dev, k)
            if prev is not None:
                res = index.collect(prev)
            prev = t
        return index.collect(prev)

    pipe_block(max(3, args.warmup))
    barrier()
    l0 = _lib.kernel_launch_count()
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    pe0.record()
    out = pipe_block(args.steps)
    pe1.record()
    barrier()
    ms_step = max_over_ranks(pe0.elapsed_time(pe1)) / args.steps
    launches = _lib.kernel_launch_count() - l0
    value = nq / (ms_step / 1e3)
    counts_ok = bool((out[2] == k).all().item()) and bool(torch.equal(out[0], out_serial[0]) and torch.equal(out[2], out_serial[2]))
    last_step = [t.cpu().numpy() for t in out] if args.dump_outputs and rank == 0 else None   # the buffers are reused by later submits
    check = verify(index, q_dev, out, k)

    # N > 1: the same step without the exchange + merge (K2 on the local shard only), to show what the exchange costs
    local_ms = None
    if world > 1:
        local_ms, _, _ = timed(lambda: index.search_local(q_dev, k), args.steps, 3)

    # ---- roofline: the dominant kernel (full-shard scan) ------------------------------------------------
    roofline, roofline_tensor = scan_rooflines(index, q_dev, k, ms_step, max(5, min(args.steps, 30)), after_idle=n_local * d * 2 < 8e9)
    small = nq <= _lib.RVO_SMALL_Q
    alg_bytes = n_local * d * 2
    roofline["traffic"] = traffic.get(args.workload)
    if roofline_tensor is not None and nq >= 1024:     # tensor-bound regime: the tensor roofline is the binding one
        roofline_tensor["traffic"] = roofline["traffic"]
        roofline, roofline_hbm = roofline_tensor, roofline
    else:
        roofline_hbm = None
        if roofline_tensor is not None:
            ai, mb = roofline_tensor["arithmetic_intensity_flop_per_byte"], roofline_tensor["machine_balance_flop_per_byte"]
            roofline["note"] = (f"Q = {nq}: arithmetic intensity {ai:.0f} FLOP/B vs machine balance {mb:.0f} — on the ridge; in back-to-back "
                                "steps the board is power-capped (clocks.reasons) and the tensor side binds: see roofline_tensor.frac_of_sustained")

    # ---- e2e: public API with HOST buffers (N=1: B200VectorDB.search_batch; N>1: H2D + sharded search + D2H) --
    q_host = q_dev.cpu().numpy()
    h2d = q_host.nbytes
    d2h = nq * k * 12 + nq * 4
    oracle_check = None
    if world == 1:
        vdb = B200VectorDB(device=dev)
        vdb.recreate_collection("bench", vectors_config=models.VectorParams(size=d, distance=models.Distance.COSINE))
        c = vdb._coll("bench")
        c.vectors, c.n = db, n_local            # adopt the resident shard (ids/payload tables are not on the hot path)

        q_pinned = torch.from_numpy(q_host).pin_memory()   # the step's inputs live in pinned host memory (bench contract)

        def step_e2e():
            return vdb.search_batch("bench", q_pinned, k)
    else:
        pin_q = torch.from_numpy(q_host).pin_memory()
        pi = torch.empty((nq, k), dtype=torch.int64).pin_memory()
        ps = torch.empty((nq, k), dtype=torch.float32).pin_memory()
        pc = torch.empty((nq,), dtype=torch.int32).pin_memory()

        qd = torch.empty_like(q_dev)
        zero_copy_in = os.environ.get("RVO_E2E_ZC_IN", "0") == "1"
        zero_copy_out = os.environ.get("RVO_E2E_ZC_OUT", "0") == "1"

        def step_e2e():
            if zero_copy_in:
                qq = pin_q                      # first kernel reads the queries from pinned host memory
            else:
                qd.copy_(pin_q, non_blocking=True)
                qq = qd
            if zero_copy_out:                   # K3 writes the results into pinned host memory
                index.search(qq, k, out=(pi, ps, pc))
            else:
                a, b, c_ = index.search(qq, k)
                pi.copy_(a, non_blocking=True); ps.copy_(b, non_blocking=True); pc.copy_(c_, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return pi, ps, pc
    e2e_ms, _, e2e_out = timed(step_e2e, args.steps, max(3, args.warmup))
    # N = 1: the same K steps through the pipelined public API (two batches in flight, each with its own stream / scratch /
    # pinned buffers): every step still copies its queries in and its results out inside the timed region
    pipe = None
    if world == 1:
        from collections import deque

        def run_pipe(steps):
            hs, last = deque(), None
            for _ in range(steps):
                hs.append(vdb.search_batch_async("bench", q_pinned, k))
                if len(hs) == 2:
                    last = hs.popleft().result()
            while hs:
                last = hs.popleft().result()
            return last
        run_pipe(max(3, args.warmup))
        torch.cuda.synchronize()
        pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        pe0.record()
        pipe_out = run_pipe(args.steps)          # result() of the last batch returns after its D2H copy has landed
        pe1.record()
        torch.cuda.synchronize()
        pipe_ms = pe0.elapsed_time(pe1) / args.steps
        pipe = {"value": nq / (pipe_ms / 1e3), "unit": "queries/s", "ms_per_step": pipe_ms, "pipeline_depth": 2,
                "api": "B200VectorDB.search_batch_async(pinned host tensor).result(), two batches in flight",
                "same_result_as_blocking_call": bool(all(np.array_equal(a, b) for a, b in zip(pipe_out, e2e_out)))}
    clocks = sampler.stop()
    # the e2e result is the same answer as the resident one
    e2e_same = bool(np.array_equal(np.asarray(e2e_out[0]), out[0].cpu().numpy()) and
                    np.array_equal(np.asarray(e2e_out[2]), out[2].cpu().numpy()))

    # N = 1: the CPU ORACLE itself on a query sample of the timed configuration (the DB is downloaded: the same bf16 values)
    if world == 1 and not args.no_cpu_baseline and n_local * d * 4 < 8e9:
        from oracle import reverso_oracle as O
        sel = sorted(set(np.linspace(0, nq - 1, min(4, nq)).astype(int).tolist()))
        dbf = np.empty((n_local, d), np.float32)
        for r0 in range(0, n_local, 1 << 18):
            r1 = min(n_local, r0 + (1 << 18))
            dbf[r0:r1] = ops.untile_rows(db, n_local, d, torch.arange(r0, r1, device=dev)).float().cpu().numpy()
        ref = O.search_batch(dbf, q_host[sel], k, None, db_is_normalized=True)
        del dbf
        gi, gs, gc = (np.asarray(t)[sel] for t in e2e_out)
        worst, bad = 0.0, 0
        for j, (rid, rsc) in enumerate(ref):
            if int(gc[j]) != len(rid):
                bad += 1
                continue
            worst = max(worst, float(np.max(np.abs(gs[j, : len(rid)] - rsc))))
            smap, rmap = dict(zip(gi[j].tolist(), gs[j].tolist())), dict(zip(rid.tolist(), rsc.tolist()))
            boundary = min(gs[j, len(rid) - 1], rsc[-1])
            bad += sum(1 for i_ in set(smap) ^ set(rmap) if abs(smap.get(i_, rmap.get(i_)) - boundary) > 1e-3)
        oracle_check = {"checker": "oracle/reverso_oracle.py (numpy restatement of qdrant-local search) on the downloaded bf16-valued DB, "
                                   "compared with the timed e2e result", "queries_checked": len(sel),
                        "max_abs_score_diff": worst, "ids_differing_beyond_1e-3_ties": bad, "ok": bool(bad == 0 and worst <= 1e-3)}

    index.disable_peer_exchange()
    del index, db
    if world == 1:
        del vdb, c
    torch.cuda.empty_cache()

    # ---- north star series (BASELINE.json metric: 100M x 1280 at 1/2/4/8 GPUs) -----------------------------------------
    # weak: every rank holds ITS 12.5M-row shard of the 8-GPU layout (N = 8 IS configs[3]);
    # strong: the full 100M x 1280 DB row-sharded over the N ranks where it fits (N = 2: 128 GB per GPU, N = 4: 64 GB; N = 8 is
    # the weak point; one GPU cannot hold 256 GB)
    def ns_series(rows_per_gpu, queries_list, seed0, what):
        ns_d = 1280
        q_all = synth.make_queries(4096, ns_d, seed=7, device=dev)
        ns_db = synth.make_db(rows_per_gpu, ns_d, q_all, n_plant=16, seed=seed0 + rank, device=dev)
        ns_index = ShardedIndex(ns_db, rows_per_gpu, ns_d, rank * rows_per_gpu)
        if world > 1 and args.exchange != "nccl":
            ns_index.enable_peer_exchange(4096, 100)
        pts = []
        for ns_q in queries_list:
            qd_ = q_all[:ns_q].contiguous()
            # small batches: the first ~20 steps after the tensor-bound phase run up to 20 % slower (measured; clocks
            # settling), so they get a longer warm-up
            ns_steps, ns_warm = ((5, 3) if rows_per_gpu <= 12_500_000 else (3, 2)) if ns_q >= 1024 else (20, 20)
            ns_ms, _, ns_out = timed(lambda: ns_index.search(qd_, 100), ns_steps, ns_warm)
            ns_check = verify(ns_index, qd_, ns_out, 100, n_sample=4)
            r_h, r_t = scan_rooflines(ns_index, qd_, 100, ns_ms, 3)
            if rows_per_gpu == 12_500_000:
                r_h["traffic"] = traffic.get({4096: "cfg3shard", 64: "cfg3shardq64", 16: "cfg3shardq16"}.get(ns_q))
                if r_t is not None:
                    r_t["traffic"] = r_h["traffic"]
            pts.append({"queries": ns_q, "value": ns_q / (ns_ms / 1e3), "unit": "queries/s", "ms_per_step": ns_ms, "steps": ns_steps,
                        "results_ok": bool((ns_out[2] == 100).all().item()) and (ns_check is None or ns_check["ok"]),
                        "verify": ns_check, "roofline": r_t if ns_q >= 1024 else r_h})
        ns_index.disable_peer_exchange()
        del ns_db, ns_index
        torch.cuda.empty_cache()
        return {"workload": what, "rows_per_gpu": rows_per_gpu, "rows_total": rows_per_gpu * world, "dim": ns_d, "points": pts}

    north = strong = None
    if extras:
        north = ns_series(12_500_000, (4096, 64, 16), 2000,
                          f"configs[3] shard layout: 12.5M x 1280 bf16 rows per GPU x {world} GPU(s) = {12.5 * world:.1f}M rows "
                          "total, top-100, exchange + K3 merge when N > 1")
        north["scaling"] = "weak"
        if world in (2, 4) and not args.no_strong:
            rows = 100_000_000 // world // 128 * 128
            strong = ns_series(rows, (4096,), 3000,
                               f"configs[3] STRONG-scaled: the full 100M x 1280 bf16 DB row-sharded over {world} GPUs "
                               f"({rows * 1280 * 2 / 1e9:.0f} GB per GPU), 4096-query batch, top-100, exchange + K3 merge")
            strong["scaling"] = "strong"
        elif world == 8:
            strong = {"scaling": "strong", "note": "at 8 GPUs the strong-scaled configs[3] IS the weak series' point (12.5M rows per GPU)",
                      "points": [p for p in north["points"] if p["queries"] == 4096]}
        else:
            strong = {"scaling": "strong", "note": "100M x 1280 bf16 = 256 GB does not fit one B200 (180 GB): strong points exist "
                                                   "for N = 2, 4, 8", "points": []}

    # ---- K1 (the other half of the path): mask pooling on BASELINE configs[2]; N > 1: independent replicas ---------------
    pool = None
    if extras:
        pB, pM, pG, pD = 256, 64, 24, 1024
        feats, masks = synth.make_maskpool_inputs(pB, pM, pG, pD, seed=11 + rank, device=dev)
        p_bufs = ops.mask_pool(feats, masks)                                            # result tensors reused across steps
        p_ms, p_launches, p_out = timed(lambda: ops.mask_pool(feats, masks, out=p_bufs), 20, 5)   # 311 MB of inputs > L2: streams HBM
        regions = int(p_out[3].item())
        alg = pB * pG * pG * pD * 2 + pB * pM * pG * pG + regions * pD * 4
        pool = {"workload": "configs[2]: 256 images x 64 masks x 24x24 patches x 1024-d bf16 features (random-init stand-in), "
                            "fp32 L2-normalised region embeddings out" + (f"; {world} independent replicas (one batch per GPU)" if world > 1 else ""),
                "value": world * pB / (p_ms / 1e3), "unit": "images/s", "ms_per_batch": p_ms, "regions_per_batch": regions,
                "gpu_launches_per_batch": p_launches / 20, "scaling": "replicas only (no collective)",
                "roofline": {"bound": "hbm", "achieved": alg / (p_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                             "frac": alg / (p_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], "algorithmic_bytes": alg,
                             "traffic": traffic.get("mask_pool"),
                             "kernel": "mask_pool_tc_kernel (whole rvo_mask_pool call: memset + one launch), per GPU",
                             "peak_kind": peaks_kind}}
        del feats, masks, p_out
        torch.cuda.empty_cache()

    # ---- configs[4]: near-duplicate self-join, 2M x 1024, cos >= 0.95; DB replicated, query blocks dealt over the ranks ----
    selfjoin = None
    if extras and not args.no_selfjoin:
        sn, sd, thr = 2_000_000, 1024, 0.95
        sdb = synth.make_selfjoin_db(sn, sd, 0.05, dev, seed=5)               # same seed on every rank: replicated DB
        ops.selfjoin_threshold(sdb, sn, sd, thr, 0, min(sn, 8192), out_cap=1 << 20)   # warm-up
        blocks = selfjoin_blocks(sn, world, rank)
        cnt = torch.zeros(1, dtype=torch.int64, device=dev)
        ovf = torch.zeros(1, dtype=torch.int64, device=dev)
        kept = []
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.kernel_launch_count()
        e0.record()
        for blo, bhi in blocks:
            pairs, scores, count, over = ops.selfjoin_threshold(sdb, sn, sd, thr, blo, bhi, out_cap=1 << 21)
            cnt += count
            ovf += over
            kept.append((blo, bhi, pairs, count))
        e1.record()
        barrier()
        sj_s = max_over_ranks(e0.elapsed_time(e1)) / 1e3
        sj_launches = _lib.kernel_launch_count() - l0
        # in-run check: for a sample of this rank's query rows, every partner j > i with fp32 cos >= 0.95 (GPU restatement)
        rows_f = None
        bad_rows, checked = 0, 0
        rs = np.random.RandomState(rank)
        for blo, bhi, pairs, count in kept[:2]:
            m = int(count.item())
            pr = pairs[:m].cpu().numpy()
            for i_ in rs.randint(blo, bhi, 8).tolist():
                vi = ops.untile_rows(sdb, sn, sd, torch.tensor([i_], device=dev)).float()[0]
                sc = torch.empty(0, device=dev)
                want, near = set(), set()
                for c0 in range((i_ + 1) // 128 * 128, sn, 1 << 19):
                    c1 = min(sn, c0 + (1 << 19))
                    blk = sdb[c0 // 128: (c1 + 127) // 128].permute(0, 2, 1, 3).reshape(-1, sdb.shape[1] * 64)[: c1 - c0, :sd].float()
                    s_ = blk @ vi
                    jj = torch.arange(c0, c1, device=dev)
                    ok_ = jj > i_
                    want |= set(jj[ok_ & (s_ >= thr)].tolist())
                    near |= set(jj[ok_ & ((s_ - thr).abs() <= 1e-3)].tolist())
                got = set(pr[pr[:, 0] == i_][:, 1].tolist())
                checked += 1
                if not ((got ^ want) <= near):
                    bad_rows += 1
        tot = torch.stack([cnt.squeeze(), ovf.squeeze(), torch.tensor(bad_rows, device=dev), torch.tensor(checked, device=dev)])
        if world > 1:
            dist.all_reduce(tot)
        flops = float(sn) * sn * sd                       # 2 * (N^2 / 2) * D: only the upper triangle is scanned
        selfjoin = {"workload": f"configs[4]: near-duplicate self-join, {sn} x {sd} bf16 frame embeddings, cos >= {thr}, 5 % planted "
                                f"near-duplicates; DB replicated on {world} GPU(s), 4096-row query blocks dealt in snake order, no "
                                "data-path collective",
                    "value": sn / sj_s, "unit": "rows joined/s", "seconds": sj_s, "pairs": int(tot[0].item()),
                    "overflowed_lists": int(tot[1].item()), "gpu_launches": int(sj_launches),
                    "verify": {"checker": "fp32 restatement on the GPU of all partners of sampled query rows", "rows_checked": int(tot[3].item()),
                               "rows_with_wrong_partner_sets": int(tot[2].item()), "ok": bool(int(tot[2].item()) == 0 and int(tot[1].item()) == 0)},
                    "roofline": {"bound": "tensor", "achieved": flops / sj_s / 1e12 / world, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                                 "frac": flops / sj_s / 1e12 / world / peaks["bf16_tflops"], "algorithmic_flops": flops,
                                 "flops_definition": "N^2 * D: upper triangle only (block b scans rows >= b), per GPU = total / N",
                                 "traffic": traffic.get("selfjoin"), "traffic_note": "every 4096-row query block re-streams the DB tail "
                                 "(~N/4096/2 passes over the 4.1 GB DB ~ 1 TB of HBM reads at N = 2M); harmless while tensor-bound",
                                 "kernel": "scan_tc2_kernel<FILTER> per 4096-row query block + pairs_kernel", "peak_kind": peaks_kind + " burst"}}
        del sdb, kept
        torch.cuda.empty_cache()

    # ---- configs[0]: the reference's own operating point — 10k x 1024, ONE query, top-10 (rank 0, N = 1 semantics) ---------
    cfg0 = None
    if extras and rank == 0:
        n0, d0, k0 = 10_000, 1024, 10
        q0 = synth.make_queries(1, d0, seed=7, device=dev)
        db0 = synth.make_db(n0, d0, q0, n_plant=32, seed=1000, device=dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def time_local(fn, steps=300, warm=30):
            for _ in range(warm):
                fn()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(steps):
                r_ = fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / steps, r_
        prep0 = ops.PreparedSearch(db0, n0, d0, q0, k0, 0.0)      # the prepared call a serving loop uses: one ctypes call per search
        res_ms, res_out = time_local(prep0)
        v0 = B200VectorDB(device=dev)
        v0.recreate_collection("c0", vectors_config=models.VectorParams(size=d0, distance=models.Distance.COSINE))
        c0 = v0._coll("c0")
        c0.vectors, c0.n = db0, n0
        c0.ids.append([f"{i:032x}" for i in range(n0)], assume_new=True)
        c0.payloads.append_or_set(np.arange(n0), [{"filename": f"f{i}.jpg"} for i in range(n0)])
        q0_pin = q0.cpu().pin_memory()
        e2e0_ms, e2e0_out = time_local(lambda: v0.search_batch("c0", q0_pin, k0, 0.0))
        q0_list = q0[0].cpu().numpy().tolist()
        t0 = time.perf_counter()
        for _ in range(200):
            hits0 = v0.search("c0", q0_list, limit=k0, score_threshold=0.0)      # exactly core_system.py:659-664
        api_ms = (time.perf_counter() - t0) / 200 * 1e3
        from oracle import reverso_oracle as O
        dbf0 = ops.untile_rows(db0, n0, d0).float().cpu().numpy()
        rid, rsc = O.search(dbf0, q0[0].cpu().numpy(), k0, 0.0, db_is_normalized=True)
        ok0 = bool(len(hits0) == len(rid) and [h.id for h in hits0] == [f"{i:032x}" for i in rid.tolist()]
                   and np.max(np.abs(np.array([h.score for h in hits0]) - rsc)) <= 1e-3)
        cpu0 = None
        if not args.no_cpu_baseline and world == 1:      # under torchrun the rank's BLAS has one thread: not a CPU baseline
            tq = []
            O.search(dbf0, q0[0].cpu().numpy(), k0, 0.0, db_is_normalized=True)
            for _ in range(50):
                t_ = time.perf_counter()
                O.search(dbf0, q0[0].cpu().numpy(), k0, 0.0, db_is_normalized=True)
                tq.append(time.perf_counter() - t_)
            cpu0 = {"value": 1.0 / statistics.median(tq), "unit": "queries/s", "cores": os.cpu_count(), "kind": "port",
                    "sample": "full size: 10k x 1024 fp32 DB, one numpy gemv + full argsort per query, median of 50 (same process as "
                              "torch: BLAS threads shared)"}
        cfg0 = {"workload": WORKLOADS["cfg0"][4] + " — what core_system.search_similar issues (core_system.py:657-664)",
                "value": 1e3 / res_ms, "unit": "queries/s", "ms_per_query": res_ms, "gpu_launches_per_query": 2,
                "e2e": {"value": 1e3 / e2e0_ms, "unit": "queries/s", "ms_per_query": e2e0_ms, "h2d_bytes_per_step": d0 * 4,
                        "d2h_bytes_per_step": k0 * 12 + 4, "api": "B200VectorDB.search_batch(pinned host query)"},
                "api_search": {"ms_per_query": api_ms, "api": "B200VectorDB.search(collection, python list, limit, score_threshold) -> "
                               "ScoredPoints with uuid + payload: the qdrant call core_system.py:659-664 makes, host clock"},
                "verify": {"checker": "oracle/reverso_oracle.py on the downloaded DB", "ok": ok0}, "cpu_baseline": cpu0}
        del db0, v0, c0
        torch.cuda.empty_cache()

    # ---- cpu baseline (rank 0, N=1): the oracle port in a numpy-only subprocess, bounded sample ----------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", args.workload,
                   "--steps", "3", "--warmup", "1", "--sample-queries", str(args.sample_queries)]
            p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
            ref_line = json.loads(p.stdout.strip().splitlines()[-1])
            cpu = ref_line["cpu_baseline"]
            cpu["fair_batched"] = ref_line.get("cpu_fair_batched")
        except Exception as e:  # the GPU numbers stand on their own
            cpu = {"value": None, "unit": "queries/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}

    if rank == 0:
        line = {
            "metric": "exact top-%d cosine queries/s" % k, "value": value, "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True,
            "serial": {"value": nq / (ms_serial / 1e3), "unit": "queries/s", "ms_per_step": ms_serial,
                       "api": "ShardedIndex.search (synchronous: every step ends with its own exchange + merge)",
                       "verify_ok": None if serial_check is None else serial_check["ok"]},
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": desc, "rows": n, "dim": d, "queries": nq, "k": k, "rows_per_gpu": n_local,
                       "parallelism": f"row-shard x{world}" if world > 1 else "single GPU", "exchange": exchange,
                       "l2": f"inputs larger than L2: each step streams the {alg_bytes / 1e9:.2f} GB shard",
                       "pipeline_depth": 2, "api": "ShardedIndex.submit / collect (two batches in flight; `serial` = ShardedIndex.search)",
                       "path": "fp32 CUDA-core scan (Q <= 4)" if small else "tcgen05 scan + fused threshold select (hot lists) + fp32 rescore"},
            "e2e": {"value": nq / (e2e_ms / 1e3), "unit": "queries/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "same_result_as_resident_step": e2e_same, "pipelined": pipe,
                    "api": "B200VectorDB.search_batch(pinned host tensor) -> numpy ids/scores/counts" if world == 1 else "ShardedIndex.search(pinned host queries, out=pinned host results): K2 + exchange + K3"},
            "gpu_launches": int(launches), "local_shard_ms_per_step": local_ms,
            "roofline": roofline, "roofline_tensor": roofline_tensor, "roofline_hbm": roofline_hbm,
            "verify": check, "verify_oracle": oracle_check,
            "north_star": north, "north_star_strong": strong, "mask_pool": pool, "selfjoin": selfjoin, "cfg0": cfg0,
            "cpu_baseline": cpu, "clocks": clocks,
            "sass": "profiles/r02_sass_excerpt.txt (cuobjdump -sass of the shipped .so: UTCHMMA / LDTM / UTMALDG per kernel)",
            "results_ok": bool(counts_ok and (check is None or check["ok"]) and e2e_same and (oracle_check is None or oracle_check["ok"])),
        }
        print(json.dumps(line), flush=True)
        if last_step is not None:
            dump_outputs(args.dump_outputs, *last_step)
    if world > 1:
        dist.destroy_process_group()
    return 0


def dump_outputs(out_dir, ids, scores, counts):
    """The merged (ids, scores, counts) of the last timed step, as ShardedIndex.collect hands them to a caller, so that two builds
    can be compared output for output (the inputs are seeded).  At most 4096 x 100 results: under 5 MB in all."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "ids.npy"), ids.astype(np.float64))          # global row ids < 2**53: exact in float64
    np.save(os.path.join(out_dir, "scores.npy"), scores.astype(np.float32))
    np.save(os.path.join(out_dir, "counts.npy"), counts.astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg1", choices=sorted(WORKLOADS))
    ap.add_argument("--sample-queries", type=int, default=8, help="queries per CPU step (bounded sample)")
    ap.add_argument("--cpu-budget", type=float, default=60.0, help="seconds of CPU work for the reference arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--exchange", default="auto", choices=["auto", "push", "nccl"],
                    help="N > 1: per-shard lists exchanged by the fused peer-memory push (default when available) or NCCL")
    ap.add_argument("--no-north-star", action="store_true",
                    help="primary workload only: skip the north-star series, K1, the self-join and configs[0]")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaled 100M x 1280 point (N = 2, 4)")
    ap.add_argument("--no-selfjoin", action="store_true", help="skip configs[4] (2M x 1024 self-join)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's ids / scores / counts to DIR/<name>.npy (float64 / float32 / float64); "
                         "B200 arm only: --impl reference times a query sample of its own, not comparable output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the result of the B200 arm's timed step")
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
