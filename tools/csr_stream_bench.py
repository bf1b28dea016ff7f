#!/usr/bin/env python
"""CSR streamed chunk by chunk (CountEngine.stream_csr, out="csr", path=...) against the in-memory out="csr".

C4 tree (15 branches x 50 steps, K=10, G=20 000), hybrid sampler, 131 072 cells per call at library size x e^m
for m = -2 and m = 0: the shape of tools/csr_bench.py, so the two files compare.  Per depth, warmed up and then
alternated, --reps calls of each arm (host clock around work that ends in a device synchronise), median:
  * stream_discard: CountEngine.stream_csr into a consumer that drops every chunk (int32 indices, int64 data),
    on the cells and scalings of the sample_density call;
  * in_memory: CountEngine.draw_to_csr on the same cells (two passes);
  * call_in_memory / call_path: sample_density(out="csr") and sample_density(out="csr", path=...) into --dir,
    whole calls; the shard is deleted outside the timed window (no fsync here, nor in disk_write);
    skipped when --dir has less free space than three shards;
  * disk_write: a plain write() loop of the shard's byte count, in 64 MB blocks, into --dir (the rate of the
    page cache and the disk under it, for the path arm to be read against);
  * the peak RSS (VmHWM after clear_refs) of one call of each arm, above the RSS before it.
Config 5 (5M cells x 30 000 genes, the bench.py c5 tree) on one GPU through stream_csr into the discarding
consumer at --c5-depths: wall time, counts/s, nnz (its zero fraction) and the peak RSS of the call.

Prints one JSON document (and writes it to --json PATH if given); GPU name and power limit are read in the
same run."""
import argparse
import gc
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
from csr_bench import gpu_info, reset_hwm, vm  # noqa: E402
from prosstt_b200 import hostpool, simulation as sim  # noqa: E402


def cells_of(tree, n, **kw):
    """(engine, rows, scalings32, seed, first) of a sample_density call, without drawing its counts."""
    got = {}
    real = sim._sample_counts

    def capture(engine, rows, s32, seed, first, dtype, out, **_):
        got.update(engine=engine, rows=rows, s32=s32, seed=seed, first=first)

    sim._sample_counts = capture
    try:
        sim.sample_density(tree, n, out="csr", **kw)
    finally:
        sim._sample_counts = real
    return got["engine"], got["rows"], got["s32"], got["seed"], got["first"]


def discard(lo, hi, indptr, indices, data):
    pass


def dir_bytes(path):
    return sum(os.path.getsize(os.path.join(path, f)) for f in os.listdir(path))


def write_loop(path, nbytes, block=64 << 20):
    buf = np.ones(block, dtype=np.uint8)
    left = nbytes
    with open(path, "wb") as fh:
        while left > 0:
            k = min(block, left)
            fh.write(memoryview(buf[:k]))
            left -= k
    os.remove(path)


def peak_of(fn):
    """(result, peak RSS above the RSS before the call, or None)."""
    hostpool.release()
    gc.collect()
    ok = reset_hwm()
    base = vm("VmRSS")
    out = fn()
    peak = vm("VmHWM")
    return out, (peak - base if ok else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=131072)
    ap.add_argument("--depths", type=float, nargs="+", default=[-2.0, 0.0])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--c5-cells", type=int, default=5000000)
    ap.add_argument("--c5-depths", type=float, nargs="*", default=[0.0, -2.0])
    ap.add_argument("--dir", default=None, help="directory for the shards (default: a new temporary directory)")
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    work = tempfile.mkdtemp(dir=a.dir, prefix="csr_stream_")
    doc = {"what": "CSR streamed per chunk (stream_csr / out='csr', path=) vs in-memory out='csr'",
           "gpu": gpu_info(), "host_threads": len(os.sched_getaffinity(0)), "c4": [], "c5": []}
    try:
        w = dict(bench.WORKLOADS["c4"])
        t0 = time.time()
        tree = bench.build_tree_gpu(w, dev)
        alpha, beta = bench.gene_hyper(w["G"])
        G, n = w["G"], a.cells
        doc["c4_tree"] = "15 branches x 50 steps, K=10, G=%d, hybrid sampler, %d cells per call" % (G, n)
        doc["c4_tree_build_s"] = time.time() - t0
        for m in a.depths:
            kw = dict(alpha=alpha, beta=beta, device=dev, sampler="hybrid", scale_mean=m)
            seed = 1000
            eng, rows, s32, dseed, first = cells_of(tree, n, seed=seed, **kw)
            shard = os.path.join(work, "x.csr")

            def sync(x):
                torch.cuda.synchronize(dev)
                return x

            arms = {
                "stream_discard": lambda: sync(eng.stream_csr(rows, s32, dseed, first, discard, np.int32, np.int64)),
                "in_memory": lambda: sync(eng.draw_to_csr(rows, s32, dseed, first)),
                "call_in_memory": lambda: sim.sample_density(tree, n, seed=seed, out="csr", **kw)[0],
                "call_path": lambda: sim.sample_density(tree, n, seed=seed, out="csr", path=shard, **kw)[0],
            }
            # the same matrix on every arm
            nnz = arms["stream_discard"]()
            mem = arms["in_memory"]()
            free = shutil.disk_usage(work).free
            if free < 3 * (16 * nnz + 8 * (n + 1)):
                del arms["call_path"]
                check = {"nnz_equal": int(mem[0][-1]) == nnz}
                shard_bytes = None
            else:
                X = arms["call_path"]()
                check = {"nnz_equal": int(mem[0][-1]) == nnz == X.nnz,
                         "arrays_equal": bool(np.array_equal(X.indptr, mem[0]) and np.array_equal(X.indices, mem[1])
                                              and np.array_equal(X.data, mem[2]))}
                shard_bytes = dir_bytes(shard)
                del X
                shutil.rmtree(shard)
            del mem
            times = {k: [] for k in list(arms) + (["disk_write"] if shard_bytes else [])}
            for r in range(a.reps + 1):                        # round 0 is the warm-up
                for k, fn in arms.items():
                    gc.collect()
                    torch.cuda.synchronize(dev)
                    c0 = time.perf_counter()
                    out = fn()
                    dt = time.perf_counter() - c0
                    del out
                    if k == "call_path":
                        shutil.rmtree(shard)
                    if r:
                        times[k].append(dt)
                if shard_bytes:
                    c0 = time.perf_counter()
                    write_loop(os.path.join(work, "plain.bin"), shard_bytes)
                    if r:
                        times["disk_write"].append(time.perf_counter() - c0)
            res = {"scale_mean": m, "nnz": nnz, "zero_fraction": 1.0 - nnz / float(n * G), "check": check,
                   "shard_bytes": shard_bytes, "dir_free_bytes": free, "arms": {}}
            for k, ts in times.items():
                med = float(np.median(ts))
                res["arms"][k] = {"seconds": ts, "median_s": med}
                if k == "disk_write":
                    res["arms"][k]["GB_per_s"] = shard_bytes / med / 1e9
                else:
                    res["arms"][k].update(counts_per_s=n * G / med, nnz_per_s=nnz / med)
                    if k == "call_path":
                        res["arms"][k]["shard_GB_per_s"] = shard_bytes / med / 1e9
            res["stream_discard_speedup_vs_in_memory"] = (res["arms"]["in_memory"]["median_s"]
                                                          / res["arms"]["stream_discard"]["median_s"])
            if "call_path" in arms:
                res["call_path_vs_call_in_memory"] = (res["arms"]["call_in_memory"]["median_s"]
                                                      / res["arms"]["call_path"]["median_s"])
            for k, fn in arms.items():
                out, peak = peak_of(fn)
                del out
                if k == "call_path":
                    shutil.rmtree(shard)
                res["arms"][k]["peak_rss_above_start_bytes"] = peak
            hostpool.release()
            del eng, rows, s32
            torch.cuda.empty_cache()
            doc["c4"].append(res)
            print(json.dumps(res, indent=1), file=sys.stderr, flush=True)
        del tree
        torch.cuda.empty_cache()
        if a.c5_depths:
            w = dict(bench.WORKLOADS["c5"])
            t0 = time.time()
            tree = bench.build_tree_gpu(w, dev)
            alpha, beta = bench.gene_hyper(w["G"])
            G, n = w["G"], a.c5_cells
            doc["c5_tree"] = "bench.py c5: 49 branches x 1000 steps, K=10, G=%d, hybrid sampler, %d cells" % (G, n)
            doc["c5_tree_build_s"] = time.time() - t0
            for m in a.c5_depths:
                eng, rows, s32, dseed, first = cells_of(tree, n, alpha=alpha, beta=beta, device=dev,
                                                        sampler="hybrid", scale_mean=m, seed=2000)
                torch.cuda.synchronize(dev)
                c0 = time.perf_counter()
                nnz, peak = peak_of(lambda: eng.stream_csr(rows, s32, dseed, first, discard, np.int64, np.int64))
                torch.cuda.synchronize(dev)
                dt = time.perf_counter() - c0
                res = {"scale_mean": m, "cells": n, "genes": G, "seconds": dt, "counts_per_s": n * G / dt,
                       "nnz": nnz, "nnz_per_s": nnz / dt, "zero_fraction": 1.0 - nnz / float(n * G),
                       "csr_bytes_int64_indices_int64_data": 16 * nnz + 8 * (n + 1),
                       "peak_rss_above_start_bytes": peak}
                doc["c5"].append(res)
                print(json.dumps(res, indent=1), file=sys.stderr, flush=True)
                del eng, rows, s32
                torch.cuda.empty_cache()
    finally:
        shutil.rmtree(work, ignore_errors=True)
    doc["gpu_after"] = gpu_info()
    text = json.dumps(doc, indent=1)
    print(text)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
