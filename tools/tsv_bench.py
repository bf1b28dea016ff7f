#!/usr/bin/env python
"""The reference's _simulation.txt from the GPU (out="tsv", path=...), plain and gzipped, against the 10x directory.

C4 cells of tools/mtx_bench.py: C4 tree (15 branches x 50 steps, K=10, G=20 000), hybrid sampler, 131 072 cells per
call at library size x e^m for m = -2 and m = 0.  Per depth, warmed up and then alternated, --reps whole
sample_density calls of each arm into the same directory (host clock; the output is deleted outside the timed
window, no fsync), median:
  * arms: out="tsv"; out="tsv", compress=True; out="tsv", compress=True, compression="lz77"; out="mtx".  Per arm:
    seconds, counts/s, the file's bytes (and bytes per count), the file write rate;
  * disk_write: a plain write() loop of the plain file's byte count, in 64 MB blocks, into the same directory.
Device rates (CUDA events, --kernel-reps launches each) on one chunk of --kernel-cells cells of the m = 0 counts
(larger than the 126 MB L2): pst_tsv_row_bytes (GB/s of int32 counts read), pst_tsv_format (GB/s of text written)
and pst_deflate_blocks over that text (GB/s of text read).
Host baseline: tree_utils.save_matrices (pandas to_csv) of the out="numpy" counts of the first --host-cells cells of
each depth, counts/s, and that rate extrapolated to the whole call (labelled as an extrapolation).

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
from csr_bench import gpu_info  # noqa: E402
from csr_npz_bench import remove  # noqa: E402
from csr_stream_bench import write_loop  # noqa: E402
from mtx_bench import event_rate  # noqa: E402
from prosstt_b200 import _native as nat, device as pdev, hostpool, simulation as sim, tree_utils  # noqa: E402


def kernel_rates(X, reps, dev):
    """Device rates of the two TSV kernels and of the deflate over their text, on the int32 chunk X."""
    lib = nat.load()
    st = nat.stream_ptr(dev)
    n, G = X.shape
    rb = torch.empty(n, dtype=torch.int32, device=dev)
    tp = torch.empty(n + 1, dtype=torch.int64, device=dev)
    nat.call("pst_tsv_row_bytes", X, n, G, G, 0, rb, st)
    nat.call("pst_csr_row_offsets", rb, n, tp, st)
    text_len = int(tp[n].item())
    text = torch.empty(text_len + 16, dtype=torch.uint8, device=dev)
    block = pdev._DEFLATE_BLOCK
    out = torch.empty(int(lib.pst_deflate_bound(text_len, block)), dtype=torch.uint8, device=dev)
    ws = int(lib.pst_deflate_workspace_bytes(text_len, block))
    work = torch.empty(max(1, ws), dtype=torch.uint8, device=dev)
    size = torch.zeros(1, dtype=torch.int64, device=dev)
    crc = torch.zeros(2, dtype=torch.int32, device=dev)
    s_rb = event_rate(lambda: nat.call("pst_tsv_row_bytes", X, n, G, G, 0, rb, st), reps, dev)
    s_fmt = event_rate(lambda: nat.call("pst_tsv_format", X, n, G, G, 0, tp, text_len, text, st), reps, dev)
    s_def = event_rate(lambda: nat.call("pst_deflate_blocks", text, None, 0, text_len, block, out, size, crc, work, ws,
                                        st), reps, dev)
    return {"cells": n, "genes": G, "counts": n * G, "text_bytes": text_len, "launches": reps,
            "tsv_row_bytes": {"seconds": s_rb, "counts_GB_per_s": 4.0 * n * G / s_rb / 1e9},
            "tsv_format": {"seconds": s_fmt, "text_GB_per_s": text_len / s_fmt / 1e9, "counts_per_s": n * G / s_fmt},
            "deflate_blocks_over_text": {"seconds": s_def, "text_GB_per_s": text_len / s_def / 1e9,
                                         "compressed_over_text": int(size.item()) / float(text_len)}}


def host_baseline(X, work):
    """counts/s of tree_utils.save_matrices (pandas to_csv) of the int64 host matrix X."""
    t0 = time.perf_counter()
    tree_utils.save_matrices("base", work, X, {}, np.zeros(1))
    dt = time.perf_counter() - t0
    path = os.path.join(work, "base_simulation.txt")
    nbytes = os.path.getsize(path)
    for f in os.listdir(work):
        if f.startswith("base_"):
            os.remove(os.path.join(work, f))
    return {"cells": X.shape[0], "counts": int(X.size), "seconds": dt, "counts_per_s": X.size / dt,
            "bytes_per_count": nbytes / float(X.size)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=131072)
    ap.add_argument("--depths", type=float, nargs="+", default=[-2.0, 0.0])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--kernel-cells", type=int, default=4096)
    ap.add_argument("--kernel-reps", type=int, default=20)
    ap.add_argument("--host-cells", type=int, default=4096)
    ap.add_argument("--dir", default=None, help="directory for the outputs (default: a new temporary directory)")
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    work = tempfile.mkdtemp(dir=a.dir, prefix="tsv_")
    doc = {"what": "the reference's _simulation.txt (out='tsv', path=), plain and gzipped, vs out='mtx'",
           "gpu": gpu_info(), "host_threads": len(os.sched_getaffinity(0)),
           "disk_free_bytes": shutil.disk_usage(work).free, "c4": []}
    try:
        w = dict(bench.WORKLOADS["c4"])
        t0 = time.time()
        tree = bench.build_tree_gpu(w, dev)
        alpha, beta = bench.gene_hyper(w["G"])
        G, n = w["G"], a.cells
        doc["c4_tree"] = "15 branches x 50 steps, K=10, G=%d, hybrid sampler, %d cells per call" % (G, n)
        doc["c4_tree_build_s"] = time.time() - t0
        for m in a.depths:
            kw = dict(alpha=alpha, beta=beta, device=dev, sampler="hybrid", scale_mean=m, seed=1000)
            paths = {"call_tsv": os.path.join(work, "x_simulation.txt"),
                     "call_tsv_gzip": os.path.join(work, "x_simulation.txt.gz"),
                     "call_tsv_gzip_lz77": os.path.join(work, "x_lz_simulation.txt.gz"),
                     "call_mtx": os.path.join(work, "x10")}
            calls = {"call_tsv": dict(out="tsv"), "call_tsv_gzip": dict(out="tsv", compress=True),
                     "call_tsv_gzip_lz77": dict(out="tsv", compress=True, compression="lz77"),
                     "call_mtx": dict(out="mtx")}
            arms = {name: (paths[name], (lambda p=paths[name], o=calls[name]: sim.sample_density(tree, n, path=p,
                                                                                                 **o, **kw)[0]))
                    for name in calls}
            sizes = {}
            for name, (p, fn) in arms.items():
                sizes[name] = fn().nbytes
                remove(p)
            # the host baseline on the first host-cells cells of the same call
            X = sim.sample_density(tree, a.host_cells, **kw)[0]
            base = host_baseline(X, work)
            del X
            times = {k: [] for k in list(arms) + ["disk_write"]}
            for r in range(a.reps + 1):                        # round 0 is the warm-up
                for name, (p, fn) in arms.items():
                    gc.collect()
                    torch.cuda.synchronize(dev)
                    c0 = time.perf_counter()
                    out = fn()
                    dt = time.perf_counter() - c0
                    del out
                    remove(p)
                    if r:
                        times[name].append(dt)
                c0 = time.perf_counter()
                write_loop(os.path.join(work, "plain.bin"), sizes["call_tsv"])
                if r:
                    times["disk_write"].append(time.perf_counter() - c0)
            counts = n * G
            res = {"scale_mean": m, "counts": counts, "text_bytes_per_count": sizes["call_tsv"] / float(counts),
                   "arms": {}}
            for name, ts in times.items():
                med = float(np.median(ts))
                res["arms"][name] = {"seconds": ts, "median_s": med}
                if name == "disk_write":
                    res["arms"][name]["GB_per_s"] = sizes["call_tsv"] / med / 1e9
                    continue
                res["arms"][name].update(counts_per_s=counts / med, file_bytes=sizes[name],
                                         bytes_per_count=sizes[name] / float(counts),
                                         written_GB_per_s=sizes[name] / med / 1e9)
            tsv_s = res["arms"]["call_tsv"]["median_s"]
            res["tsv_over_disk_write_time"] = tsv_s / res["arms"]["disk_write"]["median_s"]
            res["host_baseline_save_matrices"] = dict(base, extrapolated_full_call_s=counts / base["counts_per_s"],
                                                      note="extrapolated from the slice, not measured on the whole call")
            res["speedup_vs_host_baseline_extrapolated"] = {
                name: counts / base["counts_per_s"] / res["arms"][name]["median_s"]
                for name in ("call_tsv", "call_tsv_gzip", "call_tsv_gzip_lz77")}
            if m == a.depths[-1]:
                res["device_kernels"] = kernel_rates(
                    sim.sample_density(tree, a.kernel_cells, out="torch", **kw)[0], a.kernel_reps, dev)
            hostpool.release()
            torch.cuda.empty_cache()
            doc["c4"].append(res)
            print(json.dumps(res, indent=1), file=sys.stderr, flush=True)
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
