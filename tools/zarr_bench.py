#!/usr/bin/env python
"""AnnData Zarr output of the counts (out="zarr", path=...), plain and zlib-compressed, against the compressed CSR file
and the Parquet directory.

C4 cells of tools/mtx_bench.py: C4 tree (15 branches x 50 steps, K=10, G=20 000), hybrid sampler, 131 072 cells per
call at library size x e^m for m = -2 and m = 0.  Per depth, warmed up and then alternated, --reps whole
sample_density calls of each arm into the same path (host clock; the output is deleted outside the timed window, no
fsync), median:
  * arms: out="zarr"; out="zarr", compress=True (huffman); the same with compression="lz77"; out="csr", path=,
    compress=True; out="parquet".  Per arm: seconds, counts/s, the bytes of X (the chunk files of X, the .npz, or
    counts.parquet) and bytes per nonzero.
Device times (CUDA events, --kernel-reps launches each) on the int64 data array of one chunk of --kernel-cells cells
of the m = 0 counts (larger than the 126 MB L2), cut into Zarr chunks: pst_zarr_cut (the carry step), and the
Huffman-only compressor over the whole chunks with Adler-32 per Zarr chunk (pst_deflate_segments) and with the CRC-32
of the whole input instead (pst_deflate_blocks).
Host baseline: the raw Zarr chunks of X (indptr, indices, data) of the first --host-cells cells of each depth
compressed by zlib.compress(level=1) on all host cores, and that rate extrapolated by nonzeros to the whole call
(labelled as an extrapolation).

Prints one JSON document (and writes it to --json PATH if given); GPU name and power limit are read in the
same run."""
import argparse
import concurrent.futures
import gc
import json
import os
import shutil
import sys
import tempfile
import time
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
from csr_bench import gpu_info  # noqa: E402
from csr_npz_bench import remove  # noqa: E402
from mtx_bench import event_rate  # noqa: E402
from prosstt_b200 import _native as nat, formats, hostpool, simulation as sim  # noqa: E402
from prosstt_b200.device import _DEFLATE_BLOCK  # noqa: E402


def kernel_times(X, reps, dev):
    """Device times of the carry step and of the compressor with and without Adler-32 on the int64 data of X."""
    lib = nat.load()
    st = nat.stream_ptr(dev)
    n, G = X.shape
    row_nnz = torch.empty(n, dtype=torch.int32, device=dev)
    indptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
    nat.call("pst_csr_row_counts", X, n, G, G, row_nnz, None, st)
    nat.call("pst_csr_row_offsets", row_nnz, n, indptr, st)
    nnz = int(indptr[n].item())
    indices = torch.empty(nnz, dtype=torch.int32, device=dev)
    data = torch.empty(nnz, dtype=torch.int64, device=dev)
    flags = torch.zeros(1, dtype=torch.int32, device=dev)
    nat.call("pst_csr_pack", X, n, G, G, indptr, 0, indices, 32, data, 64, None, None, 0, None, flags, st)
    chunk_bytes = 8 * formats.ZARR_CHUNK
    most = 8 * nnz
    seg_bytes = int(lib.pst_zarr_seg_bytes(most, chunk_bytes))
    seg = torch.empty(seg_bytes, dtype=torch.uint8, device=dev)
    prev = torch.zeros(16, dtype=torch.uint8, device=dev)
    prev_state = torch.zeros(2, dtype=torch.int64, device=dev)
    state = torch.empty(2, dtype=torch.int64, device=dev)
    nseg = torch.empty(1, dtype=torch.int64, device=dev)
    count = indptr[n:n + 1]

    def cut():
        nat.call("pst_zarr_cut", prev, prev_state, data, count, 8, most, chunk_bytes, 1, seg, seg_bytes, state, nseg,
                 st)

    cut()
    whole = int(nseg.item())
    block = _DEFLATE_BLOCK
    out = torch.empty(int(lib.pst_deflate_bound(seg_bytes, block)), dtype=torch.uint8, device=dev)
    out_bytes = torch.empty(1, dtype=torch.int64, device=dev)
    offsets = torch.empty(seg_bytes // chunk_bytes + 1, dtype=torch.int64, device=dev)
    adler = torch.empty(seg_bytes // chunk_bytes, dtype=torch.int32, device=dev)
    crc = torch.empty(1, dtype=torch.int32, device=dev)
    work_bytes = int(lib.pst_deflate_workspace_bytes(seg_bytes, block))
    work = torch.empty(work_bytes, dtype=torch.uint8, device=dev)

    def segments():
        nat.call("pst_deflate_segments", seg, nseg, chunk_bytes, seg_bytes, block, chunk_bytes // block, out,
                 out_bytes, offsets, adler, work, work_bytes, st)

    def blocks():
        nat.call("pst_deflate_blocks", seg, nseg, chunk_bytes, seg_bytes, block, out, out_bytes, crc, work,
                 work_bytes, st)

    t_cut = event_rate(cut, reps, dev)
    t_seg = event_rate(segments, reps, dev)
    t_blk = event_rate(blocks, reps, dev)
    raw = whole * chunk_bytes
    return {"cells": n, "genes": G, "nonzeros": nnz, "zarr_chunks": whole, "launches": reps,
            "zarr_cut": {"seconds": t_cut, "GB_per_s_read_plus_written": (8 * nnz + raw) / t_cut / 1e9},
            "deflate_segments_adler": {"seconds": t_seg, "input_GB_per_s": raw / t_seg / 1e9},
            "deflate_blocks_crc": {"seconds": t_blk, "input_GB_per_s": raw / t_blk / 1e9}}


def host_baseline(m):
    """zlib.compress(level=1) of the raw Zarr chunks of the csr matrix m's X arrays, on all host cores."""
    chunks = []
    for a in (m.indptr.astype("<i8"), m.indices.astype("<i4"), m.data.astype("<i8")):
        chunks += [c for c in formats.zarr_chunks(a.tobytes(), formats.ZARR_CHUNK * a.itemsize, False)]
    threads = len(os.sched_getaffinity(0))
    with concurrent.futures.ThreadPoolExecutor(threads) as pool:
        t0 = time.perf_counter()
        out = list(pool.map(lambda c: zlib.compress(c, 1), chunks))
        dt = time.perf_counter() - t0
    return {"cells": m.shape[0], "nonzeros": int(m.nnz), "threads": threads, "raw_bytes": sum(len(c) for c in chunks),
            "compressed_bytes": sum(len(c) for c in out), "seconds": dt, "nonzeros_per_s": m.nnz / dt}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=131072)
    ap.add_argument("--depths", type=float, nargs="+", default=[-2.0, 0.0])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--kernel-cells", type=int, default=8192)
    ap.add_argument("--kernel-reps", type=int, default=20)
    ap.add_argument("--host-cells", type=int, default=4096)
    ap.add_argument("--dir", default=None, help="directory for the outputs (default: a new temporary directory)")
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    work = tempfile.mkdtemp(dir=a.dir, prefix="zarr_")
    doc = {"what": "AnnData Zarr output of the counts (out='zarr', path=), plain and zlib, vs out='csr', compress=True "
                   "and out='parquet'",
           "gpu": gpu_info(), "host_threads": len(os.sched_getaffinity(0)),
           "disk_free_bytes": shutil.disk_usage(work).free, "zarr_chunk": formats.ZARR_CHUNK, "c4": []}
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
            calls = {"call_zarr": dict(out="zarr"), "call_zarr_zlib": dict(out="zarr", compress=True),
                     "call_zarr_zlib_lz77": dict(out="zarr", compress=True, compression="lz77"),
                     "call_csr_npz": dict(out="csr", compress=True), "call_parquet": dict(out="parquet")}
            paths = {name: os.path.join(work, name + (".npz" if name == "call_csr_npz" else "")) for name in calls}
            arms = {name: (paths[name], (lambda p=paths[name], o=calls[name]: sim.sample_density(tree, n, path=p,
                                                                                                 **o, **kw)[0]))
                    for name in calls}
            sizes, nnz = {}, None
            for name, (p, fn) in arms.items():
                rec = fn()
                sizes[name], nnz = rec.nbytes, rec.nnz
                remove(p)
            base = host_baseline(sim.sample_density(tree, a.host_cells, out="csr", **kw)[0])
            times = {k: [] for k in arms}
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
            counts = n * G
            res = {"scale_mean": m, "counts": counts, "nonzeros": nnz, "arms": {}}
            for name, ts in times.items():
                med = float(np.median(ts))
                res["arms"][name] = {"seconds": ts, "median_s": med, "counts_per_s": counts / med,
                                     "x_bytes": sizes[name], "bytes_per_nonzero": sizes[name] / float(nnz)}
            res["host_baseline_zlib"] = dict(base, note="zlib.compress(level=1) of the raw Zarr chunks of X of the "
                                                        "first host-cells cells, on all host cores")
            res["host_baseline_extrapolated_full_call_s"] = nnz / base["nonzeros_per_s"]
            res["host_baseline_extrapolated_note"] = "extrapolated from the slice by nonzeros, not measured on the call"
            if m == a.depths[-1]:
                res["device_kernels"] = kernel_times(
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
