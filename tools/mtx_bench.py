#!/usr/bin/env python
"""10x directory (out="mtx", path=...) against the compressed CSR file (out="csr", path=..., compress=True).

C4 cells of tools/csr_npz_bench.py: C4 tree (15 branches x 50 steps, K=10, G=20 000), hybrid sampler, 131 072
cells per call at library size x e^m for m = -2 and m = 0.  Per depth, warmed up and then alternated, --reps whole
sample_density calls of each arm into the same directory (host clock; the output is deleted outside the timed
window, no fsync), median:
  * per arm: seconds, nonzeros/s, bytes per nonzero of matrix.mtx.gz / of the .npz, the file write rate, and the
    peak RSS (VmHWM after clear_refs) of one call above the RSS before it;
  * for the 10x directory: text bytes per nonzero, and the seconds close() waited for the small files
    (features, barcodes, cellparams), which a worker thread builds while the matrix streams;
  * disk_write: a plain write() loop of matrix.mtx.gz's byte count, in 64 MB blocks, into the same directory.
Device rates (CUDA events, --kernel-reps launches each) on one chunk of --kernel-cells cells of the m = 0 counts
(larger than the 126 MB L2): pst_mtx_row_bytes (GB/s of int32 counts read), pst_mtx_format (GB/s of text written)
and pst_deflate_blocks over that text (GB/s of text read).
Host baseline: scipy.io.mmwrite into gzip.open (level 6) of the first --host-cells cells of each depth, nonzeros/s,
and that rate extrapolated to the whole call (labelled as an extrapolation).
Small files alone: their host build time at the C4 and the C5 (5 000 000) cell counts.

Prints one JSON document (and writes it to --json PATH if given); GPU name and power limit are read in the
same run."""
import argparse
import concurrent.futures
import gc
import gzip
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np
import scipy.io
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
from csr_bench import gpu_info  # noqa: E402
from csr_npz_bench import remove  # noqa: E402
from csr_stream_bench import peak_of, write_loop  # noqa: E402
from prosstt_b200 import _native as nat, device as pdev, formats, hostpool, simulation as sim  # noqa: E402


class _Recorder(formats.MtxWriter):
    """The writer of the samplers, remembering the text length and the wait for the small files of its last
    close()."""
    last = None

    def close(self):
        t0 = time.perf_counter()
        concurrent.futures.wait([self._small])
        waited = time.perf_counter() - t0
        super().close()
        _Recorder.last = {"text_bytes": self._raw + formats.MTX_HEADER_BYTES, "small_files_wait_s": waited}


def event_rate(fn, reps, dev):
    """Seconds per launch of fn, CUDA events around reps launches after 3 warm-up launches."""
    for _ in range(3):
        fn()
    main = torch.cuda.current_stream(dev)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(main)
    for _ in range(reps):
        fn()
    t1.record(main)
    t1.synchronize()
    return t0.elapsed_time(t1) / 1e3 / reps


def kernel_rates(X, reps, dev):
    """Device rates of the two text kernels and of the deflate over their text, on the int32 chunk X."""
    lib = nat.load()
    st = nat.stream_ptr(dev)
    n, G = X.shape
    rb = torch.empty(n, dtype=torch.int32, device=dev)
    tp = torch.empty(n + 1, dtype=torch.int64, device=dev)
    nat.call("pst_mtx_row_bytes", X, n, G, G, 0, rb, st)
    nat.call("pst_csr_row_offsets", rb, n, tp, st)
    text_len = int(tp[n].item())
    text = torch.empty(text_len + 16, dtype=torch.uint8, device=dev)
    block = pdev._DEFLATE_BLOCK
    out = torch.empty(int(lib.pst_deflate_bound(text_len, block)), dtype=torch.uint8, device=dev)
    ws = int(lib.pst_deflate_workspace_bytes(text_len, block))
    work = torch.empty(max(1, ws), dtype=torch.uint8, device=dev)
    size = torch.zeros(1, dtype=torch.int64, device=dev)
    crc = torch.zeros(2, dtype=torch.int32, device=dev)
    s_rb = event_rate(lambda: nat.call("pst_mtx_row_bytes", X, n, G, G, 0, rb, st), reps, dev)
    s_fmt = event_rate(lambda: nat.call("pst_mtx_format", X, n, G, G, 0, tp, text_len, text, st), reps, dev)
    s_def = event_rate(lambda: nat.call("pst_deflate_blocks", text, None, 0, text_len, block, out, size, crc, work, ws,
                                        st), reps, dev)
    nnz = int((X != 0).sum().item())
    return {"cells": n, "genes": G, "nnz": nnz, "text_bytes": text_len, "launches": reps,
            "mtx_row_bytes": {"seconds": s_rb, "counts_GB_per_s": 4.0 * n * G / s_rb / 1e9},
            "mtx_format": {"seconds": s_fmt, "text_GB_per_s": text_len / s_fmt / 1e9, "nnz_per_s": nnz / s_fmt},
            "deflate_blocks_over_text": {"seconds": s_def, "text_GB_per_s": text_len / s_def / 1e9,
                                         "compressed_over_text": int(size.item()) / float(text_len)}}


def host_baseline(M, path):
    """nonzeros/s of scipy.io.mmwrite into gzip.open (genes x cells) of the csr matrix M."""
    t0 = time.perf_counter()
    with gzip.open(path, "wb") as fh:
        scipy.io.mmwrite(fh, M.T.tocoo())
    dt = time.perf_counter() - t0
    os.remove(path)
    return {"cells": M.shape[0], "nnz": int(M.nnz), "seconds": dt, "nnz_per_s": M.nnz / dt}


def small_files(n, G, work):
    """Host seconds to build and write the three small files of n cells."""
    rng = np.random.RandomState(0)
    cells = (rng.randint(0, 750, n), np.array(["b%d" % v for v in rng.randint(0, 15, n)]), rng.rand(n) * 3)
    t0 = time.perf_counter()
    for name, text in (("features", formats.mtx_features(G)), ("barcodes", formats.mtx_barcodes(0, n)),
                       ("cellparams", formats.mtx_cell_params(0, *cells))):
        with open(os.path.join(work, name + ".tsv.gz"), "wb") as fh:
            fh.write(formats.gzip_member(text))
    dt = time.perf_counter() - t0
    for name in ("features", "barcodes", "cellparams"):
        os.remove(os.path.join(work, name + ".tsv.gz"))
    return {"cells": n, "genes": G, "seconds": dt}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=131072)
    ap.add_argument("--depths", type=float, nargs="+", default=[-2.0, 0.0])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--kernel-cells", type=int, default=4096)
    ap.add_argument("--kernel-reps", type=int, default=20)
    ap.add_argument("--host-cells", type=int, default=4096)
    ap.add_argument("--c5-cells", type=int, default=5000000)
    ap.add_argument("--dir", default=None, help="directory for the outputs (default: a new temporary directory)")
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    sim.MtxWriter = _Recorder
    work = tempfile.mkdtemp(dir=a.dir, prefix="mtx_")
    doc = {"what": "10x directory (out='mtx', path=) vs the compressed CSR file (out='csr', path=, compress=True)",
           "gpu": gpu_info(), "host_threads": len(os.sched_getaffinity(0)), "c4": []}
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
            tenx, npz = os.path.join(work, "x10"), os.path.join(work, "x.npz")
            arms = {"call_mtx": (tenx, lambda: sim.sample_density(tree, n, out="mtx", path=tenx, **kw)[0]),
                    "call_npz": (npz, lambda: sim.sample_density(tree, n, out="csr", path=npz, compress=True, **kw)[0])}
            rec = arms["call_mtx"][1]()
            crec = arms["call_npz"][1]()
            nnz = int(rec.nnz)
            text_bytes = _Recorder.last["text_bytes"]
            sizes = {"call_mtx": rec.nbytes, "call_npz": crec.nbytes}
            for p, _ in arms.values():
                remove(p)
            # the host baseline on the first host-cells cells of the same call
            M = sim.sample_density(tree, a.host_cells, out="csr", **kw)[0]
            base = host_baseline(M, os.path.join(work, "base.mtx.gz"))
            del M
            times = {k: [] for k in list(arms) + ["disk_write"]}
            waits = []
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
                        if name == "call_mtx":
                            waits.append(_Recorder.last["small_files_wait_s"])
                c0 = time.perf_counter()
                write_loop(os.path.join(work, "plain.bin"), sizes["call_mtx"])
                if r:
                    times["disk_write"].append(time.perf_counter() - c0)
            res = {"scale_mean": m, "nnz": nnz, "nnz_equal": nnz == crec.nnz, "zero_fraction": 1.0 - nnz / float(n * G),
                   "text_bytes_per_nnz": text_bytes / float(nnz), "arms": {}}
            for name, ts in times.items():
                med = float(np.median(ts))
                res["arms"][name] = {"seconds": ts, "median_s": med}
                if name == "disk_write":
                    res["arms"][name]["GB_per_s"] = sizes["call_mtx"] / med / 1e9
                    continue
                res["arms"][name].update(nnz_per_s=nnz / med, file_bytes=sizes[name],
                                         bytes_per_nnz=sizes[name] / float(nnz), written_GB_per_s=sizes[name] / med / 1e9)
            mtx_s = res["arms"]["call_mtx"]["median_s"]
            res["arms"]["call_mtx"]["small_files_wait_s_median"] = float(np.median(waits))
            res["arms"]["call_mtx"]["small_files_wait_share"] = float(np.median(waits)) / mtx_s
            res["mtx_over_npz_time"] = mtx_s / res["arms"]["call_npz"]["median_s"]
            res["host_baseline_mmwrite_gzip"] = dict(base, extrapolated_full_call_s=nnz / base["nnz_per_s"],
                                                     note="extrapolated from the slice, not measured on the whole call")
            res["mtx_speedup_vs_host_baseline_extrapolated"] = nnz / base["nnz_per_s"] / mtx_s
            for name, (p, fn) in arms.items():
                out, peak = peak_of(fn)
                del out
                remove(p)
                res["arms"][name]["peak_rss_above_start_bytes"] = peak
            if m == a.depths[-1]:
                res["device_kernels"] = kernel_rates(
                    sim.sample_density(tree, a.kernel_cells, out="torch", **kw)[0], a.kernel_reps, dev)
            hostpool.release()
            torch.cuda.empty_cache()
            doc["c4"].append(res)
            print(json.dumps(res, indent=1), file=sys.stderr, flush=True)
        doc["small_files_host_build"] = [small_files(c, 20000, work) for c in (a.cells, a.c5_cells)]
        doc["small_files_note"] = ("host seconds to build and gzip features, barcodes and cellparams alone; in a call "
                                   "they overlap the matrix stream on a worker thread, and close() waits "
                                   "small_files_wait_s for them")
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
