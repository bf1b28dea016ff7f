#!/usr/bin/env python
"""compression="lz77" against the Huffman-only default, for both GPU-compressed outputs.

Whole calls: the C4 call of tools/mtx_bench.py (131 072 cells x 20 000 genes, hybrid sampler) at m = -2 and
m = 0, out="mtx" and out="csr", compress=True, each with compression="huffman" and "lz77".  After a warm-up round,
--reps rounds alternate the four arms (host clock around the whole call, output deleted outside the timed
window, no fsync); per arm the median seconds, file bytes per nonzero and the file write rate.
Kernel alone (CUDA events, --kernel-reps launches after 3 warm-up launches): pst_deflate_blocks and
pst_deflate_lz_blocks over one chunk of --kernel-cells cells of the m = 0 counts: its Matrix Market text and its
int64 indices and data (each larger than the 126 MB L2); GB/s of input and compressed / input.
Host baseline: zlib level 1 and 6 over the first --zlib-mb MB of the same three streams, in independent
32 KiB blocks each ended by a sync flush (the kernels' framing).

Prints one JSON document (and writes it to --json PATH); GPU name and power limit are read in the same run."""
import argparse
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
from prosstt_b200 import _native as nat, device as pdev, hostpool, simulation as sim  # noqa: E402

KERNELS = {"huffman": ("pst_deflate_blocks", "pst_deflate_workspace_bytes"),
           "lz77": ("pst_deflate_lz_blocks", "pst_deflate_lz_workspace_bytes")}


def streams(X, dev):
    """The mtx text (pst_mtx_format) and the int64 indices / data bytes of the int32 chunk X, on the device."""
    st = nat.stream_ptr(dev)
    n, G = X.shape
    rb = torch.empty(n, dtype=torch.int32, device=dev)
    tp = torch.empty(n + 1, dtype=torch.int64, device=dev)
    nat.call("pst_mtx_row_bytes", X, n, G, G, 0, rb, st)
    nat.call("pst_csr_row_offsets", rb, n, tp, st)
    text_len = int(tp[n].item())
    text = torch.empty(text_len + 16, dtype=torch.uint8, device=dev)
    nat.call("pst_mtx_format", X, n, G, G, 0, tp, text_len, text, st)
    nz = X.flatten().nonzero().flatten()
    return {"mtx_text": text[:text_len],
            "indices_int64": (nz % G).to(torch.int64).view(torch.uint8),
            "data_int64": X.flatten()[nz].to(torch.int64).view(torch.uint8)}


def kernel_rates(data, reps, dev):
    lib = nat.load()
    st = nat.stream_ptr(dev)
    block = pdev._DEFLATE_BLOCK
    n = int(data.numel())
    out = torch.empty(int(lib.pst_deflate_bound(n, block)), dtype=torch.uint8, device=dev)
    size = torch.zeros(1, dtype=torch.int64, device=dev)
    crc = torch.zeros(2, dtype=torch.int32, device=dev)
    res = {"input_bytes": n}
    for mode, (fn, wfn) in KERNELS.items():
        ws = int(getattr(lib, wfn)(n, block))
        work = torch.empty(max(1, ws), dtype=torch.uint8, device=dev)
        s = event_rate(lambda: nat.call(fn, data, None, 0, n, block, out, size, crc, work, ws, st), reps, dev)
        res[mode] = {"seconds": s, "input_GB_per_s": n / s / 1e9, "compressed_over_input": int(size.item()) / n}
        del work
    return res


def zlib_blocks(raw, level, block=32768):
    t0, total = time.perf_counter(), 0
    for i in range(0, len(raw), block):
        c = zlib.compressobj(level, zlib.DEFLATED, -15)
        total += len(c.compress(raw[i:i + block]) + c.flush(zlib.Z_SYNC_FLUSH))
    return {"compressed_over_input": total / len(raw), "host_seconds": time.perf_counter() - t0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=131072)
    ap.add_argument("--depths", type=float, nargs="+", default=[-2.0, 0.0])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--kernel-cells", type=int, default=4096)
    ap.add_argument("--kernel-reps", type=int, default=20)
    ap.add_argument("--zlib-mb", type=int, default=64)
    ap.add_argument("--dir", default=None, help="directory for the outputs (default: a new temporary directory)")
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    work = tempfile.mkdtemp(dir=a.dir, prefix="lz_")
    doc = {"what": "compression='lz77' vs 'huffman' for out='mtx' and out='csr', compress=True",
           "gpu": gpu_info(), "host_threads": len(os.sched_getaffinity(0)), "c4": []}
    try:
        w = dict(bench.WORKLOADS["c4"])
        tree = bench.build_tree_gpu(w, dev)
        alpha, beta = bench.gene_hyper(w["G"])
        G, n = w["G"], a.cells
        doc["c4_tree"] = "15 branches x 50 steps, K=10, G=%d, hybrid sampler, %d cells per call" % (G, n)
        for m in a.depths:
            kw = dict(alpha=alpha, beta=beta, device=dev, sampler="hybrid", scale_mean=m, seed=1000)
            arms = {}
            for mode in ("huffman", "lz77"):
                tenx, npz = os.path.join(work, "x10_" + mode), os.path.join(work, "x_%s.npz" % mode)
                arms["mtx_" + mode] = (tenx, lambda p=tenx, c=mode: sim.sample_density(
                    tree, n, out="mtx", path=p, compression=c, **kw)[0])
                arms["npz_" + mode] = (npz, lambda p=npz, c=mode: sim.sample_density(
                    tree, n, out="csr", path=p, compress=True, compression=c, **kw)[0])
            times = {k: [] for k in arms}
            sizes, nnz = {}, None
            for r in range(a.reps + 1):                        # round 0 is the warm-up
                for name, (p, fn) in arms.items():
                    gc.collect()
                    torch.cuda.synchronize(dev)
                    c0 = time.perf_counter()
                    rec = fn()
                    dt = time.perf_counter() - c0
                    sizes[name], nnz = rec.nbytes, rec.nnz
                    del rec
                    remove(p)
                    if r:
                        times[name].append(dt)
            res = {"scale_mean": m, "nnz": nnz, "arms": {}}
            for name, ts in times.items():
                med = float(np.median(ts))
                res["arms"][name] = {"seconds": ts, "median_s": med, "file_bytes": sizes[name],
                                     "bytes_per_nnz": sizes[name] / float(nnz), "nnz_per_s": nnz / med,
                                     "written_GB_per_s": sizes[name] / med / 1e9}
            for out in ("mtx", "npz"):
                h, z = res["arms"][out + "_huffman"], res["arms"][out + "_lz77"]
                res[out + "_lz77_over_huffman"] = {"size": z["file_bytes"] / h["file_bytes"],
                                                   "time": z["median_s"] / h["median_s"]}
            if m == a.depths[-1]:
                X = sim.sample_density(tree, a.kernel_cells, out="torch", **kw)[0]
                res["kernel_chunk"] = {"cells": a.kernel_cells, "genes": G, "launches": a.kernel_reps}
                for name, data in streams(X, dev).items():
                    r_ = kernel_rates(data, a.kernel_reps, dev)
                    raw = data[:a.zlib_mb << 20].cpu().numpy().tobytes()
                    r_["zlib_host_first_MB"] = len(raw) / float(1 << 20)
                    r_["zlib_level1"] = zlib_blocks(raw, 1)
                    r_["zlib_level6"] = zlib_blocks(raw, 6)
                    res["kernel_chunk"][name] = r_
                del X
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
