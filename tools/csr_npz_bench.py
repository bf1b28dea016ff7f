#!/usr/bin/env python
"""Compressed CSR file (out="csr", path=..., compress=True) against the uncompressed shard (out="csr", path=...).

C4 cells of tools/csr_stream_bench.py: C4 tree (15 branches x 50 steps, K=10, G=20 000), hybrid sampler, 131 072
cells per call at library size x e^m for m = -2 and m = 0.  Per depth, warmed up and then alternated, --reps whole
sample_density calls of each arm into the same directory (host clock; the output is deleted outside the timed
window, no fsync), median:
  * call_path: the shard directory (16 B per nonzero with int64 indices and data);
  * call_compress: the compressed .npz (pst_deflate_blocks on the GPU, formats.CsrNpzWriter on the host);
  * disk_write: a plain write() loop of the shard's byte count, in 64 MB blocks, into the same directory;
  * per arm: nonzeros/s, the file bytes per nonzero per member and in total, and the peak RSS (VmHWM after
    clear_refs) of one call above the RSS before it; for call_compress the bytes copied at close.
The rate of pst_deflate_blocks alone: CUDA events around --kernel-reps launches on the first --kernel-mb MB of
the int64 indices and data bytes of the m = 0 matrix (larger than the 126 MB L2), GB/s of input.

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
import zipfile
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
from csr_bench import gpu_info  # noqa: E402
from csr_stream_bench import peak_of, write_loop  # noqa: E402
from prosstt_b200 import _native as nat, device as pdev, formats, hostpool, simulation as sim  # noqa: E402

MEMBERS = ("indptr", "indices", "data")


class _Recorder(formats.CsrNpzWriter):
    """The writer of the samplers, remembering the bytes its last close() copied."""
    last_copied = None

    def close(self):
        super().close()
        _Recorder.last_copied = self.copied_at_close


def member_bytes(path):
    """{member: bytes on disk} of a shard directory or of a compressed file (compressed member sizes)."""
    if os.path.isdir(path):
        return {m: os.path.getsize(os.path.join(path, m + ".npy")) for m in MEMBERS}
    with zipfile.ZipFile(path) as z:
        return {m: z.getinfo(m + ".npy").compress_size for m in MEMBERS}


def same_members(shard, npz):
    """Whether every member of the compressed file decompresses to the shard's file of the same name (same
    length and CRC-32; both use the same dtypes), without decompressing it."""
    with zipfile.ZipFile(npz) as z:
        for name in z.namelist():
            info, crc = z.getinfo(name), 0
            with open(os.path.join(shard, name), "rb") as fh:
                for block in iter(lambda: fh.read(64 << 20), b""):
                    crc = zlib.crc32(block, crc)
            if crc != info.CRC or os.path.getsize(os.path.join(shard, name)) != info.file_size:
                return False
    return True


def remove(path):
    if os.path.isdir(path):
        shutil.rmtree(path)
    elif os.path.exists(path):
        os.remove(path)


def deflate_rate(buf, reps, dev):
    """(GB/s of input, compressed / raw) of pst_deflate_blocks over the device bytes `buf`."""
    lib = nat.load()
    n, block = buf.numel(), pdev._DEFLATE_BLOCK
    out = torch.empty(int(lib.pst_deflate_bound(n, block)), dtype=torch.uint8, device=dev)
    ws = int(lib.pst_deflate_workspace_bytes(n, block))
    work = torch.empty(ws, dtype=torch.uint8, device=dev)
    size = torch.zeros(1, dtype=torch.int64, device=dev)
    crc = torch.zeros(2, dtype=torch.int32, device=dev)
    st = nat.stream_ptr(dev)

    def run():
        nat.call("pst_deflate_blocks", buf, None, 0, n, block, out, size, crc, work, ws, st)

    for _ in range(3):
        run()
    main = torch.cuda.current_stream(dev)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(main)
    for _ in range(reps):
        run()
    t1.record(main)
    t1.synchronize()
    sec = t0.elapsed_time(t1) / 1e3 / reps
    return n / sec / 1e9, int(size.item()) / float(n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=131072)
    ap.add_argument("--depths", type=float, nargs="+", default=[-2.0, 0.0])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--kernel-mb", type=int, default=1024)
    ap.add_argument("--kernel-reps", type=int, default=20)
    ap.add_argument("--dir", default=None, help="directory for the outputs (default: a new temporary directory)")
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    sim.CsrNpzWriter = _Recorder
    work = tempfile.mkdtemp(dir=a.dir, prefix="csr_npz_")
    doc = {"what": "compressed CSR file (out='csr', path=, compress=True) vs the CSR shard (out='csr', path=)",
           "gpu": gpu_info(), "host_threads": len(os.sched_getaffinity(0)), "c4": [], "deflate_kernel": []}
    try:
        w = dict(bench.WORKLOADS["c4"])
        t0 = time.time()
        tree = bench.build_tree_gpu(w, dev)
        alpha, beta = bench.gene_hyper(w["G"])
        G, n = w["G"], a.cells
        doc["c4_tree"] = "15 branches x 50 steps, K=10, G=%d, hybrid sampler, %d cells per call" % (G, n)
        doc["c4_tree_build_s"] = time.time() - t0
        for m in a.depths:
            kw = dict(alpha=alpha, beta=beta, device=dev, sampler="hybrid", scale_mean=m, seed=1000, out="csr")
            shard, npz = os.path.join(work, "x.csr"), os.path.join(work, "x.npz")
            arms = {"call_path": (shard, lambda: sim.sample_density(tree, n, path=shard, **kw)[0]),
                    "call_compress": (npz, lambda: sim.sample_density(tree, n, path=npz, compress=True, **kw)[0])}
            # the same matrix on both arms, and the files' sizes
            X = arms["call_path"][1]()
            rec = arms["call_compress"][1]()
            nnz = int(X.nnz)
            check = {"nnz_equal": nnz == rec.nnz, "members_equal": same_members(shard, npz)}
            if m == 0.0 or m == a.depths[-1]:
                # member-sized inputs for the kernel rate: the first kernel-mb MB of the int64 streams
                k = min(nnz, (a.kernel_mb << 20) // 8)
                doc["deflate_kernel_inputs"] = {
                    "indices_int64": torch.from_numpy(np.ascontiguousarray(X.indices[:k], dtype=np.int64)),
                    "data_int64": torch.from_numpy(np.ascontiguousarray(X.data[:k], dtype=np.int64))}
            del X
            sizes = {name: member_bytes(p) for name, (p, _) in arms.items()}
            for p, _ in arms.values():
                remove(p)
            times = {k: [] for k in list(arms) + ["disk_write"]}
            copied = []
            for r in range(a.reps + 1):                        # round 0 is the warm-up
                for name, (p, fn) in arms.items():
                    gc.collect()
                    torch.cuda.synchronize(dev)
                    c0 = time.perf_counter()
                    out = fn()
                    dt = time.perf_counter() - c0
                    del out
                    if name == "call_compress":
                        copied.append(_Recorder.last_copied)
                    remove(p)
                    if r:
                        times[name].append(dt)
                c0 = time.perf_counter()
                write_loop(os.path.join(work, "plain.bin"), sum(sizes["call_path"].values()))
                if r:
                    times["disk_write"].append(time.perf_counter() - c0)
            res = {"scale_mean": m, "nnz": nnz, "zero_fraction": 1.0 - nnz / float(n * G), "check": check,
                   "arms": {}}
            for name, ts in times.items():
                med = float(np.median(ts))
                res["arms"][name] = {"seconds": ts, "median_s": med}
                if name == "disk_write":
                    res["arms"][name]["GB_per_s"] = sum(sizes["call_path"].values()) / med / 1e9
                    continue
                total = sum(sizes[name].values())
                res["arms"][name].update(nnz_per_s=nnz / med, counts_per_s=n * G / med, file_member_bytes=sizes[name],
                                         bytes_per_nnz={k: v / float(nnz) for k, v in sizes[name].items()},
                                         bytes_per_nnz_total=total / float(nnz), written_GB_per_s=total / med / 1e9)
            res["arms"]["call_compress"]["bytes_copied_at_close"] = copied[-1]
            res["compress_speedup_vs_path"] = (res["arms"]["call_path"]["median_s"]
                                               / res["arms"]["call_compress"]["median_s"])
            res["compressed_over_shard_bytes"] = (res["arms"]["call_compress"]["bytes_per_nnz_total"]
                                                  / res["arms"]["call_path"]["bytes_per_nnz_total"])
            for name, (p, fn) in arms.items():
                out, peak = peak_of(fn)
                del out
                remove(p)
                res["arms"][name]["peak_rss_above_start_bytes"] = peak
            hostpool.release()
            torch.cuda.empty_cache()
            doc["c4"].append(res)
            print(json.dumps(res, indent=1), file=sys.stderr, flush=True)
        del tree
        torch.cuda.empty_cache()
        for name, host in doc.pop("deflate_kernel_inputs").items():
            buf = host.view(torch.uint8).reshape(-1).to(dev)
            gbs, ratio = deflate_rate(buf, a.kernel_reps, dev)
            res = {"input": name + " of the m = %g matrix" % a.depths[-1], "bytes": buf.numel(),
                   "launches": a.kernel_reps, "block_bytes": pdev._DEFLATE_BLOCK, "input_GB_per_s": gbs,
                   "compressed_over_raw": ratio}
            doc["deflate_kernel"].append(res)
            print(json.dumps(res, indent=1), file=sys.stderr, flush=True)
            del buf
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
