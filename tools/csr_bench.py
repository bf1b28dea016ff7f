#!/usr/bin/env python
"""out="csr" against the dense host result on the C4 tree (15 branches x 50 steps, K=10, G=20 000), hybrid
sampler, 131 072 cells per call, at library size x e^m for m = -2 and m = 0.

For each depth:
  * end-to-end: the dense default call (int64 ndarray), dense int32, CSR with int64 data and CSR with int32
    data, warmed up and then alternated, --reps calls each (host clock around the call, which returns host
    memory after a device synchronise): counts/s, nnz/s and result bytes; the pass-1 share of the CSR calls
    from the CUDA events draw_to_csr records (start -> row pointer ready, over the call's wall time);
  * peak RSS (VmHWM) of one call of each arm, with the result pool emptied and the high-water mark reset
    before the call;
  * kernels on one device-resident matrix of the same cells (10.5 GB, far larger than L2): pst_csr_row_counts,
    pst_csr_pack (uint16 columns, uint16 values + overflow list) and pst_csr_fill (int32) in GB/s of dense
    input read (4 B per count), CUDA events over --kernel-reps launches;
  * a check that the CSR result holds the dense result's counts (nnz, total, three row blocks exactly).

Prints one JSON document (and writes it to --json PATH if given); GPU name and power limit are read in the
same run."""
import argparse
import gc
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from prosstt_b200 import _native as nat, hostpool, simulation as sim  # noqa: E402
from prosstt_b200.device import CountEngine  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return {"nvidia_smi": out, "torch_name": torch.cuda.get_device_name(0)}


def vm(key):
    with open("/proc/self/status") as fh:
        for line in fh:
            if line.startswith(key + ":"):
                return int(line.split()[1]) * 1024
    return None


def reset_hwm():
    """Reset this process's peak-RSS mark (clear_refs 5); False where the kernel does not allow it."""
    try:
        with open("/proc/self/clear_refs", "w") as fh:
            fh.write("5")
        return True
    except OSError:
        return False


def result_bytes(X):
    if hasattr(X, "indptr"):
        return int(X.indptr.nbytes + X.indices.nbytes + X.data.nbytes)
    return int(X.nbytes)


def kernel_rates(X, reps):
    n, G = X.shape
    dev = X.device
    st = nat.stream_ptr(dev)
    row_nnz = torch.empty(n, dtype=torch.int32, device=dev)
    sat = torch.zeros(1, dtype=torch.int64, device=dev)
    indptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
    nat.call("pst_csr_row_counts", X.data_ptr(), n, G, G, row_nnz, sat, st)
    nat.call("pst_csr_row_offsets", row_nnz, n, indptr, st)
    nnz, n_sat = int(indptr[-1].item()), int(sat.item())
    idx16 = torch.empty(max(1, nnz), dtype=torch.int16, device=dev)
    val16 = torch.empty(max(1, nnz), dtype=torch.int16, device=dev)
    ovf_pos = torch.empty(max(1, n_sat), dtype=torch.int64, device=dev)
    ovf_val = torch.empty(max(1, n_sat), dtype=torch.int32, device=dev)
    ovf_count = torch.zeros(1, dtype=torch.int64, device=dev)
    flags = torch.zeros(1, dtype=torch.int32, device=dev)

    def row_counts():
        nat.call("pst_csr_row_counts", X.data_ptr(), n, G, G, row_nnz, sat, st)

    def offsets():
        nat.call("pst_csr_row_offsets", row_nnz, n, indptr, st)

    def pack():
        ovf_count.zero_()
        nat.call("pst_csr_pack", X.data_ptr(), n, G, G, indptr, 0, idx16.data_ptr(), 16, val16.data_ptr(), 16,
                 ovf_pos, ovf_val, n_sat, ovf_count, flags, st)

    res = {"cells": n, "genes": G, "nnz": nnz, "saturated": n_sat, "dense_bytes_read": 4 * n * G}

    def timed(fn):
        fn()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize(dev)
        return a.elapsed_time(b) / reps

    ms = timed(row_counts)
    res["pst_csr_row_counts"] = {"ms": ms, "GB_per_s_dense_read": 4.0 * n * G / ms / 1e6}
    ms = timed(offsets)
    res["pst_csr_row_offsets"] = {"ms": ms}
    ms = timed(pack)
    res["pst_csr_pack_u16_u16"] = {"ms": ms, "GB_per_s_dense_read": 4.0 * n * G / ms / 1e6,
                                   "bytes_written": 4 * nnz + 12 * n_sat}
    assert int(flags.item()) == 0 and int(ovf_count.item()) == n_sat
    del idx16, val16
    indices = torch.empty(max(1, nnz), dtype=torch.int32, device=dev)
    data = torch.empty(max(1, nnz), dtype=torch.int32, device=dev)

    def fill():
        nat.call("pst_csr_fill", X.data_ptr(), n, G, G, indptr, indices, data, flags, st)

    ms = timed(fill)
    res["pst_csr_fill_i32_i32"] = {"ms": ms, "GB_per_s_dense_read": 4.0 * n * G / ms / 1e6,
                                   "bytes_written": 8 * nnz}
    assert int(flags.item()) == 0
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=131072)
    ap.add_argument("--depths", type=float, nargs="+", default=[-2.0, 0.0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--kernel-reps", type=int, default=10)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    w = dict(bench.WORKLOADS["c4"])
    t0 = time.time()
    tree = bench.build_tree_gpu(w, dev)
    alpha, beta = bench.gene_hyper(w["G"])
    G, n = w["G"], a.cells
    doc = {"what": "out='csr' vs dense host result, C4 tree (15 branches x 50 steps, K=10, G=%d), hybrid sampler, "
                   "%d cells per call" % (G, n),
           "gpu": gpu_info(), "host_threads": len(os.sched_getaffinity(0)), "tree_build_s": time.time() - t0,
           "depths": []}
    arms = [("dense_int64", {}), ("dense_int32", {"dtype": np.int32}),
            ("csr_int64", {"out": "csr"}), ("csr_int32", {"out": "csr", "dtype": np.int32})]
    for m in a.depths:
        kw = dict(alpha=alpha, beta=beta, device=dev, sampler="hybrid", scale_mean=m)
        seed = 1000

        def call(opts, s):
            return sim.sample_density(tree, n, seed=s, **kw, **opts)[0]

        # correctness on the timed cells: the CSR result holds the dense counts
        dense = call({"dtype": np.int32}, seed)
        csr = call({"out": "csr"}, seed)
        nnz = int(np.count_nonzero(dense))
        check = {"nnz_equal": csr.nnz == nnz, "total_equal": int(csr.data.sum()) == int(dense.sum(dtype=np.int64))}
        for lo in (0, n // 2, n - 64):
            check["rows_%d" % lo] = bool(np.array_equal(csr[lo:lo + 64].toarray(), dense[lo:lo + 64]))
        zero_frac = 1.0 - nnz / float(n * G)
        del dense, csr
        gc.collect()
        # timing: warm-up of every arm, then the arms alternate
        times = {k: [] for k, _ in arms}
        pass1 = {k: [] for k, _ in arms}
        sizes = {}
        for k, opts in arms:
            X = call(opts, seed)
            sizes[k] = result_bytes(X)
            del X
        for r in range(a.reps):
            for k, opts in arms:
                CountEngine.csr_timers = [] if "csr" in k else None
                gc.collect()
                torch.cuda.synchronize(dev)
                c0 = time.perf_counter()
                X = call(opts, seed + 1 + r)
                dt = time.perf_counter() - c0
                times[k].append(dt)
                if CountEngine.csr_timers:
                    ev = CountEngine.csr_timers[-1]
                    pass1[k].append(ev[0].elapsed_time(ev[1]) / 1e3 / dt)
                del X
        CountEngine.csr_timers = None
        res = {"scale_mean": m, "zero_fraction": zero_frac, "nnz": nnz, "check": check, "arms": {}}
        for k, _ in arms:
            med = float(np.median(times[k]))
            res["arms"][k] = {"seconds": times[k], "median_s": med, "counts_per_s": n * G / med,
                              "nnz_per_s": nnz / med, "result_bytes": sizes[k],
                              "result_bytes_vs_dense_int64": sizes[k] / float(8 * n * G)}
            if pass1[k]:
                res["arms"][k]["pass1_share"] = pass1[k]
                res["arms"][k]["pass1_share_median"] = float(np.median(pass1[k]))
        res["csr_int64_speedup_vs_dense_int64"] = res["arms"]["dense_int64"]["median_s"] / res["arms"]["csr_int64"]["median_s"]
        # peak RSS of one call per arm, from an emptied result pool
        for k, opts in arms:
            hostpool.release()
            gc.collect()
            ok = reset_hwm()
            base = vm("VmRSS")
            X = call(opts, seed)
            peak = vm("VmHWM")
            del X
            res["arms"][k]["peak_rss_bytes"] = peak
            res["arms"][k]["peak_rss_above_start_bytes"] = peak - base if ok else None
        hostpool.release()
        # kernels on one device-resident matrix of the same cells
        Xd = call({"out": "torch"}, seed)
        res["kernels"] = kernel_rates(Xd, a.kernel_reps)
        del Xd
        torch.cuda.empty_cache()
        doc["depths"].append(res)
        print(json.dumps(res, indent=1), file=sys.stderr, flush=True)
    doc["gpu_after"] = gpu_info()
    text = json.dumps(doc, indent=1)
    print(text)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
