#!/usr/bin/env python
"""Headline benchmark: NB counts sampled per second (cells x genes / s) by PROSSTT's samplers on the
BASELINE.json configs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload c1|c2|c3|c4|c5] [--scaling weak|strong] [--dump-outputs DIR]

Default = config 4, the one the metric is quoted on: 15-branch tree, T=50, K=10, G=20 000,
sample_density, 1M cells per GPU ("weak"; every rank samples its own slab with globally numbered
cells).  The same JSON line carries the STRONG split of config 4 (1M cells in total, N/world per
rank) under "strong".  Other workloads:
  c1  minimal example: 3 branches x 50 steps, G=500, sample_whole_tree (n_factor cells per position)
  c2  generate_simN style: 5 branches, G=10k, K=10, 10k cells, sample_density
  c3  sample_pseudotime_series: 10 branches, G=20k, 100k cells
  c5  many_branches_cells: 50 branches x 1000 steps, G=30k, 5M cells, streamed (never resident):
      "value" samples chunk after chunk into one reused HBM buffer, "e2e" streams every chunk to the
      host into a checksum sink (pst_host_checksum over the pinned staging buffers)

One process per GPU (torchrun for N>1; NCCL only for the barrier / max-over-ranks timing: the path
shards by cells with no data-path collective).  A "step" is one complete pass of the sampler:
index map -> library sizes -> NB draw of cells x genes counts into HBM.  Prints ONE JSON line on rank 0.

--impl reference times the reference's CPU algorithm (the oracle port: NumPy gather + get_pr_umi +
legacy RandomState.negative_binomial, i.e. what scipy's nbinom.rvs executes at
prosstt/simulation.py:647-648) on all host cores, on a bounded cell sample of the same workload.

--dump-outputs DIR writes what the last timed step computed (rank 0's cells), so that two builds can be
compared output for output; the inputs depend only on the arguments (fixed seeds):
  X.npy          float32 (k, G): counts of k cells, all of them if they fit 30 MB, else a fixed seeded sample
  cell.npy       float64 (k,): global index of each of those cells
  pseudotime.npy, branch.npy, scalings.npy   float64: per cell, for every cell of the step if the three fit
                 30 MB, else for the k cells of X.npy
(at most 60 MB in all; counts are exact in float32 up to 2^24).
c5 keeps only the last chunk of a step resident: its files describe that chunk.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

UNIT = "counts/s"
SEEDS = dict(tree=42, lineage=43, sampling=44)

# branch_points, chained extra branch, steps per branch, genes, programs (None: the Tree default,
# 5*branch_points + randint(1, 20), tree.py:67-68), total cells, sampler
WORKLOADS = {
    "c1": dict(bp=1, chain=0, T=50, G=500, K=None, cells=150 * 1000, fn="whole_tree",
               what="minimal example, sample_whole_tree with n_factor=1000"),
    "c2": dict(bp=2, chain=0, T=50, G=10000, K=10, cells=10000, fn="density",
               what="generate_simN style, sample_density"),
    "c3": dict(bp=4, chain=1, T=50, G=20000, K=10, cells=100000, fn="series",
               what="sample_pseudotime_series, 5 sample points"),
    "c4": dict(bp=7, chain=0, T=50, G=20000, K=10, cells=1000000, fn="density",
               what="sample_density"),
    "c5": dict(bp=24, chain=1, T=1000, G=30000, K=10, cells=5000000, fn="density",
               what="many_branches_cells, sample_density streamed in chunks"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"],
                    help="weak: --cells per GPU; strong: --cells in total.  Default: weak for c4, strong otherwise")
    ap.add_argument("--cells", type=int, default=None, help="cells (per GPU if weak, total if strong)")
    ap.add_argument("--genes", type=int, default=None)
    ap.add_argument("--chunk-cells", type=int, default=None, help="c5: cells per streamed chunk")
    ap.add_argument("--sampler", default=None)
    ap.add_argument("--e2e-cells", type=int, default=131072, help="cells per e2e step (host buffers)")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--cpu-cells", type=int, default=4096, help="cells of the cpu_baseline sample")
    ap.add_argument("--ref-cells-per-core", type=int, default=256)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (at most 60 MB)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm keeps only checksums)")
    w = dict(WORKLOADS[a.workload])
    if a.genes:
        w["G"] = a.genes
    if a.cells:
        w["cells"] = a.cells
    if a.scaling is None:
        a.scaling = "weak" if a.workload == "c4" else "strong"
    a.w = w
    return a


def metric_name(a):
    fn = {"density": "sample_density", "whole_tree": "sample_whole_tree", "series": "sample_pseudotime_series"}[a.w["fn"]]
    return "NB counts sampled/sec (cells x genes / s), %s" % fn


def config_dict(a):
    """Identical in both arms (the driver compares them)."""
    w = a.w
    nb = 2 * w["bp"] + 1 + w["chain"]
    return {"workload": "%s %s: %d-branch tree x %d steps, K=%s, G=%d, %d cells %s"
                        % (a.workload.upper(), w["what"], nb, w["T"], w["K"] if w["K"] else "default", w["G"],
                           w["cells"], "per GPU" if a.scaling == "weak" else "in total"),
            "seeds": SEEDS, "cells": w["cells"], "genes": w["G"], "scaling": a.scaling,
            "l2": "every step writes a count slab far larger than the 126 MB L2 (self-flushing), except c1/c2 "
                  "whose whole output fits L2: those lines are launch/latency-bound by construction"}


def gene_hyper(G):
    """alpha, beta as in examples/generate_simN.py:94-95 (SURVEY.md 8d)."""
    rng = np.random.RandomState(SEEDS["sampling"])
    alpha = np.exp(rng.normal(np.log(0.2), np.log(1.5), size=G))
    beta = np.exp(rng.normal(np.log(1.0), np.log(1.5), size=G)) + 1
    return alpha, beta


def topology(w):
    """Random binary topology (Tree.gen_random_topology under the tree seed); an even branch count gets one
    chained branch below the last leaf (SURVEY.md 8: as in probabilistic_branching.ipynb)."""
    from prosstt_b200 import tree as ptree
    np.random.seed(SEEDS["tree"])
    top = [[int(p), int(c)] for p, c in ptree.Tree.gen_random_topology(w["bp"])]
    nb = 2 * w["bp"] + 1
    if w["chain"]:
        top.append([nb - 1, nb])
        nb += 1
    return top, {b: w["T"] for b in range(nb)}


def tree_depth(top, time_):
    start = {0: 0}
    for p, c in top:
        start[c] = start[p] + time_[p]
    return max(start[b] + time_[b] for b in time_)


def series_points(w, top, time_):
    depth = tree_depth(top, time_)
    pts = [int(round(depth * f)) for f in (0.1, 0.3, 0.5, 0.7, 0.9)]
    return pts, [w["cells"] // len(pts)] * len(pts), [6.0] * len(pts)


# ------------------------------------------------------------------------------ ours
def build_tree_gpu(a, dev):
    from prosstt_b200 import simulation as sim, sim_utils as sut, tree as ptree
    w = a.w if hasattr(a, "w") else a
    top, time_ = topology(w)
    kw = dict(topology=top, time=time_, num_branches=len(time_), branch_points=w["bp"], G=w["G"])
    if w["K"]:
        kw["modules"] = w["K"]
    t = ptree.Tree(**kw)
    np.random.seed(SEEDS["lineage"])
    if t.G * sum(time_.values()) > 5e7:
        # big tables stay in HBM (no host round trip of the P x G arrays)
        sim.default_gene_expression_on_device(t, seed=SEEDS["lineage"], device=dev)
        return t
    rel, W, H = sim.simulate_lineage(t, a=0.05, seed=SEEDS["lineage"], device=dev)
    scale = sut.simulate_base_gene_exp(t, rel)
    t.add_genes({b: np.exp(rel[b]) * scale for b in t.branches})
    return t


class ClockSampler(object):
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8 or not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(names, f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    """(copy peak GB/s, source, write-only ceiling GB/s or None).  The write-only figure is a pure-store
    kernel timed on a B200 by tools/store_ceiling.py (profiles/store_ceiling.json)."""
    peak, src = 6650.0, "fallback (B200_PROFILING.md)"
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            peak, src = float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, read+write copy)"
    store = None
    path = os.path.join(ROOT, "profiles", "store_ceiling.json")
    if os.path.exists(path):
        with open(path) as fh:
            store = float(json.load(fh)["store_gbs"])
    return peak, src, store


def _profile_file(stem, sampler):
    """profiles/<stem>.json for the hybrid kernel, profiles/<stem>_<sampler>.json for another sampler's."""
    return os.path.join(ROOT, "profiles", stem + ("" if sampler == "hybrid" else "_" + sampler) + ".json")


def profiled_traffic(sampler="hybrid"):
    """DRAM bytes per count of the draw kernel from the committed ncu capture (NOT measured by this run)."""
    path = _profile_file("traffic", sampler)
    if not os.path.exists(path):
        return None, None
    with open(path) as fh:
        rec = json.load(fh)
    return float(rec["bytes_per_count"]), rec.get("source")


def issue_bound(sampler="hybrid"):
    """Speed of light of the instruction-bound draw kernel (profiles/issue_bound*.json, from the ncu
    capture of the committed kernel): warp-instructions per count and the issue rate of a B200."""
    path = _profile_file("issue_bound", sampler)
    if not os.path.exists(path):
        return None
    with open(path) as fh:
        return json.load(fh)


def cpu_baseline(a, sample_cells):
    """The oracle port of the workload's sampler on ONE host core (the reference is single-threaded)."""
    ot, alpha, beta, call = reference_sampler(a)
    rng = np.random.RandomState(SEEDS["sampling"])
    call(rng, 64)                                          # warm-up
    t0 = time.perf_counter()
    X = call(rng, sample_cells)
    dt = time.perf_counter() - t0
    return {"value": X.size / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "%d cells x %d genes of the same tree in %.1f s (oracle port of the sampler: "
                      "NumPy gather + get_pr_umi + legacy RandomState.negative_binomial)"
                      % (X.shape[0], a.w["G"], dt)}


DUMP_HALF_BYTES = 30 * 10 ** 6         # two halves: 60 MB of arrays in all


def dump_outputs(path, result, names, first):
    """Write one step's (X, pseudotime, branch codes, scalings) device tensors as DIR/<name>.npy (see the module
    docstring).  `names` maps branch codes to the branch names the caller receives; `first` is the global index
    of the step's first cell."""
    import torch
    X, pt, codes, s64 = result
    n, G = X.shape
    k = min(n, DUMP_HALF_BYTES // (4 * G + 32))        # a row of X and the cell's four float64 values
    cells = np.arange(n) if k == n else np.sort(np.random.RandomState(SEEDS["sampling"]).choice(n, k, replace=False))
    sel = torch.from_numpy(cells).to(X.device)
    per_cell = (lambda v: v) if 3 * 8 * n <= DUMP_HALF_BYTES else (lambda v: v.index_select(0, sel))
    arrays = {"X": X.index_select(0, sel).cpu().numpy().astype(np.float32),
              "cell": (first + cells).astype(np.float64),
              "pseudotime": per_cell(pt).cpu().numpy().astype(np.float64),
              "branch": np.asarray(names, dtype=np.float64)[per_cell(codes).cpu().numpy().astype(np.int64)],
              "scalings": per_cell(s64).cpu().numpy().astype(np.float64)}
    os.makedirs(path, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(path, name + ".npy"), arr)


def run_ours(a):
    import torch
    import torch.distributed as dist
    from prosstt_b200 import _native as nat
    from prosstt_b200.device import CountEngine, tree_tables
    from prosstt_b200.session import DensitySession
    from prosstt_b200 import simulation as sim

    w = a.w
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (ours) needs a GPU: there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert world == a.gpus or world == 1, "launch with torchrun --nproc-per-node %d" % a.gpus

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    sampler = a.sampler or sim.DEFAULT_SAMPLER
    t_setup = time.perf_counter()
    tree = build_tree_gpu(a, dev)
    torch.cuda.synchronize(dev)
    setup_s = time.perf_counter() - t_setup     # Tree + simulate_lineage + base expression + means (untimed set-up)
    G = w["G"]
    alpha, beta = gene_hyper(G)
    top, time_ = topology(w)

    # ---- the step of this workload ----------------------------------------------------------------------
    def make_stepper(total_cells, scaling):
        """Returns (step(seed), cells sampled by this rank per step, whole-job cells per step).  step(seed) returns
        the device tensors (X, pseudotime, branch codes, scalings) of this rank's cells (c5: of the last chunk)."""
        if scaling == "weak":
            mine, first, job = total_cells, rank * total_cells, total_cells * world
        else:
            lo, hi = (total_cells * rank) // world, (total_cells * (rank + 1)) // world
            mine, first, job = hi - lo, lo, total_cells
        if w["fn"] == "density":
            chunk = a.chunk_cells or (250000 if a.workload == "c5" else mine)
            chunk = max(1, min(chunk, mine))
            sess = DensitySession(tree, alpha, beta, chunk, first=first, device=dev, sampler=sampler)

            def step(seed):
                for lo in range(0, mine, chunk):          # c5: chunk after chunk into one reused buffer
                    sess.set_range(first + lo, min(chunk, mine - lo))
                    X = sess.step(seed)
                return X, sess.pt[:sess.n], sess.codes[:sess.n], sess.s64[:sess.n]
            return step, mine, job, sess
        if w["fn"] == "whole_tree":
            P = sum(time_.values())
            n_factor = max(1, job // P)

            def step(seed):
                return sim.sample_whole_tree(tree, n_factor, alpha=alpha, beta=beta, seed=seed, device=dev,
                                             shard=(rank, world) if scaling == "strong" else None, out="torch",
                                             sampler=sampler)
            per = n_factor * P
            mine = per if scaling == "weak" else (per * (rank + 1)) // world - (per * rank) // world
            return step, mine, per * (world if scaling == "weak" else 1), None
        pts, cells, std = series_points(dict(w, cells=job if scaling == "strong" else total_cells), top, time_)

        def step(seed):
            return sim.sample_pseudotime_series(tree, cells, pts, std, alpha=alpha, beta=beta, seed=seed, device=dev,
                                                shard=(rank, world) if scaling == "strong" else None, out="torch",
                                                sampler=sampler)
        per = int(np.sum(cells))
        mine = per if scaling == "weak" else (per * (rank + 1)) // world - (per * rank) // world
        return step, mine, per * (world if scaling == "weak" else 1), None

    def timed(step, steps, warmup, sample_clocks=False):
        seed = SEEDS["sampling"]
        for i in range(warmup):
            step(seed + i)
        barrier()
        clocks = ClockSampler(local) if sample_clocks else None
        if clocks:
            clocks.start()
            time.sleep(0.25)
        CountEngine.timers = []
        launches0 = nat.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        w0 = time.time()
        ev0.record()
        for i in range(steps):
            last = None                           # free the previous step's outputs before the next one allocates
            last = step(seed + 100 + i)
        ev1.record()
        barrier()
        w1 = time.time()
        launches = nat.launch_count() - launches0
        draws = [e0.elapsed_time(e1) for e0, e1 in CountEngine.timers]
        CountEngine.timers = None
        ms = max_over_ranks(ev0.elapsed_time(ev1))
        return ms, draws, launches, (clocks.stop(w0, w1) if clocks else None), last

    step, mine, job, sess = make_stepper(w["cells"], a.scaling)
    ms, draws, launches, clock_rec, last = timed(step, a.steps, a.warmup, sample_clocks=True)
    if sess is not None:
        sess.engine.check()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, last, tree_tables(tree, dev).names, sess.first if sess is not None else 0)
    del last
    value = float(job) * G * a.steps / (ms / 1e3)
    kernel_ms = float(np.sum(draws)) / a.steps            # all draw launches of one step (c5: one per chunk)

    # ---- strong split of the same workload (config 4: 1M cells in total over the ranks) ----------------
    strong = None
    if a.scaling == "weak" and not a.no_strong and w["fn"] == "density" and a.workload != "c5":
        if world == 1:
            strong = {"value": value, "unit": UNIT, "cells_total": w["cells"], "ms_per_step": ms / a.steps,
                      "draw_ms_per_step": kernel_ms, "other_ms_per_step": ms / a.steps - kernel_ms,
                      "note": "one GPU: the strong split is the weak one"}
        else:
            del sess, step
            torch.cuda.empty_cache()
            s_step, s_mine, s_job, s_sess = make_stepper(w["cells"], "strong")
            s_ms, s_draws, s_launch = timed(s_step, a.steps, a.warmup)[:3]
            s_sess.engine.check()
            d = float(np.sum(s_draws)) / a.steps
            strong = {"value": float(s_job) * G * a.steps / (s_ms / 1e3), "unit": UNIT, "cells_total": s_job,
                      "cells_per_gpu": s_mine, "ms_per_step": s_ms / a.steps, "draw_ms_per_step": d,
                      "other_ms_per_step": s_ms / a.steps - d, "launches_per_step": s_launch / a.steps,
                      "note": "%d cells in total, %d per rank; ms_per_step is the max over ranks; other = uniforms + "
                              "density index + library sizes + launch gaps (the draw includes the row grouping "
                              "and the tail fix-up kernel)" % (s_job, s_mine)}
            del s_sess, s_step
            torch.cuda.empty_cache()
            step, mine, job, sess = make_stepper(w["cells"], a.scaling)

    # ---- end to end through the public API path with HOST buffers -----------------------
    e2e = None
    if not a.no_e2e:
        e2e = run_e2e(a, tree, alpha, beta, sampler, dev, rank, world, barrier, max_over_ranks, mine, job)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src, store_peak = measured_peaks()
    per_launch_cells = mine if not draws else mine / (len(draws) / a.steps)
    algo_bytes = 4.0 * mine * G                            # per step of this rank
    achieved = algo_bytes / (kernel_ms / 1e3) / 1e9
    bpc, bpc_src = profiled_traffic(sampler)
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": None if bpc is None else bpc * per_launch_cells * G,
            "traffic_source": None if bpc is None else "NOT measured by this run: %.3f B/count from %s, scaled to "
                                                       "this launch" % (bpc, bpc_src),
            "kernel": "draw_counts (%s): row grouping + draw kernel + tail fix-up, timed together with CUDA events"
                      % sampler,
            "kernel_ms": kernel_ms, "launches_of_it_per_step": len(draws) / a.steps,
            "kernel_share_of_step": kernel_ms * a.steps / ms, "algorithmic_bytes_per_count": 4,
            "peak_source": peak_src}
    if store_peak:
        roof["store_only_peak"] = store_peak
        roof["frac_of_store_only_peak"] = achieved / store_peak
    ib = issue_bound(sampler)
    if ib:
        sol = ib["issue_slots_per_s"] / ib["speed_of_light_warp_inst_per_count"]
        roof["issue_bound"] = {"counts_per_s_at_speed_of_light": sol, "frac": (mine * G / (kernel_ms / 1e3)) / sol,
                               "warp_inst_per_count_now": ib["warp_inst_per_count"],
                               "warp_inst_per_count_speed_of_light": ib["speed_of_light_warp_inst_per_count"],
                               "source": ib["source"]}
    out = {
        "metric": metric_name(a), "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": a.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(a),
        "run": {"sampler": sampler, "output": "int32 (N,G) resident in HBM", "cells_this_rank": mine,
                "tree_lineage_means_setup_s": round(setup_s, 3),
                "means_table_mb": round(tree.G * sum(time_.values()) * 4 / 1e6, 1)},
        "clocks": clock_rec, "e2e": e2e, "gpu_launches": int(launches), "roofline": roof,
    }
    if strong is not None:
        out["strong"] = strong
    if not a.no_cpu_baseline and world == 1:
        out["cpu_baseline"] = cpu_baseline(a, a.cpu_cells)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def run_e2e(a, tree, alpha, beta, sampler, dev, rank, world, barrier, max_over_ranks, mine, job):
    """The same metric through the public API with HOST outputs.  `value`: the reference-shaped call with
    preallocated pinned int32 buffers (host_out=), as in round 1.  `default_api`: the call exactly as
    examples/generate_simN.py:113 makes it - no extra keyword, fresh int64 NumPy arrays returned."""
    import torch
    from prosstt_b200 import simulation as sim
    from prosstt_b200 import _native as nat
    w, G = a.w, a.w["G"]
    top, time_ = topology(w)
    P = sum(time_.values())
    seed = SEEDS["sampling"]

    def clock(fn, steps):
        fn(seed)                                              # warm-up (page-locks the staging buffers)
        barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            fn(seed + 200 + i)
        barrier()
        return max_over_ranks(time.perf_counter() - t0)

    if a.workload == "c5":
        # streamed: every chunk goes to the host and into the sink; nothing is kept
        from prosstt_b200.session import DensitySession
        chunk = max(1, min(a.chunk_cells or 250000, mine))
        first = (job * rank) // world if a.scaling == "strong" else rank * mine
        lib = nat.load()
        out = {}
        for transport in ("i32", "u8"):
            sess = DensitySession(tree, alpha, beta, chunk, first=first, device=dev, sampler=sampler,
                                  resident_output=False)
            sums, nbytes = [0], [0]

            def sink(staged, lo, hi, sums=sums, nbytes=nbytes):
                sums[0] += int(lib.pst_host_checksum(staged.data_ptr(), (staged.numel() // 4) * 4, 0))
                nbytes[0] += staged.numel()

            barrier()
            t0 = time.perf_counter()
            for lo in range(0, mine, chunk):
                sess.set_range(first + lo, min(chunk, mine - lo))
                sess.index_and_scalings(seed + 7)
                sess.engine.stream_chunks(sess.rows[:sess.n], sess.s32[:sess.n], nat.derive_seed(seed + 7, 2),
                                          sess.first, sink, transport=transport)
            barrier()
            dt = max_over_ranks(time.perf_counter() - t0)
            sess.engine.check()
            out[transport] = {"value": float(job) * G / dt, "unit": UNIT, "wall_s": dt,
                              "sink_gb_per_s_this_rank": nbytes[0] / dt / 1e9, "d2h_bytes_this_rank": nbytes[0],
                              "checksum_this_rank": sums[0] & 0xFFFFFFFFFFFF}
            del sess
            torch.cuda.empty_cache()
        res = dict(out["i32"])
        res.update({"h2d_bytes_per_step": 16 * P + 8 * G, "d2h_bytes_per_step": out["i32"]["d2h_bytes_this_rank"],
                    "steps": 1, "narrow_u8": out["u8"],
                    "note": "whole workload streamed once: chunks of %d cells sampled, copied as int32 into pinned "
                            "staging and summed by host threads (pst_host_checksum) while the next chunk is sampled; "
                            "narrow_u8 = uint8 transport + overflow list" % chunk})
        return res

    ecells = max(1, min(a.e2e_cells, mine))
    shard = (rank, world)
    h2d = 16 * P + 8 * G          # per call: cdf f64 + pos_pt/pos_branch i32 [P], alpha/beta-1 f32 [G]

    def api_kwargs():
        return dict(alpha=alpha, beta=beta, device=dev, sampler=sampler, shard=shard)

    if w["fn"] == "density":
        def default_call(seed_):                              # generate_simN.py:113 (+ device/shard plumbing)
            return sim.sample_density(tree, ecells * world, seed=seed_, **api_kwargs())
    elif w["fn"] == "whole_tree":
        n_factor = max(1, ecells * world // P)
        ecells = n_factor * P // world

        def default_call(seed_):
            return sim.sample_whole_tree(tree, n_factor, seed=seed_, **api_kwargs())
    else:
        pts, cells, std = series_points(dict(w, cells=ecells * world), top, time_)
        ecells = int(np.sum(cells)) // world

        def default_call(seed_):
            return sim.sample_pseudotime_series(tree, cells, pts, std, seed=seed_, **api_kwargs())

    steps = a.e2e_steps
    from prosstt_b200 import hostpool
    from prosstt_b200.device import _shared_host_transport, _host_threads
    narrow = _shared_host_transport(_host_threads()) == "u8"   # what the library picks on this host
    dt = clock(default_call, steps)
    # the same call with the result pool off: every result matrix is memory nobody has touched (what a
    # script's FIRST call sees)
    pool_env = os.environ.get("PST_HOST_POOL_GB")
    os.environ["PST_HOST_POOL_GB"] = "0"
    hostpool.release()
    try:
        dt_cold = clock(default_call, steps)
    finally:
        if pool_env is None:
            del os.environ["PST_HOST_POOL_GB"]
        else:
            os.environ["PST_HOST_POOL_GB"] = pool_env
    default_api = {"value": float(ecells) * G * world * steps / dt, "unit": UNIT, "steps": steps,
                   "cells_per_step_per_gpu": ecells,
                   "d2h_bytes_per_step": int((1 if narrow else 4) * ecells * G + 20 * ecells),
                   "host_bytes_written_per_step": int(8 * ecells * G),
                   "transport": "u8" if narrow else "i32",
                   "first_call": {"value": float(ecells) * G * world * steps / dt_cold, "unit": UNIT,
                                  "note": "PST_HOST_POOL_GB=0: every result is freshly mapped memory, the "
                                          "expansion takes a page fault per 4 KiB (what the first call of a "
                                          "script sees)"},
                   "note": "the call as the reference's scripts make it (no extra keyword): returns int64 NumPy "
                           "arrays; counts cross PCIe in `transport` format into pinned staging and are expanded "
                           "into the result by host threads while the next chunk is sampled; the memory of a "
                           "result that has been garbage-collected is reused for the next one (hostpool), so "
                           "from the second call on the expansion writes mapped memory with streaming stores"}
    if w["fn"] != "density":
        res = dict(default_api)
        res.update({"h2d_bytes_per_step": int(h2d), "default_api": default_api})
        return res

    hpt = torch.empty(ecells, dtype=torch.int64).pin_memory()
    hco = torch.empty(ecells, dtype=torch.int32).pin_memory()
    hsc = torch.empty(ecells, dtype=torch.float64).pin_memory()

    threads = _host_threads()
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    auto = _shared_host_transport(threads)                    # what the library picks on this host

    def run_pinned(x_dtype, transport=None):
        hX = torch.empty((ecells, G), dtype=x_dtype).pin_memory()
        overflow = {}

        def api_call(seed_):
            return sim.sample_density(tree, ecells * world, seed=seed_, dtype=np.int32,
                                      host_out=(hX, hpt, hco, hsc, overflow), host_transport=transport, **api_kwargs())
        dt = clock(api_call, steps)
        listed = len(overflow.get("index", ()))
        return float(ecells) * G * world * steps / dt, hX.numel(), listed

    meta = ecells * (8 + 4 + 8)
    v16, n16, listed = run_pinned(torch.uint16)
    v8, n8, listed8 = run_pinned(torch.uint8)
    d2h16 = 2 * n16 + meta + listed * 12
    d2h8 = n8 + meta + listed8 * 12
    # int32 host matrix: copied as int32 by the copy engine ("direct"), or crossing PCIe as uint8 + overflow
    # list and widened by host threads ("u8").  `value` is the call with NO transport argument (the library
    # picks one of the two from the CPU's store instructions and this rank's thread count); both are reported.
    by_transport = {}
    for tr in ("direct", "u8"):
        by_transport[tr] = run_pinned(torch.int32, tr)[0]
    v32 = run_pinned(torch.int32)[0]                          # no transport argument
    d2h = {"direct": 4 * n8 + meta, "u8": d2h8}[auto]
    return {"value": v32, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "cells_per_step_per_gpu": ecells, "steps": steps, "transport": auto,
            "host_threads_per_rank": threads, "host_cores": cores,
            "note": "simulation.sample_density(tree, N, alpha, beta, host_out=pinned buffers): tree tables, "
                    "cdf and gene parameters uploaded per call; int32 counts + pseudotime + branch + "
                    "scalings land in host memory (chunked, copy overlapped with sampling); no transport "
                    "argument: the library chose `transport` for this host (device.py:_shared_host_transport)",
            "default_api": default_api,
            "int32_direct": {"value": by_transport["direct"], "unit": UNIT, "d2h_bytes_per_step": int(4 * n8 + meta),
                             "note": "host_transport='direct': the copy engine writes the int32 matrix, 4 B per "
                                     "count over PCIe"},
            "int32_via_u8": {"value": by_transport["u8"], "unit": UNIT, "d2h_bytes_per_step": int(d2h8),
                             "note": "host_transport='u8': same int32 pinned host matrix, but the counts cross PCIe "
                                     "as uint8 + exact overflow list into pinned staging and host threads "
                                     "(pst_host_widen_stream: non-temporal stores; pst_host_apply_overflow) expand "
                                     "them: a quarter of the PCIe bytes, 4 B/count of host-memory writes by the "
                                     "CPU instead of by DMA"},
            "narrow_u16": {"value": v16, "unit": UNIT, "d2h_bytes_per_step": int(d2h16),
                           "overflow_entries_last_step": int(listed),
                           "note": "same call with a uint16 host matrix: min(count, 65535) plus an exact "
                                   "(index, value) list of the saturated elements; lossless, half the PCIe bytes"},
            "narrow_u8": {"value": v8, "unit": UNIT, "d2h_bytes_per_step": int(d2h8),
                          "overflow_entries_last_step": int(listed8),
                          "note": "uint8 host matrix, min(count, 255) plus the exact list of the counts >= 255; "
                                  "lossless, a quarter of the PCIe bytes"}}


# ------------------------------------------------------------------------------ reference arm
_REF = {}


def build_tree_cpu(a):
    """Same tree shape on the CPU with the oracle's simulate_lineage (legacy stream)."""
    from oracle import prosstt_oracle as orc
    w = a.w
    top, time_ = topology(w)
    K = w["K"] or 10
    ot = orc.OTree(top, time_, G=w["G"], modules=K)
    rng = np.random.RandomState(SEEDS["lineage"])
    if sum(time_.values()) * w["G"] > 2e8:
        # config 5: the oracle's lineage (Python loops over 50 000 steps + G pearsonr calls per sibling pair)
        # would take hours; the per-count cost of the sampler does not depend on how the means were made,
        # so the CPU tree gets log-normal means of the same scale
        ot.means = {b: np.exp(rng.normal(0.6, 1.5, size=(time_[b], w["G"]))) for b in time_}
    else:
        rel, W, H = orc.simulate_lineage(ot, rng, a=0.05)
        cap = orc.max_rel_exp(ot, rel)
        scale, _ = orc.base_gene_exp_from_normals(cap, rng.normal(0.8, 1.0, size=20 * w["G"]))
        ot.means = orc.absolute_means(rel, scale)
    alpha, beta = gene_hyper(w["G"])
    return ot, alpha, beta


def reference_sampler(a):
    """(tree, alpha, beta, call(rng, cells) -> X): the oracle port of the workload's sampler."""
    from oracle import prosstt_oracle as orc
    w = a.w
    ot, alpha, beta = build_tree_cpu(a)
    top, time_ = topology(w)
    if w["fn"] == "density":
        def call(rng, cells):
            return orc.sample_density(ot, cells, alpha, beta, rng)[0]
    elif w["fn"] == "whole_tree":
        P = sum(time_.values())

        def call(rng, cells):
            return orc.sample_whole_tree(ot, max(1, cells // P), alpha, beta, rng)[0]
    else:
        def call(rng, cells):
            pts, per, std = series_points(dict(w, cells=max(5, cells)), top, time_)
            return orc.sample_pseudotime_series(ot, per, pts, std, alpha, beta, rng)[0]
    return ot, alpha, beta, call


def _ref_worker(job):
    seed, cells = job
    X = _REF["call"](np.random.RandomState(seed), cells)
    return int(X.size), int(X.sum() & 0xFFFF)


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    _REF["call"] = reference_sampler(a)[3]
    ctx = mp.get_context("fork")
    per = a.ref_cells_per_core
    with ctx.Pool(cores) as pool:
        def step(i):
            jobs = [(1000003 * (i + 1) + k, per) for k in range(cores)]
            return sum(n for n, _ in pool.map(_ref_worker, jobs, chunksize=1))
        for i in range(a.warmup):
            step(i)
        t0 = time.perf_counter()
        total = 0
        for i in range(a.steps):
            total += step(a.warmup + i)
        dt = time.perf_counter() - t0
    value = total / dt
    sample = ("%d host processes x %d cells x %d genes per step (disjoint cell shards, own seeds) of the same "
              "workload; oracle port of the sampler = NumPy gather + get_pr_umi + legacy "
              "RandomState.negative_binomial" % (cores, per, a.w["G"]))
    out = {"impl": "reference", "metric": metric_name(a), "value": value, "unit": UNIT, "n_gpus": a.gpus,
           "steps": a.steps, "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3,
           "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None, "dtype": "f64",
           "data": "synthetic", "config": config_dict(a),
           "run": {"cells_per_step": total // a.steps // a.w["G"]},
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


if __name__ == "__main__":
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
