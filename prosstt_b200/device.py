"""Device-side view of a Tree: packed tables in HBM and the count engine.

Layout (include/prosstt_b200.h): branches in `tree.branches` order, branch b owns packed
rows [row_base[b], row_base[b]+T_b); P = sum T_b.  Everything here is small and
replicated on every GPU (a few MB; the means table is P x G fp32); only cells shard.
"""
import concurrent.futures
import os

import numpy as np
import torch

from prosstt_b200 import _native as nat
from prosstt_b200 import hostpool
from prosstt_b200.formats import sync_deflate


def tree_tables(tree, dev):
    """TreeTables of `tree` on `dev`, cached on the tree: the integer maps depend only on the topology,
    the branch lengths, the branch order and the root, which form the key - an edited tree gets new tables."""
    try:
        key = (str(dev), tuple((p, c) for p, c in tree.topology), tuple((b, int(tree.time[b])) for b in tree.branches),
               tree.root)
        hash(key)
    except TypeError:
        return TreeTables(tree, dev)
    cache = tree.__dict__.setdefault("_tables_cache", {})
    hit = cache.get(key)
    if hit is None:
        cache.clear()
        hit = cache[key] = TreeTables(tree, dev)
    return hit


class TreeTables(object):
    """Integer maps of a tree flattened for the kernels (host numpy + device copies)."""

    def __init__(self, tree, dev):
        self.dev = dev
        self.names = list(tree.branches)
        self.index = {b: i for i, b in enumerate(self.names)}
        if len(self.index) != len(self.names):
            raise ValueError("branch names must be unique")
        B = len(self.names)
        self.B = B
        self.T = np.array([int(tree.time[b]) for b in self.names], dtype=np.int32)
        if np.any(self.T < 1):
            raise ValueError("every branch needs at least one pseudotime step")
        self.row_base = np.zeros(B, dtype=np.int32)
        self.row_base[1:] = np.cumsum(self.T)[:-1]
        self.P = int(self.T.sum())
        bt = tree.branch_times()
        missing = [b for b in self.names if b not in bt or len(bt[b]) != 2]
        if missing:
            raise ValueError("branches %s are not connected to the root by the topology" % missing)
        self.branch_start = np.array([bt[b][0] for b in self.names], dtype=np.int32)
        # sample_density's concatenation (simulation.py:454-461)
        self.pos_branch = np.repeat(np.arange(B, dtype=np.int32), self.T)
        self.pos_pt = (np.arange(self.P, dtype=np.int32) - np.repeat(self.row_base, self.T)
                       + np.repeat(self.branch_start, self.T)).astype(np.int32)
        # timezones and their live branches in branch_times order (sim_utils.py:274-339)
        zones = tree.populate_timezone()
        order = [self.index[b] for b in bt.keys() if b in self.index]
        self.zone_lo = np.array([z[0] for z in zones], dtype=np.int32)
        self.zone_hi = np.array([z[1] for z in zones], dtype=np.int32)
        cand, off = [], [0]
        for lo, hi in zones:
            live = [b for b in order
                    if lo >= self.branch_start[b] and hi <= self.branch_start[b] + self.T[b] - 1]
            cand.extend(live)
            off.append(len(cand))
        self.cand_branch = np.array(cand, dtype=np.int32)
        self.cand_off = np.array(off, dtype=np.int32)
        self.max_cand = int(np.max(np.diff(self.cand_off))) if len(zones) else 0
        # cover_whole_tree (simulation.py:520-548): zone-major, branch, time
        cpt, cbr = [], []
        for z, (lo, hi) in enumerate(zones):
            for b in self.cand_branch[self.cand_off[z]:self.cand_off[z + 1]]:
                cpt.append(np.arange(lo, hi + 1, dtype=np.int32))
                cbr.append(np.full(hi + 1 - lo, b, dtype=np.int32))
        self.cover_pt = np.concatenate(cpt) if cpt else np.zeros(0, np.int32)
        self.cover_branch = np.concatenate(cbr) if cbr else np.zeros(0, np.int32)
        self.cover_row = (self.row_base[self.cover_branch] + self.cover_pt
                          - self.branch_start[self.cover_branch]).astype(np.int32)
        self.max_time = int((self.branch_start + self.T).max())
        self._dev = {}

    def d(self, name, dtype=torch.int32):
        """Device copy of one of the host tables (cached)."""
        if name not in self._dev:
            self._dev[name] = nat.to_dev(getattr(self, name), dtype, self.dev)
        return self._dev[name]

    def density_packed(self, tree):
        dens = [np.asarray(tree.density[b], dtype=np.float64) for b in self.names]
        for b, v in zip(self.names, dens):
            if v.shape != (int(tree.time[b]),):
                raise ValueError("density of branch %s has shape %s, expected (%d,)"
                                 % (str(b), str(v.shape), int(tree.time[b])))
        return np.concatenate(dens)

    def branch_codes(self, branches):
        """Branch names (any iterable) -> int32 indices into tree.branches."""
        arr = np.asarray(branches)
        if arr.dtype.kind in "iu" and all(isinstance(b, (int, np.integer)) for b in self.names):
            lut_keys = np.array(self.names, dtype=np.int64)
            sorter = np.argsort(lut_keys)
            pos = np.searchsorted(lut_keys, arr, sorter=sorter)
            pos = np.clip(pos, 0, len(lut_keys) - 1)
            codes = sorter[pos]
            if np.any(lut_keys[codes] != arr):
                raise KeyError("unknown branch name in `branches`")
            return codes.astype(np.int32)
        try:
            return np.array([self.index[b.item() if hasattr(b, "item") else b] for b in arr],
                            dtype=np.int32)
        except KeyError as err:
            raise KeyError("unknown branch name in `branches`: %s" % err)

    def branch_names(self, codes):
        """int32 indices -> array of branch names with the dtype numpy gives the names
        (reference: possible_branches[sample], simulation.py:461-467)."""
        return np.array(self.names)[np.asarray(codes, dtype=np.int64)]


def choice_cdf(p):
    """The cdf numpy's legacy RandomState.choice builds (with its validity checks)."""
    p = np.asarray(p, dtype=np.float64)
    if p.ndim != 1 or p.size == 0:
        raise ValueError("'p' must be 1-dimensional and non-empty")
    if np.any(np.isnan(p)) or np.any(p < 0):
        raise ValueError("probabilities are not non-negative")
    if abs(float(np.sum(p)) - 1.0) > np.sqrt(np.finfo(np.float64).eps):
        raise ValueError("probabilities do not sum to 1")
    cdf = np.cumsum(p)
    cdf /= cdf[-1]
    return cdf


def _content_key(m):
    """Cheap fingerprint of one branch's means for the device-table cache: buffer address, shape, the
    first and last pseudotime rows and ~4096 values at a fixed stride.  An in-place edit of the whole
    array, of a gene column (seen in the first row) or of a pseudotime row (>= G/stride samples fall in
    it) - ordinary NumPy usage in scripts written for the reference - changes it, unlike id(); after
    editing single elements call tree.invalidate_device_cache().  ~0.05 ms per branch."""
    if isinstance(m, torch.Tensor):
        return ("t", m.data_ptr(), tuple(m.shape), m._version)
    a = np.asarray(m)
    flat = a.reshape(-1)
    step = max(1, flat.size // 4096) | 1
    edge = (a[0].tobytes(), a[-1].tobytes()) if a.ndim >= 2 and a.shape[0] else ()
    return (a.__array_interface__["data"][0], a.shape, flat[::step].tobytes()) + edge


def means_table(tree, tables, dev):
    """(P, G) fp32 means table in HBM, built once per tree.means and cached on the tree."""
    if tree.means is None:
        raise ValueError("the tree has no mean expression yet: call add_genes() or "
                         "default_gene_expression() first")
    if hasattr(tree.means, "table32"):                 # simulation.DeviceMeans: already in HBM
        if tuple(tree.means.table32.shape) != (tables.P, int(tree.G)):
            raise ValueError("the device-resident means table has shape %s, the tree needs %s"
                             % (tuple(tree.means.table32.shape), (tables.P, int(tree.G))))
        if tree.means.table32.device == dev:
            return tree.means.table32
        return tree.means.table32.to(dev)
    key = ("means32", str(dev)) + tuple(_content_key(tree.means[b]) for b in tables.names)
    cache = tree.__dict__.setdefault("_device_cache", {})
    hit = cache.get(key)
    if hit is not None:
        return hit
    G = int(tree.G)
    out = torch.empty((tables.P, G), dtype=torch.float32, device=dev)
    st = nat.stream_ptr(dev)
    for i, b in enumerate(tables.names):
        m = tree.means[b]
        if isinstance(m, torch.Tensor):
            m64 = m.to(device=dev, dtype=torch.float64).contiguous()
        else:
            m64 = nat.to_dev(m, torch.float64, dev)
        if tuple(m64.shape) != (int(tables.T[i]), G):
            raise ValueError("means of branch %s have shape %s, expected %s"
                             % (str(b), tuple(m64.shape), (int(tables.T[i]), G)))
        dst = out[int(tables.row_base[i]):int(tables.row_base[i]) + int(tables.T[i])]
        nat.call("pst_f64_to_f32", nat.ptr(m64), m64.numel(), 1e-30, dst.data_ptr(), st)
    cache.clear()
    cache[key] = out
    return out


def gene_params(alpha, beta, G, dev):
    """Per-gene alpha and beta-1 as fp32 device vectors (beta-1 formed in fp64)."""
    a = np.broadcast_to(np.asarray(alpha, dtype=np.float64), (G,)) if np.ndim(alpha) == 0 \
        else np.asarray(alpha, dtype=np.float64)
    b = np.broadcast_to(np.asarray(beta, dtype=np.float64), (G,)) if np.ndim(beta) == 0 \
        else np.asarray(beta, dtype=np.float64)
    if a.shape != (G,) or b.shape != (G,):
        raise ValueError("alpha and beta must be scalars or have one value per gene (G=%d)" % G)
    return nat.to_dev(a, torch.float32, dev), nat.to_dev(b - 1.0, torch.float32, dev)


def raise_flags(word):
    """Translate the device status word into the reference's exceptions."""
    if word & nat.FLAG_ROW:
        raise IndexError("a cell's pseudotime lies outside its branch")
    if word & nat.FLAG_NOZONE:
        raise IndexError("a pseudotime value lies outside the lineage tree")
    if word & nat.FLAG_DOMAIN:
        raise ValueError("Domain error in arguments. The mean expression must be positive "
                         "and alpha*mean + beta must exceed 1 for every cell and gene.")
    if word & nat.FLAG_SCRATCH:
        raise RuntimeError("the tail list of pst_draw_counts overflowed (scratch too small)")
    if word & nat.FLAG_CLAMPED:
        raise OverflowError("a sampled count exceeded the int32 range")


_NP_TO_TORCH = {np.dtype(np.int32): torch.int32, np.dtype(np.int64): torch.int64,
                np.dtype(np.uint16): torch.uint16, np.dtype(np.uint8): torch.uint8}
_STAGE_BYTES = int(os.environ.get("PST_STAGE_MB", "256")) << 20   # one pinned staging buffer (two per device)
_STAGING = {}
_DEFLATE_BLOCK = 32768                        # bytes per DEFLATE block of the compressed CSR file (at most 32 KiB)
# stream_csr's `compression`: the device compressor, its workspace size and the workspace's token bytes per input byte
_DEFLATE = {"huffman": ("pst_deflate_blocks", "pst_deflate_workspace_bytes", 0),
            "lz77": ("pst_deflate_lz_blocks", "pst_deflate_lz_workspace_bytes", 2)}
# stream_csr's per-chunk record of int64 slots, read by the host one chunk late: those of every format, then its own
_REC_SAT, _REC_NNZ, _REC_STATUS, _REC_OWN = range(4)
_REC_SLOTS = _REC_OWN + 6                     # the .npz has the most slots of its own


_AUTO_STATE = {"narrow_overflowed": False}     # an automatically chosen uint8 transport overflowed its list once


def _shared_host_transport(threads):
    """Transport of a host matrix when nothing was asked for.  "direct" / "i32": the counts cross PCIe as
    int32, 4 B per count (55-57 GB/s = 1.4e10 counts/s for one B200).  "u8": they cross as uint8 + exact
    overflow list (a quarter of the bytes) and host threads expand them with non-temporal stores
    (pst_host_widen_stream: 5.7e9 counts/s per thread, 3.4e10 with 16).  Measured: one rank with 16 threads
    2.4e10 against 1.3e10 counts/s; eight ranks with 4 threads each on a 32-vCPU box, where the host MEMORY
    system is the limit, 3.0e10 against 2.3e10 (6 B of host traffic per count instead of the 10 B of an
    expansion with ordinary stores, which lost to "direct" there).  So "u8" wherever the CPU has the streaming
    stores and this rank has at least 3 threads, or 10 threads without them.  A fixed rule, not a timing trial:
    every rank of a job must pick the same transport (a trial run by eight ranks at once measured their
    contention and split them).  PST_HOST_TRANSPORT=direct|i32|u16|u8 overrides."""
    forced = os.environ.get("PST_HOST_TRANSPORT")
    if forced:
        return forced
    need = 3 if nat.load().pst_host_stream_stores() else 10
    return "u8" if threads >= need else "direct"


def _host_threads():
    """Host threads of this rank for the expansion: its share of the cores when several ranks share a host."""
    try:
        local_world = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
    except ValueError:
        local_world = 1
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    return max(1, cores // local_world)


def _pinned_staging(dev, nbytes):
    """Two pinned host buffers of at least nbytes for the staged device->host path, allocated once per
    device and kept (page-locking costs ~0.2 s per GB)."""
    key = str(dev)
    have = _STAGING.get(key)
    if have is None or have[0].numel() < nbytes:
        size = max(int(nbytes), 1)
        have = [torch.empty(size, dtype=torch.uint8).pin_memory() for _ in range(2)]
        _STAGING[key] = have
    return have


def _mtx_slot_bytes(G, n):
    """Matrix Market text bytes budgeted per gene slot of a chunk of a file of n cells: one line
    "<gene> <cell> <count>\n" with a count of up to 3 digits.  A chunk with more text is formatted again into
    a larger buffer (CountEngine.stream_csr)."""
    return len(str(G)) + len(str(n)) + 6


def _tsv_slot_bytes(G, n):
    """Tab-separated text bytes budgeted per gene slot of a chunk of a file of n cells: a tab and a count of up to 3
    digits.  A chunk with more text is formatted again into a larger buffer (CountEngine.stream_csr)."""
    return 4


def _plan_chunks(n, chunk_cells, cell_bytes, budget):
    """The cell chunks of a chunked device->host call: (chunk, [(lo, hi), ...]) covering [0, n) in order, where
    chunk is the largest chunk (the size of the buffers).  Owns the chunk size and the ramp-up.
    chunk_cells=None: chunks of `budget` bytes at `cell_bytes` per cell, and the first chunks are 1/8, 1/4 and 1/2
    of that so that the copy (and the host threads) start almost immediately.  An explicit chunk_cells (at least
    1, at most n) has no ramp."""
    ramp_up = chunk_cells is None
    if ramp_up:
        chunk_cells = budget // max(1, cell_bytes)
    chunk = max(1, min(n, int(chunk_cells)))
    ramp = [max(1, chunk // 8), max(1, chunk // 4), max(1, chunk // 2)] if ramp_up else []
    bounds, lo = [], 0
    while lo < n:
        size = ramp.pop(0) if ramp else chunk
        bounds.append((lo, min(n, lo + size)))
        lo = bounds[-1][1]
    return chunk, bounds


_TRANSPORTS = {"i32": torch.int32, "u16": torch.uint16, "u8": torch.uint8}


def _host_route(is_np, hdt, pinned, transport, threads):
    """How draw_to_host moves the counts into a host matrix of dtype `hdt` (the table in its docstring):
    returns (route, retry).  route is "direct" (the copy engine writes the matrix) or the staged transport
    "i32" / "u16" / "u8"; retry is the route to sample again through when an automatically chosen "u8"
    overflows its list, else None.  Raises ValueError for a combination that has no route."""
    if hdt in (torch.uint16, torch.uint8):
        if is_np or transport not in (None, "direct"):
            raise ValueError("a uint16 / uint8 host matrix must be a CPU tensor and takes transport 'direct'")
        return "direct", None
    if transport is None:
        # nothing asked for: the copy engine writes a pinned int32 matrix itself ("direct"), every other
        # target is filled by host threads from int32 staging ("i32") - or, where this rank's share of
        # the host cores expands uint8 well above the PCIe rate, from uint8 staging ("u8")
        wide = "direct" if (not is_np and hdt == torch.int32 and pinned) else "i32"
        if not _AUTO_STATE["narrow_overflowed"] and _shared_host_transport(threads) == "u8":
            return "u8", wide
        return wide, None
    if transport == "direct":
        if is_np or hdt != torch.int32:
            raise ValueError("transport 'direct' needs an int32, uint16 or uint8 CPU tensor")
        return "direct", None
    if transport not in _TRANSPORTS:
        raise ValueError("transport must be 'direct', 'i32', 'u16' or 'u8'")
    return transport, None


class _OverflowList(object):
    """The exact list of the counts a narrow format cannot hold, on the device: int64 positions, int32 values,
    an int64 count and the capacity.  Owns the check that the list held every such count."""

    def __init__(self, capacity, dev):
        self.capacity = int(capacity)
        self.pos = torch.empty(max(1, self.capacity), dtype=torch.int64, device=dev)
        self.value = torch.empty(max(1, self.capacity), dtype=torch.int32, device=dev)
        self.count = torch.zeros(1, dtype=torch.int64, device=dev)
        # in the order pst_narrow_counts and pst_csr_pack take them
        self.kernel_args = (self.pos, self.value, self.capacity, self.count)

    def read(self, fmt):
        """(positions, values) device tensors of the listed counts, in the order the kernels appended them."""
        count = int(self.count.item())
        if count > self.capacity:
            raise OverflowError("%d counts reach the saturation value of %s but the overflow list holds %d: "
                                "use a wider format or a larger overflow_cap"
                                % (count, str(fmt).replace("torch.", ""), self.capacity))
        return self.pos[:count], self.value[:count]


class CountEngine(object):
    """draw_counts on one GPU: replicated small state + a cell range to sample."""

    timers = None     # set to a list to collect (start, end) CUDA events around every draw (bench.py)
    csr_timers = None  # set to a list to collect (start, end of pass 1, end of pass 2) events of draw_to_csr

    def __init__(self, tree, tables, alpha, beta, dev, sampler="gamma_poisson"):
        self.dev = dev
        self.G = int(tree.G)
        self.P = tables.P
        self.means = means_table(tree, tables, dev)
        self.alpha, self.beta_m1 = gene_params(alpha, beta, self.G, dev)
        self.sampler = nat.SAMPLERS[sampler]
        self.flags = torch.zeros(4, dtype=torch.int32, device=dev)   # status word (+3 reserved)
        self._scratch = None
        self.overflow = None                                    # filled by draw_to_host (uint16 format)

    def draw(self, rows, scaling32, seed, cell0, out=None, gene_stats=None):
        """Sample X for the cells described by rows/scaling32 (device tensors); global
        index of the first cell is cell0.  Returns an (n, G) int32 device tensor.
        gene_stats: dict with int64 (G,) device tensors "gene_sum", "gene_sumsq", "gene_zeros"
        (stats.new_gene_stats) that the draw adds this call's per-gene summaries to - fused into
        the kernel, no second pass over the matrix; equals stats.count_stats(X) bit for bit."""
        n = int(rows.numel())
        if out is None:
            out = torch.empty((n, self.G), dtype=torch.int32, device=self.dev)
        st = nat.stream_ptr(self.dev)
        timers = CountEngine.timers
        if timers is not None:
            t0 = torch.cuda.Event(enable_timing=True)
            t0.record(torch.cuda.current_stream(self.dev))
        # scratch of the call: visiting order of the cells (grouped by tree row) and the list of the counts
        # that the fix-up kernel finishes with a 64-bit uniform (top 2^-14 of the uniforms)
        words = int(nat.load().pst_draw_scratch_words(n, self.G, self.P))
        if self._scratch is None or self._scratch.numel() < words:
            self._scratch = torch.empty(words, dtype=torch.int32, device=self.dev)
        nat.call("pst_draw_counts", nat.ptr(self.means), self.P, self.G, nat.ptr(rows),
                 nat.ptr(scaling32), nat.ptr(self.alpha), nat.ptr(self.beta_m1),
                 seed, int(cell0), n, out.data_ptr(), out.stride(0) if n else self.G,
                 nat.ptr(self.flags), self.sampler, self._scratch, words,
                 *((gene_stats["gene_sum"], gene_stats["gene_sumsq"], gene_stats["gene_zeros"])
                   if gene_stats is not None else (None, None, None)), st)
        if timers is not None:
            t1 = torch.cuda.Event(enable_timing=True)
            t1.record(torch.cuda.current_stream(self.dev))
            timers.append((t0, t1))
        return out

    def draw_to_host(self, rows, scaling32, seed, cell0, host_out, chunk_cells=None, overflow_cap=None,
                     transport=None, threads=0, fresh=False):
        """Sample in cell chunks and stream them into `host_out`, an (n, G) CPU tensor or C-contiguous
        NumPy array: sampling of chunk i+1 overlaps the transfer (and host-side expansion) of chunk i.

        Direct: the counts are copied in the dtype of host_out straight into it (4 / 2 / 1 B per count over
          PCIe).  For uint16 / uint8 that is min(count, SAT) with SAT = 65535 / 255, and every element that
          reads SAT is listed exactly in `self.overflow` = (flat index into host_out, int32 value) NumPy arrays
          sorted by index (formats.widen rebuilds int32); on every other route self.overflow is None.  At
          default depth about 2 in 10^4 counts reach 255 and none reaches 65535.
        Staged through transport "u8" / "u16" / "i32": the chunk crosses PCIe in the transport format into
          pinned staging buffers (cached per device) and host threads (pst_host_widen) expand it into host_out,
          the overflow list is applied at the end: the caller receives exact int32 / int64 counts.  This is the
          path of the reference-shaped call, which returns a fresh (pageable) int64 array.  The expansion uses
          streaming stores (pst_host_widen_stream) unless `fresh` says that host_out was just allocated and
          never touched (its pages are zeroed into the cache by the first-touch faults).

        | host_out                                | transport            | route                      |
        |-----------------------------------------|----------------------|----------------------------|
        | pinned int32 tensor                     | None                 | "u8" (*), else direct      |
        | int32 tensor, not pinned                | None                 | "u8" (*), else "i32"       |
        | int32 tensor, pinned or not             | "direct"             | direct                     |
        | uint16 / uint8 tensor                   | None or "direct"     | direct, narrow             |
        | uint16 / uint8 tensor                   | anything else        | ValueError                 |
        | uint16 / uint8 NumPy array              | any                  | ValueError                 |
        | int64 tensor, int32 / int64 NumPy array | None                 | "u8" (*), else "i32"       |
        | int64 tensor, int32 / int64 NumPy array | "direct"             | ValueError                 |
        | int32 / int64 tensor or NumPy array     | "i32" / "u16" / "u8" | staged with that transport |
        | wrong shape or dtype                    | any                  | ValueError                 |

        (*) "u8" where _shared_host_transport says it is faster on this host and no automatically chosen "u8"
        has overflowed in this process: its overflow list does not fit in deep regimes, and then the call is
        sampled again through the wide route and the process keeps to it - the counts are the same either way."""
        n = int(rows.numel())
        is_np = isinstance(host_out, np.ndarray)
        if is_np:
            if not host_out.flags.c_contiguous or not host_out.flags.writeable:
                raise ValueError("host_out must be a writeable C-contiguous array")
            hdt = _NP_TO_TORCH.get(host_out.dtype)
            pinned = False
        else:
            hdt = host_out.dtype
            pinned = host_out.is_pinned() and host_out.is_contiguous()
        if hdt not in (torch.int32, torch.int64, torch.uint16, torch.uint8) or tuple(host_out.shape) != (n, self.G):
            raise ValueError("host_out must be an int32, int64, uint16 or uint8 CPU matrix of shape (%d, %d)"
                             % (n, self.G))
        if not threads:
            threads = _host_threads()
        route, retry = _host_route(is_np, hdt, pinned, transport, threads)
        self.overflow = None

        def fill(route, overflow_cap, fresh):
            if route == "direct":
                ovf = self._dense_chunks(rows, scaling32, seed, cell0, hdt, chunk_cells, overflow_cap,
                                         host_out=host_out)
                if ovf is not None:
                    index, value = ovf.read(hdt)
                    index, order = torch.sort(index)            # appended in no particular order
                    self.overflow = (index.cpu().numpy(), value[order].cpu().numpy())
                return host_out
            G, width = self.G, _TRANSPORTS[route].itemsize
            dst_bits = 32 if hdt == torch.int32 else 64
            dst_ptr = host_out.ctypes.data if is_np else host_out.data_ptr()
            lib = nat.load()
            widen = lib.pst_host_widen if fresh else lib.pst_host_widen_stream

            def expand(staged, lo, hi):
                rc = widen(staged.data_ptr(), 8 * width, dst_ptr + lo * G * (dst_bits // 8), dst_bits,
                           (hi - lo) * G, int(threads))
                if rc != 0:
                    raise nat.NativeError("pst_host_widen failed")

            listed = self.stream_chunks(rows, scaling32, seed, cell0, expand, route, chunk_cells, overflow_cap)
            if listed is not None:
                index, value = listed
                lib.pst_host_apply_overflow(dst_ptr, dst_bits, 0, n * G, index.data_ptr(), value.data_ptr(),
                                            int(index.numel()))
            return host_out

        try:
            return fill(route, overflow_cap, fresh)
        except OverflowError:
            if retry is None:
                raise
        # A deep regime (more than 1 % of the counts above 254): the uint8 transport nobody asked for does not
        # pay here.  The draw is a pure function of (seed, cell, gene): sample again through the wide transport,
        # and keep to it for the rest of the process.
        _AUTO_STATE["narrow_overflowed"] = True
        return fill(retry, None, False)

    def stream_chunks(self, rows, scaling32, seed, cell0, consume, transport="i32", chunk_cells=None,
                      overflow_cap=None):
        """Sample in cell chunks, move each chunk over PCIe in the transport format ("i32", "u16", "u8")
        into one of two pinned staging buffers and hand it to `consume(staged, lo, hi)` on a worker
        thread (`staged`: pinned uint8 tensor holding rows [lo, hi) in the transport format) while the
        next chunk is sampled and copied.  The matrix is never resident anywhere: this is the streamed
        path for outputs larger than HBM (config 5: 600 GB).  Returns the overflow list of the narrow
        transports as CPU tensors (flat index, exact value), unsorted, or None."""
        tdt = _TRANSPORTS.get(transport)
        if tdt is None:
            raise ValueError("transport must be 'i32', 'u16' or 'u8'")
        ovf = self._dense_chunks(rows, scaling32, seed, cell0, tdt, chunk_cells, overflow_cap, consume=consume)
        if ovf is None:
            return None
        index, value = ovf.read(tdt)
        return index.cpu(), value.cpu()

    def draw_to_csr(self, rows, scaling32, seed, cell0, data_dtype=np.int64, chunk_cells=None, threads=0):
        """Sample the cells as CSR arrays on the host: (indptr, indices, data) NumPy arrays, columns ascending
        in every row, no explicit zeros; the same counts as draw().  The dense matrix exists only one chunk at
        a time in HBM.

        Pass 1 draws each chunk and counts its nonzeros per row (pst_csr_row_counts) and the counts >= 65535;
        one scan (pst_csr_row_offsets) gives the row pointer, which is the only thing read back.  So nnz is
        known before any result memory exists: indices and data are allocated once at their final size, with
        int32 indptr/indices when nnz < 2^31 and int64 otherwise (scipy wants the two of one dtype).
        Pass 2 draws each chunk again (a pure function of (seed, cell, gene)), packs it into a uint16 (G <=
        65536) or int32 column stream and a uint16 value stream (pst_csr_pack), copies both into pinned
        staging and host threads widen them into indices[p0:p1] / data[p0:p1] while the next chunk is
        sampled; the values that saturated uint16 are written from the exact overflow list at the end.
        data_dtype: np.int64 or np.int32."""
        data_dtype = np.dtype(data_dtype)
        if data_dtype not in (np.dtype(np.int32), np.dtype(np.int64)):
            raise ValueError("CSR data must be int32 or int64, not %s" % data_dtype)
        n, G, dev = int(rows.numel()), self.G, self.dev
        if not threads:
            threads = _host_threads()
        if n == 0 or G == 0:
            return np.zeros(n + 1, np.int32), np.zeros(0, np.int32), np.zeros(0, data_dtype)
        ibits = 16 if G <= 65536 else 32                 # width of the column stream
        chunk_cells, bounds = _plan_chunks(n, chunk_cells, (ibits // 8 + 2) * G, _STAGE_BYTES)
        st = nat.stream_ptr(dev)
        main = torch.cuda.current_stream(dev)
        events = CountEngine.csr_timers
        if events is not None:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record(main)
        # ---- pass 1: row sizes and the number of saturated values
        work = torch.empty((chunk_cells, G), dtype=torch.int32, device=dev)
        row_nnz = torch.empty(n, dtype=torch.int32, device=dev)
        sat = torch.zeros(1, dtype=torch.int64, device=dev)
        for lo, hi in bounds:
            self.draw(rows[lo:hi], scaling32[lo:hi], seed, cell0 + lo, out=work[:hi - lo])
            nat.call("pst_csr_row_counts", work.data_ptr(), hi - lo, G, G, row_nnz[lo:hi], sat, st)
        indptr_d = torch.empty(n + 1, dtype=torch.int64, device=dev)
        nat.call("pst_csr_row_offsets", row_nnz, n, indptr_d, st)
        if events is not None:
            ev[1].record(main)
            ev[2].record(main)                           # and again behind every pack kernel of pass 2
        indptr64 = indptr_d.cpu().numpy()
        n_sat = int(sat.item())
        self.check()                                     # domain / range errors before any result memory
        # ---- allocate once, at the final size
        nnz = int(indptr64[-1])
        idx_dtype = np.dtype(np.int32) if nnz < (1 << 31) else np.dtype(np.int64)
        indptr = indptr64.astype(np.int32) if idx_dtype == np.int32 else indptr64
        indices, fresh_i = hostpool.result_array((nnz,), idx_dtype)
        data, fresh_d = hostpool.result_array((nnz,), data_dtype)
        lib = nat.load()
        widen_i = lib.pst_host_widen if fresh_i else lib.pst_host_widen_stream
        widen_d = lib.pst_host_widen if fresh_d else lib.pst_host_widen_stream
        ibytes, ibits_out, dbits_out = ibits // 8, 8 * idx_dtype.itemsize, 8 * data_dtype.itemsize

        def value_offset(m):                            # the value stream starts on a 64-byte boundary
            return (m * ibytes + 63) // 64 * 64

        def window(lo, hi):                             # first nonzero, nonzeros and packed bytes of cells [lo, hi)
            p0, m = int(indptr64[lo]), int(indptr64[hi] - indptr64[lo])
            return p0, m, value_offset(m) + 2 * m

        stage_bytes = max(window(lo, hi)[2] for lo, hi in bounds)
        stage_dev = [torch.empty(max(1, stage_bytes), dtype=torch.uint8, device=dev) for _ in range(2)]
        stage_host = _pinned_staging(dev, stage_bytes)
        ovf = _OverflowList(n_sat, dev)
        pack_flags = torch.zeros(1, dtype=torch.int32, device=dev)

        # ---- pass 2: redraw, pack, stream
        def produce(k, lo, hi):
            p0, m, used = window(lo, hi)
            self.draw(rows[lo:hi], scaling32[lo:hi], seed, cell0 + lo, out=work[:hi - lo])
            buf = stage_dev[k]
            nat.call("pst_csr_pack", work.data_ptr(), hi - lo, G, G, indptr_d[lo:hi + 1], p0, buf.data_ptr(),
                     ibits, buf.data_ptr() + value_offset(m), 16, *ovf.kernel_args, pack_flags, st)
            if events is not None:
                ev[2].record(main)
            return [(buf[:used], stage_host[k][:used])]

        def consume(dsts, lo, hi):
            p0, m, _ = window(lo, hi)
            src = dsts[0].data_ptr()
            rc = widen_i(src, ibits, indices.ctypes.data + p0 * idx_dtype.itemsize, ibits_out, m, int(threads))
            rc |= widen_d(src + value_offset(m), 16, data.ctypes.data + p0 * data_dtype.itemsize, dbits_out, m,
                          int(threads))
            if rc != 0:
                raise nat.NativeError("pst_host_widen failed")

        # a chunk without nonzeros has nothing to pack: the redraw would have no nonzero either
        self._copy_chunks([(lo, hi) for lo, hi in bounds if window(lo, hi)[1]], produce, consume)
        if events is not None:
            events.append(tuple(ev))
        self.check()
        if int(pack_flags.item()) != 0:
            raise RuntimeError("the redrawn counts do not match the row sizes of the first pass")
        listed = int(ovf.count.item())
        if listed != n_sat:
            raise RuntimeError("%d counts >= 65535 in the second pass, %d in the first" % (listed, n_sat))
        if n_sat:
            pos, value = ovf.pos[:n_sat].cpu(), ovf.value[:n_sat].cpu()
            lib.pst_host_apply_overflow(data.ctypes.data, dbits_out, 0, nnz, pos.data_ptr(), value.data_ptr(), n_sat)
        return indptr, indices, data

    def stream_csr(self, rows, scaling32, seed, cell0, consume, index_dtype=np.int64, data_dtype=np.int64,
                   chunk_cells=None, threads=0, overflow_cap=None, compress=False, mtx=False, compression="huffman",
                   tsv=False):
        """Sample the cells in chunks and hand each one as CSR to consume(lo, hi, indptr, indices, data), on a
        worker thread, once per chunk, in cell order.  indptr is chunk-local int64 (hi - lo + 1 entries from 0);
        indices and data are the chunk's nonzeros in `index_dtype` / `data_dtype` (int32 or int64), columns
        ascending in every row.  They are reused host buffers, valid during the call only.  Returns the total
        nnz.  Concatenated over the chunks, the arrays are draw_to_csr's, so the counts are those of draw().

        Nothing is sized by the whole matrix, and every chunk is drawn once, into int32 work buffer k = i & 1,
        which survives until chunk i+2 is drawn: a chunk that did not fit a device buffer of k is encoded again
        from it.  The host reads the chunk's record (_REC_*) one chunk late (_copy_chunks' collect); an error in
        its status word raises as draw() would (raise_flags) and ends the stream.

        compress=True: consume(lo, hi, parts) receives the chunk compressed instead, parts = [(member,
        compressed, crc, raw_len)] for "indptr", "indices" and "data" in the order formats.CsrNpzWriter.append
        takes them: `compressed` (a reused uint8 host buffer) is raw DEFLATE that decompresses to the raw_len
        bytes of the member's part, whose CRC-32 is crc.  indptr is the chunk's row ends in index_dtype, offset
        by the nonzeros of the chunks before it (the file's leading 0 is not included).

        mtx=True: consume(lo, hi, compressed, crc, text_len, nnz) receives the chunk as Matrix Market text
        (formats.MtxWriter.append): `compressed` (a reused uint8 host buffer) is raw DEFLATE that decompresses to
        the text_len bytes of the chunk's nnz lines "<g+1> <c+1> <v>\n", c = lo + row within the chunk, whose
        CRC-32 is crc; index_dtype and data_dtype do not apply.

        tsv=True: consume(lo, hi, text, crc, text_len) receives the chunk as dense tab-separated text
        (formats.TsvWriter.append): the text_len bytes of its rows "cell_<cell0+c>" "\t<v>" for every gene "\n",
        c = lo + row within the chunk.  `text` (a reused uint8 host buffer) is that text itself, crc 0; with
        compress=True it is raw DEFLATE that decompresses to it, whose CRC-32 is crc.  index_dtype and data_dtype
        do not apply.

        compression ("huffman" or "lz77", with compress=True or mtx=True): the device compressor,
        pst_deflate_blocks (Huffman-only) or pst_deflate_lz_blocks (LZ77 matches within each 32 KiB block,
        smaller output, a larger workspace).  Both write the same framing, so the consumer is the same."""
        index_dtype, data_dtype = np.dtype(index_dtype), np.dtype(data_dtype)
        for what, dt in (("indices", index_dtype), ("data", data_dtype)):
            if dt not in (np.dtype(np.int32), np.dtype(np.int64)):
                raise ValueError("CSR %s must be int32 or int64, not %s" % (what, dt))
        if compression not in _DEFLATE:
            raise ValueError("compression must be 'huffman' or 'lz77', not %r" % (compression,))
        n, G, dev = int(rows.numel()), self.G, self.dev
        if n == 0:
            return 0
        # an encoder gives its budget per cell, its output when G == 0 and start(), which allocates its buffers and
        # returns step, grow (True if a buffer of k grew for the chunk), encode (what then runs again), copies, deliver
        cell_bytes, empty, start = (
            self._mtx_encoder(n, consume, compression) if mtx else
            self._tsv_encoder(n, consume, compress, compression, cell0) if tsv else
            self._npz_encoder(n, consume, index_dtype, data_dtype, compression) if compress else
            self._shard_encoder(n, consume, index_dtype, data_dtype, threads, overflow_cap))
        if G == 0:
            empty()
            return 0
        chunk, bounds = _plan_chunks(n, chunk_cells, cell_bytes, _STAGE_BYTES)
        st = nat.stream_ptr(dev)
        work = [torch.empty((chunk, G), dtype=torch.int32, device=dev) for _ in range(2)]
        row_nnz = torch.empty(chunk, dtype=torch.int32, device=dev)      # read by the scan right after the count
        indptr = [torch.empty(chunk + 1, dtype=torch.int64, device=dev) for _ in range(2)]
        info = torch.zeros((2, _REC_SLOTS), dtype=torch.int64, device=dev)
        info_host = torch.zeros((2, _REC_SLOTS), dtype=torch.int64).pin_memory()
        pack_flags = torch.zeros(1, dtype=torch.int32, device=dev)
        total = [0]
        step, grow, encode, copies, deliver = start(chunk, work, indptr, info, pack_flags)

        def produce(k, lo, hi):
            cells = hi - lo
            self.draw(rows[lo:hi], scaling32[lo:hi], seed, cell0 + lo, out=work[k][:cells])
            info[k].zero_()                     # the compressors write each CRC into the low word of a zeroed slot
            nat.call("pst_csr_row_counts", work[k].data_ptr(), cells, G, G, row_nnz, info[k, _REC_SAT], st)
            nat.call("pst_csr_row_offsets", row_nnz, cells, indptr[k], st)
            step(k, lo, cells)
            info[k, _REC_NNZ].copy_(indptr[k][cells])
            info[k, _REC_STATUS].copy_(self.flags[0])
            info_host[k].copy_(info[k], non_blocking=True)

        def collect(k, lo, hi):
            record = info_host[k].tolist()
            if record[_REC_STATUS]:
                self.flags[0].zero_()
                raise_flags(record[_REC_STATUS])
            total[0] += record[_REC_NNZ]
            if grow(k, record):
                encode(k, lo, hi - lo)
                record = info[k].tolist()                # waits for it: the copies wait for the first encode only
            return copies(k, hi - lo, record), record

        self._copy_chunks(bounds, produce, deliver, collect)
        if int(pack_flags.item()) != 0:
            raise RuntimeError("the packed counts do not match the row sizes of their chunk")
        return total[0]

    def _shard_encoder(self, n, consume, index_dtype, data_dtype, threads, overflow_cap):
        """stream_csr's CSR shard.  pst_csr_pack writes chunk k into device staging k: a uint16 column stream (int32
        when G > 65536) and, at the fixed offset of chunk x G column entries, a uint16 value stream (4 B per
        nonzero over PCIe), plus the saturated values in overflow list k, which grows when they do not fit."""
        G, dev, st, lib = self.G, self.dev, nat.stream_ptr(self.dev), nat.load()
        ibytes = 2 if G <= 65536 else 4                  # bytes per entry of the column stream
        threads = int(threads or _host_threads())

        def empty():
            consume(0, n, np.zeros(n + 1, np.int64), np.zeros(0, index_dtype), np.zeros(0, data_dtype))

        def start(chunk, work, indptr, info, pack_flags):
            value_at = (chunk * G * ibytes + 63) // 64 * 64  # the value stream, after the worst-case column stream
            stage = [torch.empty(value_at + 2 * chunk * G, dtype=torch.uint8, device=dev) for _ in range(2)]
            ovf = [_OverflowList(overflow_cap or (1 << 16), dev) for _ in range(2)]
            ovf_host = [torch.empty(12 * ovf[k].capacity, dtype=torch.uint8).pin_memory() for k in range(2)]
            # host side: the row pointer, then the streams of the nonzeros, values on a 64-byte boundary
            stage_host = _pinned_staging(dev, 8 * (chunk + 1) + value_at + 64 + 2 * chunk * G)
            # the widened chunk, reused from chunk to chunk (by the one worker): its pages are touched as the chunks'
            # nnz needs them and hostpool keeps them mapped for the next call.  Past the first chunk they are mapped
            # and out of cache, which is what the streaming stores are for.
            indices_w = hostpool.result_array((chunk * G,), index_dtype)[0]
            data_w = hostpool.result_array((chunk * G,), data_dtype)[0]
            widen = lib.pst_host_widen_stream

            def pack(k, lo, cells):
                ovf[k].count.zero_()
                nat.call("pst_csr_pack", work[k].data_ptr(), cells, G, G, indptr[k], 0, stage[k].data_ptr(),
                         8 * ibytes, stage[k].data_ptr() + value_at, 16, *ovf[k].kernel_args, pack_flags, st)

            def grow(k, record):
                if record[_REC_SAT] <= ovf[k].capacity:
                    return False
                ovf[k] = _OverflowList(max(record[_REC_SAT], 2 * ovf[k].capacity), dev)
                ovf_host[k] = torch.empty(12 * ovf[k].capacity, dtype=torch.uint8).pin_memory()
                return True

            def copies(k, cells, record):
                n_sat, nnz = record[_REC_SAT], record[_REC_NNZ]
                at = 8 * (cells + 1)
                vat = (at + nnz * ibytes + 63) // 64 * 64
                h = stage_host[k]
                pairs = [(indptr[k][:cells + 1].view(torch.uint8), h[:at]),
                         (stage[k][:nnz * ibytes], h[at:at + nnz * ibytes]),
                         (stage[k][value_at:value_at + 2 * nnz], h[vat:vat + 2 * nnz])]
                if n_sat:
                    pairs += [(ovf[k].pos[:n_sat].view(torch.uint8), ovf_host[k][:8 * n_sat]),
                              (ovf[k].value[:n_sat].view(torch.uint8), ovf_host[k][8 * n_sat:12 * n_sat])]
                return pairs

            def deliver(dsts, lo, hi, record):
                n_sat, nnz = record[_REC_SAT], record[_REC_NNZ]
                indices, data = indices_w[:nnz], data_w[:nnz]
                rc = widen(dsts[1].data_ptr(), 8 * ibytes, indices.ctypes.data, 8 * index_dtype.itemsize, nnz, threads)
                rc |= widen(dsts[2].data_ptr(), 16, data.ctypes.data, 8 * data_dtype.itemsize, nnz, threads)
                if rc != 0:
                    raise nat.NativeError("pst_host_widen failed")
                if n_sat:
                    lib.pst_host_apply_overflow(data.ctypes.data, 8 * data_dtype.itemsize, 0, nnz, dsts[3].data_ptr(),
                                                dsts[4].data_ptr(), n_sat)
                consume(lo, hi, dsts[0].numpy().view(np.int64), indices, data)

            return pack, grow, pack, copies, deliver

        return (ibytes + 2) * G, empty, start

    def _npz_encoder(self, n, consume, index_dtype, data_dtype, compression):
        """stream_csr(compress=True): pst_csr_pack writes the final index_dtype / data_dtype bytes, pst_csr_indptr_bytes
        the indptr bytes after a running nnz kept on the device, and the compressor each member, reading its length
        from the device.  That running nnz adds up the chunks in order, so a chunk is never encoded again."""
        G, dev, st, lib, block = self.G, self.dev, nat.stream_ptr(self.dev), nat.load(), _DEFLATE_BLOCK
        isz, dsz = index_dtype.itemsize, data_dtype.itemsize
        deflate, deflate_work, tokens = _DEFLATE[compression]
        SIZE, CRC = _REC_OWN, _REC_OWN + 3               # record: the members' compressed sizes, then their CRCs
        members = ("indptr", "indices", "data")

        def empty():
            consume(0, n, [(m,) + sync_deflate(raw) for m, raw in zip(members, (bytes(n * isz), b"", b""))])

        def start(chunk, work, indptr, info, pack_flags):
            wide = [torch.empty(max(1, size), dtype=torch.uint8, device=dev)                # indptr, indices, data
                    for size in (chunk * isz, chunk * G * isz, chunk * G * dsz)]
            bound = [int(lib.pst_deflate_bound(w.numel(), block)) for w in wide]
            packed = [[torch.empty(b, dtype=torch.uint8, device=dev) for b in bound] for _ in range(2)]
            dwork_bytes = max(int(getattr(lib, deflate_work)(w.numel(), block)) for w in wide)
            dwork = torch.empty(dwork_bytes, dtype=torch.uint8, device=dev)
            running = torch.zeros(1, dtype=torch.int64, device=dev)     # nonzeros of the chunks before
            stage_host = _pinned_staging(dev, sum(bound) + 3 * 64)

            def step(k, lo, cells):
                nat.call("pst_csr_pack", work[k].data_ptr(), cells, G, G, indptr[k], 0, wide[1], 8 * isz, wide[2],
                         8 * dsz, None, None, 0, None, pack_flags, st)
                nat.call("pst_csr_indptr_bytes", indptr[k], cells, running, wide[0], 8 * isz, st)
                nnz = indptr[k][cells:cells + 1]
                for j, (count, scale, most) in enumerate(((None, 0, cells * isz), (nnz, isz, cells * G * isz),
                                                          (nnz, dsz, cells * G * dsz))):
                    nat.call(deflate, wide[j], count, scale, most, block, packed[k][j], info[k, SIZE + j],
                             info[k, CRC + j].data_ptr(), dwork, dwork_bytes, st)

            def copies(k, cells, record):
                pairs, at = [], 0
                for j in range(3):
                    size = record[SIZE + j]
                    pairs.append((packed[k][j][:size], stage_host[k][at:at + size]))
                    at = (at + size + 63) // 64 * 64
                return pairs

            def deliver(dsts, lo, hi, record):
                raw = ((hi - lo) * isz, record[_REC_NNZ] * isz, record[_REC_NNZ] * dsz)
                consume(lo, hi, [(members[j], dsts[j].numpy(), record[CRC + j] & 0xFFFFFFFF, raw[j]) for j in range(3)])

            return step, (lambda k, record: False), None, copies, deliver

        # the wide streams of a chunk and their compressed form, bounded by about as many bytes again, and the
        # tokens of the largest stream
        return (2 * (isz + dsz) + tokens * max(isz, dsz)) * G, empty, start

    def _mtx_encoder(self, n, consume, compression):
        """stream_csr(mtx=True): pst_mtx_row_bytes and pst_csr_row_offsets (the text pointer), pst_mtx_format into the
        text buffer, shared by both k, of _mtx_slot_bytes per gene slot, and the compressor over the text.  A chunk
        with more text is not formatted (pst_mtx_format writes nothing), and is formatted again in a larger buffer."""
        G, dev, st, lib, block = self.G, self.dev, nat.stream_ptr(self.dev), nat.load(), _DEFLATE_BLOCK
        deflate, deflate_work, tokens = _DEFLATE[compression]
        slot = _mtx_slot_bytes(G, n)
        TEXT_LEN, SIZE, CRC = range(_REC_OWN, _REC_OWN + 3)     # record: text length, compressed size, CRC

        def empty():
            consume(0, n, *sync_deflate(b""), 0)

        def start(chunk, work, indptr, info, pack_flags):
            row_bytes = torch.empty(chunk, dtype=torch.int32, device=dev)
            text_ptr = [torch.empty(chunk + 1, dtype=torch.int64, device=dev) for _ in range(2)]
            buf = {"cap": -1}                             # the text buffer, its deflate workspace and capacity
            packed = [None, None]
            formatted_cap = [0, 0]                        # the capacity chunk k was formatted against
            # a copy of the cached pair, so that growing one k leaves the cache as it is
            stage_host = list(_pinned_staging(dev, int(lib.pst_deflate_bound(chunk * G * slot, block))))

            def reserve(k, cap):
                """Text buffer of at least cap bytes, and room in packed[k] for its compressed form."""
                if cap > buf["cap"]:
                    buf["cap"] = cap
                    buf["text"] = torch.empty(max(16, cap), dtype=torch.uint8, device=dev)
                    buf["work_bytes"] = int(getattr(lib, deflate_work)(cap, block))
                    buf["work"] = torch.empty(max(1, buf["work_bytes"]), dtype=torch.uint8, device=dev)
                bound = int(lib.pst_deflate_bound(buf["cap"], block))
                if packed[k] is None or packed[k].numel() < bound:
                    packed[k] = torch.empty(max(1, bound), dtype=torch.uint8, device=dev)

            def encode(k, lo, cells):
                """Format chunk k from its work buffer and compress the text."""
                reserve(k, buf["cap"])
                formatted_cap[k] = buf["cap"]
                nat.call("pst_mtx_format", work[k], cells, G, G, lo, text_ptr[k], buf["cap"], buf["text"], st)
                nat.call(deflate, buf["text"], text_ptr[k][cells:cells + 1], 1, buf["cap"], block,
                         packed[k], info[k, SIZE], info[k, CRC].data_ptr(), buf["work"], buf["work_bytes"], st)

            reserve(0, chunk * G * slot)

            def step(k, lo, cells):
                nat.call("pst_mtx_row_bytes", work[k], cells, G, G, lo, row_bytes, st)
                nat.call("pst_csr_row_offsets", row_bytes, cells, text_ptr[k], st)
                info[k, TEXT_LEN].copy_(text_ptr[k][cells])
                encode(k, lo, cells)

            def grow(k, record):
                # the text did not fit the buffer as it was when the chunk was queued: nothing was formatted.  The
                # buffer may have grown since (for the chunk before), so the test is against that capacity.
                if record[TEXT_LEN] <= formatted_cap[k]:
                    return False
                reserve(k, max(record[TEXT_LEN], 2 * formatted_cap[k]))
                return True

            def copies(k, cells, record):
                size = record[SIZE]
                if stage_host[k].numel() < size:
                    stage_host[k] = torch.empty(size, dtype=torch.uint8).pin_memory()
                return [(packed[k][:size], stage_host[k][:size])]

            def deliver(dsts, lo, hi, record):
                consume(lo, hi, dsts[0].numpy(), record[CRC] & 0xFFFFFFFF, record[TEXT_LEN], record[_REC_NNZ])

            return step, grow, encode, copies, deliver

        # the text of a chunk and its compressed form, bounded by about as many bytes again, and the tokens
        return (2 + tokens) * slot * G, empty, start

    def _tsv_encoder(self, n, consume, compress, compression, row0):
        """stream_csr(tsv=True): pst_tsv_row_bytes and pst_csr_row_offsets (the text pointer), pst_tsv_format into text
        buffer k, of _tsv_slot_bytes per gene slot and the label per cell, and, with compress, the compressor over the
        text.  A chunk with more text is not formatted (pst_tsv_format writes nothing), and is formatted again in a
        larger buffer.  Without compress the text itself is copied, so it needs one buffer per k."""
        G, dev, st, lib, block = self.G, self.dev, nat.stream_ptr(self.dev), nat.load(), _DEFLATE_BLOCK
        deflate, deflate_work, tokens = _DEFLATE[compression]
        cell_text = _tsv_slot_bytes(G, n) * G + len("cell_%d\n" % (row0 + n))
        TEXT_LEN, SIZE, CRC = range(_REC_OWN, _REC_OWN + 3)     # record: text length, compressed size, CRC

        def empty():
            text = "".join("cell_%d\n" % i for i in range(row0, row0 + n)).encode("ascii")
            consume(0, n, *(sync_deflate(text) if compress else (np.frombuffer(text, np.uint8), 0, len(text))))

        def start(chunk, work, indptr, info, pack_flags):
            row_bytes = torch.empty(chunk, dtype=torch.int32, device=dev)
            text_ptr = [torch.empty(chunk + 1, dtype=torch.int64, device=dev) for _ in range(2)]
            text, packed = [None, None], [None, None]
            dwork = {"bytes": -1}                         # the deflate workspace, shared by both k
            formatted_cap = [0, 0]                        # the capacity chunk k was formatted against
            out_bytes = chunk * cell_text
            if compress:
                out_bytes = int(lib.pst_deflate_bound(out_bytes, block))
            # a copy of the cached pair, so that growing one k leaves the cache as it is
            stage_host = list(_pinned_staging(dev, out_bytes))

            def reserve(k, cap):
                """Text buffer k of cap bytes and, with compress, room for its compressed form."""
                text[k] = torch.empty(max(16, cap), dtype=torch.uint8, device=dev)
                if compress:
                    packed[k] = torch.empty(max(1, int(lib.pst_deflate_bound(cap, block))), dtype=torch.uint8,
                                            device=dev)
                    need = int(getattr(lib, deflate_work)(cap, block))
                    if need > dwork["bytes"]:
                        dwork["bytes"] = need
                        dwork["buf"] = torch.empty(max(1, need), dtype=torch.uint8, device=dev)

            def encode(k, lo, cells):
                """Format chunk k from its work buffer and, with compress, compress the text."""
                cap = formatted_cap[k] = text[k].numel()
                nat.call("pst_tsv_format", work[k], cells, G, G, row0 + lo, text_ptr[k], cap, text[k], st)
                if compress:
                    nat.call(deflate, text[k], text_ptr[k][cells:cells + 1], 1, cap, block, packed[k], info[k, SIZE],
                             info[k, CRC].data_ptr(), dwork["buf"], dwork["bytes"], st)

            for k in range(2):
                reserve(k, chunk * cell_text)

            def step(k, lo, cells):
                nat.call("pst_tsv_row_bytes", work[k], cells, G, G, row0 + lo, row_bytes, st)
                nat.call("pst_csr_row_offsets", row_bytes, cells, text_ptr[k], st)
                info[k, TEXT_LEN].copy_(text_ptr[k][cells])
                encode(k, lo, cells)

            def grow(k, record):
                # the text did not fit the buffer the chunk was formatted against: nothing was formatted
                if record[TEXT_LEN] <= formatted_cap[k]:
                    return False
                reserve(k, max(record[TEXT_LEN], 2 * formatted_cap[k]))
                return True

            def copies(k, cells, record):
                size = record[SIZE] if compress else record[TEXT_LEN]
                if stage_host[k].numel() < size:
                    stage_host[k] = torch.empty(size, dtype=torch.uint8).pin_memory()
                return [((packed if compress else text)[k][:size], stage_host[k][:size])]

            def deliver(dsts, lo, hi, record):
                consume(lo, hi, dsts[0].numpy(), record[CRC] & 0xFFFFFFFF if compress else 0, record[TEXT_LEN])

            return step, grow, encode, copies, deliver

        # the text of a chunk and, with compress, its compressed form, bounded by about as many bytes again, and the
        # tokens
        return ((2 + tokens) if compress else 1) * cell_text, empty, start

    def _dense_chunks(self, rows, scaling32, seed, cell0, tdt, chunk_cells, overflow_cap, host_out=None,
                      consume=None):
        """The counts of the cells in the transfer dtype `tdt` through _copy_chunks: straight into `host_out`
        (a CPU tensor of dtype tdt) or through pinned staging into `consume`.  Owns the dense chunk sizes and
        the narrowing: int32 is drawn into the copy buffer itself; uint16 / uint8 are drawn into an int32 work
        buffer and pst_narrow_counts writes min(count, SAT) into the copy buffer and lists the saturated counts.
        Returns that _OverflowList, or None for int32."""
        n, G, dev = int(rows.numel()), self.G, self.dev
        width = tdt.itemsize
        # ~1 GiB copies keep the copy engine at its large-transfer rate; staged chunks fit the pinned staging
        chunk, bounds = _plan_chunks(n, chunk_cells, width * G, (1 << 30) if host_out is not None else _STAGE_BYTES)
        stage = [torch.empty((chunk, G), dtype=tdt, device=dev) for _ in range(2)]
        ovf = None
        if width < 4:
            # the int32 chunk is consumed by the narrowing kernel on the sampling stream, so one is enough
            work = torch.empty((chunk, G), dtype=torch.int32, device=dev)
            if overflow_cap is None:
                # uint8 lists every count >= 255 (2e-4 of them at default depth; allow 50x that)
                overflow_cap = (1 << 20) if width == 2 else max(1 << 20, n * G // 100)
            ovf = _OverflowList(overflow_cap, dev)
        if host_out is None:
            stage_host = _pinned_staging(dev, chunk * G * width)

        def produce(k, lo, hi):
            buf = stage[k][:hi - lo]
            if ovf is None:
                self.draw(rows[lo:hi], scaling32[lo:hi], seed, cell0 + lo, out=buf)
            else:
                self.draw(rows[lo:hi], scaling32[lo:hi], seed, cell0 + lo, out=work[:hi - lo])
                nat.call("pst_narrow_counts", work.data_ptr(), hi - lo, G, G, buf.data_ptr(), G, 8 * width, lo,
                         *ovf.kernel_args, nat.stream_ptr(dev))
            if host_out is not None:
                return [(buf, host_out[lo:hi])]
            return [(buf.view(torch.uint8).view(-1), stage_host[k][:(hi - lo) * G * width])]

        self._copy_chunks(bounds, produce, consume and (lambda dsts, lo, hi: consume(dsts[0], lo, hi)))
        return ovf

    def _copy_chunks(self, bounds, produce, consume=None, collect=None):
        """The double-buffered device->host loop behind every chunked result.  For chunk i, with buffer
        k = i & 1, produce(k, lo, hi) queues the device work that fills device buffer k on the current stream
        and returns the chunk's copies: a list of (src, dst) pairs, device bytes and their host destination.
        One side stream copies every src into its dst while the next chunk is produced.  Before buffer k is
        produced again, the current stream waits on the device for its copies, so without `consume` the host
        never waits per chunk.  With `consume`, one worker thread calls consume(dsts, lo, hi) once the copies
        have landed, and the host waits for it before it copies into buffer k again (the dsts are pinned
        staging that the next use of k overwrites).
        With `collect`, the copies run one chunk late: once chunk i+1's work is queued and chunk i's has finished,
        collect(k, lo, hi) reads what chunk i left on the device while the device works on and returns (chunk i's
        copies, a record for consume(dsts, lo, hi, record)).  The copies wait for chunk i's work only: device work
        that collect queues itself must have finished when it returns.
        Owns the overlap and its teardown: whatever ends the loop, the side stream and the worker are drained
        before the buffers can go back to the allocator."""
        main = torch.cuda.current_stream(self.dev)
        copy_stream = torch.cuda.Stream(device=self.dev)
        pool = concurrent.futures.ThreadPoolExecutor(max_workers=1)
        filled = [None, None]                           # the device work on buffer k has finished
        copied = [None, None]                           # the copies out of buffer k have finished
        pending = [None, None]                          # consume still reading the host side of buffer k

        def landed(event, dsts, *args):
            event.synchronize()                         # the chunk is in dsts
            consume(dsts, *args)

        def copy(k, pairs, *args):                      # args: lo, hi and, with collect, the chunk's record
            if pending[k] is not None:
                pending[k].result()
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(filled[k])
                for src, dst in pairs:
                    dst.copy_(src, non_blocking=True)
                copied[k] = torch.cuda.Event()
                copied[k].record(copy_stream)
            if consume is not None:
                pending[k] = pool.submit(landed, copied[k], [dst for _, dst in pairs], *args)

        lag = 0 if collect is None else 1
        try:
            for i in range(len(bounds) + lag):
                if i < len(bounds):
                    k = i & 1
                    if copied[k] is not None:
                        main.wait_event(copied[k])
                    pairs = produce(k, *bounds[i])
                    filled[k] = torch.cuda.Event()
                    filled[k].record(main)
                    if not lag:
                        copy(k, pairs, *bounds[i])
                if lag and i:
                    k = (i - 1) & 1
                    filled[k].synchronize()
                    pairs, record = collect(k, *bounds[i - 1])
                    copy(k, pairs, *bounds[i - 1], record)
            for f in pending:
                if f is not None:
                    f.result()
        finally:
            copy_stream.synchronize()
            pool.shutdown(wait=True)

    def check(self):
        """One device->host read of the status word; raises like the reference would."""
        word = int(self.flags[0].item())
        if word:
            self.flags[0].zero_()
            raise_flags(word)
