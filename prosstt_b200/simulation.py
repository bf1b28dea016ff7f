"""Simulation entry points: lineage (mean expression along the tree) and the three cell
samplers with their negative-binomial count draw.

Mirror of prosstt/simulation.py (same names, arguments, defaults, return tuples and
exceptions); the numeric work is done by the sm_100a kernels behind include/prosstt_b200.h.
Extra keyword-only arguments (never required):

  seed     64-bit key of the counter-based generator; None draws it from the global
           legacy numpy stream, so `np.random.seed(s)` makes a script reproducible
  device   CUDA device (default: current)
  shard    (rank, world): sample only this rank's contiguous slice of the cells; every
           random quantity is keyed by the GLOBAL cell index, so the union over ranks is
           bit-identical to the unsharded call
  dtype    dtype of the returned count matrix (reference: int64; int32 avoids a host pass); with
           out="csr" the dtype of its data, int64 or int32
  out      "numpy" (reference behaviour), "torch" (leave everything on the GPU) or "csr": X is a
           scipy.sparse.csr_matrix (canonical: columns ascending, no explicit zeros; int32 indptr/indices,
           int64 when it has 2^31 nonzeros or more) with the same counts as "numpy".  The GPU compacts
           each chunk and only the nonzeros cross PCIe (CountEngine.draw_to_csr); not with host_out
  path     with out="csr": stream the counts chunk by chunk to a CSR shard directory at `path`
           (formats.CsrShardWriter, with the cells' pseudotime, branches and scalings) instead of holding
           them in host memory; X is then the shard's memory-mapped matrix (formats.load_csr_shard).  The
           counts are those of the in-memory call; every chunk is drawn once (CountEngine.stream_csr)
  compress with out="csr" and path: write one compressed `.npz` at `path` instead (formats.CsrNpzWriter:
           zip64, DEFLATE members, read by scipy.sparse.load_npz and np.load); the GPU compresses every chunk, so
           only compressed bytes cross PCIe and reach the disk.  X is then a formats.CompressedCsr record
           (path, shape, nnz, dtype, index_dtype, nbytes, load()), not the loaded matrix
           out="mtx" with path: write a 10x directory at `path` (formats.MtxWriter: matrix.mtx.gz genes x cells,
           features.tsv.gz, barcodes.tsv.gz named by the global cell index, cellparams.tsv.gz), read by
           Seurat::Read10X, DropletUtils::read10xCounts, Matrix::readMM and scanpy.read_10x_mtx.  The GPU formats
           and compresses every chunk, so only gzipped text crosses PCIe and reaches the disk.  X is then a
           formats.MtxRecord (path, shape, nnz, nbytes, load()); the counts are those of out="csr".  The file is
           always gzipped (compress=True is an error), and dtype must be int64 or int32 as for "csr"
           out="tsv" with path: write the reference's own counts file at `path`, the dense tab-separated table of
           tree_utils.save_matrices' `<job>_simulation.txt`, byte for byte (formats.TsvWriter: header line
           "\tgene_0\tgene_1...", rows "cell_<global index>\t<count>..."), read by
           pd.read_csv(path, sep="\t", index_col=0); with compress=True one gzip member of those bytes.  The GPU
           formats (and compresses) every chunk, so only the file's bytes cross PCIe.  X is then a
           formats.TsvRecord (path, shape, nbytes, compressed, load()); dtype must be int64 or int32 and does not
           change the text.  Under shard=, each rank writes a complete file with its own header line
  compression  "huffman" (default) or "lz77", where the GPU compresses (compress=True, out="mtx"): "lz77" adds
           LZ77 matches within each 32 KiB DEFLATE block (pst_deflate_lz_blocks), so the same content is written
           in a smaller file; "huffman" writes Huffman-only blocks.  Both files decompress to the same bytes
  sampler  "hybrid" (default): direct inversion of the NB cdf for mean <= 32, sd <= 20, gamma scale <= 32 and
           shape <= 48 - in fp32 below the 1 - 2^-14 quantile of its uniform, with a 64-bit uniform against an
           fp64-accumulated cdf above it, so body and far tail match the exact pmf (checked at 1e9 draws per
           regime) - and the gamma-Poisson mixture for everything else;
           "gamma_poisson": the mixture (NumPy's legacy algorithm family) for every count, 4.6x slower.
           Both are keyed by (seed, global cell, gene): counts never depend on the partition over GPUs
  host_transport, host_threads (sample_density with host_out): see sample_density
  host_out (sample_density) preallocated, ideally pinned, CPU tensors (X int32 (n,G), pseudotime
           int64, branch codes int32, scalings float64) that receive the result in overlapped
           chunks: the zero-allocation path for repeated or very large calls
"""
import warnings
from collections.abc import Mapping

import numpy as np
import pandas as pd
import torch

from prosstt_b200 import _native as nat
from prosstt_b200 import count_model as cm
from prosstt_b200 import hostpool
from prosstt_b200 import sim_utils as sut
from prosstt_b200.device import CountEngine, TreeTables, choice_cdf, raise_flags, tree_tables
from prosstt_b200.formats import CsrNpzWriter, CsrShardWriter, MtxWriter, TsvWriter, _csr_matrix, load_csr_shard
from prosstt_b200.sharding import shard_range

DEFAULT_SAMPLER = "hybrid"


# =============================================================================== lineage
def _walk_programs(lengths, K, seed, branch_ids, attempts, dev, draws=None):
    """Raw (un-carried) momentum walks of several branches: packed (sum T, K) device
    tensor.  `draws` = (u0, v0, eta, eps) host arrays replace the Philox draws."""
    nb = len(lengths)
    T = np.asarray(lengths, dtype=np.int32)
    row_base = np.zeros(nb, dtype=np.int32)
    row_base[1:] = np.cumsum(T)[:-1]
    eps_off = np.zeros(nb + 1, dtype=np.int64)
    eps_off[1:] = np.cumsum((T.astype(np.int64) - 1) * K)
    st = nat.stream_ptr(dev)
    d_T = nat.to_dev(T, torch.int32, dev)
    d_off = nat.to_dev(eps_off, torch.int64, dev)
    if draws is None:
        u0 = torch.empty(nb * K, dtype=torch.float64, device=dev)
        v0 = torch.empty_like(u0)
        eta = torch.empty_like(u0)
        eps = torch.empty(max(1, int(eps_off[-1])), dtype=torch.float64, device=dev)
        nat.call("pst_walk_draws", seed, nb, K, int(T.max()), nat.to_dev(branch_ids, torch.int32, dev),
                 nat.to_dev(attempts, torch.int32, dev), nat.ptr(d_T), nat.ptr(d_off),
                 nat.ptr(u0), nat.ptr(v0), nat.ptr(eta), nat.ptr(eps), st)
    else:
        u0, v0, eta = (nat.to_dev(np.ravel(x), torch.float64, dev) for x in draws[:3])
        flat = np.concatenate([np.ravel(e) for e in draws[3]]) if len(draws[3]) else np.zeros(0)
        eps = nat.to_dev(flat if flat.size else np.zeros(1), torch.float64, dev)
    W = torch.empty((int(T.sum()), K), dtype=torch.float64, device=dev)
    nat.call("pst_walk_scan", nb, K, nat.to_dev(row_base, torch.int32, dev), nat.ptr(d_T),
             nat.ptr(d_off), nat.ptr(u0), nat.ptr(v0), nat.ptr(eta), nat.ptr(eps), nat.ptr(W), st)
    return W


def diffusion(steps, seed=None, device=None):
    """One momentum random walk of `steps` points (simulation.py:89-124):
    walk[0]=log U(0,1.5), v[0]~N(0,.2), eta~U(0,1), v[t+1]=eta v[t]+N(0,2/steps),
    walk[t+1]=walk[t]+v[t]."""
    dev = nat.device(device)
    W = _walk_programs([steps], 1, nat.split_seed(seed), [0], [0], dev)
    return W[:, 0].cpu().numpy()


def sim_expr_branch(branch_length, expr_progr, cutoff=0.2, max_loops=100, seed=None, device=None):
    """K = expr_progr walks of one branch as a (T, K) array (simulation.py:21-86).  The
    reference's correlation rejection never triggers (SURVEY.md Q1); cutoff/max_loops are
    accepted and ignored."""
    dev = nat.device(device)
    W = _walk_programs([branch_length], expr_progr, nat.split_seed(seed), [0], [0], dev)
    return W.cpu().numpy()


def _sim_coeff_gamma(tree, a=0.05):
    """H[k,g] ~ Gamma(a, 1), shape (K, G) (simulation.py:192-212); global legacy stream."""
    return np.random.standard_gamma(a, size=tree.modules * tree.G).reshape((tree.modules, tree.G))


def _sim_coeff_beta(tree, groups, a=2, b=2):
    """H[k,g] += Beta(a,b) for each membership of gene g in program k
    (simulation.py:164-189)."""
    H = np.zeros((tree.modules, tree.G))
    for k in range(tree.modules):
        for gene in groups[k]:
            H[k][gene] += np.random.beta(a, b)
    return H


def simulate_coefficients(tree, fallback_a=0.04, **kwargs):
    """Program -> gene weights H (simulation.py:127-161): no 'a' -> warn, Gamma(0.04);
    'a' and 'b' -> Beta(2,2) over random groups (the values are ignored, SURVEY.md Q4);
    'a' only -> Gamma(a)."""
    if "a" not in kwargs:
        warnings.warn("No argument 'a' specified in kwargs: using gamma and a=0.04", UserWarning)
        return _sim_coeff_gamma(tree, fallback_a)
    if "b" in kwargs:
        return _sim_coeff_beta(tree, sut.create_groups(tree.modules, tree.G))
    return _sim_coeff_gamma(tree, a=kwargs["a"])


class _LineageState(object):
    """Device buffers of simulate_lineage: packed W (P,K) and rel (P,G) in fp64, followed by scratch
    rows that hold the candidate branches of the level being simulated."""

    SCRATCH_BYTES = 8 << 30                      # rel rows of the candidates of one round

    def __init__(self, tree, H, dev):
        self.dev = dev
        self.tables = tree_tables(tree, dev)
        self.K, self.G = int(tree.modules), int(tree.G)
        self.H = nat.to_dev(H, torch.float64, dev)
        self.P = P = self.tables.P
        Tmax = int(self.tables.T.max())
        # room for at least one candidate of the longest branch, at most SCRATCH_BYTES of rel rows
        self.S = max(Tmax, min(4 * P, self.SCRATCH_BYTES // max(1, 8 * self.G)))
        self.Wall = torch.zeros((P + self.S, max(1, self.K)), dtype=torch.float64, device=dev)
        self.relall = torch.empty((P + self.S, self.G), dtype=torch.float64, device=dev)
        self.W, self.rel = self.Wall[:P], self.relall[:P]
        self.colmax = torch.empty(self.G, dtype=torch.float64, device=dev)
        top = tree.topology
        self.parent = {}
        for p, c in top:
            self.parent.setdefault(c, p)             # first row wins (sim_utils.py:632-635)

    def rows(self, b):
        i = self.tables.index[b]
        lo = int(self.tables.row_base[i])
        return lo, lo + int(self.tables.T[i])

    def gene_maxima(self):
        """Per-gene maximum of rel over the whole tree (sim_utils.py:406-426 before the exp), recomputed
        from W and H without reading the (P, G) table back."""
        self.colmax.fill_(float("-inf"))
        nat.call("pst_rel_means", nat.ptr(self.Wall), nat.ptr(self.H), None, 0, self.P, self.K, self.G,
                 None, None, None, nat.ptr(self.colmax), nat.stream_ptr(self.dev))
        return self.colmax

    def try_candidates(self, seed, cands):
        """One batched round of the rejection loop.  cands = [(branch, attempt), ...] in visiting order.
        Draws, scans, carries and multiplies every candidate into the scratch rows with one launch per
        stage.  Returns the scratch row of each candidate."""
        dev, K, G, P = self.dev, self.K, self.G, self.P
        st = nat.stream_ptr(dev)
        tb = self.tables
        ids = np.array([tb.index[b] for b, _ in cands], dtype=np.int32)
        att = np.array([a for _, a in cands], dtype=np.int32)
        T = tb.T[ids].astype(np.int32)
        row = np.zeros(len(cands), dtype=np.int64)
        row[1:] = np.cumsum(T.astype(np.int64))[:-1]
        row += P
        if K > 0:
            eps_off = np.zeros(len(cands) + 1, dtype=np.int64)
            eps_off[1:] = np.cumsum((T.astype(np.int64) - 1) * K)
            d_T = nat.to_dev(T, torch.int32, dev)
            d_off = nat.to_dev(eps_off, torch.int64, dev)
            d_row = nat.to_dev(row.astype(np.int32), torch.int32, dev)
            n = len(cands) * K
            u0 = torch.empty(n, dtype=torch.float64, device=dev)
            v0, eta = torch.empty_like(u0), torch.empty_like(u0)
            eps = torch.empty(max(1, int(eps_off[-1])), dtype=torch.float64, device=dev)
            nat.call("pst_walk_draws", seed, len(cands), K, int(T.max()), nat.to_dev(ids, torch.int32, dev),
                     nat.to_dev(att, torch.int32, dev), d_T, d_off, u0, v0, eta, eps, st)
            nat.call("pst_walk_scan", len(cands), K, d_row, d_T, d_off, u0, v0, eta, eps, self.Wall, st)
            plast = np.array([self.rows(self.parent[b])[1] - 1 if b in self.parent else -1 for b, _ in cands],
                             dtype=np.int32)
            if np.any(plast >= 0):
                nat.call("pst_walk_carry", len(cands), K, d_row, d_T, nat.to_dev(plast, torch.int32, dev),
                         self.Wall, st)
        nrows = int(T.sum())
        nat.call("pst_rel_means", nat.ptr(self.Wall), nat.ptr(self.H), None, P, nrows, K, G,
                 nat.ptr(self.relall), None, None, None, st)
        return row, T

    def accept(self, b, row):
        lo, hi = self.rows(b)
        self.Wall[lo:hi].copy_(self.Wall[row:row + hi - lo])
        self.relall[lo:hi].copy_(self.relall[row:row + hi - lo])


def _bfs_levels(tree):
    """Branches in the reference's visiting order (sut.breadth_first_branches) cut into runs of equal
    depth: the branches of one run depend only on earlier runs (their parents) and on each other
    through the sibling test."""
    order = [b.item() if hasattr(b, "item") else b for b in sut.breadth_first_branches(tree)]
    depth = {tree.root: 0}
    for _ in range(len(order)):
        for p, c in tree.topology:
            if p in depth and c not in depth:
                depth[c] = depth[p] + 1
    levels = []
    for b in order:
        d = depth.get(b, -1)
        if levels and levels[-1][0] == d:
            levels[-1][1].append(b)
        else:
            levels.append((d, [b]))
    return order, [lv for _, lv in levels]


def simulate_lineage(tree, rel_exp_cutoff=8, intra_branch_tol=0.5, inter_branch_tol=0,
                     seed=None, device=None, max_attempts=10000, _return_state=False, **kwargs):
    """Relative mean expression of every gene at every tree position
    (simulation.py:215-286).  Branches are visited breadth first; each gets K momentum
    walks (device scan), is shifted to start where its parent ended, and rel = W.H is
    formed; the branch is redrawn while its largest relative expression exceeds
    rel_exp_cutoff or some pair of already simulated siblings has no more than
    inter_branch_tol of its genes anticorrelated.

    The rejection loop runs a whole breadth-first level at a time: attempt a of branch b is a pure
    function of (seed, b, a), so several attempts of every branch of the level are drawn, scanned,
    carried, multiplied and tested (pst_lineage_checks: maximum per candidate, anticorrelated genes
    per sibling pair) with one launch per stage and ONE device->host read per round; the host then
    takes, branch by branch in the reference's visiting order, the first attempt that passes - the
    same attempt the one-at-a-time loop would have taken.

    Returns (pd.Series rel_means, pd.Series programs, H), indexed in visiting order."""
    if not len(tree.time) == tree.num_branches:
        raise ValueError("the parameters are not enough for %i branches" % tree.num_branches)
    dev = nat.device(device)
    H = simulate_coefficients(tree, **kwargs)
    walk_seed = nat.split_seed(seed)
    state = _LineageState(tree, H, dev)
    tables = state.tables
    K, G = state.K, state.G
    order, levels = _bfs_levels(tree)
    position = {b: i for i, b in enumerate(order)}
    group_of = {}
    for siblings in tree.get_parallel_branches().values():
        members = [s.item() if hasattr(s, "item") else s for s in siblings]
        for b in members:
            group_of.setdefault(b, members)          # first group that lists the branch (sim_utils.py:663-667)
    st = nat.stream_ptr(dev)
    done = set()
    for level in levels:
        pending = list(level)
        base = {b: 0 for b in level}
        want = 4
        while pending:
            # candidates of this round: `A` consecutive attempts of a prefix of the pending branches
            T_of = {b: int(tables.T[tables.index[b]]) for b in pending}
            A = max(1, min(want, state.S // max(1, sum(T_of.values()))))
            batch, used = [], 0
            for b in pending:
                if used + A * T_of[b] > state.S and batch:
                    break
                batch.append(b)
                used += A * T_of[b]
            cands = [(b, base[b] + a) for b in batch for a in range(A)]
            if max(a for _, a in cands) >= max_attempts:
                b = batch[0]
                raise RuntimeError("branch %s: no acceptable expression programs after %d "
                                   "attempts (rel_exp_cutoff=%g, inter_branch_tol=%g)"
                                   % (str(b), max_attempts, rel_exp_cutoff, inter_branch_tol))
            row, T = state.try_candidates(walk_seed, cands)
            slot = {c: i for i, c in enumerate(cands)}
            # sibling pairs: candidate x (accepted sibling | every candidate of a sibling visited earlier)
            pairs, pa, pb, pn = {}, [], [], []
            for b in batch:
                older = [s for s in group_of.get(b, [b]) if s != b and position.get(s, 1 << 60) < position[b]
                         and (s in done or s in batch)]
                for a in range(A):
                    i = slot[(b, base[b] + a)]
                    for s in older:
                        if s in done:
                            lo, hi = state.rows(s)
                            keys = [((b, a, s, None), lo, hi - lo)]
                        else:
                            keys = [((b, a, s, a2), int(row[slot[(s, base[s] + a2)]]), T_of[s]) for a2 in range(A)]
                        for key, other_row, other_T in keys:
                            pairs[key] = len(pa)
                            pa.append(int(row[i]))
                            pb.append(other_row)
                            pn.append(min(int(T[i]), other_T))
            slot_max = torch.full((len(cands),), float("-inf"), dtype=torch.float64, device=dev)
            pair_neg = torch.zeros(max(1, len(pa)), dtype=torch.int32, device=dev)
            nat.call("pst_lineage_checks", state.relall, G, len(cands), nat.to_dev(row, torch.int64, dev),
                     nat.to_dev(T, torch.int32, dev), len(pa),
                     nat.to_dev(pa, torch.int64, dev) if pa else None, nat.to_dev(pb, torch.int64, dev) if pa else None,
                     nat.to_dev(pn, torch.int32, dev) if pa else None, slot_max, pair_neg, st)
            tops = slot_max.cpu().numpy()                     # the one device->host read of the round
            negs = pair_neg.cpu().numpy()
            taken = {}                                         # branch -> attempt index accepted in this round
            for b in batch:
                siblings = [s for s in group_of.get(b, [b]) if s != b and position.get(s, 1 << 60) < position[b]]
                if any(s not in done and s not in taken for s in siblings):
                    continue                                   # an earlier sibling is still open: next round
                for a in range(A):
                    ok = not tops[slot[(b, base[b] + a)]] > rel_exp_cutoff            # simulation.py:270
                    for s in siblings:
                        key = (b, a, s, None) if (b, a, s, None) in pairs else (b, a, s, taken[s])
                        ok = ok and (negs[pairs[key]] / (G * 1.0) > inter_branch_tol)  # sim_utils.py:249-251
                    if ok:
                        taken[b] = a
                        break
                else:
                    base[b] += A
            for b, a in taken.items():
                state.accept(b, int(row[slot[(b, base[b] + a)]]))
                done.add(b)
            pending = [b for b in pending if b not in done]
            want = 8
    if _return_state:
        return state, H
    rel_host = state.rel.cpu().numpy()
    W_host = state.W.cpu().numpy()[:, :K]
    rel_means, programs = {}, {}
    for branch in sut.breadth_first_branches(tree):
        b = branch.item() if hasattr(branch, "item") else branch
        lo, hi = state.rows(b)
        rel_means[branch] = rel_host[lo:hi]
        programs[branch] = W_host[lo:hi]
    return pd.Series(rel_means), pd.Series(programs), H


class DeviceMeans(Mapping):
    """`tree.means` kept on the GPU: the fp32 (P, G) table the samplers read, plus W, H and the
    gene scale from which a branch's fp64 (T_b, G) array is rebuilt on the device and copied to
    the host the first time `tree.means[branch]` is read.  A read-only Mapping like the reference's
    dict (`tree.add_genes(tree.means)` works); `to_host()` gives a plain dict of ndarrays, which is
    also what pickling / copying a tree should carry."""

    def __init__(self, tables, W, H, gene_scale, table32):
        self.tables, self.W, self.H, self.gene_scale, self.table32 = tables, W, H, gene_scale, table32
        self._host = {}

    def __getitem__(self, branch):
        b = branch.item() if hasattr(branch, "item") else branch
        if b not in self._host:
            i = self.tables.index[b]
            lo, T = int(self.tables.row_base[i]), int(self.tables.T[i])
            K, G = self.H.shape
            buf = torch.empty((T, G), dtype=torch.float64, device=self.W.device)
            # pst_rel_means indexes its outputs from packed row 0: shift the pointer back by lo rows
            nat.call("pst_rel_means", nat.ptr(self.W), nat.ptr(self.H), nat.ptr(self.gene_scale), lo, T, K, G,
                     None, buf.data_ptr() - lo * G * 8, None, None, nat.stream_ptr(self.W.device))
            self._host[b] = buf.cpu().numpy()
        return self._host[b]

    def __iter__(self):
        return iter(self.tables.names)

    def __len__(self):
        return len(self.tables.names)

    def __contains__(self, b):
        return b in self.tables.index

    def to_host(self):
        """Plain dict branch -> (T_b, G) float64 ndarray, as the reference keeps it."""
        return {b: self[b] for b in self.tables.names}

    def __reduce__(self):                      # pickling / deepcopy carry host arrays, not CUDA tensors
        return (dict, (self.to_host(),))


def default_gene_expression_on_device(tree, seed=None, device=None, abs_max=5000, gene_mean=0.8,
                                      gene_std=1, base_seed=None, **kwargs):
    """simulate_lineage + simulate_base_gene_exp + exp(rel)*scale + add_genes (tree.py:436-446)
    without the host round trip of the (P, G) tables: the per-gene maximum comes from the device
    and the means table is built in HBM.  The O(G) base-expression draw runs on the host (global
    legacy stream, reference draw order) unless `base_seed` is given, in which case it is the
    counter-based device draw (sut.base_gene_exp_on_device).  Sets tree.means to a DeviceMeans.
    Returns (H, gene_scale)."""
    kwargs.setdefault("a", 0.05)
    state, H = simulate_lineage(tree, seed=seed, device=device, _return_state=True, **kwargs)
    dev, tb = state.dev, state.tables
    st = nat.stream_ptr(dev)
    # max over the tree of exp(rel) per gene (sim_utils.py:406-426,461): exp is monotone; the per-gene
    # maximum comes out of the W.H kernel, the (P, G) table is not read back
    colmax = state.gene_maxima()
    if base_seed is not None:
        scale = sut.base_gene_exp_on_device(torch.exp(colmax), base_seed, abs_max, gene_mean, gene_std)
        base = scale.cpu().numpy()
    else:
        base = sut._base_gene_exp_legacy(np.exp(colmax.cpu().numpy()), abs_max, gene_mean, gene_std)  # sim_utils.py:463-469
        scale = nat.to_dev(base, torch.float64, dev)
    table32 = torch.empty((tb.P, state.G), dtype=torch.float32, device=dev)
    nat.call("pst_rel_means", nat.ptr(state.Wall), nat.ptr(state.H), nat.ptr(scale), 0, tb.P, state.K, state.G,
             None, None, nat.ptr(table32), None, st)
    tree.means = DeviceMeans(tb, state.W.clone(), state.H, scale, table32)      # drops the scratch rows
    del state
    tree.invalidate_device_cache()
    return H, base


# =============================================================================== samplers
def _shard_range(n, shard):
    if shard is None:
        return 0, n
    rank, world = shard
    return shard_range(n, rank, world)


def _check_csr_request(out, dtype, host_out=None, path=None, compress=False, compression="huffman"):
    """out="csr" takes int64 (default) or int32 data and no preallocated host_out; path needs out="csr";
    compress needs both.  out="mtx" needs path, takes int64 or int32 and neither host_out nor compress.
    out="tsv" needs path, takes int64 or int32, compress and no host_out.
    compression is "huffman" or "lz77"; "lz77" only where the GPU compresses (compress=True or out="mtx")."""
    if compression not in ("huffman", "lz77"):
        raise ValueError("compression must be 'huffman' or 'lz77', not %r" % (compression,))
    if out == "tsv":
        if path is None:
            raise ValueError("out='tsv' writes the reference's _simulation.txt: it needs path=")
        if host_out is not None:
            raise ValueError("host_out cannot be combined with out='tsv'")
        if np.dtype(dtype) not in (np.dtype(np.int64), np.dtype(np.int32)):
            raise ValueError("out='tsv' takes dtype int64 or int32, not %s" % np.dtype(dtype))
        if compression == "lz77" and not compress:
            raise ValueError("compression='lz77' applies where the GPU compresses: out='tsv' needs compress=True")
        return
    if compression == "lz77" and out != "mtx" and not compress:
        raise ValueError("compression='lz77' applies where the GPU compresses: out='csr', path=, compress=True "
                         "or out='mtx', path=")
    if out == "mtx":
        if path is None:
            raise ValueError("out='mtx' writes a 10x directory: it needs path=")
        if compress:
            raise ValueError("out='mtx' always gzips its files: compress=True does not apply")
        if host_out is not None:
            raise ValueError("host_out cannot be combined with out='mtx'")
        if np.dtype(dtype) not in (np.dtype(np.int64), np.dtype(np.int32)):
            raise ValueError("out='mtx' takes dtype int64 or int32, not %s" % np.dtype(dtype))
        return
    if compress and (path is None or out != "csr"):
        raise ValueError("compress=True writes a compressed CSR file: it needs out='csr' and path=")
    if path is not None and out != "csr":
        raise ValueError("path= writes a CSR shard: it needs out='csr'")
    if out != "csr":
        return
    if host_out is not None:
        raise ValueError("host_out cannot be combined with out='csr'")
    if np.dtype(dtype) not in (np.dtype(np.int64), np.dtype(np.int32)):
        raise ValueError("out='csr' stores int64 or int32 counts, not %s" % np.dtype(dtype))


def _sample_counts(engine, rows, s32, seed, first, dtype, out, path=None, cells=None, compress=False,
                   compression="huffman"):
    """The count matrix of the cells described by rows/s32: a device int32 tensor (out="torch"), a
    scipy.sparse.csr_matrix with `dtype` data (out="csr", CountEngine.draw_to_csr: only the nonzeros cross
    PCIe) or a fresh host array of `dtype` (reference: int64, simulation.py:651).  The host forms never hold
    the whole matrix on the GPU: chunks are sampled, copied into pinned staging and expanded into the result
    by host threads while the next chunk is sampled (CountEngine.draw_to_host).
    out="csr" with `path`: the chunks go to a CSR shard at path (CountEngine.stream_csr into a
    formats.CsrShardWriter, which also stores `cells` = (pseudotime, branches, scalings) host arrays) and the
    shard's memory-mapped matrix is returned; with `compress`, into one compressed file (formats.CsrNpzWriter,
    stream_csr(compress=True)), and its formats.CompressedCsr record is returned.
    out="mtx": the chunks go to a 10x directory at path (stream_csr(mtx=True) into a formats.MtxWriter, whose
    barcodes count from the global cell index `first`), and its formats.MtxRecord is returned.
    out="tsv": the chunks go to the reference's _simulation.txt at path, gzipped with `compress`
    (stream_csr(tsv=True) into a formats.TsvWriter, whose rows are named from the global cell index `first`), and
    its formats.TsvRecord is returned.  `compression` picks the device compressor of the compressed forms
    (stream_csr)."""
    if out == "torch":
        X = engine.draw(rows, s32, seed, first)
        engine.check()
        return X
    if out == "mtx":
        _check_csr_request(out, dtype, path=path)
        with MtxWriter(path, (int(rows.numel()), engine.G), *cells, first=first) as w:
            engine.stream_csr(rows, s32, seed, first, lambda lo, hi, *text: w.append(hi - lo, text[3], *text[:3]),
                              mtx=True, compression=compression)
        return w.record()
    if out == "tsv":
        _check_csr_request(out, dtype, path=path, compress=compress, compression=compression)
        with TsvWriter(path, (int(rows.numel()), engine.G), first=first, compress=compress) as w:
            engine.stream_csr(rows, s32, seed, first, lambda lo, hi, *text: w.append(hi - lo, *text), tsv=True,
                              compress=compress, compression=compression)
        return w.record()
    if out == "csr":
        _check_csr_request(out, dtype)
        n = int(rows.numel())
        if path is not None and compress:
            with CsrNpzWriter(path, (n, engine.G), *cells, dtype=dtype) as w:
                engine.stream_csr(rows, s32, seed, first, lambda lo, hi, parts: [w.append(*p) for p in parts],
                                  w.index_dtype, dtype, compress=True, compression=compression)
            return w.record()
        if path is not None:
            with CsrShardWriter(path, (n, engine.G), *cells, dtype=dtype) as shard:
                engine.stream_csr(rows, s32, seed, first, lambda lo, hi, *chunk: shard.append(*chunk),
                                  shard.index_dtype, dtype)
            return load_csr_shard(path)[0]
        indptr, indices, data = engine.draw_to_csr(rows, s32, seed, first, data_dtype=dtype)
        torch.cuda.current_stream(engine.dev).synchronize()
        engine.check()
        return _csr_matrix(indptr, indices, data, (n, engine.G))
    want = np.dtype(dtype)
    n = int(rows.numel())
    direct = want in (np.dtype(np.int32), np.dtype(np.int64))
    # a fresh matrix - or the memory of an earlier result that has been garbage-collected (hostpool: no page
    # faults from the second call on)
    host, fresh = hostpool.result_array((n, engine.G), want if direct else np.int64)
    if n and engine.G:
        engine.draw_to_host(rows, s32, seed, first, host, fresh=fresh)    # untouched pages: ordinary stores
    torch.cuda.current_stream(engine.dev).synchronize()
    engine.check()
    return host if direct else host.astype(want)


def _draw_for_cells(tree, tables, pt, codes, rows, alpha, beta, scale, scale_mean, scale_v,
                    seed, first, dev, dtype, out, sampler, host_out=None, host_transport=None, host_threads=0,
                    path=None, compress=False, compression="huffman"):
    """Common tail of every sampler (simulation.py:590-599): scalings, then counts.
    host_out = (X, pseudotime, branch_codes, scalings) preallocated CPU tensors (int32 (n,G),
    int64, int32, float64; ideally pinned): the counts are streamed into them in cell chunks
    while the next chunk is being sampled, and numpy views of them are returned.  X may also be
    uint16 or uint8 (a half / a quarter of the PCIe bytes): elements read min(count, 65535 / 255)
    and a fifth entry of host_out, a dict, receives the exact values of the saturated elements as
    "index" (flat, into X) and "value" arrays (formats.widen rebuilds the int32 matrix); without
    the dict a saturated element raises OverflowError instead of passing silently."""
    _check_csr_request(out, dtype, host_out, path, compress, compression)
    n = int(rows.numel())
    s64, s32 = sut.calc_scalings(n, scale, scale_mean, scale_v, seed=nat.derive_seed(seed, 1),
                                 first=first, device=dev, return_device=True)
    engine = CountEngine(tree, tables, alpha, beta, dev, sampler=sampler)
    if host_out is not None:
        hX, hpt, hcodes, hs = host_out[:4]
        overflow = host_out[4] if len(host_out) > 4 else None
        if tuple(hX.shape) != (n, engine.G) or hX.dtype not in (torch.int32, torch.int64, torch.uint16, torch.uint8):
            raise ValueError("host_out[0] must be an int32 (or int64 / uint16 / uint8) CPU tensor of shape (%d, %d)"
                             % (n, engine.G))
        hpt.copy_(pt, non_blocking=True)
        hcodes.copy_(codes, non_blocking=True)
        hs.copy_(s64, non_blocking=True)
        engine.draw_to_host(rows, s32, nat.derive_seed(seed, 2), first, hX, transport=host_transport,
                            threads=host_threads)
        torch.cuda.current_stream(dev).synchronize()
        engine.check()
        if engine.overflow is not None:
            if overflow is not None:
                overflow["index"], overflow["value"] = engine.overflow
            elif len(engine.overflow[0]):
                raise OverflowError("%d counts saturate the %s matrix: pass a dict as host_out[4] to receive them, "
                                    "or use an int32 buffer"
                                    % (len(engine.overflow[0]), str(hX.dtype).replace("torch.", "")))
        return hX.numpy(), hpt.numpy(), tables.branch_names(hcodes.numpy()), hs.numpy()
    if out == "torch":
        return _sample_counts(engine, rows, s32, nat.derive_seed(seed, 2), first, dtype, out), pt, codes, s64
    cells = pt.cpu().numpy(), tables.branch_names(codes.cpu().numpy()), s64.cpu().numpy()
    X = _sample_counts(engine, rows, s32, nat.derive_seed(seed, 2), first, dtype, out, path=path, cells=cells,
                       compress=compress, compression=compression)
    return (X,) + cells


def sample_density(tree, no_cells, alpha=0.3, beta=2, scale=True, scale_v=0.7, scale_mean=0.,
                   seed=None, device=None, shard=None, dtype=np.int64, out="numpy",
                   sampler=DEFAULT_SAMPLER, uniforms=None, host_out=None, host_transport=None, host_threads=0, *,
                   path=None, compress=False, compression="huffman"):
    """Sample `no_cells` (pseudotime, branch) pairs according to tree.density and draw
    their counts (simulation.py:416-471).  Returns (X, pseudotime, branches, scalings).
    `uniforms` (one per cell) replays externally supplied draws through the index map.
    host_transport ("direct", "i32", "u16", "u8"; with host_out): the format in which the counts cross
    PCIe; the narrow ones are expanded into the int32 / int64 host matrix by `host_threads` host threads
    (0 = all) together with their exact overflow list - the caller receives the same counts either way.
    out="csr" / "mtx" / "tsv", path, compress, compression: the sparse and on-disk forms of the module docstring;
    out="mtx", path="counts_10x" writes a 10x directory and returns its formats.MtxRecord; out="tsv",
    path="job_simulation.txt" writes the reference's counts file and returns its formats.TsvRecord."""
    dev = nat.device(device)
    seed = nat.split_seed(seed)
    tables = tree_tables(tree, dev)
    cdf = nat.to_dev(choice_cdf(tables.density_packed(tree)), torch.float64, dev)
    lo, hi = _shard_range(int(no_cells), shard)
    n = hi - lo
    st = nat.stream_ptr(dev)
    if uniforms is None:
        u = torch.empty(n, dtype=torch.float64, device=dev)
        nat.call("pst_uniform_f64", nat.derive_seed(seed, 0), nat.TAG_DENSITY_U, lo, n, nat.ptr(u), st)
    else:
        u = nat.to_dev(np.asarray(uniforms)[lo:hi], torch.float64, dev)
    rows = torch.empty(n, dtype=torch.int32, device=dev)
    pt = torch.empty(n, dtype=torch.int64, device=dev)
    codes = torch.empty(n, dtype=torch.int32, device=dev)
    nat.call("pst_density_index", nat.ptr(cdf), tables.P, nat.ptr(u), n, nat.ptr(tables.d("pos_pt")),
             nat.ptr(tables.d("pos_branch")), nat.ptr(rows), nat.ptr(pt), nat.ptr(codes), st)
    return _draw_for_cells(tree, tables, pt, codes, rows, alpha, beta, scale, scale_mean, scale_v,
                           seed, lo, dev, dtype, out, sampler, host_out=host_out, host_transport=host_transport,
                           host_threads=host_threads, path=path, compress=compress, compression=compression)


def cover_whole_tree(tree):
    """All (pseudotime, branch) pairs of the tree: timezone-major, then branch, then time
    (simulation.py:520-548)."""
    zones = tree.populate_timezone()
    live = sut.assign_branches(tree.branch_times(), zones)
    pseudotime, branches = [], []
    for i, (lo, hi) in enumerate(zones):
        for branch in live[i]:
            pseudotime.extend(range(lo, hi + 1))
            branches.extend([branch] * (hi + 1 - lo))
    return pseudotime, branches


def sample_whole_tree(tree, n_factor, alpha=0.3, beta=2, scale=True, scale_mean=0., scale_v=0.7,
                      seed=None, device=None, shard=None, dtype=np.int64, out="numpy",
                      sampler=DEFAULT_SAMPLER, *, path=None, compress=False, compression="huffman"):
    """Every tree position sampled n_factor times (simulation.py:474-517).  out / path / compress /
    compression: see sample_density."""
    dev = nat.device(device)
    seed = nat.split_seed(seed)
    tables = tree_tables(tree, dev)
    total = len(tables.cover_pt) * int(n_factor)
    lo, hi = _shard_range(total, shard)
    n = hi - lo
    rows = torch.empty(n, dtype=torch.int32, device=dev)
    pt = torch.empty(n, dtype=torch.int64, device=dev)
    codes = torch.empty(n, dtype=torch.int32, device=dev)
    nat.call("pst_whole_tree_index", nat.ptr(tables.d("cover_pt")), nat.ptr(tables.d("cover_branch")),
             nat.ptr(tables.d("cover_row")), len(tables.cover_pt), int(n_factor), lo, n,
             nat.ptr(pt), nat.ptr(codes), nat.ptr(rows), nat.stream_ptr(dev))
    return _draw_for_cells(tree, tables, pt, codes, rows, alpha, beta, scale, scale_mean, scale_v,
                           seed, lo, dev, dtype, out, sampler, path=path, compress=compress, compression=compression)


def draw_times(timepoint, no_cells, max_time, var=4, seed=None, first=0, device=None,
               return_device=False, normals=None):
    """Pseudotimes around a sample point: N(timepoint, var) truncated toward zero and
    clipped to [0, max_time-1] (simulation.py:382-413; `var` is used as a std)."""
    dev = nat.device(device)
    st = nat.stream_ptr(dev)
    if normals is None:
        z = torch.empty(no_cells, dtype=torch.float64, device=dev)
        nat.call("pst_normal_f64", nat.split_seed(seed), nat.TAG_SERIES_Z, int(first), no_cells,
                 float(timepoint), float(var), None, None, nat.ptr(z), st)
    else:
        z = nat.to_dev(normals, torch.float64, dev)
    pt = torch.empty(no_cells, dtype=torch.int64, device=dev)
    nat.call("pst_times_from_normals", nat.ptr(z), no_cells, int(max_time), nat.ptr(pt), st)
    return pt if return_device else pt.cpu().numpy()


def sample_pseudotime_series(tree, cells, series_points, point_std, alpha=0.3, beta=2, scale=True,
                             scale_mean=0, scale_v=0.7, seed=None, device=None, shard=None,
                             dtype=np.int64, out="numpy", sampler=DEFAULT_SAMPLER, *, path=None, compress=False,
                             compression="huffman"):
    """Time-series experiment: normally distributed pseudotimes around each sample point,
    branches picked by density (simulation.py:319-379).  out / path / compress / compression: see
    sample_density."""
    dev = nat.device(device)
    seed = nat.split_seed(seed)
    series_points, cells, point_std = sut.process_timeseries_input(series_points, cells, point_std)
    max_time = tree.get_max_time()
    total = int(np.sum(cells))
    lo, hi = _shard_range(total, shard)
    # N(point, std) per cell of the global range [lo, hi): one launch per sample point over its own cells
    # (element index = global cell index), no per-cell loc/scale arrays to build and upload
    n = hi - lo
    st = nat.stream_ptr(dev)
    z = torch.empty(n, dtype=torch.float64, device=dev)
    start = 0
    for point, count, std in zip(series_points, cells, point_std):
        a, b = max(lo, start), min(hi, start + int(count))
        if b > a:
            nat.call("pst_normal_f64", nat.derive_seed(seed, 0), nat.TAG_SERIES_Z, a, b - a, float(point), float(std),
                     None, None, z[a - lo:b - lo], st)
        start += int(count)
    pt = torch.empty(n, dtype=torch.int64, device=dev)
    if n:
        nat.call("pst_times_from_normals", nat.ptr(z), n, int(max_time), nat.ptr(pt), st)
    return _sample_data_at_times(tree, pt, alpha=alpha, beta=beta, scale=scale, scale_mean=scale_mean,
                                 scale_v=scale_v, seed=nat.derive_seed(seed, 3), device=dev,
                                 dtype=dtype, out=out, sampler=sampler, _first=lo, path=path, compress=compress,
                                 compression=compression)


def sample_whole_tree_restricted(tree, alpha=0.2, beta=3, seed=None, device=None, dtype=np.int64,
                                 out="numpy", sampler=DEFAULT_SAMPLER, *, path=None, compress=False,
                                 compression="huffman"):
    """Bare-bones run with default lineage parameters (simulation.py:289-316): one cell
    per pseudotime value, random branch, per-gene alpha/beta around the given means.  out / path / compress /
    compression: see sample_density."""
    sample_time = np.arange(0, tree.get_max_time())
    tree.default_gene_expression()
    alphas, betas = cm.generate_negbin_params(tree, mean_alpha=alpha, mean_beta=beta)
    return _sample_data_at_times(tree, sample_time, alpha=alphas, beta=betas, seed=seed,
                                 device=device, dtype=dtype, out=out, sampler=sampler, path=path,
                                 compress=compress, compression=compression)


def _sample_data_at_times(tree, sample_pt, branches=None, alpha=0.3, beta=2, scale=True,
                          scale_mean=0., scale_v=0.7, seed=None, device=None, dtype=np.int64,
                          out="numpy", sampler=DEFAULT_SAMPLER, _first=0, path=None, compress=False,
                          compression="huffman"):
    """Cells at given pseudotimes (simulation.py:551-599): pick branches if they are not
    supplied, draw library sizes, draw counts.  `_first` is the global index of the first
    cell (sharded callers).  out / path / compress / compression: see sample_density."""
    dev = nat.device(device)
    seed = nat.split_seed(seed)
    tables = tree_tables(tree, dev)
    pt = sample_pt if isinstance(sample_pt, torch.Tensor) else \
        nat.to_dev(np.asarray(sample_pt), torch.int64, dev)
    n = int(pt.numel())
    if branches is None:
        codes, rows, flags = sut._pick_branch_codes(tree, pt, nat.derive_seed(seed, 0), _first, dev,
                                                    tables=tables)
    else:
        codes, rows, flags = _rows_for(tables, pt, branches, dev)
    # a bad pseudotime / branch gives an out-of-range row, which the draw samples from row 0 and flags too;
    # the index map's own status word is read after the draw has been queued (no stall in front of it)
    try:
        result = _draw_for_cells(tree, tables, pt, codes, rows, alpha, beta, scale, scale_mean, scale_v,
                                 seed, _first, dev, dtype, out, sampler, path=path, compress=compress,
                                 compression=compression)
    except IndexError:
        sut.check_flags(flags)
        raise
    sut.check_flags(flags)
    return result


def _rows_for(tables, pt, branches, dev):
    codes = branches if isinstance(branches, torch.Tensor) else \
        nat.to_dev(tables.branch_codes(branches), torch.int32, dev)
    n = int(pt.numel())
    if int(codes.numel()) != n:
        raise ValueError("pseudotime and branches must have the same length")
    rows = torch.empty(n, dtype=torch.int32, device=dev)
    flags = torch.zeros(1, dtype=torch.int32, device=dev)
    nat.call("pst_rows_from_branch", nat.ptr(pt), nat.ptr(codes), n, tables.B,
             nat.ptr(tables.d("branch_start")), nat.ptr(tables.d("row_base")), nat.ptr(tables.d("T")),
             nat.ptr(rows), nat.ptr(flags), nat.stream_ptr(dev))
    return codes, rows, flags


def draw_counts(tree, pseudotime, branches, scalings, alpha, beta, seed=None, device=None,
                dtype=np.int64, out="numpy", sampler=DEFAULT_SAMPLER, first=0, *, path=None, compress=False,
                compression="huffman"):
    """UMI counts of cells at (pseudotime, branch) with library sizes `scalings`
    (simulation.py:602-651): X[n,g] ~ NB(mean = means[branch_n][t_n - start, g]*scaling_n,
    variance = alpha_g mean^2 + beta_g mean).  out="csr", path=p writes the CSR shard with the
    pseudotime, branches and scalings given here and returns its memory-mapped matrix; with compress=True the
    compressed file, and its formats.CompressedCsr record.  out="mtx", path=p writes the 10x directory with
    them (barcodes cell_<first + i>) and returns its formats.MtxRecord.  out="tsv", path=p writes the reference's
    _simulation.txt (rows cell_<first + i>) and returns its formats.TsvRecord.  compression="lz77": see
    sample_density."""
    dev = nat.device(device)
    _check_csr_request(out, dtype, path=path, compress=compress, compression=compression)
    seed = nat.split_seed(seed)
    tables = tree_tables(tree, dev)
    pt = pseudotime if isinstance(pseudotime, torch.Tensor) else \
        nat.to_dev(np.asarray(pseudotime), torch.int64, dev)
    codes, rows, flags = _rows_for(tables, pt, branches, dev)
    sut.check_flags(flags)
    s32 = nat.to_dev(scalings, torch.float32, dev)
    if np.ndim(alpha) == 0:
        alpha = [alpha] * tree.G
    if np.ndim(beta) == 0:
        beta = [beta] * tree.G
    engine = CountEngine(tree, tables, alpha, beta, dev, sampler=sampler)
    cells = None
    if path is not None:
        given = scalings.detach().cpu().numpy() if isinstance(scalings, torch.Tensor) else scalings
        cells = pt.cpu().numpy(), tables.branch_names(codes.cpu().numpy()), np.asarray(given, dtype=np.float64)
    return _sample_counts(engine, rows, s32, seed, first, dtype, out, path=path, cells=cells, compress=compress,
                          compression=compression)


def add_non_diff_genes(inform_expr_matrix, genes, gene_params, cell_scalings, seed=None,
                       device=None, sampler=DEFAULT_SAMPLER):
    """Append `genes` constant-mean genes (mu = scaling * base_expr) to a count matrix
    (simulation.py:654-675): the same NB kernel on a tree of one branch and one pseudotime step
    whose means row is base_expr.  Returns a float64 (N, G + genes) array like the reference."""
    from prosstt_b200.tree import Tree
    dev = nat.device(device)
    X0 = np.asarray(inform_expr_matrix)
    N, G = X0.shape
    base = np.asarray(gene_params["base_expr"], dtype=np.float64).reshape(1, genes)
    flat = Tree(topology=[], time={0: 1}, num_branches=1, branch_points=0, modules=1, G=genes)
    flat.add_genes({0: base})
    engine = CountEngine(flat, TreeTables(flat, dev), gene_params["alpha"], gene_params["beta"], dev, sampler=sampler)
    rows = torch.zeros(N, dtype=torch.int32, device=dev)
    s32 = nat.to_dev(cell_scalings, torch.float32, dev)
    fusion = np.zeros((N, G + genes))
    fusion[:, :G] = X0
    fusion[:, G:] = _sample_counts(engine, rows, s32, nat.split_seed(seed), 0, np.int64, "numpy")
    return fusion
