"""CPU oracle for the PROSSTT simulation hot path.  TEST INFRASTRUCTURE ONLY.

This file is a plain-NumPy restatement of what the reference (soedinglab/prosstt
1.2.0, pure Python) computes on the path named by BASELINE.json -> north_star.
It is the *checker*: only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s
`cpu_baseline` / `--impl reference` legs may import it.  Nothing under
`prosstt_b200/` imports it, and the product path has no CPU fallback.

Parity status: PINNED.  The reference has no tests or golden vectors of its own
(SURVEY.md section 4), so the pins are fixtures produced by running the reference
itself in the build container (tests/golden/make_golden.py -> tests/golden/*.npz,
maps.json); tests/test_oracle_golden.py checks every function below against them
bit for bit (integer maps, draws-in deterministic stages, and complete sampler
runs replayed through the legacy MT19937 stream).

Third-party arithmetic: the per-count draw is not in the reference tree; it is
scipy.stats.nbinom.rvs -> numpy.random.RandomState.negative_binomial (unpinned in
the reference's setup.py:12; this image: numpy 2.3.5 / scipy 1.18.1; NumPy freezes
the legacy RandomState stream).  `nb_draw_legacy` below calls that very function;
its published algorithm (gamma-Poisson mixture: Marsaglia-Tsang gamma, PTRS
Poisson for lam >= 10, multiplication method below) is what the CUDA sampler
re-implements on a counter-based generator, so counts are compared in
distribution, not bit for bit (north star, correctness part 3).  Our own counter-based
sampler is, in addition, replayed count by count from its Philox words
(oracle/count_replay.py, tests/test_count_replay.py).

All file:line citations are relative to /root/reference/prosstt/.
"""
from collections import OrderedDict

import numpy as np


# ---------------------------------------------------------------------------
# tree integer maps
# ---------------------------------------------------------------------------
class OTree:
    """The fields of tree.Tree (tree.py:51-80) the hot path reads."""

    def __init__(self, topology, time, root=None, G=0, modules=0, density=None):
        self.topology = [list(p) for p in topology]
        self.time = OrderedDict(time)
        self.branches = list(self.time.keys())            # tree.py:65
        self.root = self.branches[0] if root is None else root   # tree.py:72-75
        self.G = G
        self.modules = modules
        if density is None:                               # tree.py:138-151
            total = 0
            for v in self.time.values():
                total += v
            density = {b: np.array([1.0 / total] * int(self.time[b])) for b in self.branches}
        self.density = density
        self.means = None


def branch_times(tree):
    """tree.py:376-399 - [start, end] (inclusive) per branch; insertion order is
    root first, then children in topology-row order."""
    bt = OrderedDict()
    bt[tree.root] = [0, tree.time[tree.root] - 1]
    for parent, child in tree.topology:
        end = bt[parent][1]
        bt[child] = [end + 1, end + tree.time[child]]
    return bt


def paths(tree, start):
    """tree.py:302-330 - all root-to-leaf paths, depth first in topology order."""
    kids = [c for p, c in tree.topology if p == start]
    if not kids:
        return [[start]]
    out = []
    for k in kids:
        for tail in paths(tree, k):
            out.append([start] + tail)
    return out


def max_time(tree):
    """tree.py:267-285."""
    return int(max(sum(tree.time[b] for b in p) for p in paths(tree, tree.root)))


def populate_timezone(tree):
    """tree.py:332-374 with morph_stack (tree.py:402-423): per path a stack of
    half-open [start, end) intervals; cut all stacks at the smallest current end."""
    stacks = []
    for p in paths(tree, tree.root):
        acc, st = 0, []
        for b in p:
            st.append([acc, acc + tree.time[b]])
            acc += tree.time[b]
        stacks.append(st)
    zones = []
    while stacks:
        starts = [s[0][0] for s in stacks]
        ends = [s[0][1] for s in stacks]
        lo, hi = min(ends), max(ends)
        if lo == hi:
            zones.append([max(starts), hi - 1])
            for s in stacks:
                s.pop(0)
        else:
            zones.append([max(starts), lo - 1])
            for s in stacks:
                if s[0][1] != lo:
                    s.insert(1, [lo, s[0][1]])
                s.pop(0)
        stacks = [s for s in stacks if s]
    return zones


def assign_branches(bt, zones):
    """sim_utils.py:274-339 - branches whose [start,end] contains the zone, in
    branch_times order."""
    res = OrderedDict()
    for i, (z0, z1) in enumerate(zones):
        live = [k for k, (s, e) in bt.items() if z0 >= s and z1 <= e]
        if live:
            res[i] = live
    return res


def cover_whole_tree(tree):
    """simulation.py:520-548 - zone-major, then branch, then time."""
    zones = populate_timezone(tree)
    assign = assign_branches(branch_times(tree), zones)
    pt, br = [], []
    for i, (z0, z1) in enumerate(zones):
        for b in assign.get(i, []):
            pt.extend(range(z0, z1 + 1))
            br.extend([b] * (z1 + 1 - z0))
    return pt, br


def bfs_branches(tree):
    """sim_utils.py:545-608 - stable sort of tree.branches by depth below the root
    (unreached branches keep -1 and sort first)."""
    level = OrderedDict((b, -1) for b in tree.branches)
    level[tree.root] = 0
    frontier = [tree.root]
    seen = set()
    while frontier:
        nxt = []
        for node in frontier:
            if node in seen:
                continue
            seen.add(node)
            for p, c in tree.topology:
                if p == node:
                    level[c] = level[node] + 1
                    nxt.append(c)
        frontier = nxt
    return [b for b, _ in sorted(level.items(), key=lambda kv: kv[1])]


def parent_of(tree, branch):
    """sim_utils.py:632-635 - first topology row whose child is `branch`."""
    for p, c in tree.topology:
        if c == branch:
            return p
    return None


# ---------------------------------------------------------------------------
# lineage: walks, carry, relative means, absolute means
# ---------------------------------------------------------------------------
def diffusion_from_draws(u0, v0, eta, eps):
    """simulation.py:89-124 given its draws (u0~U(0,1.5), v0~N(0,.2), eta~U(0,1),
    eps[t]~N(0,2/T)): walk[0]=log(u0); walk[t+1]=walk[t]+v[t]; v[t+1]=eta*v[t]+eps[t]."""
    T = len(eps) + 1
    walk = np.zeros(T)
    v = v0
    walk[0] = np.log(u0)
    for t in range(T - 1):
        walk[t + 1] = walk[t] + v
        v = eta * v + eps[t]
    return walk


def branch_programs_from_draws(u0, v0, eta, eps):
    """simulation.py:21-86 - K walks stacked and transposed to (T, K); the
    correlation rejection is dead code (SURVEY.md Q1)."""
    K = len(u0)
    return np.stack([diffusion_from_draws(u0[k], v0[k], eta[k], eps[k]) for k in range(K)]).T


def carry_from_parent(child, parent):
    """sim_utils.py:129-142 - shift child so its first row equals parent's last."""
    return child - (child[0] - parent[-1])


def lineage_from_draws(tree, draws, H):
    """simulation.py:264-269 for the ACCEPTED attempt of each branch:
    draws[b] = (u0[K], v0[K], eta[K], eps[K,T_b-1]).  Returns programs, rel_means."""
    W, rel = {}, {}
    for b in bfs_branches(tree):
        w = branch_programs_from_draws(*draws[b])
        p = parent_of(tree, b)
        if p is not None:
            w = carry_from_parent(w, W[p])
        W[b] = w
        rel[b] = np.dot(w, H)
    return W, rel


def max_rel_exp(tree, rel):
    """sim_utils.py:406-426 + :461 - per gene max over the tree of exp(rel)."""
    return np.max(np.stack([np.max(np.exp(rel[b]), axis=0) for b in tree.branches], axis=1), axis=1)


def base_gene_exp_from_normals(max_per_gene, normals, abs_max=5000):
    """sim_utils.py:463-469 - per gene consume normals (already loc/scale-shifted)
    until exp(z)*max <= abs_max.  Returns (scale, number of normals consumed)."""
    out = np.zeros(len(max_per_gene))
    i = 0
    for g in range(len(max_per_gene)):
        while True:
            s = np.exp(normals[i])
            i += 1
            if not s * max_per_gene[g] > abs_max:
                break
        out[g] = s
    return out, i


def absolute_means(rel, gene_scale):
    """tree.py:180-183 / generate_simN.py:109-111."""
    return {b: np.exp(rel[b]) * gene_scale for b in rel}


def pearson_anticorrelated(rel_a, rel_b):
    """sim_utils.py:145-168 + :249-251 - number of genes whose Pearson r over the
    first min(T_a,T_b) rows is < 0 (NaN for constant columns counts as not < 0)."""
    n = min(rel_a.shape[0], rel_b.shape[0])
    a = rel_a[:n] - rel_a[:n].mean(axis=0)
    b = rel_b[:n] - rel_b[:n].mean(axis=0)
    with np.errstate(invalid="ignore", divide="ignore"):
        r = (a * b).sum(axis=0) / np.sqrt((a * a).sum(axis=0) * (b * b).sum(axis=0))
    return int(np.sum(r < 0))


# ---------------------------------------------------------------------------
# count model
# ---------------------------------------------------------------------------
def negbin_params_from_normals(za, zb):
    """count_model.py:42-48 with za~N(log mean_alpha, log a_scale), zb likewise."""
    return np.exp(za), np.exp(zb) + 1


def get_pr_umi(a, b, m):
    """count_model.py:156-161."""
    a, b, m = np.asarray(a, float), np.asarray(b, float), np.asarray(m, float)
    with np.errstate(invalid="ignore", divide="ignore"):
        s2 = a * m ** 2 + b * m
        p = (s2 - m) / s2
        r = m ** 2 / (s2 - m)
    p = np.where(s2 <= 0, 0.0, p)
    r = np.where(s2 <= 0, 0.0, r)
    return p, r


def scalings_from_normals(z):
    """sim_utils.py:494-495."""
    return np.exp(z)


# ---------------------------------------------------------------------------
# samplers' index maps
# ---------------------------------------------------------------------------
def choice_index(p, u):
    """numpy legacy RandomState.choice(replace=True, p=p): cdf=cumsum(p);
    cdf/=cdf[-1]; searchsorted(cdf, u, 'right')  (call sites simulation.py:464,
    sim_utils.py:399)."""
    cdf = np.cumsum(np.asarray(p, float))
    cdf /= cdf[-1]
    return np.searchsorted(cdf, u, side="right")


def density_positions(tree):
    """simulation.py:452-461 - flat (abs pseudotime, branch, density) over
    tree.branches order."""
    bt = branch_times(tree)
    pt = np.concatenate([np.arange(bt[b][0], bt[b][1] + 1) for b in tree.branches])
    br = [b for b in tree.branches for _ in range(tree.time[b])]
    pr = np.concatenate([np.asarray(tree.density[b], float) for b in tree.branches])
    return pt, br, pr


def sample_density_index(tree, u):
    """simulation.py:464-467 given the N uniforms consumed by random.choice."""
    pt, br, pr = density_positions(tree)
    idx = choice_index(pr, u)
    return pt[idx], [br[i] for i in idx], idx


def draw_times_from_normals(z, max_t):
    """simulation.py:409-413 given z = norm.rvs(loc=t, scale=std): truncate toward
    zero, clip to [0, max_t-1]."""
    t = np.asarray(z).astype(int)
    t[t < 0] = 0
    t[t >= max_t] = max_t - 1
    return t


def pick_branches_from_uniforms(tree, pseudotime, u):
    """sim_utils.py:342-403 - first zone containing t, density indexed with
    t - zone_start (SURVEY.md Q5), one uniform per cell."""
    zones = populate_timezone(tree)
    assign = assign_branches(branch_times(tree), zones)
    out = []
    for t, ui in zip(pseudotime, u):
        zi = next(i for i, (z0, z1) in enumerate(zones) if z0 <= t <= z1)
        cand = assign[zi]
        w = np.array([tree.density[b][t - zones[zi][0]] for b in cand])
        out.append(cand[int(choice_index(w / w.sum(), ui))])
    return out


def timeseries_input(series_points, cells, point_std):
    """sim_utils.py:501-542 (SURVEY.md Q7)."""
    n = len(series_points)
    if np.ndim(cells) == 0:
        cells = np.array([cells / n] * n, dtype=int)
    else:
        cells = np.array(cells, dtype=int)
    if np.ndim(point_std) == 0:
        point_std = np.array([point_std / n] * n, dtype=float)
    else:
        point_std = np.array(point_std, dtype=float)
    return np.asarray(series_points, dtype=int) if not isinstance(series_points, np.ndarray) \
        else series_points, cells, point_std


# ---------------------------------------------------------------------------
# the hot loop: draw_counts
# ---------------------------------------------------------------------------
def cell_means(tree, pseudotime, branches, scalings):
    """simulation.py:633-640 - mu[n,g] = means[branch_n][pt_n - start(branch_n), g]*scaling_n."""
    bt = branch_times(tree)
    rows = np.stack([tree.means[b][int(t) - bt[b][0]] for t, b in zip(pseudotime, branches)])
    return rows * np.asarray(scalings)[:, None]


def nb_draw_legacy(r, p_success, rng):
    """simulation.py:647-648: scipy nbinom(n=r, p=1-p).rvs() == legacy
    RandomState.negative_binomial(n, p) (SURVEY.md section 5 [probe])."""
    return rng.negative_binomial(r, p_success)


def draw_counts(tree, pseudotime, branches, scalings, alpha, beta, rng):
    """simulation.py:602-651 with an explicit legacy RandomState."""
    mu = cell_means(tree, pseudotime, branches, scalings)
    a = np.broadcast_to(np.asarray(alpha, float), (tree.G,))
    b = np.broadcast_to(np.asarray(beta, float), (tree.G,))
    p, r = get_pr_umi(a[None, :], b[None, :], mu)
    if not (np.all(r > 0) and np.all((1 - p) > 0) and np.all((1 - p) <= 1)):
        raise ValueError("Domain error in arguments.")  # scipy _argcheck (SURVEY.md Q9)
    return nb_draw_legacy(r.ravel(), (1 - p).ravel(), rng).reshape(mu.shape)


def sample_density(tree, no_cells, alpha, beta, rng, scale=True, scale_v=0.7, scale_mean=0.0):
    """simulation.py:416-471 end to end on an explicit legacy RandomState
    (draw order: N uniforms, N normals, N*G NB draws; SURVEY.md appendix B)."""
    u = rng.random_sample(no_cells)
    pt, br, _ = sample_density_index(tree, u)
    sc = np.exp(rng.normal(scale_mean, scale_v, size=no_cells)) if scale else np.ones(no_cells)
    X = draw_counts(tree, pt, br, sc, alpha, beta, rng)
    return X, pt, br, sc


def sample_whole_tree(tree, n_factor, alpha, beta, rng, scale=True, scale_mean=0.0, scale_v=0.7):
    """simulation.py:474-517."""
    pt, br = cover_whole_tree(tree)
    pt = np.repeat(pt, n_factor)
    br = list(np.repeat(np.array(br, dtype=object), n_factor))
    sc = np.exp(rng.normal(scale_mean, scale_v, size=len(pt))) if scale else np.ones(len(pt))
    return draw_counts(tree, pt, br, sc, alpha, beta, rng), pt, br, sc


def sample_pseudotime_series(tree, cells, series_points, point_std, alpha, beta, rng,
                             scale=True, scale_mean=0.0, scale_v=0.7):
    """simulation.py:319-379."""
    pts, cells, std = timeseries_input(series_points, cells, point_std)
    mt = max_time(tree)
    times = np.concatenate([draw_times_from_normals(rng.normal(t, s, size=n), mt)
                            for t, n, s in zip(pts, cells, std)])
    br = pick_branches_from_uniforms(tree, times, [rng.random_sample() for _ in times])
    sc = np.exp(rng.normal(scale_mean, scale_v, size=len(times))) if scale else np.ones(len(times))
    return draw_counts(tree, times, br, sc, alpha, beta, rng), times, br, sc


# ---------------------------------------------------------------------------
# counter-based generator used by the CUDA kernels (integer part only): the
# published Philox4x32-10 (Salmon et al., SC'11; Random123).  Used by the tests
# to pin the device generator bit for bit; known-answer vectors in
# tests/test_oracle_golden.py.
# ---------------------------------------------------------------------------
PHILOX_M0, PHILOX_M1 = 0xD2511F53, 0xCD9E8D57
PHILOX_W0, PHILOX_W1 = 0x9E3779B9, 0xBB67AE85


def philox4x32_10(counter, key):
    """counter: (...,4) uint32, key: (...,2) uint32 -> (...,4) uint32."""
    c = [np.asarray(counter[..., i], dtype=np.uint64) for i in range(4)]
    k0 = np.asarray(key[..., 0], dtype=np.uint64)
    k1 = np.asarray(key[..., 1], dtype=np.uint64)
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(PHILOX_M0) * c[0]
        p1 = np.uint64(PHILOX_M1) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & mask,
             (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & mask]
        k0 = (k0 + np.uint64(PHILOX_W0)) & mask
        k1 = (k1 + np.uint64(PHILOX_W1)) & mask
    return np.stack(c, axis=-1).astype(np.uint32)


# ---------------------------------------------------------------------------
# simulate_lineage on an explicit legacy RandomState (used to build the bench tree on
# the CPU for the reference arm, and pinned against the golden lineage fixtures)
# ---------------------------------------------------------------------------
def diffusion(steps, rng):
    """simulation.py:104-124 with its draw order: U(0,1.5), N(0,.2), U(0,1), then one
    N(0, 2/steps) per step."""
    u0 = rng.uniform(0, 1.5)
    v0 = rng.normal(0, 0.2)
    eta = rng.uniform()
    eps = np.array([rng.normal(0, 2 / steps) for _ in range(steps - 1)])
    return diffusion_from_draws(u0, v0, eta, eps)


def simulate_lineage(tree, rng, a=0.05, rel_exp_cutoff=8, inter_branch_tol=0):
    """simulation.py:254-286 (gamma coefficients): H, then per BFS branch redraw until the
    cutoff and sibling-divergence tests pass.  Returns (rel_means, programs, H)."""
    K, G = tree.modules, tree.G
    H = rng.standard_gamma(a, size=K * G).reshape(K, G)          # simulation.py:211
    kids_of = {}
    for p, c in tree.topology:
        kids_of.setdefault(p, []).append(c)
    W, rel = {}, {}
    for b in bfs_branches(tree):
        while True:
            w = np.stack([diffusion(tree.time[b], rng) for _ in range(K)]).T
            p = parent_of(tree, b)
            if p is not None:
                w = carry_from_parent(w, W[p])
            W[b] = w
            rel[b] = np.dot(w, H)
            above = np.max(rel[b]) > rel_exp_cutoff
            # find_parallel (sim_utils.py:663-667): parents in np.unique order; first
            # sibling group containing b, restricted to branches that have programs
            sibs = None
            for parent in sorted(kids_of, key=lambda x: x):
                if b in kids_of[parent]:
                    sibs = sorted(s for s in set(kids_of[parent]) if s in W)
                    break
            ok = True
            if sibs is not None and len(sibs) > 1:
                for i in range(len(sibs) - 1):
                    for j in range(i + 1, len(sibs)):
                        frac = pearson_anticorrelated(rel[sibs[i]], rel[sibs[j]]) / (G * 1.0)
                        ok = ok and (frac > inter_branch_tol)
            if not above and ok:
                break
    return rel, W, H
