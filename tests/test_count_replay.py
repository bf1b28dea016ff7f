"""Every count of both samplers against an fp64 replay of its own Philox words (oracle/count_replay.py).

The distributional tests (test_gpu_parity.py) cannot see errors that keep the distribution or are rare: a
word taken from the wrong slot of a Philox block, a result written to the wrong (cell, gene), a redraw that
reads the wrong block, a search hand-off one term off.  Here each count is replayed from (seed, cell, gene)
and the kernel's fp32 parameters (pst_nb_params_f32); a count the replay determines must come out exactly,
the others inside the replay's interval.  The CPU tests check the replay itself.
"""
import numpy as np
import pytest
import scipy.stats

from oracle import count_replay as cr
from oracle.prosstt_oracle import philox4x32_10

INT_MAX = cr.INT_MAX


def _params_f32(mu, th):
    """The NB parameters in fp32 with exact functions where the kernel uses MUFU instructions."""
    mu = np.asarray(mu, np.float32); th = np.asarray(th, np.float32)
    r = (mu / th).astype(np.float32)
    q = (th / (np.float32(1) + th)).astype(np.float32)
    a = (q * r).astype(np.float32)
    e2 = (-r.astype(np.float64) * np.log2(1.0 + th.astype(np.float64))).astype(np.float32)
    return {"mu": mu, "theta": th, "q": q, "a": a, "log2p0": e2}


def _nb_pmf(q, a, kmax):
    q = float(q); r = float(a) / q
    return scipy.stats.nbinom.pmf(np.arange(kmax + 1), r, 1.0 - q)


def _chi2_pvalue(values, pmf):
    n = values.size
    hist = np.bincount(values, minlength=pmf.size)[:pmf.size].astype(float)
    exp = pmf * n
    keep = exp >= 20
    o = np.append(hist[keep], n - hist[keep].sum())
    e = np.append(exp[keep], n - exp[keep].sum())
    if e[-1] < 5:
        o, e = o[:-1], e[:-1]
    return scipy.stats.chi2.sf(((o - e) ** 2 / e).sum(), len(e) - 1)


# -------------------------------------------------------------------------------- CPU: the replay
def test_philox_known_answers_and_counter_layout():
    """Random123's known-answer vectors, and the counter words of every stream of pst_draw_counts:
    (gene or quad, cell lo, tag << 16 | cell hi, block) - the layout test_philox_words_bit_exact pins for
    the generator itself."""
    z = philox4x32_10(np.zeros((1, 4), np.uint32), np.zeros((1, 2), np.uint32))[0]
    assert [int(x) for x in z] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    f = philox4x32_10(np.full((1, 4), 0xFFFFFFFF, np.uint32), np.full((1, 2), 0xFFFFFFFF, np.uint32))[0]
    assert [int(x) for x in f] == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    seed, cell, gene = 0x0123456789ABCDEF, (1 << 33) + 5, 77
    got = cr.philox_block(seed, gene, cell, cr.TAG_COUNT, 0xFFFFFFFE)
    ctr = np.array([[gene, 5, (0x200 << 16) | 2, 0xFFFFFFFE]], np.uint32)
    key = np.array([[0x89ABCDEF, 0x01234567]], np.uint32)
    assert np.array_equal(got.reshape(1, 4), philox4x32_10(ctr, key))


def test_u01_is_the_kernels_conversion():
    w = np.array([0, 1, 2 ** 24, 2 ** 31, 0xFFFFFF7F, 0xFFFFFF80, 0xFFFFFFFF], np.uint32)
    u = cr.u01(w)
    assert u.dtype == np.float32 and u[0] == np.float32(2.0 ** -33) and u[-1] == np.float32(0.99999994)
    assert np.all(u > 0) and np.all(u < 1) and np.all(np.diff(u) >= 0)


@pytest.mark.parametrize("mu,th", [(0.5, 0.3), (3.0, 1.5), (14.0, 6.0), (30.0, 12.0), (5.0, 1e-8), (5.0, 0.05)])
def test_inversion_point_values_follow_the_nb_pmf_and_its_quantile(mu, th):
    """The inversion's point value for uniform Philox words is NB(r = a/q, 1 - q) distributed (chi-square at
    4e5 draws), and equals scipy's quantile function of u / c (c the common pmf factor of the fp32 log2 P(0))
    wherever the replay calls the count determined."""
    n = 400000
    p = _params_f32(np.full(n, mu), np.full(n, th))
    w = cr.philox_block(99, np.arange(n) % 1000, np.arange(n) // 1000, cr.TAG_QUAD, 0)[:, 0]
    fw = w.astype(np.float32)
    U = fw.astype(np.float64) * 2.0 ** -32 * (1 + 2.0 ** -15)
    pt, lo, hi, _ = cr.nb_inversion(U, p["q"], p["a"], p["log2p0"], False, p["mu"])
    q, a = float(p["q"][0]), float(p["a"][0])
    c = 2.0 ** (float(p["log2p0"][0]) - (a / q) * np.log1p(-q) / np.log(2.0))
    keep = U < c                                            # above the top: the kernel redraws
    pmf = _nb_pmf(q, a, int(pt.max()) + 1)
    assert _chi2_pvalue(pt[keep], pmf) > 1e-4
    det = (lo == hi) & keep
    assert det.mean() > 0.99
    ppf = scipy.stats.nbinom.ppf(U[det] / c, a / q, 1 - q)
    assert np.array_equal(pt[det], ppf.astype(np.int64))
    assert np.all(lo[keep] <= pt[keep]) and np.all(pt[keep] <= hi[keep])


@pytest.mark.parametrize("mu,th", [(2.0, 0.5), (14.0, 6.0), (30.0, 12.0), (5.0, 0.05)])
def test_fp32_emulation_of_the_head_lands_in_the_band(mu, th):
    """The kernel's t_k recursion and fp32 accumulation of d = cdf - u, emulated in NumPy float32 with exact
    functions in place of the MUFU instructions (and the drain's P(k) form from k = 33 with a + q k advanced
    by additions), for 1e6 uniforms: every result lies inside the replay's [lo, hi]."""
    n = 1000000
    p = _params_f32(np.full(n, mu), np.full(n, th))
    w = cr.philox_block(7, np.arange(n) % 997, np.arange(n) // 997, cr.TAG_QUAD, 0)[:, 1]
    fw = w.astype(np.float32)
    sel = fw < np.float32(4294705152.0)
    fw, p = fw[sel], {k: v[sel] for k, v in p.items()}
    U = fw.astype(np.float64) * 2.0 ** -32 * (1 + 2.0 ** -15)
    _, lo, hi, _ = cr.nb_inversion(U, p["q"], p["a"], p["log2p0"], False, p["mu"])
    f32 = np.float32

    def fma(x, y, z):                                       # one rounding (fp64 holds x y exactly)
        return (x.astype(np.float64) * np.float64(y) + z.astype(np.float64)).astype(f32)

    q, a = p["q"], p["a"]
    t = np.exp2(p["log2p0"].astype(np.float64)).astype(f32)
    d = fma(fw, -(2.0 ** -32) * (1 + 2.0 ** -15), t)
    cnt = (d < 0).astype(np.int64)
    inv_fact = [f32(1.0 / np.prod(np.arange(1, k + 1, dtype=np.float64))) for k in range(34)]
    for k in range(33):
        t = (t * (a if k == 0 else fma(q, float(k), a))).astype(f32)
        d = fma(t, inv_fact[k + 1], d)
        cnt += (d < 0)
    pp = (t * inv_fact[33]).astype(f32)
    ak = fma(q, 33.0, a)
    k = 33
    while (d < 0).any() and k < 2000:
        pp = (pp * (ak * f32(1.0 / (k + 1))).astype(f32)).astype(f32)
        d = (d + pp).astype(f32)
        cnt += (d < 0)
        ak = (ak + q).astype(f32)
        k += 1
    assert np.all((lo <= cnt) & (cnt <= hi)), np.nonzero(~((lo <= cnt) & (cnt <= hi)))[0][:10]
    assert (lo == hi).mean() > 0.99


@pytest.mark.parametrize("sampler,mu,th", [("gamma_poisson", 0.4, 2.0), ("gamma_poisson", 4.0, 0.5),
                                           ("hybrid", 60.0, 40.0), ("gamma_poisson", 300.0, 0.3),
                                           ("hybrid", 500.0, 2.0)])
def test_mixture_point_values_follow_the_nb_pmf(sampler, mu, th):
    """The mixture replay (Marsaglia-Tsang, inversion below lambda = 10, PTRS above) gives NB(mu/theta,
    1/(1+theta)) counts: chi-square at 2e5 draws on the determined counts, which are nearly all."""
    n = 200000
    p = _params_f32(np.full(n, mu), np.full(n, th))
    p["route"] = np.zeros(n, np.int32)
    res = cr.replay(sampler, 31337, np.arange(n) // 64, np.arange(n) % 64, p)
    det = res["lo"] == res["hi"]
    assert det.mean() > 0.99
    r = float(p["mu"][0]) / float(p["theta"][0])
    pmf = scipy.stats.nbinom.pmf(np.arange(int(res["lo"][det].max()) + 1), r, 1 / (1 + float(p["theta"][0])))
    assert _chi2_pvalue(res["lo"][det], pmf) > 1e-4


# -------------------------------------------------------------------------------- GPU: every count
_STATS = {}


def _record(sampler, res):
    for k, name in enumerate(cr.PATH_NAMES):
        sel = res["path"] == k
        if sel.any():
            tot, det = _STATS.get((sampler, name), (0, 0))
            _STATS[(sampler, name)] = (tot + int(sel.sum()), det + int((res["lo"][sel] == res["hi"][sel]).sum()))


class _Gpu:
    def __init__(self):
        import torch
        from prosstt_b200 import _native as nat
        self.torch, self.nat = torch, nat
        self.dev = torch.device("cuda:0")

    def t(self, a, dtype):
        return self.nat.to_dev(np.ascontiguousarray(a), dtype, self.dev)

    def params(self, M, s, alpha, bm):
        """The hook pst_nb_params_f32 on fp32 inputs (the kernel's own __device__ functions)."""
        torch, nat = self.torch, self.nat
        n = M.size
        ins = [self.t(x.astype(np.float32).ravel(), torch.float32) for x in (M, s, alpha, bm)]
        outs = {k: torch.empty(n, dtype=torch.float32, device=self.dev) for k in ("mu", "theta", "r", "q", "a", "log2p0")}
        route = torch.empty(n, dtype=torch.int32, device=self.dev)
        nat.call("pst_nb_params_f32", *ins, n, outs["mu"], outs["theta"], outs["r"], outs["q"], outs["a"],
                 outs["log2p0"], route, nat.stream_ptr(self.dev))
        res = {k: v.cpu().numpy() for k, v in outs.items()}
        res["route"] = route.cpu().numpy()
        return res

    def draw(self, sampler, means, alpha, bm, rows, sc, seed, cell0, ldx, stats=False):
        torch, nat = self.torch, self.nat
        P, G = means.shape
        n = rows.size
        X = torch.full((n, ldx), -7, dtype=torch.int32, device=self.dev)
        status = torch.zeros(4, dtype=torch.int32, device=self.dev)
        words = int(nat.load().pst_draw_scratch_words(n, G, P))
        scratch = torch.empty(words, dtype=torch.int32, device=self.dev)
        gs = [torch.zeros(G, dtype=torch.int64, device=self.dev) for _ in range(3)] if stats else [None] * 3
        nat.call("pst_draw_counts", self.t(means.astype(np.float32), torch.float32), P, G,
                 self.t(rows.astype(np.int32), torch.int32), self.t(sc.astype(np.float32), torch.float32),
                 self.t(alpha.astype(np.float32), torch.float32), self.t(bm.astype(np.float32), torch.float32),
                 seed, cell0, n, X, ldx, status, nat.SAMPLERS[sampler], scratch, words, gs[0], gs[1], gs[2],
                 nat.stream_ptr(self.dev))
        torch.cuda.synchronize()
        return X.cpu().numpy(), int(status[0].item()), [g.cpu().numpy() if stats else None for g in gs]

    def check(self, sampler, means, alpha, bm, rows, sc, seed=2024, cell0=0, ldx=None, stats=False):
        """Draw with the raw ABI, replay every count, assert; returns (X, replay)."""
        P, G = means.shape
        n = rows.size
        ldx = G + 5 if ldx is None else ldx
        X, status, gs = self.draw(sampler, means, alpha, bm, rows, sc, seed, cell0, ldx, stats)
        assert np.all(X[:, G:] == -7), "padding beyond G written"
        got = X[:, :G].astype(np.int64).ravel()
        cells = np.repeat(np.arange(n), G); genes = np.tile(np.arange(G), n)
        prm = self.params(means[rows[cells], genes], sc[cells], alpha[genes], bm[genes])
        res = cr.replay(sampler, seed, cell0 + cells.astype(np.uint64), genes, prm)
        _record(sampler, res)
        det = res["lo"] == res["hi"]
        bad = np.nonzero(det & (got != res["lo"]))[0]
        assert bad.size == 0, _dump(sampler, "determined count differs", bad, cells, genes, got, res, prm, cell0)
        out = np.nonzero(~det & ((got < res["lo"]) | (got > res["hi"])))[0]
        assert out.size == 0, _dump(sampler, "count outside the replay's interval", out, cells, genes, got, res, prm, cell0)
        assert status == res["flags"], (status, res["flags"])
        if stats:
            Xg = X[:, :G].astype(np.int64)
            assert np.array_equal(gs[0], Xg.sum(0)) and np.array_equal(gs[1], (Xg * Xg).sum(0))
            assert np.array_equal(gs[2], (Xg == 0).sum(0))
        return X[:, :G], res


def _dump(sampler, what, idx, cells, genes, got, res, prm, cell0):
    lines = ["%s: %d counts (%s)" % (what, idx.size, sampler)]
    for i in idx[:12]:
        lines.append("  cell %d gene %d path %s kernel %d replay [%d, %d] mu %r theta %r q %r a %r log2p0 %r route %d" % (
            cell0 + cells[i], genes[i], cr.PATH_NAMES[res["path"][i]], got[i], res["lo"][i], res["hi"][i],
            float(prm["mu"][i]), float(prm["theta"][i]), float(prm["q"][i]), float(prm["a"][i]),
            float(prm["log2p0"][i]), int(prm["route"][i])))
    return "\n".join(lines)


@pytest.fixture(scope="module")
def gpu():
    yield _Gpu()
    if _STATS:
        print("\ndetermined fraction per (sampler, path):")
        for (s, name), (tot, det) in sorted(_STATS.items()):
            print("  %-14s %-18s %9d counts  %.5f" % (s, name, tot, det / tot))


SAMPLERS = ["hybrid", "gamma_poisson"]
FLOORS = {"inv_head": 0.999, "inv_search": 0.99, "mix_lambda<10": 0.99, "mix_lambda<10_far": 0.9, "domain": 1.0}


def _floors(sampler, res, extra=None):
    floors = dict(FLOORS, **(extra or {}))
    for k, name in enumerate(cr.PATH_NAMES):
        sel = res["path"] == k
        if name in floors and sel.sum() >= 100:
            frac = (res["lo"][sel] == res["hi"][sel]).mean()
            assert frac >= floors[name], (sampler, name, frac, int(sel.sum()))


def _gene_table(rng, G, P, lo=-1.0, hi=3.5):
    M = np.exp(rng.uniform(lo, hi, size=(P, G)))
    alpha = np.exp(rng.normal(np.log(0.2), 0.6, size=G))
    bm = np.exp(rng.normal(0.0, 0.6, size=G))
    return M, alpha, bm


@pytest.mark.gpu
@pytest.mark.parametrize("sampler", SAMPLERS)
def test_shapes_groups_and_cells_straddling_2_32(gpu, sampler):
    """G in {1, 3, 5, 127, 128, 129, 1003} (non-vector path, partial strips, twin edge lanes), ldx = G + 5,
    tree rows of 1, 63, 64, 65 and 200 cells in shuffled order, global cells straddling 2^32."""
    rng = np.random.RandomState(5)
    sizes = [1, 63, 64, 65, 200]
    rows = rng.permutation(np.repeat(np.arange(5), sizes))
    for G in (1, 3, 5, 127, 128, 129, 1003):
        M, alpha, bm = _gene_table(rng, G, 5)
        sc = np.exp(rng.normal(0, 0.7, size=rows.size))
        _, res = gpu.check(sampler, M, alpha, bm, rows, sc, seed=11 + G, cell0=(1 << 32) - 150)
        _floors(sampler, res)


@pytest.mark.gpu
@pytest.mark.parametrize("sampler", SAMPLERS)
def test_cells_near_the_2_48_limit_and_fused_stats(gpu, sampler):
    rng = np.random.RandomState(6)
    M, alpha, bm = _gene_table(rng, 128, 3)
    rows = rng.randint(0, 3, size=700)
    sc = np.exp(rng.normal(0, 0.7, size=700))
    gpu.check(sampler, M, alpha, bm, rows, sc, seed=(1 << 63) + 12345, cell0=(1 << 48) - 701)
    # the fused-stats instantiation, replayed like the others (and its summaries equal the counts')
    gpu.check(sampler, M, alpha, bm, rows, sc, seed=77, cell0=3, stats=True)


@pytest.mark.gpu
@pytest.mark.parametrize("sampler", SAMPLERS)
def test_hybrid_routes_head_searches_series_and_far_tail(gpu, sampler):
    """Head-only genes, stage-2 and long searches (mean 30, variance 390), the theta < 0.1 series
    (beta - 1 = 1e-8 and 0.05) and > 2e6 inversion counts, so that ~130 reach the far tail."""
    M = np.array([[0.2, 1.5, 30.0, 28.0, 5.0, 5.0, 9.0, 2.0]], np.float32)
    alpha = np.array([0.5, 0.3, 0.3, 0.35, 0.0, 0.0, 0.1, 1.0], np.float32)
    bm = np.array([0.5, 1.0, 3.0, 1.5, 1e-8, 0.05, 2.0, 1.0], np.float32)
    G = 128
    reps = G // M.shape[1]
    M, alpha, bm = np.tile(M, reps), np.tile(alpha, reps), np.tile(bm, reps)
    n = 17000
    rows = np.zeros(n, np.int64)
    sc = np.ones(n, np.float32)
    X, res = gpu.check(sampler, M, alpha, bm, rows, sc, seed=4242, cell0=10 ** 9)
    _floors(sampler, res)
    if sampler == "hybrid":
        tail = (res["path"] == cr.P_TAIL).sum()
        assert tail >= 80, tail
        assert (res["path"] == cr.P_SEARCH).sum() > 100000


def _s_max_neighbours(gpu, M, alpha, bm):
    """The largest fp32 library size the hook routes to the inversion for (M, alpha, bm), by bisection,
    and its two fp32 neighbours."""
    lo, hi = np.float32(1e-3), np.float32(1e4)
    r = gpu.params(np.array([M, M]), np.array([lo, hi]), np.array([alpha, alpha]), np.array([bm, bm]))["route"]
    assert r[0] == 1 and r[1] == 0
    a, b = lo.view(np.int32), hi.view(np.int32)
    while b - a > 1:
        mids = np.linspace(a, b, 66).astype(np.int32)[1:-1]
        rr = gpu.params(np.full(mids.size, M), mids.view(np.float32), np.full(mids.size, alpha), np.full(mids.size, bm))["route"]
        inv = np.nonzero(rr == 1)[0]
        a = mids[inv[-1]] if inv.size else a
        b = mids[inv[-1] + 1] if inv.size and inv[-1] + 1 < mids.size else mids[0] if not inv.size else b
    s = np.array([a - 1, a, b, b + 1], np.int32).view(np.float32)
    r = gpu.params(np.full(4, M), s, np.full(4, alpha), np.full(4, bm))["route"]
    assert list(r) == [1, 1, 0, 0], r
    return s


@pytest.mark.gpu
@pytest.mark.parametrize("sampler", SAMPLERS)
def test_library_sizes_one_ulp_either_side_of_s_max(gpu, sampler):
    genes = [(10.0, 0.1, 1.0), (3.0, 0.5, 2.0), (1.0, 0.0, 0.05), (20.0, 0.05, 3.0)]
    G = len(genes)
    M = np.array([[g[0] for g in genes]], np.float32)
    alpha = np.array([g[1] for g in genes], np.float32)
    bm = np.array([g[2] for g in genes], np.float32)
    cols = []
    for g in genes:
        cols.append(_s_max_neighbours(gpu, *g))
    # every gene sees its own four library sizes; 2000 cells each
    sc = np.concatenate([np.repeat(c, 500) for c in cols])
    rows = np.zeros(sc.size, np.int64)
    _, res = gpu.check(sampler, M, alpha, bm, rows, sc, seed=8, cell0=123)
    _floors(sampler, res)


@pytest.mark.gpu
@pytest.mark.parametrize("sampler", SAMPLERS)
def test_mixture_regimes_clamp_and_domain(gpu, sampler):
    """r < 1, r >> 1, lambda straddling 10, PTRS rejections (moderate lambda), lambda >= 1.6e7, a clamped
    count (PST_FLAG_CLAMPED); a gene with beta < 1 and alpha = 0 (zero column) and cells whose library size
    is NaN or 0 (zero rows), both with PST_FLAG_DOMAIN."""
    M = np.array([[100.0, 5000.0, 10.0, 60.0, 300.0, 2.0e7, 3.0e9, 4.0]], np.float32)
    alpha = np.array([5.0, 0.001, 3.9, 0.05, 0.2, 1e-4, 1e-12, 0.0], np.float32)
    bm = np.array([1.0, 0.5, 1.0, 0.5, 1.0, 1.0, 0.01, -0.5], np.float32)
    n = 3000
    rows = np.zeros(n, np.int64)
    sc = np.ones(n, np.float32)
    sc[7] = np.nan
    sc[1500] = 0.0
    X, res = gpu.check(sampler, M, alpha, bm, rows, sc, seed=99, cell0=55)
    assert np.all(X[:, 7] == 0) and np.all(X[7] == 0) and np.all(X[1500] == 0)
    assert res["flags"] == cr.FLAG_DOMAIN | cr.FLAG_CLAMPED
    live = np.ones(n, bool)
    live[[7, 1500]] = False
    assert np.all(X[live, 6] == INT_MAX)
    _floors(sampler, res, {"mix_ptrs": 0.8})
    ptrs = res["path"] == cr.P_PTRS
    assert ptrs.sum() > 5000


@pytest.mark.gpu
def test_samplers_agree_count_for_count_on_ptrs_genes(gpu):
    """Genes whose every count takes PTRS draw the same numbers in both kernels (same blocks, same
    arithmetic): equal wherever the replay determines the count."""
    rng = np.random.RandomState(3)
    G = 96
    M = np.exp(rng.uniform(np.log(200), np.log(3000), size=(2, G))).astype(np.float32)
    alpha = np.full(G, 0.05, np.float32)
    bm = np.full(G, 1.0, np.float32)
    rows = rng.randint(0, 2, size=400)
    sc = np.exp(rng.normal(0, 0.3, size=400)).astype(np.float32)
    Xh, rh = gpu.check("hybrid", M, alpha, bm, rows, sc, seed=5, cell0=1 << 40)
    Xg, rg = gpu.check("gamma_poisson", M, alpha, bm, rows, sc, seed=5, cell0=1 << 40)
    ptrs = (rh["path"] == cr.P_PTRS) & (rg["path"] == cr.P_PTRS)
    assert ptrs.mean() > 0.95
    det = ptrs & (rh["lo"] == rh["hi"])
    assert det.mean() > 0.9
    assert np.array_equal(Xh.ravel()[det], Xg.ravel()[det])
