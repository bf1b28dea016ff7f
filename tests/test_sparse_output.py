"""out="csr": the samplers' sparse result (scipy.sparse.csr_matrix) and the kernels behind it
(pst_csr_row_counts, pst_csr_row_offsets, pst_csr_pack).  The counts must equal the dense result of the
same call bit for bit, whatever the chunking, the sharding or the width of the transfer streams."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

pytestmark = pytest.mark.gpu

from prosstt_b200 import _native as nat  # noqa: E402
from prosstt_b200 import device as pdev, sim_utils as sut, simulation as sim, tree as ptree  # noqa: E402
from prosstt_b200 import hostpool, stats as pstats  # noqa: E402
from prosstt_b200.device import CountEngine, TreeTables  # noqa: E402

DEV = "cuda:0"
SAMPLERS = ["gamma_poisson", "hybrid"]


def _random_tree(G, T=12, seed=0, log_mean=0.0):
    """Three branches of T steps with log-normal means (no lineage simulation: any G is cheap)."""
    t = ptree.Tree(topology=[[0, 1], [0, 2]], time={0: T, 1: T, 2: T}, num_branches=3, branch_points=1,
                   modules=2, G=G)
    rng = np.random.RandomState(seed)
    t.add_genes({b: np.exp(rng.normal(log_mean, 1.0, size=(T, G))) for b in t.branches})
    alpha = np.exp(rng.normal(np.log(0.2), np.log(1.5), size=G))
    beta = np.exp(rng.normal(0.0, np.log(1.5), size=G)) + 1
    return t, alpha, beta


def _lineage_tree(bp, T, K, G, seed):
    np.random.seed(seed)
    top = [[int(a), int(b)] for a, b in ptree.Tree.gen_random_topology(bp)]
    t = ptree.Tree(topology=top, time={b: T for b in range(2 * bp + 1)}, num_branches=2 * bp + 1,
                   branch_points=bp, modules=K, G=G)
    rel, W, H = sim.simulate_lineage(t, a=0.05, seed=seed, device=DEV)
    scale = sut.simulate_base_gene_exp(t, rel)
    t.add_genes({b: np.exp(rel[b]) * scale for b in t.branches})
    rng = np.random.RandomState(seed)
    alpha = np.exp(rng.normal(np.log(0.2), np.log(1.5), size=G))
    beta = np.exp(rng.normal(np.log(1.0), np.log(1.5), size=G)) + 1
    return t, alpha, beta


@pytest.fixture(scope="module")
def lineage_tree():
    return _lineage_tree(2, 20, 6, 1000, seed=3)


def _check_csr(m, dense, data_dtype=np.int64, index_dtype=np.int32):
    assert isinstance(m, sp.csr_matrix) and m.shape == dense.shape
    assert m.data.dtype == data_dtype and m.indptr.dtype == index_dtype and m.indices.dtype == index_dtype
    assert m.has_canonical_format and m.has_sorted_indices
    m.check_format(full_check=True)
    assert not np.any(m.data == 0)
    assert np.array_equal(m.toarray(), dense)


def _same_rest(a, b):
    assert np.array_equal(a[1], b[1]) and list(a[2]) == list(b[2]) and np.array_equal(a[3], b[3])


# ------------------------------------------------------------------ equal to the dense result
@pytest.mark.parametrize("sampler", SAMPLERS)
def test_every_sampler_equals_the_dense_result(sampler, lineage_tree):
    t, alpha, beta = lineage_tree
    kw = dict(alpha=alpha, beta=beta, seed=12, device=DEV, sampler=sampler)
    calls = [
        lambda **o: sim.sample_density(t, 1500, **kw, **o),
        lambda **o: sim.sample_whole_tree(t, 7, **kw, **o),
        lambda **o: sim.sample_pseudotime_series(t, [300, 400], [5, 30], 4.0, **kw, **o),
    ]
    for call in calls:
        dense = call()
        for dt in (np.int64, np.int32):
            got = call(out="csr", dtype=dt)
            _check_csr(got[0], dense[0], data_dtype=dt)
            _same_rest(got, dense)
    # draw_counts returns X alone
    X, pt, br, sc = sim.sample_density(t, 800, **kw)
    dkw = dict(seed=4, device=DEV, sampler=sampler)
    dense = sim.draw_counts(t, pt, br, sc, alpha, beta, **dkw)
    for dt in (np.int64, np.int32):
        _check_csr(sim.draw_counts(t, pt, br, sc, alpha, beta, out="csr", dtype=dt, **dkw), dense, data_dtype=dt)


@pytest.mark.parametrize("sampler", SAMPLERS)
def test_restricted_sampler_equals_the_dense_result(sampler):
    results = []
    for out in ("numpy", "csr"):
        np.random.seed(92)                       # default_gene_expression and the NB parameters use it
        results.append(sim.sample_whole_tree_restricted(ptree.Tree(), seed=6, device=DEV, sampler=sampler, out=out))
    dense, got = results
    _check_csr(got[0], dense[0])
    _same_rest(got, dense)


# ------------------------------------------------------------------ shapes
@pytest.mark.parametrize("G", [1, 7, 1003])
def test_ragged_gene_counts(G):
    t, alpha, beta = _random_tree(G, seed=G)
    kw = dict(alpha=alpha, beta=beta, seed=5, device=DEV)
    dense = sim.sample_density(t, 900, **kw)
    got = sim.sample_density(t, 900, out="csr", **kw)
    _check_csr(got[0], dense[0])
    _same_rest(got, dense)


def test_more_than_65536_genes_take_the_int32_column_stream():
    G = 70003
    t, alpha, beta = _random_tree(G, T=4, seed=11)
    kw = dict(alpha=alpha, beta=beta, seed=8, device=DEV)
    dense = sim.sample_density(t, 300, dtype=np.int32, **kw)[0]
    assert dense[:, 65536:].any()                # columns that do not fit uint16 are nonzero somewhere
    _check_csr(sim.sample_density(t, 300, out="csr", dtype=np.int32, **kw)[0], dense, data_dtype=np.int32)


def test_empty_rows_all_zero_result_and_no_cells():
    t, alpha, beta = _random_tree(7, seed=2)
    kw = dict(alpha=alpha, beta=beta, seed=3, device=DEV)
    dense = sim.sample_density(t, 2000, scale_mean=-5.0, **kw)[0]
    got = sim.sample_density(t, 2000, scale_mean=-5.0, out="csr", **kw)[0]
    assert (dense.sum(axis=1) == 0).sum() > 100 and dense.any()       # many empty rows, not all
    _check_csr(got, dense)
    zero = sim.sample_density(t, 500, scale_mean=-40.0, out="csr", **kw)[0]
    assert zero.nnz == 0 and zero.indptr.tolist() == [0] * 501
    _check_csr(zero, np.zeros((500, 7), dtype=np.int64))
    none = sim.sample_density(t, 0, out="csr", **kw)
    assert none[0].shape == (0, 7) and none[0].nnz == 0 and len(none[1]) == 0
    none[0].check_format(full_check=True)
    assert sim.draw_counts(t, [], [], [], alpha, beta, seed=1, device=DEV, out="csr").shape == (0, 7)


# ------------------------------------------------------------------ values above uint16
def test_counts_above_65535_come_back_exactly():
    t, alpha, beta = _random_tree(64, T=6, seed=21, log_mean=9.0)     # means around 8e3, e^9 x e^(N(0,1))
    kw = dict(alpha=alpha, beta=beta, seed=2, device=DEV, scale_mean=1.0)
    dense = sim.sample_density(t, 600, **kw)[0]
    assert (dense >= 65535).sum() > 100 and dense.max() > 100000
    for dt in (np.int64, np.int32):
        _check_csr(sim.sample_density(t, 600, out="csr", dtype=dt, **kw)[0], dense, data_dtype=dt)


# ------------------------------------------------------------------ invariance
def test_chunking_and_ramp_up_do_not_change_the_matrix(lineage_tree, monkeypatch):
    t, alpha, beta = lineage_tree
    kw = dict(alpha=alpha, beta=beta, seed=31, device=DEV)
    whole = sim.sample_density(t, 3001, out="csr", **kw)[0]
    _check_csr(whole, sim.sample_density(t, 3001, **kw)[0])
    # a small staging size: chunks of 200 cells after a ramp-up of 25, 50 and 100
    monkeypatch.setattr(pdev, "_STAGE_BYTES", 4 * t.G * 200)
    small = sim.sample_density(t, 3001, out="csr", **kw)[0]
    assert np.array_equal(small.indptr, whole.indptr) and np.array_equal(small.indices, whole.indices)
    assert np.array_equal(small.data, whole.data)
    # explicit chunk sizes through the engine, one of them a single cell
    dev = torch.device(DEV)
    tb = TreeTables(t, dev)
    eng = CountEngine(t, tb, alpha, beta, dev, sampler="hybrid")
    rng = np.random.RandomState(1)
    rows = nat.to_dev(rng.randint(0, tb.P, size=1000), torch.int32, dev)
    sc = nat.to_dev(np.exp(rng.normal(0, 0.7, size=1000)), torch.float32, dev)
    want = eng.draw(rows, sc, 5, 77).cpu().numpy()
    for chunk in (1, 97, 1000):
        indptr, indices, data = eng.draw_to_csr(rows, sc, 5, 77, chunk_cells=chunk, threads=3)
        m = sim._csr_matrix(indptr, indices, data, want.shape)
        _check_csr(m, want)
    eng.check()


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_shards_stack_to_the_whole(world, lineage_tree):
    t, alpha, beta = lineage_tree
    kw = dict(alpha=alpha, beta=beta, seed=17, device=DEV, out="csr")
    whole = sim.sample_density(t, 1001, **kw)[0]
    parts = [sim.sample_density(t, 1001, shard=(r, world), **kw)[0] for r in range(world)]
    stacked = sp.vstack(parts, format="csr")
    assert stacked.shape == whole.shape
    assert np.array_equal(stacked.indptr, whole.indptr) and np.array_equal(stacked.indices, whole.indices)
    assert np.array_equal(stacked.data, whole.data)


# ------------------------------------------------------------------ int64 indices
def _mem_available_bytes():
    try:
        with open("/proc/meminfo") as fh:
            for line in fh:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


def test_more_than_2_31_nonzeros_use_int64_indices():
    """125 000 cells x 20 000 genes at e^3.5 x library size: ~2.3e9 nonzeros, 28 GB of int64 indices and
    int32 data.  Checked against the same cells drawn on the device without a dense host copy."""
    if _mem_available_bytes() < (80 << 30):
        pytest.skip("needs ~80 GB of available host memory")
    t, alpha, beta = _lineage_tree(7, 50, 10, 20000, seed=1)
    n = 125000
    kw = dict(alpha=alpha, beta=beta, seed=9, device=DEV, scale_mean=3.5, dtype=np.int32)
    m, pt, br, sc = sim.sample_density(t, n, out="csr", **kw)
    assert m.nnz >= (1 << 31)
    assert m.indptr.dtype == np.int64 and m.indices.dtype == np.int64 and m.data.dtype == np.int32
    assert m.shape == (n, 20000) and m.has_canonical_format
    X = sim.sample_density(t, n, out="torch", **kw)[0]
    st = pstats.count_stats(X)
    row_nnz = np.diff(m.indptr)
    assert np.array_equal(row_nnz, 20000 - st["cell_zeros"].cpu().numpy().astype(np.int64))
    nonempty = row_nnz > 0
    totals = np.zeros(n, dtype=np.int64)
    totals[nonempty] = np.add.reduceat(m.data, m.indptr[:-1][nonempty], dtype=np.int64)
    assert np.array_equal(totals, st["cell_total"].cpu().numpy())
    for lo in (0, 61234, n - 300):               # including rows whose offsets are past 2^31
        block = m[lo:lo + 300]
        assert np.array_equal(block.toarray(), X[lo:lo + 300].cpu().numpy())
    del X, st, m, block
    torch.cuda.empty_cache()
    hostpool.release()                           # do not keep 28 GB of recycled result memory for later tests


# ------------------------------------------------------------------ kernels through the raw ABI
def _random_counts(rng, n, G, zero_frac, big_frac=0.0):
    X = (rng.negative_binomial(0.7, 0.05, size=(n, G)) + 1).astype(np.int32)
    X[rng.random_sample((n, G)) < zero_frac] = 0
    big = rng.random_sample((n, G)) < big_frac
    X[big] = rng.randint(65530, 70000, size=int(big.sum()))
    X[n // 2] = 0                                                    # an empty row
    return X


def test_row_counts_and_offsets_match_numpy():
    dev = torch.device(DEV)
    st = nat.stream_ptr(dev)
    rng = np.random.RandomState(4)
    for n, G, zf, bf in ((500, 403, 0.5, 0.01), (129, 2048, 0.9, 0.0), (64, 128, 0.0, 0.2), (5, 7, 1.0, 0.0),
                         (20000, 12, 0.7, 0.001)):
        Xh = _random_counts(rng, n, G, zf, bf)
        X = torch.from_numpy(Xh).to(dev)
        row_nnz = torch.full((n,), -1, dtype=torch.int32, device=dev)
        sat = torch.full((1,), 3, dtype=torch.int64, device=dev)      # added to
        nat.call("pst_csr_row_counts", X.data_ptr(), n, G, G, row_nnz, sat, st)
        assert np.array_equal(row_nnz.cpu().numpy(), (Xh != 0).sum(axis=1)), (n, G)
        assert int(sat.item()) == 3 + int((Xh >= 65535).sum()), (n, G)
        indptr = torch.full((n + 1,), -1, dtype=torch.int64, device=dev)
        nat.call("pst_csr_row_offsets", row_nnz, n, indptr, st)
        want = np.concatenate([[0], np.cumsum((Xh != 0).sum(axis=1))])
        assert np.array_equal(indptr.cpu().numpy(), want), (n, G)
    # padded row stride
    Xh = _random_counts(rng, 40, 24, 0.5, 0.05)
    X = torch.from_numpy(Xh).to(dev)
    row_nnz = torch.empty(40, dtype=torch.int32, device=dev)
    sat = torch.zeros(1, dtype=torch.int64, device=dev)
    nat.call("pst_csr_row_counts", X.data_ptr(), 40, 21, 24, row_nnz, sat, st)
    assert np.array_equal(row_nnz.cpu().numpy(), (Xh[:, :21] != 0).sum(axis=1))
    assert int(sat.item()) == int((Xh[:, :21] >= 65535).sum())


@pytest.mark.parametrize("index_bits", [16, 32])
@pytest.mark.parametrize("data_bits", [16, 32])
def test_pack_matches_scipy(index_bits, data_bits):
    dev = torch.device(DEV)
    st = nat.stream_ptr(dev)
    rng = np.random.RandomState(index_bits + data_bits)
    it = {16: torch.uint16, 32: torch.int32}
    for n, G, zf, bf in ((500, 403, 0.5, 0.01), (129, 2048, 0.9, 0.0), (64, 128, 0.0, 0.2), (33, 7, 0.3, 0.05)):
        Xh = _random_counts(rng, n, G, zf, bf)
        want = sp.csr_matrix(Xh)
        want.sort_indices()
        X = torch.from_numpy(Xh).to(dev)
        indptr = torch.from_numpy(want.indptr.astype(np.int64)).to(dev)
        n_sat = int((Xh >= 65535).sum())
        # rows [lo, hi) into a window that starts at their first nonzero
        lo, hi = n // 3, n
        p0, p1 = int(want.indptr[lo]), int(want.indptr[hi])
        idx = torch.zeros(max(1, p1 - p0) + 8, dtype=it[index_bits], device=dev)
        val = torch.zeros(max(1, p1 - p0) + 8, dtype=it[data_bits], device=dev)
        ovf_pos = torch.full((max(1, n_sat),), -1, dtype=torch.int64, device=dev)
        ovf_val = torch.zeros(max(1, n_sat), dtype=torch.int32, device=dev)
        ovf_count = torch.zeros(1, dtype=torch.int64, device=dev)
        flags = torch.zeros(1, dtype=torch.int32, device=dev)
        nat.call("pst_csr_pack", X[lo:].data_ptr(), hi - lo, G, G, indptr[lo:], p0, idx.data_ptr(), index_bits,
                 val.data_ptr(), data_bits, ovf_pos, ovf_val, n_sat, ovf_count, flags, st)
        assert int(flags.item()) == 0
        m = p1 - p0
        got_idx = idx[:m].to(torch.int64).cpu().numpy() if index_bits == 32 else idx[:m].cpu().numpy().astype(np.int64)
        assert np.array_equal(got_idx, want.indices[p0:p1]), (n, G)
        assert not idx[m:].to(torch.int32).any() and not val[m:].to(torch.int32).any()   # nothing past the window
        vals = val[:m].cpu().numpy().astype(np.int64)
        exact = want.data[p0:p1].astype(np.int64)
        if data_bits == 32:
            assert np.array_equal(vals, exact) and int(ovf_count.item()) == 0
        else:
            assert np.array_equal(vals, np.minimum(exact, 65535))
            listed = int(ovf_count.item())
            assert listed == int((exact >= 65535).sum())
            pos = ovf_pos[:listed].cpu().numpy()
            order = np.argsort(pos)
            assert np.array_equal(pos[order], p0 + np.flatnonzero(exact >= 65535))
            assert np.array_equal(ovf_val[:listed].cpu().numpy()[order], exact[exact >= 65535])


def test_pack_reports_a_stale_row_pointer_and_writes_nothing():
    dev = torch.device(DEV)
    rng = np.random.RandomState(10)
    Xh = rng.poisson(0.5, size=(40, 24)).astype(np.int32)
    X = torch.from_numpy(Xh).to(dev)
    bad = torch.zeros(41, dtype=torch.int64, device=dev)             # every row "empty"
    flags = torch.zeros(1, dtype=torch.int32, device=dev)
    idx = torch.zeros(8, dtype=torch.uint16, device=dev)
    val = torch.zeros(8, dtype=torch.uint16, device=dev)
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    nat.call("pst_csr_pack", X.data_ptr(), 40, 24, 24, bad, 0, idx.data_ptr(), 16, val.data_ptr(), 16, None, None, 0,
             cnt, flags, nat.stream_ptr(dev))
    assert int(flags.item()) & nat.FLAG_ROW
    assert not idx.to(torch.int32).any() and not val.to(torch.int32).any()
    with pytest.raises(ValueError):                                  # 16-bit columns need G <= 65536
        nat.call("pst_csr_pack", X.data_ptr(), 1, 70000, 70000, bad, 0, idx.data_ptr(), 16, val.data_ptr(), 32,
                 None, None, 0, None, flags, nat.stream_ptr(dev))


# ------------------------------------------------------------------ errors
def test_errors_are_those_of_the_dense_path(lineage_tree):
    flat = ptree.Tree(topology=[], time={0: 1}, num_branches=1, branch_points=0, modules=1, G=4)
    flat.add_genes({0: np.array([[1.0, 2.0, 0.0, 3.0]])})
    with pytest.raises(ValueError):                                  # mu == 0: domain error
        sim.draw_counts(flat, [0], [0], [1.0], 0.2, 2.0, seed=1, device=DEV, out="csr")
    flat.add_genes({0: np.array([[1.0, 2.0, 1.0, 3.0]])})
    flat.invalidate_device_cache()
    with pytest.raises(IndexError):                                  # pseudotime outside the branch
        sim.draw_counts(flat, [5], [0], [1.0], 0.2, 2.0, seed=1, device=DEV, out="csr")
    t, alpha, beta = lineage_tree
    with pytest.raises(IndexError):                                  # pseudotime outside the tree
        sim._sample_data_at_times(t, [0, 10 ** 6], alpha=alpha, beta=beta, seed=1, device=DEV, out="csr")
    n = 50
    host = (torch.empty((n, t.G), dtype=torch.int32), torch.empty(n, dtype=torch.int64),
            torch.empty(n, dtype=torch.int32), torch.empty(n, dtype=torch.float64))
    with pytest.raises(ValueError):
        sim.sample_density(t, n, alpha, beta, seed=1, device=DEV, out="csr", host_out=host)
    for dt in (np.int16, np.uint16, np.float64):
        with pytest.raises(ValueError):
            sim.sample_density(t, n, alpha, beta, seed=1, device=DEV, out="csr", dtype=dt)
        with pytest.raises(ValueError):
            sim.draw_counts(t, [0], [t.branches[0]], [1.0], alpha, beta, seed=1, device=DEV, out="csr", dtype=dt)
