"""out="csr", path=...: CSR streamed to a shard directory chunk by chunk (CountEngine.stream_csr into
formats.CsrShardWriter).  The shard must hold the in-memory out="csr" result bit for bit, whatever the chunking,
and the stream must draw every chunk once and keep host memory bounded by the chunk, not by the matrix.
The writer and the format are checked without a GPU."""
import os
import shutil
import zipfile

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from prosstt_b200 import _native as nat
from prosstt_b200 import device as pdev, formats, sim_utils as sut, simulation as sim, tree as ptree
from prosstt_b200.device import CountEngine, TreeTables

DEV = "cuda:0"
SAMPLERS = ["gamma_poisson", "hybrid"]
gpu = pytest.mark.gpu


# ------------------------------------------------------------------ the writer and the format (no GPU)
def _cells(n, seed=0):
    rng = np.random.RandomState(seed)
    return rng.randint(0, 50, size=n), np.array(["b%d" % v for v in rng.randint(0, 3, size=n)]), rng.rand(n)


def _write(path, m, chunks, dtype=np.int64, cells=None):
    """Write the scipy matrix m as a shard, in the given row chunks."""
    n = m.shape[0]
    with formats.CsrShardWriter(path, m.shape, *(cells or _cells(n)), dtype=dtype) as w:
        for lo, hi in chunks:
            part = m[lo:hi]
            w.append(part.indptr.astype(np.int64), part.indices, part.data)
    return w


def _random_csr(n, G, density, seed):
    m = sp.random(n, G, density=density, format="csr", random_state=seed,
                  data_rvs=lambda k: np.random.RandomState(seed).randint(1, 100000, size=k)).astype(np.int64)
    m.sort_indices()
    return m


@pytest.mark.parametrize("dtype", [np.int64, np.int32])
def test_writer_round_trip(tmp_path, dtype):
    m = _random_csr(301, 57, 0.2, 1)
    m[40:90] = 0                                               # empty rows, and an empty chunk below
    m.eliminate_zeros()
    cells = _cells(301, 2)
    path = str(tmp_path / "x.csr")
    _write(path, m, [(0, 7), (7, 50), (50, 80), (80, 80), (80, 301)], dtype=dtype, cells=cells)
    assert not os.path.exists(path + ".partial")
    X, pt, br, sc = formats.load_csr_shard(path)
    for name in ("indptr", "indices", "data"):                 # views of the files: no copy
        a = getattr(X, name)
        assert isinstance(a, np.memmap) and not a.flags.writeable
        assert os.path.samefile(a.filename, os.path.join(path, name + ".npy"))
    assert X.shape == m.shape and X.has_canonical_format and X.has_sorted_indices
    X.check_format(full_check=True)
    assert X.indptr.dtype == np.int32 and X.indices.dtype == np.int32 and X.data.dtype == dtype
    assert np.array_equal(X.indptr, m.indptr) and np.array_equal(X.indices, m.indices)
    assert np.array_equal(X.data, m.data)
    assert np.array_equal(pt, cells[0]) and pt.dtype == np.int64
    assert list(br) == list(cells[1]) and np.array_equal(sc, cells[2]) and sc.dtype == np.float64
    for name in ("format", "shape", "indptr", "indices", "data", "pseudotime", "branches", "scalings"):
        np.load(os.path.join(path, name + ".npy"), mmap_mode="r", allow_pickle=False)


def test_zipped_members_load_with_scipy(tmp_path):
    m = _random_csr(120, 33, 0.3, 5)
    path = str(tmp_path / "x.csr")
    _write(path, m, [(0, 60), (60, 120)])
    npz = str(tmp_path / "x.npz")
    with zipfile.ZipFile(npz, "w", compression=zipfile.ZIP_STORED) as z:
        for name in ("format", "shape", "indptr", "indices", "data", "pseudotime", "branches", "scalings"):
            z.write(os.path.join(path, name + ".npy"), name + ".npy")
    got = sp.load_npz(npz)
    X = formats.load_csr_shard(path)[0]
    assert got.format == "csr" and got.shape == X.shape
    assert np.array_equal(got.indptr, X.indptr) and np.array_equal(got.indices, X.indices)
    assert np.array_equal(got.data, X.data)


def test_all_zero_and_empty_shards(tmp_path):
    z = sp.csr_matrix((9, 4), dtype=np.int64)
    _write(str(tmp_path / "z"), z, [(0, 4), (4, 9)])
    X = formats.load_csr_shard(str(tmp_path / "z"))[0]
    assert X.nnz == 0 and X.indptr.tolist() == [0] * 10 and len(X.indices) == 0 and len(X.data) == 0
    X.check_format(full_check=True)
    e = sp.csr_matrix((0, 4), dtype=np.int64)
    _write(str(tmp_path / "e"), e, [])
    X, pt, br, sc = formats.load_csr_shard(str(tmp_path / "e"))
    assert X.shape == (0, 4) and X.indptr.tolist() == [0] and len(pt) == len(br) == len(sc) == 0


def test_index_dtype_switches_at_2_31(tmp_path):
    for n, G, want in ((1, (1 << 31) - 1, np.int32), (2, 1 << 30, np.int64), (3, 1 << 31, np.int64)):
        path = str(tmp_path / ("s%d" % n))
        with formats.CsrShardWriter(path, (n, G), *_cells(n)) as w:
            assert w.index_dtype == want
            w.append(np.array([0] + [2] * n), np.array([5, G - 1]), np.array([3, 4]))
        X = formats.load_csr_shard(path)[0]
        assert X.indptr.dtype == want and X.indices.dtype == want and X.shape == (n, G)
        X.check_format(full_check=True)
        assert X.indices.tolist() == [5, G - 1] and X.data.tolist() == [3, 4]


def test_failed_writes_leave_nothing(tmp_path):
    m = _random_csr(20, 5, 0.5, 3)
    short = str(tmp_path / "short")
    with pytest.raises(ValueError):
        _write(short, m, [(0, 10)])                            # 10 of 20 rows
    inside = str(tmp_path / "inside")
    with pytest.raises(KeyError):
        with formats.CsrShardWriter(inside, m.shape, *_cells(20)) as w:
            w.append(m[:10].indptr, m[:10].indices, m[:10].data)
            raise KeyError("stop")
    for p in (short, inside):
        assert not os.path.exists(p) and not os.path.exists(p + ".partial")
    done = str(tmp_path / "done")
    _write(done, m, [(0, 20)])
    with pytest.raises(FileExistsError):
        formats.CsrShardWriter(done, m.shape, *_cells(20))
    with pytest.raises(ValueError):                             # data dtype
        formats.CsrShardWriter(str(tmp_path / "f"), m.shape, *_cells(20), dtype=np.float64)
    with pytest.raises(ValueError):                             # one annotation per cell
        formats.CsrShardWriter(str(tmp_path / "g"), m.shape, *_cells(19))
    assert sorted(os.listdir(tmp_path)) == ["done"]


def test_shard_path_suffix():
    assert formats.shard_path("s", 0, 1) == "s.npy" and formats.shard_path("s", 3, 8) == "s.rank3of8.npy"
    assert formats.shard_path("s", 0, 1, suffix=".csr") == "s.csr"
    assert formats.shard_path("s", 1, 3, suffix=".csr") == "s.rank1of3.csr"


# ------------------------------------------------------------------ trees (as in test_sparse_output.py)
def _random_tree(G, T=12, seed=0, log_mean=0.0):
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


def _same_matrix(got, want, data_dtype=np.int64):
    """got: a streamed shard's matrix; want: the in-memory out="csr" matrix of the same call."""
    n, G = want.shape
    idx = np.int32 if n * G < (1 << 31) else np.int64
    assert isinstance(got, sp.csr_matrix) and got.shape == want.shape
    assert got.indptr.dtype == idx and got.indices.dtype == idx and got.data.dtype == data_dtype
    assert got.has_canonical_format and got.has_sorted_indices
    got.check_format(full_check=True)
    assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)
    assert np.array_equal(got.data, want.data)


def _same_call(got, want, path, data_dtype=np.int64):
    """A sampler's (X, pseudotime, branches, scalings) with path= against the in-memory call, for the returned
    matrix and for a fresh load of the shard."""
    for res in (got, formats.load_csr_shard(path)):
        _same_matrix(res[0], want[0], data_dtype)
        assert np.array_equal(res[1], want[1]) and list(res[2]) == list(want[2]) and np.array_equal(res[3], want[3])


def _shard_bytes(path):
    return {f: open(os.path.join(path, f), "rb").read() for f in sorted(os.listdir(path))}


# ------------------------------------------------------------------ equal to the in-memory result
@gpu
@pytest.mark.parametrize("sampler", SAMPLERS)
def test_every_sampler_writes_the_in_memory_result(sampler, lineage_tree, tmp_path):
    t, alpha, beta = lineage_tree
    kw = dict(alpha=alpha, beta=beta, seed=12, device=DEV, sampler=sampler, out="csr")
    calls = [
        lambda **o: sim.sample_density(t, 1500, **kw, **o),
        lambda **o: sim.sample_whole_tree(t, 7, **kw, **o),
        lambda **o: sim.sample_pseudotime_series(t, [300, 400], [5, 30], 4.0, **kw, **o),
    ]
    for c, call in enumerate(calls):
        for dt in (np.int64, np.int32):
            path = str(tmp_path / ("c%d_%s" % (c, np.dtype(dt).name)))
            _same_call(call(dtype=dt, path=path), call(dtype=dt), path, dt)
    X, pt, br, sc = sim.sample_density(t, 800, alpha=alpha, beta=beta, seed=3, device=DEV)
    dkw = dict(seed=4, device=DEV, sampler=sampler, out="csr")
    for dt in (np.int64, np.int32):
        path = str(tmp_path / ("d_%s" % np.dtype(dt).name))
        got = sim.draw_counts(t, pt, br, sc, alpha, beta, dtype=dt, path=path, **dkw)
        want = sim.draw_counts(t, pt, br, sc, alpha, beta, dtype=dt, **dkw)
        _same_call((got, pt, br, sc), (want, pt, br, sc), path, dt)


@gpu
@pytest.mark.parametrize("sampler", SAMPLERS)
def test_restricted_sampler_writes_the_in_memory_result(sampler, tmp_path):
    results = []
    for path in (str(tmp_path / "r"), None):
        np.random.seed(92)                       # default_gene_expression and the NB parameters use it
        results.append(sim.sample_whole_tree_restricted(ptree.Tree(), seed=6, device=DEV, sampler=sampler,
                                                        out="csr", path=path))
    _same_call(results[0], results[1], str(tmp_path / "r"))


# ------------------------------------------------------------------ shapes
@gpu
@pytest.mark.parametrize("G", [1, 7, 1003, 70003])
def test_gene_counts(G, tmp_path):
    t, alpha, beta = _random_tree(G, T=4 if G > 65536 else 12, seed=G)
    n = 300 if G > 65536 else 900
    kw = dict(alpha=alpha, beta=beta, seed=5, device=DEV, out="csr")
    path = str(tmp_path / "g")
    got = sim.sample_density(t, n, path=path, **kw)
    want = sim.sample_density(t, n, **kw)
    if G > 65536:
        assert want[0].indices.max() >= 65536                  # columns beyond uint16 are present
    _same_call(got, want, path)


@gpu
def test_empty_rows_all_zero_result_and_no_cells(tmp_path):
    t, alpha, beta = _random_tree(7, seed=2)
    kw = dict(alpha=alpha, beta=beta, seed=3, device=DEV, out="csr")
    p = str(tmp_path / "sparse")
    got = sim.sample_density(t, 2000, scale_mean=-5.0, path=p, **kw)
    want = sim.sample_density(t, 2000, scale_mean=-5.0, **kw)
    assert (np.diff(want[0].indptr) == 0).sum() > 100 and want[0].nnz > 0
    _same_call(got, want, p)
    p = str(tmp_path / "zero")
    zero = sim.sample_density(t, 500, scale_mean=-40.0, path=p, **kw)
    assert zero[0].nnz == 0 and zero[0].indptr.tolist() == [0] * 501
    _same_call(zero, sim.sample_density(t, 500, scale_mean=-40.0, **kw), p)
    for name in ("indices", "data"):
        assert np.load(os.path.join(p, name + ".npy"), mmap_mode="r").shape == (0,)
    p = str(tmp_path / "none")
    none = sim.sample_density(t, 0, path=p, **kw)
    assert none[0].shape == (0, 7) and none[0].nnz == 0 and len(none[1]) == 0
    none[0].check_format(full_check=True)
    assert sim.draw_counts(t, [], [], [], alpha, beta, seed=1, device=DEV, out="csr",
                           path=str(tmp_path / "none2")).shape == (0, 7)


# ------------------------------------------------------------------ values above uint16
def _engine(t, alpha, beta, n, seed=1):
    dev = torch.device(DEV)
    tb = TreeTables(t, dev)
    eng = CountEngine(t, tb, alpha, beta, dev, sampler="hybrid")
    rng = np.random.RandomState(seed)
    rows = nat.to_dev(rng.randint(0, tb.P, size=n), torch.int32, dev)
    sc = nat.to_dev(np.exp(rng.normal(0, 0.7, size=n)), torch.float32, dev)
    return eng, rows, sc


def _stream(eng, rows, sc, seed, cell0, **kw):
    """stream_csr's chunks joined into one matrix, with the chunk bounds."""
    parts, bounds = [], []

    def consume(lo, hi, indptr, indices, data):
        assert indptr[0] == 0 and len(indptr) == hi - lo + 1
        bounds.append((lo, hi))
        parts.append((indptr.copy(), indices.copy(), data.copy()))

    nnz = eng.stream_csr(rows, sc, seed, cell0, consume, **kw)
    n = int(rows.numel())
    assert bounds == sorted(bounds) and (not bounds or (bounds[0][0] == 0 and bounds[-1][1] == n))
    assert all(a[1] == b[0] for a, b in zip(bounds, bounds[1:]))
    offsets = np.cumsum([0] + [p[0][-1] for p in parts])
    indptr = np.concatenate([[0]] + [p[0][1:] + o for p, o in zip(parts, offsets)])
    indices = np.concatenate([p[1] for p in parts]) if parts else np.zeros(0, np.int64)
    data = np.concatenate([p[2] for p in parts]) if parts else np.zeros(0, np.int64)
    assert nnz == len(data)
    return indptr, indices, data, bounds


@gpu
def test_counts_above_65535_come_back_exactly(tmp_path):
    t, alpha, beta = _random_tree(64, T=6, seed=21, log_mean=9.0)     # means around 8e3, e^9 x e^(N(0,1))
    kw = dict(alpha=alpha, beta=beta, seed=2, device=DEV, scale_mean=1.0, out="csr")
    for dt in (np.int64, np.int32):
        want = sim.sample_density(t, 600, dtype=dt, **kw)
        assert (want[0].data >= 65535).sum() > 100 and want[0].data.max() > 100000
        path = str(tmp_path / np.dtype(dt).name)
        _same_call(sim.sample_density(t, 600, dtype=dt, path=path, **kw), want, path, dt)
    # a per-chunk overflow list far too small: every chunk is packed again from its work buffer
    eng, rows, sc = _engine(t, alpha, beta, 600)
    want = eng.draw_to_csr(rows, sc, 7, 11, chunk_cells=64)
    assert (want[2] >= 65535).sum() > 100
    for cap in (1, 3, None):
        indptr, indices, data, _ = _stream(eng, rows, sc, 7, 11, chunk_cells=64, overflow_cap=cap)
        assert np.array_equal(indptr, want[0]) and np.array_equal(indices, want[1])
        assert np.array_equal(data, want[2])
    eng.check()


# ------------------------------------------------------------------ chunking
@gpu
def test_chunking_gives_identical_files(lineage_tree, tmp_path, monkeypatch):
    t, alpha, beta = lineage_tree
    n = 1000
    eng, rows, sc = _engine(t, alpha, beta, n)
    want = eng.draw(rows, sc, 5, 77).cpu().numpy()
    cells = _cells(n)
    files = []
    for chunk in (1, 97, n, 5 * n):
        path = str(tmp_path / ("c%d" % chunk))
        with formats.CsrShardWriter(path, (n, t.G), *cells) as w:
            eng.stream_csr(rows, sc, 5, 77, lambda lo, hi, *a: w.append(*a), w.index_dtype, np.int64,
                           chunk_cells=chunk, threads=3)
        X = formats.load_csr_shard(path)[0]
        assert np.array_equal(X.toarray(), want)
        files.append(_shard_bytes(path))
    assert all(f == files[0] for f in files[1:])
    eng.check()
    # the samplers' own chunk plan, and a small staging size: chunks of 200 cells after a ramp of 25, 50, 100
    kw = dict(alpha=alpha, beta=beta, seed=31, device=DEV, out="csr")
    sim.sample_density(t, 3001, path=str(tmp_path / "big"), **kw)
    monkeypatch.setattr(pdev, "_STAGE_BYTES", 4 * t.G * 200)
    sim.sample_density(t, 3001, path=str(tmp_path / "small"), **kw)
    assert _shard_bytes(str(tmp_path / "big")) == _shard_bytes(str(tmp_path / "small"))
    _same_matrix(formats.load_csr_shard(str(tmp_path / "small"))[0], sim.sample_density(t, 3001, **kw)[0])


@gpu
def test_one_draw_per_chunk(lineage_tree, monkeypatch):
    t, alpha, beta = lineage_tree
    n, chunk = 1000, 97
    eng, rows, sc = _engine(t, alpha, beta, n)
    calls = []
    real = CountEngine.draw

    def spy(self, *a, **k):
        calls.append(1)
        return real(self, *a, **k)

    monkeypatch.setattr(CountEngine, "draw", spy)
    planned = len(pdev._plan_chunks(n, chunk, 4 * t.G, pdev._STAGE_BYTES)[1])
    assert planned == 11
    got = _stream(eng, rows, sc, 5, 0, chunk_cells=chunk)
    assert len(calls) == planned and len(got[3]) == planned
    del calls[:]
    want = eng.draw_to_csr(rows, sc, 5, 0, chunk_cells=chunk)
    assert len(calls) == 2 * planned
    assert all(np.array_equal(a, b) for a, b in zip(got[:3], want))


# ------------------------------------------------------------------ shards
@gpu
@pytest.mark.parametrize("world", [2, 3])
def test_rank_shards_stack_to_the_whole(world, lineage_tree, tmp_path):
    t, alpha, beta = lineage_tree
    kw = dict(alpha=alpha, beta=beta, seed=17, device=DEV, out="csr")
    whole = sim.sample_density(t, 1001, **kw)[0]
    stem = str(tmp_path / "sim")
    paths = [formats.shard_path(stem, r, world, suffix=".csr") for r in range(world)]
    for r, p in enumerate(paths):
        sim.sample_density(t, 1001, shard=(r, world), path=p, **kw)
    assert sorted(os.listdir(tmp_path)) == sorted(os.path.basename(p) for p in paths)
    stacked = sp.vstack([formats.load_csr_shard(p)[0] for p in paths], format="csr")
    assert stacked.shape == whole.shape
    assert np.array_equal(stacked.indptr, whole.indptr) and np.array_equal(stacked.indices, whole.indices)
    assert np.array_equal(stacked.data, whole.data)


# ------------------------------------------------------------------ errors
@gpu
def test_errors(lineage_tree, tmp_path):
    flat = ptree.Tree(topology=[], time={0: 1}, num_branches=1, branch_points=0, modules=1, G=4)
    flat.add_genes({0: np.array([[1.0, 2.0, 0.0, 3.0]])})
    p = str(tmp_path / "domain")
    with pytest.raises(ValueError):                                  # mu == 0: domain error
        sim.draw_counts(flat, [0] * 5, [0] * 5, [1.0] * 5, 0.2, 2.0, seed=1, device=DEV, out="csr", path=p)
    assert not os.path.exists(p) and not os.path.exists(p + ".partial")
    # a domain error in a later chunk of a long stream
    t, alpha, beta = _random_tree(16, seed=4)
    means = {b: np.array(t.means[b]) for b in t.branches}
    for b in t.branches:                                             # the last step of every branch
        means[b][-1, 3] = 0.0
    t.add_genes(means)
    t.invalidate_device_cache()
    eng, rows, sc = _engine(t, alpha, beta, 5000)
    rows = torch.full((5000,), 5, dtype=torch.int32, device=DEV)
    rows[4000:] = TreeTables(t, torch.device(DEV)).P - 1
    with pytest.raises(ValueError):
        _stream(eng, rows, sc, 1, 0, chunk_cells=100)
    eng.flags.zero_()
    flat.add_genes({0: np.array([[1.0, 2.0, 1.0, 3.0]])})
    flat.invalidate_device_cache()
    p = str(tmp_path / "branch")
    with pytest.raises(IndexError):                                  # pseudotime outside the branch
        sim.draw_counts(flat, [5], [0], [1.0], 0.2, 2.0, seed=1, device=DEV, out="csr", path=p)
    assert not os.path.exists(p) and not os.path.exists(p + ".partial")
    t, alpha, beta = lineage_tree
    p = str(tmp_path / "tree")
    with pytest.raises(IndexError):                                  # pseudotime outside the tree
        sim._sample_data_at_times(t, [0, 10 ** 6], alpha=alpha, beta=beta, seed=1, device=DEV, out="csr", path=p)
    assert not os.path.exists(p) and not os.path.exists(p + ".partial")
    n = 50
    p = str(tmp_path / "bad")
    host = (torch.empty((n, t.G), dtype=torch.int32), torch.empty(n, dtype=torch.int64),
            torch.empty(n, dtype=torch.int32), torch.empty(n, dtype=torch.float64))
    with pytest.raises(ValueError):
        sim.sample_density(t, n, alpha, beta, seed=1, device=DEV, path=p)
    with pytest.raises(ValueError):
        sim.draw_counts(t, [0], [t.branches[0]], [1.0], alpha, beta, seed=1, device=DEV, path=p)
    with pytest.raises(ValueError):
        sim.sample_density(t, n, alpha, beta, seed=1, device=DEV, out="csr", path=p, host_out=host)
    with pytest.raises(ValueError):
        sim.sample_density(t, n, alpha, beta, seed=1, device=DEV, out="csr", path=p, dtype=np.int16)
    assert not os.path.exists(p)
    p = str(tmp_path / "twice")
    sim.sample_density(t, n, alpha, beta, seed=1, device=DEV, out="csr", path=p)
    with pytest.raises(FileExistsError):
        sim.sample_density(t, n, alpha, beta, seed=1, device=DEV, out="csr", path=p)


# ------------------------------------------------------------------ bounded host memory
def _vm(key):
    with open("/proc/self/status") as fh:
        for line in fh:
            if line.startswith(key + ":"):
                return int(line.split()[1]) * 1024
    return None


def _reset_hwm():
    try:
        with open("/proc/self/clear_refs", "w") as fh:
            fh.write("5")
        return True
    except OSError:
        return False


@gpu
def test_host_memory_is_bounded_by_the_chunk(tmp_path):
    """~400 000 cells x 4000 genes: about 9e8 nonzeros, some 14 GB of int64 indices and data on disk."""
    if shutil.disk_usage(str(tmp_path)).free < (40 << 30):
        pytest.skip("needs ~40 GB of free space in the temporary directory")
    if not _reset_hwm() or _vm("VmHWM") is None:
        pytest.skip("the peak-RSS mark cannot be reset here")
    t, alpha, beta = _random_tree(4000, seed=8)
    kw = dict(alpha=alpha, beta=beta, seed=9, device=DEV, out="csr")
    sim.sample_density(t, 1000, path=str(tmp_path / "warm"), **kw)   # pinned staging, modules
    shutil.rmtree(str(tmp_path / "warm"))
    path = str(tmp_path / "big")
    _reset_hwm()
    base = _vm("VmRSS")
    X = sim.sample_density(t, 400000, path=path, **kw)[0]
    peak = _vm("VmHWM") - base
    written = sum(os.path.getsize(os.path.join(path, f)) for f in os.listdir(path))
    assert X.nnz > 5e8 and written > 8e9
    assert peak < 0.25 * written, (peak, written)
    del X
    shutil.rmtree(path)
