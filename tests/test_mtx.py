"""out="mtx", path=...: a 10x directory (gzipped Matrix Market genes x cells, features, barcodes, cell parameters)
formatted and compressed on the GPU chunk by chunk (pst_mtx_row_bytes, pst_mtx_format, pst_deflate_blocks) and
assembled by formats.MtxWriter.  scipy.io.mmread must read back the out="csr" result of the same call, whatever the
chunking.  The writer and the format are checked without a GPU, by feeding it zlib-made sync-flushed blocks."""
import gzip
import os
import shutil
import subprocess
import zlib

import numpy as np
import pytest
import scipy.io
import scipy.sparse as sp
import torch

from prosstt_b200 import _native as nat
from prosstt_b200 import device as pdev, formats, simulation as sim, tree_utils
from prosstt_b200.device import CountEngine, TreeTables
from test_csr_stream import _cells, _engine, _lineage_tree, _random_csr, _random_tree

DEV = "cuda:0"
SAMPLERS = ["gamma_poisson", "hybrid"]
FILES = ["barcodes.tsv.gz", "cellparams.tsv.gz", "features.tsv.gz", "matrix.mtx.gz"]
gpu = pytest.mark.gpu


# ------------------------------------------------------------------ the writer and the format (no GPU)
def _lines(m, col0=0):
    """The Matrix Market lines of the cells x genes csr matrix m, cell number col0 + row + 1."""
    out = []
    for i in range(m.shape[0]):
        for p in range(m.indptr[i], m.indptr[i + 1]):
            out.append("%d %d %d\n" % (m.indices[p] + 1, col0 + i + 1, m.data[p]))
    return "".join(out).encode("ascii")


def _text(m):
    """The whole decompressed matrix.mtx.gz of m: the 128-byte header, then the lines."""
    size = "%d %d %d\n" % (m.shape[1], m.shape[0], m.nnz)
    banner = "%%MatrixMarket matrix coordinate integer general\n"
    pad = 128 - len(banner) - len(size) - 2
    return (banner + "%" + " " * pad + "\n" + size).encode("ascii") + _lines(m)


def _huffman_sync(raw):
    """(bytes, crc, len): raw as zlib Huffman-only blocks ended by a sync flush, the form of pst_deflate_blocks."""
    c = zlib.compressobj(6, zlib.DEFLATED, -15, 9, zlib.Z_HUFFMAN_ONLY)
    return c.compress(raw) + c.flush(zlib.Z_SYNC_FLUSH), zlib.crc32(raw), len(raw)


def _write(path, m, chunks, cells=None, first=0):
    n = m.shape[0]
    with formats.MtxWriter(path, m.shape, *(cells or _cells(n)), first=first) as w:
        for lo, hi in chunks:
            part = m[lo:hi]
            w.append(hi - lo, part.nnz, *_huffman_sync(_lines(part, lo)))
    return w


def _gunzip(path):
    return gzip.decompress(open(path, "rb").read())


def _check_dir(path, m, cells, first=0):
    n, G = m.shape
    assert sorted(os.listdir(path)) == FILES
    for f in FILES:
        head = open(os.path.join(path, f), "rb").read(10)
        assert head == b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff", f      # MTIME 0, XFL 0, OS 255
    mat = os.path.join(path, "matrix.mtx.gz")
    assert _gunzip(mat) == _text(m)
    assert scipy.io.mminfo(mat) == (G, n, m.nnz, "coordinate", "integer", "general")
    if n and G:
        got = sp.csr_matrix(scipy.io.mmread(mat, spmatrix=False).T)
        assert got.shape == m.shape and (got != m).nnz == 0
    assert _gunzip(os.path.join(path, "features.tsv.gz")) == "".join(
        "gene_%d\tgene_%d\tGene Expression\n" % (j, j) for j in range(G)).encode()
    assert _gunzip(os.path.join(path, "barcodes.tsv.gz")) == "".join(
        "cell_%d\n" % (first + i) for i in range(n)).encode()
    frame = tree_utils.cell_params_frame(*cells, index=["cell_%d" % (first + i) for i in range(n)])
    assert _gunzip(os.path.join(path, "cellparams.tsv.gz")) == frame.to_csv(sep="\t").encode()
    if shutil.which("gzip"):
        r = subprocess.run(["gzip", "-t"] + [os.path.join(path, f) for f in FILES], capture_output=True)
        assert r.returncode == 0, r.stderr


def test_writer_round_trip(tmp_path):
    m = _random_csr(301, 57, 0.2, 1)
    m[40:90] = 0                                               # empty rows, and an empty chunk below
    m.eliminate_zeros()
    cells = _cells(301, 2)
    path = str(tmp_path / "x")
    w = _write(path, m, [(0, 7), (7, 50), (50, 80), (80, 80), (80, 301)], cells=cells)
    assert sorted(os.listdir(tmp_path)) == ["x"]
    _check_dir(path, m, cells)
    rec = w.record()
    assert isinstance(rec, formats.MtxRecord)
    assert rec.path == path and rec.shape == m.shape and rec.nnz == m.nnz
    assert rec.nbytes == os.path.getsize(os.path.join(path, "matrix.mtx.gz"))
    got = rec.load()
    assert isinstance(got, sp.csr_matrix) and got.dtype == np.int64 and (got != m).nnz == 0


def test_cellparams_match_save_cell_params(tmp_path):
    m = _random_csr(40, 9, 0.3, 4)
    cells = _cells(40, 5)
    path = str(tmp_path / "x")
    _write(path, m, [(0, 40)], cells=cells)
    tree_utils.save_cell_params("job", str(tmp_path), *cells)
    assert _gunzip(os.path.join(path, "cellparams.tsv.gz")) == open(str(tmp_path / "job_cellparams.txt"), "rb").read()


def test_edge_cases(tmp_path):
    z = sp.csr_matrix((9, 4), dtype=np.int64)                  # nnz = 0
    _write(str(tmp_path / "z"), z, [(0, 4), (4, 9)])
    _check_dir(str(tmp_path / "z"), z, _cells(9))
    e = sp.csr_matrix((0, 4), dtype=np.int64)                  # zero cells
    w = _write(str(tmp_path / "e"), e, [])
    _check_dir(str(tmp_path / "e"), e, _cells(0))
    assert w.record().nnz == 0 and w.record().load().shape == (0, 4)
    g1 = _random_csr(50, 1, 0.5, 6)                            # G = 1
    _write(str(tmp_path / "g1"), g1, [(0, 20), (20, 50)])
    _check_dir(str(tmp_path / "g1"), g1, _cells(50))
    m = _random_csr(30, 6, 0.4, 8)                             # the cells of rank k: global barcode names
    first = 10 ** 15
    _write(str(tmp_path / "far"), m, [(0, 30)], first=first)
    _check_dir(str(tmp_path / "far"), m, _cells(30), first=first)


def test_header_fits_the_widest_numbers():
    big = 10 ** 19 - 1
    h = formats.mtx_header((1 << 31) - 1, big, big)
    assert len(h) == formats.MTX_HEADER_BYTES == 128
    assert h.endswith(b"%d %d %d\n" % ((1 << 31) - 1, big, big))
    assert h.splitlines()[1].strip(b" ") == b"%"
    assert formats.mtx_header(1, 0, 0).splitlines()[2] == b"1 0 0"


def test_chunking_and_repeats_give_identical_files(tmp_path):
    m = _random_csr(200, 40, 0.3, 7)
    cells = _cells(200, 1)
    files = []
    for i, chunks in enumerate(([(0, 200)], [(0, 200)], [(0, 1), (1, 100), (100, 200)])):
        p = str(tmp_path / ("f%d" % i))
        _write(p, m, chunks, cells=cells)
        files.append({f: open(os.path.join(p, f), "rb").read() for f in FILES})
    assert files[1] == files[0]
    assert _gunzip(str(tmp_path / "f2" / "matrix.mtx.gz")) == _gunzip(str(tmp_path / "f0" / "matrix.mtx.gz"))


def test_failed_writes_leave_nothing(tmp_path):
    m = _random_csr(20, 5, 0.5, 3)
    short = str(tmp_path / "short")
    with pytest.raises(ValueError):
        _write(short, m, [(0, 10)])                            # 10 of 20 rows
    inside = str(tmp_path / "inside")
    with pytest.raises(KeyError):
        with formats.MtxWriter(inside, m.shape, *_cells(20)) as w:
            w.append(3, m[:3].nnz, *_huffman_sync(_lines(m[:3])))
            raise KeyError("stop")
    aborted = str(tmp_path / "aborted")
    w = formats.MtxWriter(aborted, m.shape, *_cells(20))
    w.abort()
    too_many = str(tmp_path / "too_many")
    with pytest.raises(ValueError):
        with formats.MtxWriter(too_many, (2, 5), *_cells(2)) as w:
            w.append(3, 0, *_huffman_sync(b""))
    for p in (short, inside, aborted, too_many):
        assert not os.path.exists(p) and not os.path.exists(p + ".partial")
    os.makedirs(str(tmp_path / "stale.partial"))                # left behind by an interrupted writer
    _write(str(tmp_path / "stale"), m, [(0, 20)])
    done = str(tmp_path / "done")
    _write(done, m, [(0, 20)])
    with pytest.raises(FileExistsError):
        formats.MtxWriter(done, m.shape, *_cells(20))
    with pytest.raises(ValueError):                             # one annotation per cell
        formats.MtxWriter(str(tmp_path / "g"), m.shape, *_cells(19))
    assert sorted(os.listdir(tmp_path)) == ["done", "stale"]


def test_mtx_argument_errors():
    for kw in (dict(path=None), dict(path="p", compress=True), dict(path="p", host_out=object()),
               dict(path="p", dtype=np.uint16), dict(path="p", dtype=np.float64)):
        with pytest.raises(ValueError):
            sim._check_csr_request("mtx", kw.pop("dtype", np.int64), **kw)
    for dt in (np.int64, np.int32):
        sim._check_csr_request("mtx", dt, path="p")


def test_shard_path_directory():
    assert formats.shard_path("s", 0, 1, suffix="") == "s"
    assert formats.shard_path("s", 2, 3, suffix="") == "s.rank2of3"


# ------------------------------------------------------------------ the kernels
def _format(X, col0=0, cap_short=0):
    """(row_bytes, text_ptr, text) of pst_mtx_row_bytes + pst_csr_row_offsets + pst_mtx_format over the int32 host
    matrix X; with cap_short, the cap is that many bytes below the text and the text buffer comes back whole."""
    dev = torch.device(DEV)
    st = nat.stream_ptr(dev)
    n, G = X.shape
    x = torch.from_numpy(np.ascontiguousarray(X, np.int32)).to(dev)
    rb = torch.empty(max(1, n), dtype=torch.int32, device=dev)
    tp = torch.empty(n + 1, dtype=torch.int64, device=dev)
    nat.call("pst_mtx_row_bytes", x, n, G, G, col0, rb, st)
    nat.call("pst_csr_row_offsets", rb, n, tp, st)
    total = int(tp[n].item())
    out = torch.full((total + 64,), 0xA5, dtype=torch.uint8, device=dev)
    nat.call("pst_mtx_format", x, n, G, G, col0, tp, total - cap_short, out, st)
    text = out.cpu().numpy().tobytes()
    return rb[:n].cpu().numpy(), tp.cpu().numpy(), text if cap_short else text[:total]


@gpu
@pytest.mark.parametrize("G", [1, 7, 70003])
def test_format_kernels_match_python(G):
    rng = np.random.RandomState(G)
    values = np.array([1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 99, 100, 65535, (1 << 31) - 1], np.int64)
    n = 40 if G > 65536 else 300
    X = np.where(rng.rand(n, G) < 0.3, rng.choice(values, size=(n, G)), 0)
    X[rng.rand(n) < 0.2] = 0                                   # all-zero rows
    if G > 1:
        X[:, -1] = 65535                                       # the last gene of every row
    for col0 in (0, 123456, 10 ** 17):
        rb, tp, text = _format(X, col0)
        m = sp.csr_matrix(X)
        want = _lines(m, col0)
        assert text == want, (G, col0)
        lens = [len(_lines(m[i], col0 + i)) for i in range(n)]
        assert rb.tolist() == lens and tp[n] == len(want)
    if G > 65536:
        assert m.indices.max() >= 65536
    _, _, untouched = _format(X, 5, cap_short=1)               # a cap one byte short: nothing written
    assert untouched == b"\xa5" * len(untouched)


@gpu
def test_format_kernel_every_alignment():
    """Rows of 0 ... 40 single nonzeros put the row starts at every offset of a 16-byte piece."""
    rng = np.random.RandomState(3)
    n, G = 600, 260
    X = np.zeros((n, G), np.int64)
    for i in range(n):
        k = i % 41
        X[i, rng.choice(G, size=k, replace=False)] = rng.randint(1, 10 ** rng.randint(1, 10), size=k)
    rb, tp, text = _format(X, 7)
    assert text == _lines(sp.csr_matrix(X), 7)
    assert len(set((tp % 16).tolist())) == 16


# ------------------------------------------------------------------ end to end
@pytest.fixture(scope="module")
def lineage_tree():
    return _lineage_tree(2, 20, 6, 1000, seed=3)


def _same_dir(got, want, path, first=0):
    """An out="mtx" call's (X, pseudotime, branches, scalings) against the out="csr" call."""
    rec, M = got[0], want[0]
    assert isinstance(rec, formats.MtxRecord) and rec.path == path and rec.shape == M.shape
    assert rec.nnz == M.nnz and rec.nbytes == os.path.getsize(os.path.join(path, "matrix.mtx.gz"))
    for a, b in zip(got[1:], want[1:]):
        assert list(a) == list(b)
    _check_dir(path, sp.csr_matrix(M, dtype=np.int64), want[1:], first)
    L = rec.load()
    assert L.dtype == np.int64 and L.shape == M.shape and (L != M).nnz == 0


@gpu
@pytest.mark.parametrize("sampler", SAMPLERS)
def test_every_sampler_writes_the_csr_result(sampler, lineage_tree, tmp_path):
    t, alpha, beta = lineage_tree
    kw = dict(alpha=alpha, beta=beta, seed=12, device=DEV, sampler=sampler)
    calls = [
        lambda **o: sim.sample_density(t, 1500, **kw, **o),
        lambda **o: sim.sample_whole_tree(t, 7, **kw, **o),
        lambda **o: sim.sample_pseudotime_series(t, [300, 400], [5, 30], 4.0, **kw, **o),
        lambda **o: sim._sample_data_at_times(t, np.arange(0, 60), **kw, **o),
    ]
    for c, call in enumerate(calls):
        path = str(tmp_path / ("c%d" % c))
        _same_dir(call(out="mtx", path=path), call(out="csr"), path)
    path = str(tmp_path / "i32")
    _same_dir(sim.sample_density(t, 700, dtype=np.int32, out="mtx", path=path, **kw),
              sim.sample_density(t, 700, dtype=np.int32, out="csr", **kw), path)
    X, pt, br, sc = sim.sample_density(t, 800, alpha=alpha, beta=beta, seed=3, device=DEV)
    dkw = dict(seed=4, device=DEV, sampler=sampler, first=5000)
    path = str(tmp_path / "d")
    got = sim.draw_counts(t, pt, br, sc, alpha, beta, out="mtx", path=path, **dkw)
    want = sim.draw_counts(t, pt, br, sc, alpha, beta, out="csr", **dkw)
    _same_dir((got, pt, br, sc), (want, pt, br, sc), path, first=5000)
    from prosstt_b200 import tree as ptree
    np.random.seed(92)
    p = str(tmp_path / "r")
    got = sim.sample_whole_tree_restricted(ptree.Tree(), seed=6, device=DEV, sampler=sampler, out="mtx", path=p)
    np.random.seed(92)
    _same_dir(got, sim.sample_whole_tree_restricted(ptree.Tree(), seed=6, device=DEV, sampler=sampler, out="csr"), p)


@gpu
@pytest.mark.parametrize("G", [1, 7, 70003])
def test_gene_counts(G, tmp_path):
    t, alpha, beta = _random_tree(G, T=4 if G > 65536 else 12, seed=G)
    n = 300 if G > 65536 else 900
    kw = dict(alpha=alpha, beta=beta, seed=5, device=DEV)
    path = str(tmp_path / "g")
    want = sim.sample_density(t, n, out="csr", **kw)
    if G > 65536:
        assert want[0].indices.max() >= 65536
    _same_dir(sim.sample_density(t, n, out="mtx", path=path, **kw), want, path)


@gpu
def test_empty_rows_all_zero_result_and_no_cells(tmp_path):
    t, alpha, beta = _random_tree(7, seed=2)
    kw = dict(alpha=alpha, beta=beta, seed=3, device=DEV)
    p = str(tmp_path / "sparse")
    want = sim.sample_density(t, 2000, scale_mean=-5.0, out="csr", **kw)
    assert (np.diff(want[0].indptr) == 0).sum() > 100 and want[0].nnz > 0
    _same_dir(sim.sample_density(t, 2000, scale_mean=-5.0, out="mtx", path=p, **kw), want, p)
    p = str(tmp_path / "zero")
    zero = sim.sample_density(t, 500, scale_mean=-40.0, out="mtx", path=p, **kw)
    assert zero[0].nnz == 0
    _same_dir(zero, sim.sample_density(t, 500, scale_mean=-40.0, out="csr", **kw), p)
    p = str(tmp_path / "none")
    none = sim.sample_density(t, 0, out="mtx", path=p, **kw)
    assert none[0].shape == (0, 7) and none[0].nnz == 0 and len(none[1]) == 0
    assert scipy.io.mminfo(os.path.join(p, "matrix.mtx.gz"))[:3] == (7, 0, 0)


def _stream_text(eng, rows, sc, seed, cell0, **kw):
    """stream_csr(mtx=True)'s chunks decompressed and joined, with the chunk bounds."""
    parts, bounds = [], []

    def consume(lo, hi, compressed, crc, text_len, nnz):
        raw = zlib.decompress(bytes(compressed) + b"\x03\x00", -15)
        assert len(raw) == text_len and zlib.crc32(raw) == crc and raw.count(b"\n") == nnz
        parts.append(raw)
        bounds.append((lo, hi))

    eng.stream_csr(rows, sc, seed, cell0, consume, mtx=True, **kw)
    return b"".join(parts), bounds


@gpu
def test_counts_above_3_digits_and_forced_reformat(lineage_tree, tmp_path, monkeypatch):
    t, alpha, beta = _random_tree(64, T=6, seed=21, log_mean=9.0)     # counts of 4 to 6 digits: more text than
    kw = dict(alpha=alpha, beta=beta, seed=2, device=DEV, scale_mean=1.0)   # the budget, re-formatted
    want = sim.sample_density(t, 600, out="csr", **kw)
    assert (want[0].data >= 65535).sum() > 100
    path = str(tmp_path / "deep")
    _same_dir(sim.sample_density(t, 600, out="mtx", path=path, **kw), want, path)
    # a budget of one byte per gene slot: every chunk is formatted again from its work buffer, never redrawn
    t, alpha, beta = lineage_tree
    n, chunk = 1000, 97
    eng, rows, sc = _engine(t, alpha, beta, n)
    ref, ref_bounds = _stream_text(eng, rows, sc, 5, 0, chunk_cells=chunk)
    assert ref == _lines(sp.csr_matrix(eng.draw(rows, sc, 5, 0).cpu().numpy()))
    calls = []
    real = CountEngine.draw

    def spy(self, *a, **k):
        calls.append(1)
        return real(self, *a, **k)

    monkeypatch.setattr(CountEngine, "draw", spy)
    monkeypatch.setattr(pdev, "_mtx_slot_bytes", lambda G, n: 1)
    got, bounds = _stream_text(eng, rows, sc, 5, 0, chunk_cells=chunk)
    assert got == ref and bounds == ref_bounds and len(calls) == len(bounds) == 11
    cells = _cells(n)
    files = []
    for p in ("tiny", "tiny_again"):
        with formats.MtxWriter(str(tmp_path / p), (n, t.G), *cells) as w:
            eng.stream_csr(rows, sc, 5, 0, lambda lo, hi, *a: w.append(hi - lo, a[3], *a[:3]), mtx=True,
                           chunk_cells=chunk)
        files.append(open(str(tmp_path / p / "matrix.mtx.gz"), "rb").read())
    monkeypatch.undo()
    with formats.MtxWriter(str(tmp_path / "budget"), (n, t.G), *cells) as w:
        eng.stream_csr(rows, sc, 5, 0, lambda lo, hi, *a: w.append(hi - lo, a[3], *a[:3]), mtx=True, chunk_cells=chunk)
    assert files[0] == files[1] == open(str(tmp_path / "budget" / "matrix.mtx.gz"), "rb").read()
    eng.check()


@gpu
def test_chunking_gives_identical_text_and_repeats_identical_files(lineage_tree, tmp_path, monkeypatch):
    t, alpha, beta = lineage_tree
    n = 1000
    eng, rows, sc = _engine(t, alpha, beta, n)
    want = _lines(sp.csr_matrix(eng.draw(rows, sc, 5, 77).cpu().numpy()))
    for chunk in (1, 97, n, 5 * n):
        assert _stream_text(eng, rows, sc, 5, 77, chunk_cells=chunk)[0] == want, chunk
    eng.check()
    kw = dict(alpha=alpha, beta=beta, seed=31, device=DEV, out="mtx")
    sim.sample_density(t, 3001, path=str(tmp_path / "big"), **kw)
    sim.sample_density(t, 3001, path=str(tmp_path / "again"), **kw)
    for f in FILES:
        assert open(str(tmp_path / "big" / f), "rb").read() == open(str(tmp_path / "again" / f), "rb").read(), f
    monkeypatch.setattr(pdev, "_STAGE_BYTES", 2 * 16 * t.G * 200)
    sim.sample_density(t, 3001, path=str(tmp_path / "small"), **kw)
    assert _gunzip(str(tmp_path / "big" / "matrix.mtx.gz")) == _gunzip(str(tmp_path / "small" / "matrix.mtx.gz"))


@gpu
def test_rank_directories_stack_to_the_whole(lineage_tree, tmp_path):
    t, alpha, beta = lineage_tree
    world = 3
    kw = dict(alpha=alpha, beta=beta, seed=17, device=DEV)
    whole = sim.sample_density(t, 1001, out="csr", **kw)[0]
    stem = str(tmp_path / "sim")
    paths = [formats.shard_path(stem, r, world, suffix="") for r in range(world)]
    for r, p in enumerate(paths):
        sim.sample_density(t, 1001, shard=(r, world), out="mtx", path=p, **kw)
    assert sorted(os.listdir(tmp_path)) == sorted(os.path.basename(p) for p in paths)
    stacked = sp.csr_matrix(sp.hstack([scipy.io.mmread(os.path.join(p, "matrix.mtx.gz"), spmatrix=False)
                                       for p in paths]))
    assert stacked.shape == whole.T.shape and (stacked != whole.T).nnz == 0
    barcodes = b"".join(_gunzip(os.path.join(p, "barcodes.tsv.gz")) for p in paths)
    assert barcodes == "".join("cell_%d\n" % i for i in range(1001)).encode()


@gpu
def test_errors_leave_nothing(lineage_tree, tmp_path):
    t, alpha, beta = _random_tree(16, seed=4)
    means = {b: np.array(t.means[b]) for b in t.branches}
    for b in t.branches:                                             # the last step of every branch
        means[b][-1, 3] = 0.0
    t.add_genes(means)
    t.invalidate_device_cache()
    eng, rows, sc = _engine(t, alpha, beta, 5000)
    rows = torch.full((5000,), 5, dtype=torch.int32, device=DEV)
    rows[4000:] = TreeTables(t, torch.device(DEV)).P - 1
    p = str(tmp_path / "domain")
    with pytest.raises(ValueError):                                  # a domain error in a later chunk
        with formats.MtxWriter(p, (5000, t.G), *_cells(5000)) as w:
            eng.stream_csr(rows, sc, 1, 0, lambda lo, hi, *a: w.append(hi - lo, a[3], *a[:3]), mtx=True,
                           chunk_cells=100)
    eng.flags.zero_()
    from prosstt_b200 import tree as ptree
    flat = ptree.Tree(topology=[], time={0: 1}, num_branches=1, branch_points=0, modules=1, G=4)
    flat.add_genes({0: np.array([[1.0, 2.0, 0.0, 3.0]])})
    with pytest.raises(ValueError):
        sim.draw_counts(flat, [0] * 5, [0] * 5, [1.0] * 5, 0.2, 2.0, seed=1, device=DEV, out="mtx",
                        path=str(tmp_path / "flat"))
    t2, alpha2, beta2 = lineage_tree
    with pytest.raises(IndexError):                                  # a pseudotime outside the tree
        sim._sample_data_at_times(t2, [0, 5, 10 ** 6], alpha=alpha2, beta=beta2, seed=1, device=DEV, out="mtx",
                                  path=str(tmp_path / "badpt"))
    with pytest.raises(ValueError):
        sim.sample_density(t2, 50, alpha2, beta2, seed=1, device=DEV, out="mtx")
    with pytest.raises(ValueError):
        sim.sample_density(t2, 50, alpha2, beta2, seed=1, device=DEV, out="mtx", path=str(tmp_path / "c"),
                           compress=True)
    twice = str(tmp_path / "twice")
    sim.sample_density(t2, 50, alpha2, beta2, seed=1, device=DEV, out="mtx", path=twice)
    with pytest.raises(FileExistsError):
        sim.sample_density(t2, 50, alpha2, beta2, seed=1, device=DEV, out="mtx", path=twice)
    assert sorted(os.listdir(tmp_path)) == ["twice"]
