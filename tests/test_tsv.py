"""out="tsv", path=...: the reference's `<job>_simulation.txt` (tree_utils.save_matrices), plain or gzipped, formatted
and compressed on the GPU chunk by chunk (pst_tsv_row_bytes, pst_tsv_format, pst_deflate_blocks) and assembled by
formats.TsvWriter.  The file must equal, byte for byte, what save_matrices writes for the out="numpy" result of the
same call, whatever the chunking: the installed pandas is the definition, so every expected byte comes from it.  The
writer is checked without a GPU, by feeding it pandas' text and zlib-made sync-flushed blocks."""
import gzip
import os
import shutil
import subprocess
import tempfile
import zlib

import numpy as np
import pandas as pd
import pytest
import torch

from prosstt_b200 import _native as nat
from prosstt_b200 import device as pdev, formats, simulation as sim, tree_utils
from prosstt_b200.device import CountEngine, TreeTables
from test_csr_stream import _engine, _lineage_tree, _random_tree
from test_mtx import _huffman_sync

DEV = "cuda:0"
SAMPLERS = ["gamma_poisson", "hybrid"]
GZIP_HEADER = b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff"      # MTIME 0, XFL 0, OS 255
gpu = pytest.mark.gpu


# ------------------------------------------------------------------ the writer and the format (no GPU)
def _saved(X):
    """The bytes of save_matrices' _simulation.txt for the matrix X."""
    d = tempfile.mkdtemp()
    try:
        tree_utils.save_matrices("job", d, np.asarray(X), {}, np.zeros(1))
        return open(os.path.join(d, "job_simulation.txt"), "rb").read()
    finally:
        shutil.rmtree(d)


def _expected(X, first=0):
    """(header, [row lines]) of save_matrices' file for X, the rows renamed cell_<first + i>."""
    lines = _saved(X).split(b"\n")[:-1]
    rows = []
    for i, line in enumerate(lines[1:]):
        label, sep, rest = line.partition(b"\t")
        assert label == b"cell_%d" % i
        rows.append(b"cell_%d" % (first + i) + sep + rest + b"\n")
    return lines[0] + b"\n", rows


def _matrix(n, G, seed):
    """Counts with zeros, every digit count from 1 to 10 and the int32 maximum."""
    rng = np.random.RandomState(seed)
    values = np.array([0, 0, 0, 1, 9, 10, 99, 100, 999, 1000, 12345, 123456, 1234567, 12345678, 123456789,
                       1234567890, (1 << 31) - 1], np.int64)
    return rng.choice(values, size=(n, G))


def _write(path, X, chunks, compress=False, first=0):
    _, rows = _expected(X, first)
    with formats.TsvWriter(path, X.shape, first=first, compress=compress) as w:
        for lo, hi in chunks:
            text = b"".join(rows[lo:hi])
            if compress:
                w.append(hi - lo, *_huffman_sync(text))
            else:
                w.append(hi - lo, text, 0, len(text))
    return w


def _content(path, compress):
    raw = open(path, "rb").read()
    if compress:
        assert raw[:10] == GZIP_HEADER
        return gzip.decompress(raw)
    return raw


def _check_file(path, X, compress, first=0):
    header, rows = _expected(X, first)
    assert _content(path, compress) == header + b"".join(rows)
    if first == 0:
        assert _content(path, compress) == _saved(X)
    frame = pd.read_csv(path, sep="\t", index_col=0, compression="gzip" if compress else None)
    assert frame.shape == X.shape
    if X.size:
        assert np.array_equal(frame.values, X)
    assert list(frame.index) == ["cell_%d" % (first + i) for i in range(X.shape[0])]
    if compress and shutil.which("gzip"):
        r = subprocess.run(["gzip", "-t", path], capture_output=True)
        assert r.returncode == 0, r.stderr


@pytest.mark.parametrize("compress", [False, True])
def test_writer_round_trip(tmp_path, compress):
    X = _matrix(301, 57, 1)
    files = []
    for i, chunks in enumerate(([(0, 301)], [(0, 301)], [(0, 1), (1, 50), (50, 50), (50, 300), (300, 301)])):
        path = str(tmp_path / ("x%d" % i))
        w = _write(path, X, chunks, compress)
        _check_file(path, X, compress)
        files.append(open(path, "rb").read())
        rec = w.record()
        assert isinstance(rec, formats.TsvRecord) and rec.path == path and rec.shape == X.shape
        assert rec.compressed == compress and rec.nbytes == os.path.getsize(path)
        assert rec.load().equals(pd.read_csv(path, sep="\t", index_col=0, compression="gzip" if compress else None))
    assert files[0] == files[1]
    if not compress:
        assert files[2] == files[0]
    assert sorted(os.listdir(tmp_path)) == ["x0", "x1", "x2"]


@pytest.mark.parametrize("compress", [False, True])
def test_edge_cases(tmp_path, compress):
    for name, X, chunks, first in (("none", np.zeros((0, 5), np.int64), [], 0),          # the header line only
                                   ("nogenes", np.zeros((7, 0), np.int64), [(0, 3), (3, 7)], 0),
                                   ("neither", np.zeros((0, 0), np.int64), [], 0),
                                   ("g1", _matrix(40, 1, 2), [(0, 40)], 0),
                                   ("decade", _matrix(30, 6, 3), [(0, 9), (9, 30)], 9990),   # cell_9999, cell_10000
                                   ("far", _matrix(5, 3, 4), [(0, 5)], 10 ** 15)):
        path = str(tmp_path / name)
        _write(path, X, chunks, compress, first)
        _check_file(path, X, compress, first)
    assert formats.tsv_header(0) == _saved(np.zeros((0, 0), np.int64))


def test_wide_header_spans_stored_blocks(tmp_path):
    X = _matrix(3, 70003, 5)                                  # a header line of 0.8 MB: many stored blocks
    _write(str(tmp_path / "w"), X, [(0, 3)], True)
    _check_file(str(tmp_path / "w"), X, True)


@pytest.mark.parametrize("compress", [False, True])
def test_failed_writes_leave_nothing(tmp_path, compress):
    X = _matrix(20, 5, 3)
    short = str(tmp_path / "short")
    with pytest.raises(ValueError):
        _write(short, X, [(0, 10)], compress)                 # 10 of 20 rows
    inside = str(tmp_path / "inside")
    with pytest.raises(KeyError):
        with formats.TsvWriter(inside, X.shape, compress=compress) as w:
            w.append(3, *(_huffman_sync(b"x") if compress else (b"x", 0, 1)))
            raise KeyError("stop")
    aborted = str(tmp_path / "aborted")
    formats.TsvWriter(aborted, X.shape, compress=compress).abort()
    too_many = str(tmp_path / "too_many")
    with pytest.raises(ValueError):
        with formats.TsvWriter(too_many, (2, 5), compress=compress) as w:
            w.append(3, b"", 0, 0)
    for p in (short, inside, aborted, too_many):
        assert not os.path.exists(p) and not os.path.exists(p + ".partial")
    open(str(tmp_path / "stale.partial"), "wb").write(b"left behind")
    _write(str(tmp_path / "stale"), X, [(0, 20)], compress)
    _check_file(str(tmp_path / "stale"), X, compress)
    with pytest.raises(FileExistsError):
        formats.TsvWriter(str(tmp_path / "stale"), X.shape, compress=compress)
    assert sorted(os.listdir(tmp_path)) == ["stale"]


def test_tsv_argument_errors():
    for kw in (dict(path=None), dict(path="p", host_out=object()), dict(path="p", dtype=np.uint16),
               dict(path="p", dtype=np.float64), dict(path="p", compression="lz77"),
               dict(path="p", compress=True, compression="zstd")):
        with pytest.raises(ValueError):
            sim._check_csr_request("tsv", kw.pop("dtype", np.int64), **kw)
    for dt in (np.int64, np.int32):
        for kw in (dict(), dict(compress=True), dict(compress=True, compression="lz77")):
            sim._check_csr_request("tsv", dt, path="p", **kw)


def test_shard_path_file():
    assert formats.shard_path("sim", 0, 1, suffix="_simulation.txt") == "sim_simulation.txt"
    assert formats.shard_path("sim", 1, 3, suffix="_simulation.txt.gz") == "sim.rank1of3_simulation.txt.gz"


# ------------------------------------------------------------------ the kernels
def _format(X, row0=0, cap_short=0):
    """(row_bytes, text_ptr, text) of pst_tsv_row_bytes + pst_csr_row_offsets + pst_tsv_format over the int32 host
    matrix X; with cap_short, the cap is that many bytes below the text and the text buffer comes back whole."""
    dev = torch.device(DEV)
    st = nat.stream_ptr(dev)
    n, G = X.shape
    x = torch.from_numpy(np.ascontiguousarray(X, np.int32)).to(dev)
    rb = torch.empty(max(1, n), dtype=torch.int32, device=dev)
    tp = torch.empty(n + 1, dtype=torch.int64, device=dev)
    nat.call("pst_tsv_row_bytes", x if G else None, n, G, G, row0, rb, st)
    nat.call("pst_csr_row_offsets", rb, n, tp, st)
    total = int(tp[n].item())
    out = torch.full((total + 64,), 0xA5, dtype=torch.uint8, device=dev)
    nat.call("pst_tsv_format", x if G else None, n, G, G, row0, tp, total - cap_short, out, st)
    text = out.cpu().numpy().tobytes()
    return rb[:n].cpu().numpy(), tp.cpu().numpy(), text if cap_short else text[:total]


def _rows(X, row0=0):
    return ["cell_%d" % (row0 + i) + "".join("\t%d" % v for v in row) + "\n" for i, row in enumerate(X)]


@gpu
@pytest.mark.parametrize("G", [0, 1, 7, 70003])
def test_format_kernels_match_python(G):
    n = 12 if G > 65536 else 300
    X = _matrix(n, G, G)
    if G:
        X[:, -1] = (1 << 31) - 1                              # the last gene of every row
        X[::7] = 0
    for row0 in (0, 9990, 10 ** 17):
        rb, tp, text = _format(X, row0)
        rows = _rows(X, row0)
        assert text == "".join(rows).encode(), (G, row0)
        assert rb.tolist() == [len(r) for r in rows] and tp[n] == len(text)
        if 0 < G < 100:                                       # the row starts fall on every offset of a piece
            assert len(set((tp % 16).tolist())) == 16
    _, _, untouched = _format(X, 5, cap_short=1)              # a cap one byte short: nothing written
    assert untouched == b"\xa5" * len(untouched)


@gpu
def test_format_kernel_strided_rows():
    """ldx > G and a matrix whose genes are not a multiple of 4: the unvectorised loads."""
    dev = torch.device(DEV)
    st = nat.stream_ptr(dev)
    X = _matrix(50, 13, 9)
    wide = np.zeros((50, 20), np.int32)
    wide[:, :13] = X
    x = torch.from_numpy(wide).to(dev)
    rb = torch.empty(50, dtype=torch.int32, device=dev)
    tp = torch.empty(51, dtype=torch.int64, device=dev)
    nat.call("pst_tsv_row_bytes", x, 50, 13, 20, 3, rb, st)
    nat.call("pst_csr_row_offsets", rb, 50, tp, st)
    out = torch.empty(int(tp[50].item()), dtype=torch.uint8, device=dev)
    nat.call("pst_tsv_format", x, 50, 13, 20, 3, tp, out.numel(), out, st)
    assert out.cpu().numpy().tobytes() == "".join(_rows(X, 3)).encode()


# ------------------------------------------------------------------ end to end
@pytest.fixture(scope="module")
def lineage_tree():
    return _lineage_tree(2, 20, 6, 1000, seed=3)


def _same_file(got, want, path, compress, first=0):
    """An out="tsv" call's (X, pseudotime, branches, scalings) against the out="numpy" call."""
    rec, X = got[0], np.asarray(want[0])
    assert isinstance(rec, formats.TsvRecord) and rec.path == path and rec.shape == X.shape
    assert rec.compressed == compress and rec.nbytes == os.path.getsize(path)
    for a, b in zip(got[1:], want[1:]):
        assert list(a) == list(b)
    _check_file(path, X, compress, first)
    frame = rec.load()
    assert frame.shape == X.shape and np.array_equal(frame.values, X)
    assert list(frame.columns) == ["gene_%d" % j for j in range(X.shape[1])]


@gpu
@pytest.mark.parametrize("sampler", SAMPLERS)
def test_every_entry_point_writes_save_matrices(sampler, lineage_tree, tmp_path):
    t, alpha, beta = lineage_tree
    kw = dict(alpha=alpha, beta=beta, seed=12, device=DEV, sampler=sampler)
    calls = [
        lambda **o: sim.sample_density(t, 1500, **kw, **o),
        lambda **o: sim.sample_whole_tree(t, 7, **kw, **o),
        lambda **o: sim.sample_pseudotime_series(t, [300, 400], [5, 30], 4.0, **kw, **o),
        lambda **o: sim._sample_data_at_times(t, np.arange(0, 60), **kw, **o),
    ]
    for c, call in enumerate(calls):
        want = call()
        for compress in (False, True):
            path = str(tmp_path / ("c%d_%d" % (c, compress)))
            _same_file(call(out="tsv", path=path, compress=compress), want, path, compress)
    want = sim.sample_density(t, 700, dtype=np.int32, **kw)
    for compress in (False, True):
        path = str(tmp_path / ("i32_%d" % compress))
        _same_file(sim.sample_density(t, 700, dtype=np.int32, out="tsv", path=path, compress=compress, **kw),
                   want, path, compress)
    X, pt, br, sc = sim.sample_density(t, 800, alpha=alpha, beta=beta, seed=3, device=DEV)
    dkw = dict(seed=4, device=DEV, sampler=sampler, first=5000)
    want = sim.draw_counts(t, pt, br, sc, alpha, beta, **dkw)
    for compress in (False, True):
        path = str(tmp_path / ("d%d" % compress))
        got = sim.draw_counts(t, pt, br, sc, alpha, beta, out="tsv", path=path, compress=compress, **dkw)
        _same_file((got, pt, br, sc), (want, pt, br, sc), path, compress, first=5000)
    from prosstt_b200 import tree as ptree
    np.random.seed(92)
    want = sim.sample_whole_tree_restricted(ptree.Tree(), seed=6, device=DEV, sampler=sampler)
    for compress in (False, True):
        np.random.seed(92)
        p = str(tmp_path / ("r%d" % compress))
        got = sim.sample_whole_tree_restricted(ptree.Tree(), seed=6, device=DEV, sampler=sampler, out="tsv", path=p,
                                               compress=compress)
        _same_file(got, want, p, compress)


@gpu
def test_no_cells(tmp_path):
    t, alpha, beta = _random_tree(7, seed=2)
    kw = dict(alpha=alpha, beta=beta, seed=3, device=DEV)
    for compress in (False, True):
        p = str(tmp_path / ("none%d" % compress))
        _same_file(sim.sample_density(t, 0, out="tsv", path=p, compress=compress, **kw), sim.sample_density(t, 0, **kw),
                   p, compress)
        assert _content(p, compress) == formats.tsv_header(7)


@gpu
def test_no_genes(tmp_path):
    from prosstt_b200 import tree as ptree
    flat = ptree.Tree(topology=[], time={0: 3}, num_branches=1, branch_points=0, modules=1, G=0)
    flat.add_genes({0: np.zeros((3, 0))})
    for compress in (False, True):
        p = str(tmp_path / ("g0_%d" % compress))
        got = sim.draw_counts(flat, [0, 1, 2, 1], [0] * 4, [1.0] * 4, 0.2, 2.0, seed=1, device=DEV, out="tsv",
                              path=p, compress=compress, first=98)
        assert got.shape == (4, 0)
        _check_file(p, np.zeros((4, 0), np.int64), compress, first=98)


def _stream_text(eng, rows, sc, seed, cell0, compress=False, **kw):
    """stream_csr(tsv=True)'s chunks (decompressed) and joined, with the chunk bounds."""
    parts, bounds = [], []

    def consume(lo, hi, data, crc, text_len):
        raw = zlib.decompress(bytes(data) + b"\x03\x00", -15) if compress else bytes(data)
        assert len(raw) == text_len and raw.count(b"\n") == hi - lo
        if compress:
            assert zlib.crc32(raw) == crc
        parts.append(raw)
        bounds.append((lo, hi))

    eng.stream_csr(rows, sc, seed, cell0, consume, tsv=True, compress=compress, **kw)
    return b"".join(parts), bounds


@gpu
@pytest.mark.parametrize("compress", [False, True])
def test_counts_above_3_digits_and_forced_reformat(lineage_tree, tmp_path, monkeypatch, compress):
    t, alpha, beta = _random_tree(64, T=6, seed=21, log_mean=9.0)     # counts of 4 to 6 digits: more text than
    kw = dict(alpha=alpha, beta=beta, seed=2, device=DEV, scale_mean=1.0)   # the budget, re-formatted
    want = sim.sample_density(t, 600, **kw)
    assert (want[0] >= 1000).mean() > 0.3
    path = str(tmp_path / "deep")
    _same_file(sim.sample_density(t, 600, out="tsv", path=path, compress=compress, **kw), want, path, compress)
    # a budget of one byte per gene slot: every chunk is formatted again from its work buffer, never redrawn
    t, alpha, beta = lineage_tree
    n, chunk = 1000, 97
    eng, rows, sc = _engine(t, alpha, beta, n)
    ref, ref_bounds = _stream_text(eng, rows, sc, 5, 0, compress, chunk_cells=chunk)
    assert ref == "".join(_rows(eng.draw(rows, sc, 5, 0).cpu().numpy())).encode()
    calls = []
    real = CountEngine.draw

    def spy(self, *a, **k):
        calls.append(1)
        return real(self, *a, **k)

    monkeypatch.setattr(CountEngine, "draw", spy)
    monkeypatch.setattr(pdev, "_tsv_slot_bytes", lambda G, n: 1)
    got, bounds = _stream_text(eng, rows, sc, 5, 0, compress, chunk_cells=chunk)
    assert got == ref and bounds == ref_bounds and len(calls) == len(bounds) == 11
    files = []
    for p in ("tiny", "tiny_again"):
        with formats.TsvWriter(str(tmp_path / p), (n, t.G), compress=compress) as w:
            eng.stream_csr(rows, sc, 5, 0, lambda lo, hi, *a: w.append(hi - lo, *a), tsv=True, compress=compress,
                           chunk_cells=chunk)
        files.append(open(str(tmp_path / p), "rb").read())
    monkeypatch.undo()
    with formats.TsvWriter(str(tmp_path / "budget"), (n, t.G), compress=compress) as w:
        eng.stream_csr(rows, sc, 5, 0, lambda lo, hi, *a: w.append(hi - lo, *a), tsv=True, compress=compress,
                       chunk_cells=chunk)
    assert files[0] == files[1] == open(str(tmp_path / "budget"), "rb").read()
    eng.check()


@gpu
def test_chunking_gives_identical_text_and_repeats_identical_files(lineage_tree, tmp_path, monkeypatch):
    t, alpha, beta = lineage_tree
    n = 1000
    eng, rows, sc = _engine(t, alpha, beta, n)
    want = "".join(_rows(eng.draw(rows, sc, 5, 77).cpu().numpy(), 77)).encode()
    for compress in (False, True):
        for chunk in (1, 97, n, 5 * n):
            assert _stream_text(eng, rows, sc, 5, 77, compress, chunk_cells=chunk)[0] == want, (compress, chunk)
    eng.check()
    kw = dict(alpha=alpha, beta=beta, seed=31, device=DEV, out="tsv")
    for compress in (False, True):
        big, again, small = (str(tmp_path / ("%s%d" % (s, compress))) for s in ("big", "again", "small"))
        sim.sample_density(t, 3001, path=big, compress=compress, **kw)
        sim.sample_density(t, 3001, path=again, compress=compress, **kw)
        assert open(big, "rb").read() == open(again, "rb").read()
        with monkeypatch.context() as m:
            m.setattr(pdev, "_STAGE_BYTES", 2 * 16 * t.G * 200)
            sim.sample_density(t, 3001, path=small, compress=compress, **kw)
        assert _content(big, compress) == _content(small, compress)


@gpu
def test_lz77_is_smaller_and_decompresses_to_the_same_text(lineage_tree, tmp_path):
    t, alpha, beta = lineage_tree
    kw = dict(alpha=alpha, beta=beta, seed=8, device=DEV, out="tsv", compress=True)
    huff, lz = str(tmp_path / "huffman"), str(tmp_path / "lz77")
    a = sim.sample_density(t, 4000, path=huff, **kw)[0]
    b = sim.sample_density(t, 4000, path=lz, compression="lz77", **kw)[0]
    assert _content(huff, True) == _content(lz, True)
    _check_file(lz, sim.sample_density(t, 4000, alpha=alpha, beta=beta, seed=8, device=DEV)[0], True)
    assert b.nbytes < a.nbytes, (a.nbytes, b.nbytes)


@gpu
def test_rank_files_stack_to_the_whole(lineage_tree, tmp_path):
    t, alpha, beta = lineage_tree
    world = 3
    kw = dict(alpha=alpha, beta=beta, seed=17, device=DEV, out="tsv")
    whole = str(tmp_path / "whole.txt")
    sim.sample_density(t, 1001, path=whole, **kw)
    stem = str(tmp_path / "sim")
    for compress in (False, True):
        suffix = "_simulation.txt.gz" if compress else "_simulation.txt"
        paths = [formats.shard_path(stem, r, world, suffix=suffix) for r in range(world)]
        for r, p in enumerate(paths):
            sim.sample_density(t, 1001, shard=(r, world), path=p, compress=compress, **kw)
        texts = [_content(p, compress) for p in paths]
        header = formats.tsv_header(t.G)
        assert all(x.startswith(header) for x in texts)
        assert texts[0] + b"".join(x[len(header):] for x in texts[1:]) == open(whole, "rb").read()


@gpu
@pytest.mark.parametrize("compress", [False, True])
def test_errors_leave_nothing(lineage_tree, tmp_path, compress):
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
        with formats.TsvWriter(p, (5000, t.G), compress=compress) as w:
            eng.stream_csr(rows, sc, 1, 0, lambda lo, hi, *a: w.append(hi - lo, *a), tsv=True, compress=compress,
                           chunk_cells=100)
    eng.flags.zero_()
    t2, alpha2, beta2 = lineage_tree
    with pytest.raises(IndexError):                                  # a pseudotime outside the tree
        sim._sample_data_at_times(t2, [0, 5, 10 ** 6], alpha=alpha2, beta=beta2, seed=1, device=DEV, out="tsv",
                                  path=str(tmp_path / "badpt"), compress=compress)
    with pytest.raises(ValueError):
        sim.sample_density(t2, 50, alpha2, beta2, seed=1, device=DEV, out="tsv", compress=compress)
    twice = str(tmp_path / "twice")
    sim.sample_density(t2, 50, alpha2, beta2, seed=1, device=DEV, out="tsv", path=twice, compress=compress)
    with pytest.raises(FileExistsError):
        sim.sample_density(t2, 50, alpha2, beta2, seed=1, device=DEV, out="tsv", path=twice, compress=compress)
    assert sorted(os.listdir(tmp_path)) == ["twice"]
