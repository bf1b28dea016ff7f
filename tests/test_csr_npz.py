"""out="csr", path=..., compress=True: one zip64 `.npz` with DEFLATE members, compressed on the GPU chunk by chunk
(pst_deflate_blocks) and assembled by formats.CsrNpzWriter.  scipy.sparse.load_npz must read the in-memory
out="csr" result back, whatever the chunking, and every decompressed member must be the bytes np.save writes.
The writer and the format are checked without a GPU, by feeding it zlib-made sync-flushed blocks."""
import io
import os
import shutil
import struct
import zipfile
import zlib

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from prosstt_b200 import _native as nat
from prosstt_b200 import device as pdev, formats, simulation as sim
from prosstt_b200.device import TreeTables
from test_csr_stream import _cells, _engine, _lineage_tree, _random_csr, _random_tree, _reset_hwm, _vm

DEV = "cuda:0"
SAMPLERS = ["gamma_poisson", "hybrid"]
MEMBERS = ("format", "shape", "indptr", "indices", "data", "pseudotime", "branches", "scalings")
gpu = pytest.mark.gpu


# ------------------------------------------------------------------ the writer and the format (no GPU)
def _npy(a):
    buf = io.BytesIO()
    np.save(buf, a, allow_pickle=False)
    return buf.getvalue()


def _write(path, m, chunks, dtype=np.int64, cells=None):
    """Write the scipy matrix m as a compressed file, in the given row chunks."""
    n = m.shape[0]
    with formats.CsrNpzWriter(path, m.shape, *(cells or _cells(n)), dtype=dtype) as w:
        before = 0
        for lo, hi in chunks:
            part = m[lo:hi]
            w.append("indptr", *formats.sync_deflate((part.indptr[1:] + before).astype(w.index_dtype).tobytes()))
            w.append("indices", *formats.sync_deflate(part.indices.astype(w.index_dtype).tobytes()))
            w.append("data", *formats.sync_deflate(part.data.astype(dtype).tobytes()))
            before += part.nnz
    return w


def _check_file(path, m, cells, dtype):
    idx = np.int32 if m.shape[0] * m.shape[1] < (1 << 31) else np.int64
    with zipfile.ZipFile(path) as z:
        assert z.testzip() is None
        assert sorted(z.namelist()) == sorted(n + ".npy" for n in MEMBERS)
        assert all(i.compress_type == zipfile.ZIP_DEFLATED for i in z.infolist())
        want = dict(indptr=m.indptr.astype(idx), indices=m.indices.astype(idx), data=m.data.astype(dtype),
                    format=np.array(b"csr"), shape=np.array(m.shape, dtype=np.int64),
                    pseudotime=np.asarray(cells[0], np.int64), branches=np.asarray(cells[1]),
                    scalings=np.asarray(cells[2], np.float64))
        for name, a in want.items():
            assert z.read(name + ".npy") == _npy(a), name
    got = sp.load_npz(path)
    assert got.shape == m.shape and (got != m).nnz == 0 and got.data.dtype == dtype
    with np.load(path) as z:
        assert sorted(z.files) == sorted(MEMBERS)
    X, pt, br, sc = formats.load_csr_shard(path)
    assert X.indptr.dtype == idx and X.indices.dtype == idx and X.data.dtype == dtype
    X.check_format(full_check=True)
    assert np.array_equal(X.indptr, m.indptr) and np.array_equal(X.indices, m.indices)
    assert np.array_equal(X.data, m.data)
    assert np.array_equal(pt, cells[0]) and list(br) == list(cells[1]) and np.array_equal(sc, cells[2])


@pytest.mark.parametrize("dtype", [np.int64, np.int32])
def test_writer_round_trip(tmp_path, dtype):
    m = _random_csr(301, 57, 0.2, 1)
    m[40:90] = 0                                               # empty rows, and an empty chunk below
    m.eliminate_zeros()
    cells = _cells(301, 2)
    path = str(tmp_path / "x.npz")
    w = _write(path, m, [(0, 7), (7, 50), (50, 80), (80, 80), (80, 301)], dtype=dtype, cells=cells)
    assert sorted(os.listdir(tmp_path)) == ["x.npz"]
    _check_file(path, m, cells, dtype)
    rec = w.record()
    assert isinstance(rec, formats.CompressedCsr)
    assert rec.path == path and rec.shape == m.shape and rec.nnz == m.nnz and rec.dtype == dtype
    assert rec.index_dtype == np.int32 and rec.nbytes == os.path.getsize(path)
    assert (rec.load() != m).nnz == 0
    with zipfile.ZipFile(path) as z:                           # indptr and data went through temporaries
        assert w.copied_at_close == sum(z.getinfo(n + ".npy").compress_size for n in ("indptr", "data")) - 2 * (
            5 + 128 + 2)


def test_chunking_and_repeats_give_identical_files(tmp_path):
    m = _random_csr(200, 40, 0.3, 7)
    cells = _cells(200, 1)
    files = []
    for i, chunks in enumerate(([(0, 200)], [(0, 200)], [(0, 1), (1, 100), (100, 200)])):
        p = str(tmp_path / ("f%d.npz" % i))
        _write(p, m, chunks, cells=cells)
        with zipfile.ZipFile(p) as z:
            files.append({n: z.read(n) for n in z.namelist()})
        if i == 1:
            assert open(p, "rb").read() == open(str(tmp_path / "f0.npz"), "rb").read()
    assert files[2] == files[0]


def test_every_streamed_member_is_zip64(tmp_path):
    m = _random_csr(50, 20, 0.3, 3)
    path = str(tmp_path / "x.npz")
    _write(path, m, [(0, 50)])
    raw = open(path, "rb").read()
    with zipfile.ZipFile(path) as z:
        for info in z.infolist():
            assert info.extract_version >= 45
            at = info.header_offset
            sig, _, _, method, _, _, crc, csize, usize, nlen, xlen = struct.unpack("<IHHHHHIIIHH", raw[at:at + 30])
            assert sig == 0x04034B50 and method == 8 and crc == info.CRC
            assert csize == usize == 0xFFFFFFFF and xlen == 20
            tag, size, u64, c64 = struct.unpack("<HHQQ", raw[at + 30 + nlen:at + 50 + nlen])
            assert (tag, size, u64, c64) == (1, 16, info.file_size, info.compress_size)
    assert struct.unpack("<I", raw[-22 - 20:-22 - 16])[0] == 0x07064B50       # zip64 end-of-directory locator


def test_index_dtype_switches_at_2_31(tmp_path):
    for n, G, want in ((1, (1 << 31) - 1, np.int32), (2, 1 << 30, np.int64), (3, 1 << 31, np.int64)):
        m = sp.csr_matrix((n, G), dtype=np.int64)             # rows of zeros, announced shape only
        path = str(tmp_path / ("s%d.npz" % n))
        w = _write(path, m, [(0, n)])
        assert w.index_dtype == want
        X = formats.load_csr_shard(path)[0]
        assert X.indptr.dtype == want and X.indices.dtype == want and X.shape == (n, G) and X.nnz == 0
        with zipfile.ZipFile(path) as z:
            assert z.read("indptr.npy") == _npy(np.zeros(n + 1, want))


def test_all_zero_and_empty_matrices(tmp_path):
    z = sp.csr_matrix((9, 4), dtype=np.int64)
    cells = _cells(9)
    _write(str(tmp_path / "z.npz"), z, [(0, 4), (4, 9)], cells=cells)
    _check_file(str(tmp_path / "z.npz"), z, cells, np.int64)
    e = sp.csr_matrix((0, 4), dtype=np.int64)
    _write(str(tmp_path / "e.npz"), e, [])
    X, pt, br, sc = formats.load_csr_shard(str(tmp_path / "e.npz"))
    assert X.shape == (0, 4) and X.indptr.tolist() == [0] and len(pt) == len(br) == len(sc) == 0
    assert sp.load_npz(str(tmp_path / "e.npz")).shape == (0, 4)


def test_failed_writes_leave_nothing(tmp_path):
    m = _random_csr(20, 5, 0.5, 3)
    short = str(tmp_path / "short.npz")
    with pytest.raises(ValueError):
        _write(short, m, [(0, 10)])                            # 10 of 20 rows
    inside = str(tmp_path / "inside.npz")
    with pytest.raises(KeyError):
        with formats.CsrNpzWriter(inside, m.shape, *_cells(20)) as w:
            w.append("indices", *formats.sync_deflate(m.indices[:3].astype(np.int32).tobytes()))
            raise KeyError("stop")
    aborted = str(tmp_path / "aborted.npz")
    w = formats.CsrNpzWriter(aborted, m.shape, *_cells(20))
    w.append("data", *formats.sync_deflate(m.data[:3].tobytes()))
    w.abort()
    mismatch = str(tmp_path / "mismatch.npz")
    with pytest.raises(ValueError):                            # indices and data of different lengths
        with formats.CsrNpzWriter(mismatch, (1, 5), *_cells(1)) as w:
            w.append("indptr", *formats.sync_deflate(np.array([2], np.int32).tobytes()))
            w.append("indices", *formats.sync_deflate(np.array([0, 1], np.int32).tobytes()))
            w.append("data", *formats.sync_deflate(np.array([4], np.int64).tobytes()))
    with pytest.raises(ValueError):                            # not whole values
        with formats.CsrNpzWriter(str(tmp_path / "odd.npz"), (1, 5), *_cells(1)) as w:
            w.append("data", *formats.sync_deflate(b"abc"))
    for p in (short, inside, aborted, mismatch, str(tmp_path / "odd.npz")):
        assert not os.path.exists(p) and not os.path.exists(p + ".partial")
    done = str(tmp_path / "done.npz")
    _write(done, m, [(0, 20)])
    with pytest.raises(FileExistsError):
        formats.CsrNpzWriter(done, m.shape, *_cells(20))
    with pytest.raises(ValueError):                             # data dtype
        formats.CsrNpzWriter(str(tmp_path / "f.npz"), m.shape, *_cells(20), dtype=np.float64)
    with pytest.raises(ValueError):                             # one annotation per cell
        formats.CsrNpzWriter(str(tmp_path / "g.npz"), m.shape, *_cells(19))
    assert sorted(os.listdir(tmp_path)) == ["done.npz"]


def test_shard_path_npz_suffix():
    assert formats.shard_path("s", 0, 1, suffix=".npz") == "s.npz"
    assert formats.shard_path("s", 2, 3, suffix=".npz") == "s.rank2of3.npz"


def test_compress_argument_errors():
    for kw in (dict(out="csr", path=None), dict(out="numpy", path="p.npz"), dict(out="torch", path=None)):
        with pytest.raises(ValueError):
            sim._check_csr_request(kw["out"], np.int64, path=kw["path"], compress=True)
    sim._check_csr_request("csr", np.int64, path="p.npz", compress=True)


def test_host_crc32_combine():
    rng = np.random.RandomState(0)
    lib = nat.load()
    for la, lb in ((0, 0), (5, 0), (0, 7), (1000, 33333), (70000, 1)):
        a, b = rng.bytes(la), rng.bytes(lb)
        assert lib.pst_host_crc32_combine(zlib.crc32(a), zlib.crc32(b), lb) == zlib.crc32(a + b)


# ------------------------------------------------------------------ the kernels
def _deflate(data, block=32768, count=None, scale=1):
    """(compressed bytes, crc) of pst_deflate_blocks over the bytes `data`."""
    lib = nat.load()
    n = len(data)
    x = torch.from_numpy(np.frombuffer(data, np.uint8).copy()).to(DEV) if n else torch.empty(16, dtype=torch.uint8,
                                                                                               device=DEV)
    out = torch.empty(max(1, lib.pst_deflate_bound(n, block)), dtype=torch.uint8, device=DEV)
    ws = int(lib.pst_deflate_workspace_bytes(n, block))
    work = torch.empty(max(1, ws), dtype=torch.uint8, device=DEV)
    size = torch.full((1,), -1, dtype=torch.int64, device=DEV)
    crc = torch.zeros(2, dtype=torch.int32, device=DEV)
    cnt = None if count is None else torch.tensor([count], dtype=torch.int64, device=DEV)
    nat.call("pst_deflate_blocks", x, cnt, scale, n, block, out, size, crc, work, ws, nat.stream_ptr(torch.device(DEV)))
    k = int(size.item())
    assert 0 <= k <= lib.pst_deflate_bound(n, block)
    return out[:k].cpu().numpy().tobytes(), int(crc[0].item()) & 0xFFFFFFFF


def _fibonacci_bytes(n, rng):
    """n bytes whose counts, with the end-of-block symbol's 1, are 1, 1, 2, 3, 5, ...: an optimal code needs one
    more bit per symbol, past 15 bits."""
    f = [1, 2]
    while sum(f) + f[-1] + f[-2] <= n:
        f.append(f[-1] + f[-2])
    vals = np.concatenate([np.full(c, 7 * i % 256, np.uint8) for i, c in enumerate(f)])
    vals = np.concatenate([vals, np.full(n - len(vals), 7 * (len(f) - 1) % 256, np.uint8)])
    return rng.permutation(vals).tobytes()


@gpu
def test_deflate_blocks_decode_with_zlib():
    rng = np.random.RandomState(1)
    cases = {"empty": b"", "one": b"\x05"}
    for n in (3, 4, 8, 13, 1000, 32767, 32768, 32769, 100003):
        cases["len%d" % n] = rng.randint(0, 7, size=n).astype(np.uint8).tobytes()
    cases["repeated"] = b"\x07" * 100000
    cases["uniform"] = np.tile(np.arange(256, dtype=np.uint8), 500).tobytes()
    cases["random"] = rng.bytes(3 * 32768 + 11)
    cases["fibonacci"] = _fibonacci_bytes(32768, rng) * 2
    cases["int64_counts"] = np.minimum(rng.negative_binomial(0.5, 0.1, size=40000), 70000).astype(np.int64).tobytes()
    for name, data in cases.items():
        for block in (32768, 1024):
            comp, crc = _deflate(data, block)
            assert zlib.decompress(comp + b"\x03\x00", -15) == data, (name, block)
            assert crc == zlib.crc32(data), (name, block)
            nblocks = (len(data) + block - 1) // block
            if name == "random":                                 # incompressible: every block stored
                assert len(comp) == len(data) + 5 * nblocks
            if name in ("repeated", "fibonacci", "int64_counts") and block == 32768:
                assert len(comp) < 0.8 * len(data), name
    # the Fibonacci histogram needs codes longer than 15 bits without the limit
    comp, _ = _deflate(cases["fibonacci"][:32768])
    assert zlib.decompress(comp + b"\x03\x00", -15) == cases["fibonacci"][:32768]
    # the length from device memory: count x scale bytes of a larger buffer; blocks concatenate
    data = cases["int64_counts"]
    comp, crc = _deflate(data, count=1001, scale=8)
    assert zlib.decompress(comp + b"\x03\x00", -15) == data[:8008] and crc == zlib.crc32(data[:8008])
    a, _ = _deflate(data[:16384])
    b, _ = _deflate(data[16384:])
    assert zlib.decompress(a + b + b"\x03\x00", -15) == data


@gpu
def test_crc32_matches_zlib():
    rng = np.random.RandomState(2)
    for n in (0, 1, 2, 5, 1000, 32767, 32768, 32769, 65536 * 3 + 7, 1000003):
        data = rng.bytes(n)
        x = torch.from_numpy(np.frombuffer(data, np.uint8).copy()).to(DEV) if n else None
        crc = torch.zeros(2, dtype=torch.int32, device=DEV)
        nat.call("pst_crc32", x, n, crc, nat.stream_ptr(torch.device(DEV)))
        assert int(crc[0].item()) & 0xFFFFFFFF == zlib.crc32(data), n


# ------------------------------------------------------------------ end to end
@pytest.fixture(scope="module")
def lineage_tree():
    return _lineage_tree(2, 20, 6, 1000, seed=3)


def _same_file(got, want, path, data_dtype=np.int64):
    """A compress=True call's (X, pseudotime, branches, scalings) against the in-memory call."""
    rec, M = got[0], want[0]
    assert isinstance(rec, formats.CompressedCsr) and rec.path == path and rec.shape == M.shape
    assert rec.nnz == M.nnz and rec.dtype == data_dtype and rec.nbytes == os.path.getsize(path)
    idx = np.int32 if M.shape[0] * M.shape[1] < (1 << 31) else np.int64
    assert rec.index_dtype == idx
    L = sp.load_npz(path)
    assert L.shape == M.shape and L.format == "csr"
    for name in ("indptr", "indices", "data"):
        assert np.array_equal(getattr(L, name), getattr(M, name)) and getattr(L, name).dtype == getattr(M, name).dtype
    X, pt, br, sc = formats.load_csr_shard(path)
    assert X.indptr.dtype == idx and X.indices.dtype == idx and X.data.dtype == data_dtype
    assert np.array_equal(X.indptr, M.indptr) and np.array_equal(X.indices, M.indices)
    assert np.array_equal(X.data, M.data)
    for res in ((pt, br, sc), got[1:]):
        assert np.array_equal(res[0], want[1]) and list(res[1]) == list(want[2]) and np.array_equal(res[2], want[3])
    with zipfile.ZipFile(path) as z:
        assert z.testzip() is None
        for name, a in (("indptr", M.indptr.astype(idx)), ("indices", M.indices.astype(idx)), ("data", M.data)):
            assert z.read(name + ".npy") == _npy(a), name


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
            path = str(tmp_path / ("c%d_%s.npz" % (c, np.dtype(dt).name)))
            _same_file(call(dtype=dt, path=path, compress=True), call(dtype=dt), path, dt)
    X, pt, br, sc = sim.sample_density(t, 800, alpha=alpha, beta=beta, seed=3, device=DEV)
    dkw = dict(seed=4, device=DEV, sampler=sampler, out="csr")
    for dt in (np.int64, np.int32):
        path = str(tmp_path / ("d_%s.npz" % np.dtype(dt).name))
        got = sim.draw_counts(t, pt, br, sc, alpha, beta, dtype=dt, path=path, compress=True, **dkw)
        want = sim.draw_counts(t, pt, br, sc, alpha, beta, dtype=dt, **dkw)
        _same_file((got, pt, br, sc), (want, pt, br, sc), path, dt)
    np.random.seed(92)
    p = str(tmp_path / "r.npz")
    got = sim.sample_whole_tree_restricted(ptree_Tree(), seed=6, device=DEV, sampler=sampler, out="csr", path=p,
                                           compress=True)
    np.random.seed(92)
    _same_file(got, sim.sample_whole_tree_restricted(ptree_Tree(), seed=6, device=DEV, sampler=sampler, out="csr"), p)


def ptree_Tree():
    from prosstt_b200 import tree as ptree
    return ptree.Tree()


@gpu
@pytest.mark.parametrize("G", [1, 7, 70003])
def test_gene_counts(G, tmp_path):
    t, alpha, beta = _random_tree(G, T=4 if G > 65536 else 12, seed=G)
    n = 300 if G > 65536 else 900
    kw = dict(alpha=alpha, beta=beta, seed=5, device=DEV, out="csr")
    path = str(tmp_path / "g.npz")
    got = sim.sample_density(t, n, path=path, compress=True, **kw)
    want = sim.sample_density(t, n, **kw)
    if G > 65536:
        assert want[0].indices.max() >= 65536
    _same_file(got, want, path)


@gpu
def test_empty_rows_all_zero_result_and_no_cells(tmp_path):
    t, alpha, beta = _random_tree(7, seed=2)
    kw = dict(alpha=alpha, beta=beta, seed=3, device=DEV, out="csr")
    p = str(tmp_path / "sparse.npz")
    got = sim.sample_density(t, 2000, scale_mean=-5.0, path=p, compress=True, **kw)
    want = sim.sample_density(t, 2000, scale_mean=-5.0, **kw)
    assert (np.diff(want[0].indptr) == 0).sum() > 100 and want[0].nnz > 0
    _same_file(got, want, p)
    p = str(tmp_path / "zero.npz")
    zero = sim.sample_density(t, 500, scale_mean=-40.0, path=p, compress=True, **kw)
    assert zero[0].nnz == 0
    _same_file(zero, sim.sample_density(t, 500, scale_mean=-40.0, **kw), p)
    p = str(tmp_path / "none.npz")
    none = sim.sample_density(t, 0, path=p, compress=True, **kw)
    assert none[0].shape == (0, 7) and none[0].nnz == 0 and len(none[1]) == 0
    assert sp.load_npz(p).shape == (0, 7)


@gpu
def test_counts_above_65535_come_back_exactly(tmp_path):
    t, alpha, beta = _random_tree(64, T=6, seed=21, log_mean=9.0)
    kw = dict(alpha=alpha, beta=beta, seed=2, device=DEV, scale_mean=1.0, out="csr")
    for dt in (np.int64, np.int32):
        want = sim.sample_density(t, 600, dtype=dt, **kw)
        assert (want[0].data >= 65535).sum() > 100 and want[0].data.max() > 100000
        path = str(tmp_path / ("%s.npz" % np.dtype(dt).name))
        _same_file(sim.sample_density(t, 600, dtype=dt, path=path, compress=True, **kw), want, path, dt)


def _members(path):
    with zipfile.ZipFile(path) as z:
        return {n: z.read(n) for n in z.namelist()}


@gpu
def test_chunking_gives_identical_members_and_repeats_identical_files(lineage_tree, tmp_path, monkeypatch):
    t, alpha, beta = lineage_tree
    n = 1000
    eng, rows, sc = _engine(t, alpha, beta, n)
    want = eng.draw(rows, sc, 5, 77).cpu().numpy()
    cells = _cells(n)
    files = []
    for chunk in (1, 97, n, 5 * n):
        path = str(tmp_path / ("c%d.npz" % chunk))
        with formats.CsrNpzWriter(path, (n, t.G), *cells) as w:
            eng.stream_csr(rows, sc, 5, 77, lambda lo, hi, parts: [w.append(*p) for p in parts], w.index_dtype,
                           np.int64, chunk_cells=chunk, threads=3, compress=True)
        assert np.array_equal(formats.load_csr_shard(path)[0].toarray(), want)
        files.append(_members(path))
    assert all(f == files[0] for f in files[1:])
    eng.check()
    kw = dict(alpha=alpha, beta=beta, seed=31, device=DEV, out="csr", compress=True)
    sim.sample_density(t, 3001, path=str(tmp_path / "big.npz"), **kw)
    sim.sample_density(t, 3001, path=str(tmp_path / "again.npz"), **kw)
    assert open(str(tmp_path / "big.npz"), "rb").read() == open(str(tmp_path / "again.npz"), "rb").read()
    monkeypatch.setattr(pdev, "_STAGE_BYTES", 32 * t.G * 200)
    sim.sample_density(t, 3001, path=str(tmp_path / "small.npz"), **kw)
    assert _members(str(tmp_path / "big.npz")) == _members(str(tmp_path / "small.npz"))


@gpu
def test_compressed_size_matches_zlib_huffman_only(tmp_path):
    """Per streamed member, the file's compressed bytes against zlib's Huffman-only DEFLATE of the same bytes."""
    t, alpha, beta = _lineage_tree(2, 50, 10, 2000, seed=5)
    for m in (-2.0, 0.0):
        p = str(tmp_path / ("m%d.npz" % int(m)))
        rec = sim.sample_density(t, 40000, alpha=alpha, beta=beta, seed=8, device=DEV, scale_mean=m, out="csr",
                                 path=p, compress=True)[0]
        assert rec.nnz > 1e7
        with zipfile.ZipFile(p) as z:
            for name in ("indptr", "indices", "data"):
                raw = z.read(name + ".npy")
                c = zlib.compressobj(6, zlib.DEFLATED, -15, 9, zlib.Z_HUFFMAN_ONLY)
                ref = len(c.compress(raw) + c.flush())
                assert z.getinfo(name + ".npy").compress_size <= 1.02 * ref, (m, name, ref)


@gpu
@pytest.mark.parametrize("world", [2, 3])
def test_rank_files_stack_to_the_whole(world, lineage_tree, tmp_path):
    t, alpha, beta = lineage_tree
    kw = dict(alpha=alpha, beta=beta, seed=17, device=DEV, out="csr")
    whole = sim.sample_density(t, 1001, **kw)[0]
    stem = str(tmp_path / "sim")
    paths = [formats.shard_path(stem, r, world, suffix=".npz") for r in range(world)]
    for r, p in enumerate(paths):
        sim.sample_density(t, 1001, shard=(r, world), path=p, compress=True, **kw)
    assert sorted(os.listdir(tmp_path)) == sorted(os.path.basename(p) for p in paths)
    stacked = sp.vstack([sp.load_npz(p) for p in paths], format="csr")
    assert stacked.shape == whole.shape
    assert np.array_equal(stacked.indptr, whole.indptr) and np.array_equal(stacked.indices, whole.indices)
    assert np.array_equal(stacked.data, whole.data)


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
    p = str(tmp_path / "domain.npz")
    with pytest.raises(ValueError):                                  # a domain error in a later chunk
        with formats.CsrNpzWriter(p, (5000, t.G), *_cells(5000)) as w:
            eng.stream_csr(rows, sc, 1, 0, lambda lo, hi, parts: [w.append(*q) for q in parts], w.index_dtype,
                           np.int64, chunk_cells=100, compress=True)
    eng.flags.zero_()
    flat_p = str(tmp_path / "flat.npz")
    from prosstt_b200 import tree as ptree
    flat = ptree.Tree(topology=[], time={0: 1}, num_branches=1, branch_points=0, modules=1, G=4)
    flat.add_genes({0: np.array([[1.0, 2.0, 0.0, 3.0]])})
    with pytest.raises(ValueError):
        sim.draw_counts(flat, [0] * 5, [0] * 5, [1.0] * 5, 0.2, 2.0, seed=1, device=DEV, out="csr", path=flat_p,
                        compress=True)
    t2, alpha2, beta2 = lineage_tree
    with pytest.raises(ValueError):
        sim.sample_density(t2, 50, alpha2, beta2, seed=1, device=DEV, path=str(tmp_path / "nocsr.npz"), compress=True)
    with pytest.raises(ValueError):
        sim.sample_density(t2, 50, alpha2, beta2, seed=1, device=DEV, out="csr", compress=True)
    twice = str(tmp_path / "twice.npz")
    sim.sample_density(t2, 50, alpha2, beta2, seed=1, device=DEV, out="csr", path=twice, compress=True)
    with pytest.raises(FileExistsError):
        sim.sample_density(t2, 50, alpha2, beta2, seed=1, device=DEV, out="csr", path=twice, compress=True)
    assert sorted(os.listdir(tmp_path)) == ["twice.npz"]


@gpu
def test_host_memory_is_bounded_by_the_chunk(tmp_path):
    """~400 000 cells x 4000 genes: about 9e8 nonzeros, some 14 GB of int64 indices and data before compression."""
    if shutil.disk_usage(str(tmp_path)).free < (20 << 30):
        pytest.skip("needs ~20 GB of free space in the temporary directory")
    if not _reset_hwm() or _vm("VmHWM") is None:
        pytest.skip("the peak-RSS mark cannot be reset here")
    t, alpha, beta = _random_tree(4000, seed=8)
    kw = dict(alpha=alpha, beta=beta, seed=9, device=DEV, out="csr", compress=True)
    sim.sample_density(t, 1000, path=str(tmp_path / "warm.npz"), **kw)
    os.remove(str(tmp_path / "warm.npz"))
    path = str(tmp_path / "big.npz")
    _reset_hwm()
    base = _vm("VmRSS")
    rec = sim.sample_density(t, 400000, path=path, **kw)[0]
    peak = _vm("VmHWM") - base
    raw = rec.nnz * (rec.index_dtype.itemsize + rec.dtype.itemsize)
    assert rec.nnz > 5e8 and raw > 8e9
    assert peak < 0.1 * raw, (peak, raw)
    os.remove(path)


@gpu
def test_data_member_over_4_gib_reads_back(tmp_path):
    """About 6e8 int64 values: the data member is past 4 GiB, which only zip64 sizes can describe."""
    if shutil.disk_usage(str(tmp_path)).free < (20 << 30):
        pytest.skip("needs ~20 GB of free space in the temporary directory")
    t, alpha, beta = _random_tree(1000, seed=11, log_mean=2.0)
    path = str(tmp_path / "big.npz")
    rec = sim.sample_density(t, 700000, alpha=alpha, beta=beta, seed=4, device=DEV, out="csr", path=path,
                             compress=True)[0]
    assert rec.nnz * 8 > (4 << 30) and rec.index_dtype == np.int32
    with zipfile.ZipFile(path) as z:
        info = z.getinfo("data.npy")
        assert info.file_size > (4 << 30)
        assert z.testzip() is None
        with z.open("data.npy") as fh:
            np.lib.format.read_magic(fh)
            shape, _, dtype = np.lib.format.read_array_header_1_0(fh)
            assert shape == (rec.nnz,) and dtype == np.int64
        with z.open("indptr.npy") as fh:
            indptr = np.load(io.BytesIO(fh.read()))
    assert indptr[-1] == rec.nnz
    os.remove(path)
