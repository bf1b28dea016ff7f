"""out="zarr", path=...: an AnnData store in Zarr v2 format, X's chunks cut on the GPU across the engine's cell chunks
(pst_zarr_cut) and, with compress=True, compressed into one zlib stream each (pst_deflate_segments) before
formats.ZarrWriter writes them.  The reader here is written from the Zarr v2 and AnnData on-disk specifications with
json, zlib and NumPy only, so every byte of a store is checked without anndata or zarr; when anndata is installed,
anndata.read_zarr is checked too.  Without a GPU the writer is fed chunks made by Python's zlib."""
import json
import os
import struct
import zlib

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from prosstt_b200 import _native as nat
from prosstt_b200 import formats, simulation as sim
from prosstt_b200.device import TreeTables
from prosstt_b200.tree_utils import cell_params_frame
from test_csr_stream import _engine, _lineage_tree, _random_tree

DEV = "cuda:0"
SAMPLERS = ["gamma_poisson", "hybrid"]
gpu = pytest.mark.gpu
GROUPS = {"": ("anndata", "0.1.0"), "X": ("csr_matrix", "0.1.0"), "obs": ("dataframe", "0.2.0"),
          "obs/branches": ("categorical", "0.2.0"), "var": ("dataframe", "0.2.0"), "obsm": ("dict", "0.1.0"),
          "varm": ("dict", "0.1.0"), "obsp": ("dict", "0.1.0"), "varp": ("dict", "0.1.0"),
          "layers": ("dict", "0.1.0"), "uns": ("dict", "0.1.0")}


# ------------------------------------------------------------------ the reader (Zarr v2 + AnnData specifications)
def _json(path):
    with open(path, "rb") as fh:
        return json.loads(fh.read())


def read_array(store, key, chunk, compress, dtype=None, attrs=None):
    """The values of array `key`, checking its .zarray, its .zattrs and that padded tails are zeros (or "")."""
    folder = os.path.join(store, key)
    meta = _json(os.path.join(folder, ".zarray"))
    strings = dtype is None
    length = meta["shape"][0]
    assert meta == {"chunks": [chunk], "compressor": {"id": "zlib", "level": 1} if compress else None,
                    "dtype": "|O" if strings else np.dtype(dtype).str,
                    "fill_value": None if strings else (0.0 if np.dtype(dtype).kind == "f" else 0),
                    "filters": [{"id": "vlen-utf8"}] if strings else None, "order": "C", "shape": [length],
                    "zarr_format": 2}, (key, meta)
    if attrs is None:
        assert not os.path.exists(os.path.join(folder, ".zattrs"))
    else:
        assert _json(os.path.join(folder, ".zattrs")) == {"encoding-type": attrs, "encoding-version": "0.2.0"}
    files = sorted(f for f in os.listdir(folder) if not f.startswith("."))
    assert files == sorted(str(c) for c in range(-(-length // chunk))), (key, files)
    values = []
    for c in range(len(files)):
        with open(os.path.join(folder, str(c)), "rb") as fh:
            raw = fh.read()
        if compress:
            assert raw[:2] == b"\x78\x01" or key.startswith(("obs", "var"))
            raw = zlib.decompress(raw)
        keep = min(chunk, length - c * chunk)
        if strings:
            count, = struct.unpack_from("<I", raw)
            assert count == chunk
            at, items = 4, []
            for _ in range(count):
                size, = struct.unpack_from("<I", raw, at)
                items.append(raw[at + 4:at + 4 + size].decode("utf-8"))
                at += 4 + size
            assert at == len(raw) and all(v == "" for v in items[keep:])
            values += items[:keep]
        else:
            piece = np.frombuffer(raw, np.dtype(dtype))
            assert len(piece) == chunk and not piece[keep:].any(), key
            values.append(piece[:keep])
    if strings:
        return values
    return np.concatenate(values) if values else np.zeros(0, dtype)


def check_store(store, m, cells, compress, chunk, first=0, dtype=np.int64):
    """The whole store against the csr matrix m and the cells' (pseudotime, branches, scalings)."""
    n, G = m.shape
    meta = {}
    for root, dirs, files in os.walk(store):
        for f in files:
            if f.startswith(".") and f != ".zmetadata":
                key = os.path.relpath(os.path.join(root, f), store)
                meta[key] = _json(os.path.join(root, f))
    assert _json(os.path.join(store, ".zmetadata")) == {"metadata": meta, "zarr_consolidated_format": 1}
    groups = {os.path.dirname(k) for k in meta if k.endswith(".zgroup")}
    assert groups == set(GROUPS)
    for g, (kind, version) in GROUPS.items():
        key = os.path.join(g, ".zattrs")
        assert meta[os.path.join(g, ".zgroup")] == {"zarr_format": 2}
        assert {k: meta[key][k] for k in ("encoding-type", "encoding-version")} == {"encoding-type": kind,
                                                                                    "encoding-version": version}
    assert meta["X/.zattrs"]["shape"] == [n, G]
    assert meta["obs/.zattrs"] == {"_index": "_index", "column-order": ["pseudotime", "branches", "scalings"],
                                   "encoding-type": "dataframe", "encoding-version": "0.2.0"}
    assert meta["var/.zattrs"] == {"_index": "_index", "column-order": [], "encoding-type": "dataframe",
                                   "encoding-version": "0.2.0"}
    assert meta["obs/branches/.zattrs"]["ordered"] is False
    m = m.tocsr()
    m.sort_indices()
    indptr = read_array(store, "X/indptr", chunk, compress, "<i8")
    indices = read_array(store, "X/indices", chunk, compress, "<i4")
    data = read_array(store, "X/data", chunk, compress, np.dtype(dtype).newbyteorder("<"))
    assert np.array_equal(indptr, m.indptr) and np.array_equal(indices, m.indices)
    assert np.array_equal(data, m.data)
    frame = cell_params_frame(*cells, index=["cell_%d" % i for i in range(first, first + n)])
    assert read_array(store, "obs/_index", chunk, compress, None, "string-array") == list(frame.index)
    assert np.array_equal(read_array(store, "obs/pseudotime", chunk, compress, "<i8", "array"), frame["pseudotime"])
    assert np.array_equal(read_array(store, "obs/scalings", chunk, compress, "<f8", "array"), frame["scalings"])
    names = np.asarray(frame["branches"]).astype(str)
    cats, inv = np.unique(names, return_inverse=True)
    ct = np.int8 if len(cats) < 127 else np.int16
    assert read_array(store, "obs/branches/categories", chunk, compress, None, "string-array") == list(cats)
    assert np.array_equal(read_array(store, "obs/branches/codes", chunk, compress, ct, "array"), inv.reshape(-1))
    assert read_array(store, "var/_index", chunk, compress, None, "string-array") == ["gene_%d" % j for j in range(G)]
    _check_anndata(store, m, frame)


def _check_anndata(store, m, frame):
    try:
        import anndata
    except ImportError:
        return
    a = anndata.read_zarr(store)
    assert a.shape == m.shape and (sp.csr_matrix(a.X) != m).nnz == 0
    assert list(a.obs_names) == list(frame.index) and list(a.var_names) == ["gene_%d" % j for j in range(m.shape[1])]
    assert np.array_equal(a.obs["pseudotime"], frame["pseudotime"])
    assert np.array_equal(a.obs["scalings"], frame["scalings"])
    assert list(a.obs["branches"].astype(str)) == list(np.asarray(frame["branches"]).astype(str))


def test_anndata_round_trip(tmp_path):
    """anndata.read_zarr of a store the writer makes (skipped where anndata is not installed)."""
    pytest.importorskip("anndata")
    m = _random_csr(40, 9, 1)
    for compress in (False, True):
        p = str(tmp_path / ("a%d" % compress))
        _write(p, m, [(0, 40)], compress, chunk=8192, cells=_cells(40))
        frame = cell_params_frame(*_cells(40))
        _check_anndata(p, m, frame)


# ------------------------------------------------------------------ the writer, fed by zlib
def _random_csr(n, G, seed, dtype=np.int64, density=0.3):
    rng = np.random.RandomState(seed)
    d = rng.poisson(3.0, (n, G)) * (rng.random_sample((n, G)) < density)
    d[rng.random_sample(n) < 0.2] = 0
    return sp.csr_matrix(d.astype(dtype))


def _cells(n, seed=0):
    rng = np.random.RandomState(seed)
    return (rng.randint(0, 50, n).astype(np.int64), np.array(["1", "10", "2"] * n)[:n],
            rng.random_sample(n) * 2)


def feed(w, m, bounds, compress, chunk, dtype=np.int64):
    """Append the csr matrix m to w in the row chunks `bounds`, cutting each array into Zarr chunks as the engine does:
    the complete chunks of every append, the tail padded by the last one."""
    arrays = [m.indptr.astype("<i8"), m.indices.astype("<i4"), m.data.astype(np.dtype(dtype).newbyteorder("<"))]
    done = [0, 0, 0]
    for i, (lo, hi) in enumerate(bounds):
        final = i == len(bounds) - 1
        ends = (hi + 1, m.indptr[hi], m.indptr[hi])
        parts = []
        for j, a in enumerate(arrays):
            upto = int(ends[j]) if final else int(ends[j]) // chunk * chunk
            raw = a[done[j]:upto].tobytes()
            parts.append(formats.zarr_chunks(raw, chunk * a.itemsize, compress))
            done[j] = upto
        w.append(hi - lo, int(m.indptr[hi] - m.indptr[lo]), parts)


def _write(path, m, bounds, compress, chunk, cells=None, first=0, dtype=np.int64):
    old = formats.ZARR_CHUNK
    formats.ZARR_CHUNK = chunk
    try:
        with formats.ZarrWriter(path, m.shape, *(cells or _cells(m.shape[0])), first=first, dtype=dtype,
                                compress=compress) as w:
            feed(w, m, bounds, compress, chunk, dtype)
    finally:
        formats.ZARR_CHUNK = old
    return w.record()


def _files(store):
    out = {}
    for root, _, files in os.walk(store):
        for f in files:
            with open(os.path.join(root, f), "rb") as fh:
                out[os.path.relpath(os.path.join(root, f), store)] = fh.read()
    return out


@pytest.mark.parametrize("compress", [False, True])
@pytest.mark.parametrize("dtype", [np.int64, np.int32])
def test_writer_round_trip(tmp_path, compress, dtype):
    m = _random_csr(20000, 7, 3, dtype)
    cells = _cells(20000)
    bounds = [(0, 1), (1, 4000), (4000, 4000), (4000, 13111), (13111, 20000)]
    p = str(tmp_path / "s")
    rec = _write(p, m, bounds, compress, 8192, cells, first=70, dtype=dtype)
    assert rec == formats.ZarrRecord(p, m.shape, m.nnz, rec.nbytes, compress) and rec.nbytes > 0
    check_store(p, m, cells, compress, 8192, first=70, dtype=dtype)
    assert len(os.listdir(os.path.join(p, "X", "data"))) > 3
    loaded = rec.load()
    assert loaded.dtype == np.dtype(dtype) and (loaded != m).nnz == 0
    q = str(tmp_path / "again")
    _write(q, m, [(0, 20000)], compress, 8192, cells, first=70, dtype=dtype)
    assert _files(p) == _files(q)                          # the same store whatever the appends


@pytest.mark.parametrize("compress", [False, True])
def test_empty_shapes(tmp_path, compress):
    for n, G in ((0, 5), (6, 0), (0, 0), (3, 4)):
        m = sp.csr_matrix((n, G), dtype=np.int64)
        p = str(tmp_path / ("e%d_%d_%d" % (n, G, compress)))
        rec = _write(p, m, [(0, n)] if n else [], compress, 8192, _cells(n))
        check_store(p, m, _cells(n), compress, 8192)
        assert sorted(os.listdir(os.path.join(p, "X", "indptr"))) == [".zarray", "0"]
        if m.nnz == 0:
            assert sorted(os.listdir(os.path.join(p, "X", "data"))) == [".zarray"]
        assert rec.load().shape == (n, G)


@pytest.mark.parametrize("compress", [False, True])
def test_failed_writes_leave_nothing(tmp_path, compress):
    m = _random_csr(100, 5, 2)
    p = str(tmp_path / "s")
    with pytest.raises(RuntimeError):
        with formats.ZarrWriter(p, m.shape, *_cells(100), compress=compress) as w:
            w.append(50, 0, [[], [], []])
            raise RuntimeError("boom")
    assert os.listdir(tmp_path) == []
    w = formats.ZarrWriter(p, m.shape, *_cells(100), compress=compress)
    w.append(100, m.nnz, [[], [], []])
    with pytest.raises(ValueError):                        # the chunks are missing
        w.close()
    assert os.listdir(tmp_path) == []
    w = formats.ZarrWriter(p, m.shape, *_cells(100), compress=compress)
    with pytest.raises(ValueError):                        # a short chunk
        w.append(1, 0, [[b"\0" * 8] if not compress else [(b"", 1, 8)], [], []])
    w.abort()
    assert os.listdir(tmp_path) == []
    with pytest.raises(ValueError):                        # rows missing
        with formats.ZarrWriter(p, m.shape, *_cells(100), compress=compress) as w:
            w.append(10, 0, [[], [], []])
    assert os.listdir(tmp_path) == []
    _write(p, m, [(0, 100)], compress, 8192)
    with pytest.raises(FileExistsError):
        formats.ZarrWriter(p, m.shape, *_cells(100))
    assert os.listdir(tmp_path) == ["s"]


def test_zarr_argument_errors():
    for kw in (dict(), dict(path="p", host_out=(1,)), dict(path="p", compression="lz77")):
        with pytest.raises(ValueError):
            sim._check_csr_request("zarr", np.int64, **kw)
    with pytest.raises(ValueError):
        sim._check_csr_request("zarr", np.uint16, path="p")
    with pytest.raises(ValueError, match="AnnData Zarr store"):
        sim._check_csr_request("zarr", np.int64)
    sim._check_csr_request("zarr", np.int32, path="p", compress=True, compression="lz77")


def test_zarr_symbols_declared_and_exported():
    header = open(os.path.join(os.path.dirname(__file__), "..", "include", "prosstt_b200.h")).read()
    lib = nat.load()
    for name in ("pst_deflate_segments", "pst_deflate_lz_segments", "pst_zarr_cut", "pst_zarr_seg_bytes"):
        assert name + "(" in header and name in nat._SIGNATURES and getattr(lib, name) is not None
    assert lib.pst_abi_version() == 2
    assert lib.pst_zarr_seg_bytes(0, 32768) == 65536 and lib.pst_zarr_seg_bytes(100000, 32768) == 5 * 32768


# ------------------------------------------------------------------ the kernels
def _segments(data, length, seg_blocks, block, lz):
    """(compressed bytes, seg_offsets, seg_adler) of pst_deflate_segments over the first `length` of data, the launch
    sized for all of it."""
    dev = torch.device(DEV)
    st = nat.stream_ptr(dev)
    lib = nat.load()
    x = torch.from_numpy(np.frombuffer(data, np.uint8).copy()).to(dev)
    nb = -(-len(data) // block)
    nseg = -(-nb // seg_blocks)
    count = torch.tensor([length], dtype=torch.int64, device=dev)
    out = torch.zeros(int(lib.pst_deflate_bound(len(data), block)), dtype=torch.uint8, device=dev)
    out_bytes = torch.zeros(1, dtype=torch.int64, device=dev)
    offs = torch.full((nseg + 1,), -1, dtype=torch.int64, device=dev)
    adler = torch.zeros(nseg, dtype=torch.int32, device=dev)
    work_fn = "pst_deflate_lz_workspace_bytes" if lz else "pst_deflate_workspace_bytes"
    work = torch.empty(int(getattr(lib, work_fn)(len(data), block)), dtype=torch.uint8, device=dev)
    nat.call("pst_deflate_lz_segments" if lz else "pst_deflate_segments", x, count, 1, len(data), block, seg_blocks,
             out, out_bytes, offs, adler, work, work.numel(), st)
    total = int(out_bytes.item())
    return out[:total].cpu().numpy().tobytes(), offs.cpu().numpy(), adler.cpu().numpy().view(np.uint32)


@gpu
@pytest.mark.parametrize("lz", [False, True])
def test_segments_are_zlib_streams(lz):
    rng = np.random.RandomState(5)
    block = 32768
    inputs = [rng.randint(0, 256, 9 * block + 1000).astype(np.uint8).tobytes(), b"\xff" * (8 * block),
              bytes(8 * block), (np.arange(7 * block + 77) % 7).astype(np.uint8).tobytes()]
    for data in inputs:
        for seg_blocks in (1, 2, 3):
            for length in (len(data), len(data) - 1000, 2 * block + 5, block * seg_blocks, 0):
                blocks, offs, adler = _segments(data, length, seg_blocks, block, lz)
                seg_bytes = seg_blocks * block
                assert offs[0] == 0 and offs[-1] == len(blocks) and np.all(np.diff(offs) >= 0)
                for s in range(len(adler)):
                    raw = data[s * seg_bytes:min(length, (s + 1) * seg_bytes)] if s * seg_bytes < length else b""
                    if not raw:
                        assert offs[s + 1] == offs[s]
                        continue
                    assert int(adler[s]) == zlib.adler32(raw), (s, length, seg_blocks)
                    stream = b"\x78\x01" + blocks[offs[s]:offs[s + 1]] + b"\x03\x00" + struct.pack(">I", int(adler[s]))
                    assert zlib.decompress(stream) == raw


@gpu
def test_cut_carries_across_calls():
    dev = torch.device(DEV)
    st = nat.stream_ptr(dev)
    lib = nat.load()
    rng = np.random.RandomState(2)
    chunk = 32768
    values = rng.randint(-2 ** 31, 2 ** 31, 300000).astype(np.int32)
    sizes = [0, 5, 8191, 8192, 8193, 100000, 1, 0, 60000]
    sizes.append(len(values) - sum(sizes))
    most = max(sizes) * 4 + 64
    seg_bytes = int(lib.pst_zarr_seg_bytes(most, chunk))
    seg = [torch.full((seg_bytes,), 0xEE, dtype=torch.uint8, device=dev) for _ in range(2)]
    state = torch.zeros((2, 2), dtype=torch.int64, device=dev)
    prev, prev_state = torch.zeros(16, dtype=torch.uint8, device=dev), torch.zeros(2, dtype=torch.int64, device=dev)
    src = torch.empty(most, dtype=torch.uint8, device=dev)
    nchunks = torch.zeros(1, dtype=torch.int64, device=dev)
    got, at = [], 0
    for i, size in enumerate(sizes):
        k = i & 1
        src[:size * 4] = torch.from_numpy(values[at:at + size].view(np.uint8).copy()).to(dev)
        count = torch.tensor([size], dtype=torch.int64, device=dev)
        final = int(i == len(sizes) - 1)
        nat.call("pst_zarr_cut", prev, prev_state, src, count, 4, most, chunk, final, seg[k], seg_bytes, state[k],
                 nchunks, st)
        whole = int(nchunks.item())
        got.append(seg[k][:whole * chunk].cpu().numpy().tobytes())
        prev, prev_state = seg[k], state[k]
        at += size
    raw = b"".join(got)
    assert len(raw) == -(-len(values) * 4 // chunk) * chunk
    assert raw[:len(values) * 4] == values.tobytes() and not any(raw[len(values) * 4:])


# ------------------------------------------------------------------ end to end
@pytest.fixture(scope="module")
def lineage_tree():
    return _lineage_tree(2, 20, 6, 1000, seed=3)


def _same(got, want, path, chunk, compress=False, first=0, dtype=np.int64):
    """An out="zarr" call's (X, pseudotime, branches, scalings) against the out="csr" call."""
    rec, m = got[0], want[0]
    assert isinstance(rec, formats.ZarrRecord) and rec.path == path and rec.shape == m.shape
    assert rec.nnz == m.nnz and rec.compressed == compress
    for a, b in zip(got[1:], want[1:]):
        assert list(a) == list(b)
    check_store(path, m, tuple(want[1:]), compress, chunk, first, dtype)
    loaded = rec.load()
    assert loaded.dtype == np.dtype(dtype) and (loaded != m).nnz == 0


@pytest.fixture
def small_chunks(monkeypatch):
    monkeypatch.setattr(formats, "ZARR_CHUNK", 8192)
    return 8192


ARMS = [(False, "huffman"), (True, "huffman"), (True, "lz77")]


@gpu
@pytest.mark.parametrize("sampler", SAMPLERS)
def test_every_entry_point_writes_the_csr_counts(sampler, lineage_tree, tmp_path, small_chunks):
    t, alpha, beta = lineage_tree
    kw = dict(alpha=alpha, beta=beta, seed=12, device=DEV, sampler=sampler)
    calls = [
        lambda **o: sim.sample_density(t, 1500, **kw, **o),
        lambda **o: sim.sample_whole_tree(t, 7, **kw, **o),
        lambda **o: sim.sample_pseudotime_series(t, [300, 400], [5, 30], 4.0, **kw, **o),
    ]
    for c, call in enumerate(calls):
        for dtype in (np.int64, np.int32):
            want = call(out="csr", dtype=dtype)
            for compress, compression in ARMS:
                path = str(tmp_path / ("c%d_%d_%s_%d" % (c, compress, compression, np.dtype(dtype).itemsize)))
                got = call(out="zarr", path=path, compress=compress, compression=compression, dtype=dtype)
                _same(got, want, path, small_chunks, compress, dtype=dtype)
    X, pt, br, sc = sim.sample_density(t, 800, alpha=alpha, beta=beta, seed=3, device=DEV)
    dkw = dict(seed=4, device=DEV, sampler=sampler, first=5000)
    want = sim.draw_counts(t, pt, br, sc, alpha, beta, out="csr", **dkw)
    for compress, compression in ARMS:
        path = str(tmp_path / ("d%d_%s" % (compress, compression)))
        got = sim.draw_counts(t, pt, br, sc, alpha, beta, out="zarr", path=path, compress=compress,
                              compression=compression, **dkw)
        _same((got, pt, br, sc), (want, pt, br, sc), path, small_chunks, compress, first=5000)


@gpu
def test_default_chunk_and_compressors(lineage_tree, tmp_path):
    t, alpha, beta = lineage_tree
    kw = dict(alpha=alpha, beta=beta, seed=8, device=DEV)
    want = sim.sample_density(t, 4000, out="csr", **kw)
    recs = []
    for compress, compression in ARMS:
        p = str(tmp_path / ("%d%s" % (compress, compression)))
        got = sim.sample_density(t, 4000, out="zarr", path=p, compress=compress, compression=compression, **kw)
        _same(got, want, p, formats.ZARR_CHUNK, compress)
        recs.append(got[0])
    assert recs[2].nbytes < recs[1].nbytes < recs[0].nbytes, [r.nbytes for r in recs]


@gpu
def test_engine_chunking_leaves_no_trace(lineage_tree, tmp_path, small_chunks):
    t, alpha, beta = lineage_tree
    eng, rows, sc = _engine(t, alpha, beta, 3001)
    cells = _cells(3001)
    for compress, compression in ARMS:
        stores = []
        for chunk_cells in (None, 1, 37, 1000):
            p = str(tmp_path / ("s%d%s%s" % (compress, compression, chunk_cells)))
            with formats.ZarrWriter(p, (3001, t.G), *cells, compress=compress) as w:
                eng.stream_csr(rows, sc, 31, 0, lambda lo, hi, *a: w.append(hi - lo, *a), zarr=True,
                               compress=compress, compression=compression, chunk_cells=chunk_cells)
            stores.append(_files(p))
        assert len(stores[0]) > 20
        for s in stores[1:]:
            assert s == stores[0]
    eng.check()
    m = sp.csr_matrix(eng.draw(rows, sc, 31, 0).cpu().numpy().astype(np.int64))
    check_store(p, m, cells, True, small_chunks)



@gpu
def test_indptr_spans_several_zarr_chunks(lineage_tree, tmp_path, small_chunks):
    """More cells than a Zarr chunk: indptr (the leading 0 and one value per cell) fills chunks of its own, also for
    a cell count that is a multiple of the chunk, where the leading 0 alone makes one more chunk."""
    t, alpha, beta = lineage_tree
    kw = dict(alpha=alpha, beta=beta, seed=21, device=DEV)
    for n in (2 * small_chunks, 2 * small_chunks - 1, small_chunks + 5):
        want = sim.sample_density(t, n, out="csr", **kw)
        for compress, compression in ARMS:
            path = str(tmp_path / ("n%d_%d%s" % (n, compress, compression)))
            got = sim.sample_density(t, n, out="zarr", path=path, compress=compress, compression=compression, **kw)
            _same(got, want, path, small_chunks, compress)
            assert len([f for f in os.listdir(os.path.join(path, "X", "indptr")) if f[0] != "."]) == \
                n // small_chunks + 1
    # engine chunks that end at every row, at rows C - 1 and C, and across them
    t2, alpha2, beta2 = _random_tree(12, seed=6)
    n = small_chunks + 3
    eng, rows, sc = _engine(t2, alpha2, beta2, n)
    cells = _cells(n)
    m = sp.csr_matrix(eng.draw(rows, sc, 5, 0).cpu().numpy().astype(np.int64))
    stores = []
    for chunk_cells in (None, 1, 37, small_chunks - 1, small_chunks):
        p = str(tmp_path / ("c%s" % chunk_cells))
        with formats.ZarrWriter(p, (n, t2.G), *cells) as w:
            eng.stream_csr(rows, sc, 5, 0, lambda lo, hi, *a: w.append(hi - lo, *a), zarr=True, chunk_cells=chunk_cells)
        stores.append(_files(p))
    eng.check()
    check_store(p, m, cells, False, small_chunks)
    for s in stores[1:]:
        assert s == stores[0]

@gpu
def test_rank_stores_concatenate_to_the_whole(lineage_tree, tmp_path, small_chunks):
    t, alpha, beta = lineage_tree
    kw = dict(alpha=alpha, beta=beta, seed=17, device=DEV, out="zarr", compress=True)
    whole = str(tmp_path / "whole")
    m = sim.sample_density(t, 1001, path=whole, **kw)[0].load()
    for world in (2, 3):
        stem = str(tmp_path / ("sim%d" % world))
        paths = [formats.shard_path(stem, r, world, suffix="") for r in range(world)]
        parts = []
        for r, p in enumerate(paths):
            rec = sim.sample_density(t, 1001, shard=(r, world), path=p, **kw)[0]
            lo, hi = sim.shard_range(1001, r, world)
            assert rec.shape == (hi - lo, t.G)
            assert read_array(p, "obs/_index", small_chunks, True, None, "string-array") == \
                ["cell_%d" % i for i in range(lo, hi)]
            parts.append(rec.load())
        assert (sp.vstack(parts).tocsr() != m).nnz == 0


@gpu
def test_no_cells_and_no_genes(tmp_path):
    t, alpha, beta = _random_tree(7, seed=2)
    kw = dict(alpha=alpha, beta=beta, seed=3, device=DEV)
    for compress in (False, True):
        p = str(tmp_path / ("none%d" % compress))
        got = sim.sample_density(t, 0, out="zarr", path=p, compress=compress, **kw)
        _same(got, sim.sample_density(t, 0, out="csr", **kw), p, formats.ZARR_CHUNK, compress)
    from prosstt_b200 import tree as ptree
    flat = ptree.Tree(topology=[], time={0: 3}, num_branches=1, branch_points=0, modules=1, G=0)
    flat.add_genes({0: np.zeros((3, 0))})
    for compress in (False, True):
        p = str(tmp_path / ("g0_%d" % compress))
        got = sim.draw_counts(flat, [0, 1, 2, 1], [0] * 4, [1.0] * 4, 0.2, 2.0, seed=1, device=DEV, out="zarr",
                              path=p, compress=compress, first=98)
        assert got.shape == (4, 0) and got.nnz == 0
        check_store(p, sp.csr_matrix((4, 0), dtype=np.int64), ([0, 1, 2, 1], [0] * 4, [1.0] * 4), compress,
                    formats.ZARR_CHUNK, first=98)


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
        with formats.ZarrWriter(p, (5000, t.G), *_cells(5000), compress=compress) as w:
            eng.stream_csr(rows, sc, 1, 0, lambda lo, hi, *a: w.append(hi - lo, *a), zarr=True, compress=compress,
                           chunk_cells=100)
    eng.flags.zero_()
    t2, alpha2, beta2 = lineage_tree
    twice = str(tmp_path / "twice")
    sim.sample_density(t2, 50, alpha2, beta2, seed=1, device=DEV, out="zarr", path=twice, compress=compress)
    with pytest.raises(FileExistsError):
        sim.sample_density(t2, 50, alpha2, beta2, seed=1, device=DEV, out="zarr", path=twice, compress=compress)
    assert sorted(os.listdir(tmp_path)) == ["twice"]
