"""compression="lz77": LZ77 matching in the GPU DEFLATE (pst_deflate_lz_blocks) for the compressed `.npz`
(out="csr", path=..., compress=True) and the 10x directory (out="mtx", path=...).  The kernel is checked against
zlib's decoder and a small Python decoder that lists each block's tokens and code lengths; the files must hold the
same content as the Huffman-only calls, in fewer bytes."""
import gzip
import os
import shutil
import subprocess
import zipfile
import zlib

import numpy as np
import pytest
import scipy.io
import scipy.sparse as sp
import torch

from prosstt_b200 import _native as nat
from prosstt_b200 import device as pdev, formats, simulation as sim
from prosstt_b200.device import CountEngine, TreeTables
from test_csr_stream import _cells, _engine, _lineage_tree, _random_tree

DEV = "cuda:0"
SAMPLERS = ["gamma_poisson", "hybrid"]
FILES = ["barcodes.tsv.gz", "cellparams.tsv.gz", "features.tsv.gz", "matrix.mtx.gz"]
NEW_SYMBOLS = ("pst_deflate_lz_workspace_bytes", "pst_deflate_lz_blocks")
gpu = pytest.mark.gpu

LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195,
            227, 258]
LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
             4097, 6145, 8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0] + [i // 2 for i in range(2, 28)]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]


# ------------------------------------------------------------------ arguments and symbols (no GPU)
def test_lz77_argument_errors():
    bad = [dict(out="csr"), dict(out="csr", path="p"), dict(out="numpy"), dict(out="torch"),
           dict(out="numpy", path="p")]
    for kw in bad:                                                   # outputs the GPU does not compress
        with pytest.raises(ValueError, match="lz77"):
            sim._check_csr_request(kw["out"], np.int64, path=kw.get("path"), compression="lz77")
    for out, kw in (("mtx", dict(path="p")), ("csr", dict(path="p.npz", compress=True))):
        with pytest.raises(ValueError, match="compression"):
            sim._check_csr_request(out, np.int64, compression="zstd", **kw)
        with pytest.raises(ValueError, match="compression"):
            sim._check_csr_request(out, np.int64, compression=None, **kw)
        sim._check_csr_request(out, np.int64, compression="lz77", **kw)
        sim._check_csr_request(out, np.int64, compression="huffman", **kw)
    # the rules of compress= and out="mtx" still hold with lz77
    for out, kw in (("mtx", dict()), ("mtx", dict(path="p", compress=True)), ("csr", dict(compress=True)),
                    ("numpy", dict(path="p.npz", compress=True)), ("mtx", dict(path="p", host_out=1))):
        with pytest.raises(ValueError):
            sim._check_csr_request(out, np.int64, compression="lz77", **kw)
    with pytest.raises(ValueError):
        sim._check_csr_request("mtx", np.uint16, path="p", compression="lz77")


def test_lz77_symbols_declared_and_exported():
    header = open(os.path.join(os.path.dirname(__file__), "..", "include", "prosstt_b200.h")).read()
    lib = nat.load()
    for name in NEW_SYMBOLS:
        assert name + "(" in header and name in nat._SIGNATURES
        assert getattr(lib, name) is not None
    assert lib.pst_abi_version() == 2
    for n, block in ((0, 32768), (1, 1024), (100003, 32768), (100003, 4096)):
        plain = lib.pst_deflate_workspace_bytes(n, block)
        nb = (n + block - 1) // block
        assert lib.pst_deflate_lz_workspace_bytes(n, block) == plain + 2 * block * nb
    assert lib.pst_deflate_lz_workspace_bytes(-1, 32768) == -1


# ------------------------------------------------------------------ a DEFLATE decoder that keeps the tokens
class _Bits:
    def __init__(self, data):
        self.data, self.pos = data, 0

    def get(self, n):
        v = 0
        for i in range(n):
            v |= ((self.data[self.pos >> 3] >> (self.pos & 7)) & 1) << i
            self.pos += 1
        return v


def _canonical(lengths):
    count = [0] * 16
    for l in lengths:
        count[l] += 1
    count[0] = 0
    code, nxt = 0, [0] * 16
    for l in range(1, 16):
        code = (code + count[l - 1]) << 1
        nxt[l] = code
    table = {}
    for s, l in enumerate(lengths):
        if l:
            table[(l, nxt[l])] = s
            nxt[l] += 1
    return table


def _sym(br, table):
    code = 0
    for l in range(1, 16):
        code = (code << 1) | br.get(1)
        if (l, code) in table:
            return table[(l, code)]
    raise AssertionError("invalid Huffman code")


def _blocks(comp):
    """The blocks of a pst_deflate*_blocks output: (kind, lit/len lengths, distance lengths, tokens, bytes); a
    token is a literal byte or (length, distance).  The empty stored blocks of the sync flushes are left out."""
    br, out = _Bits(comp), []
    while br.pos + 8 <= 8 * len(comp):
        assert br.get(1) == 0                                        # never final
        kind = br.get(2)
        if kind == 0:
            br.pos = (br.pos + 7) & ~7
            n = br.get(16)
            assert br.get(16) == n ^ 0xFFFF
            raw = bytes(comp[br.pos // 8:br.pos // 8 + n])
            br.pos += 8 * n
            if n:
                out.append(("stored", None, None, list(raw), raw))
            continue
        assert kind == 2
        hlit, hdist, hclen = br.get(5) + 257, br.get(5) + 1, br.get(4) + 4
        cl = [0] * 19
        for i in range(hclen):
            cl[CL_ORDER[i]] = br.get(3)
        ctab, lens = _canonical(cl), []
        while len(lens) < hlit + hdist:
            s = _sym(br, ctab)
            if s < 16:
                lens.append(s)
            elif s == 16:
                lens += [lens[-1]] * (3 + br.get(2))
            elif s == 17:
                lens += [0] * (3 + br.get(3))
            else:
                lens += [0] * (11 + br.get(7))
        lit, dist = lens[:hlit], lens[hlit:]
        ltab, dtab = _canonical(lit), _canonical(dist)
        toks, buf = [], bytearray()
        while True:
            s = _sym(br, ltab)
            if s < 256:
                toks.append(s)
                buf.append(s)
            elif s == 256:
                break
            else:
                length = LEN_BASE[s - 257] + br.get(LEN_EXTRA[s - 257])
                ds = _sym(br, dtab)
                d = DIST_BASE[ds] + br.get(DIST_EXTRA[ds])
                assert d <= len(buf), "a match reaches back past its block"
                for _ in range(length):
                    buf.append(buf[-d])
                toks.append((length, d))
        out.append(("dynamic", lit, dist, toks, bytes(buf)))
    return out


def _len_code(length):
    return max(i for i, b in enumerate(LEN_BASE) if b <= length) if length < 258 else 28


def _dist_code(d):
    return max(i for i, b in enumerate(DIST_BASE) if b <= d)


# ------------------------------------------------------------------ the kernel
def _run(name, data, block=32768, count=None, scale=1, offset=0, max_bytes=None):
    """(compressed bytes, crc) of `name` over data (at `offset` bytes into a device buffer)."""
    lib = nat.load()
    n = len(data) if max_bytes is None else max_bytes
    buf = np.zeros(offset + max(len(data), n, 16), np.uint8)
    buf[offset:offset + len(data)] = np.frombuffer(data, np.uint8)
    x = torch.from_numpy(buf).to(DEV)[offset:]
    out = torch.empty(max(1, lib.pst_deflate_bound(n, block)), dtype=torch.uint8, device=DEV)
    ws = int((lib.pst_deflate_lz_workspace_bytes if "lz" in name else lib.pst_deflate_workspace_bytes)(n, block))
    work = torch.empty(max(1, ws), dtype=torch.uint8, device=DEV)
    size = torch.full((1,), -1, dtype=torch.int64, device=DEV)
    crc = torch.zeros(2, dtype=torch.int32, device=DEV)
    cnt = None if count is None else torch.tensor([count], dtype=torch.int64, device=DEV)
    nat.call(name, x, cnt, scale, n, block, out, size, crc, work, ws, nat.stream_ptr(torch.device(DEV)))
    k = int(size.item())
    assert 0 <= k <= lib.pst_deflate_bound(n, block)
    return out[:k].cpu().numpy().tobytes(), int(crc[0].item()) & 0xFFFFFFFF


def _lz(data, **kw):
    return _run("pst_deflate_lz_blocks", data, **kw)


def _check(data, block=32768, **kw):
    comp, crc = _lz(data, block=block, **kw)
    assert zlib.decompress(comp + b"\x03\x00", -15) == data
    assert crc == zlib.crc32(data)
    return comp


def _zlib_blocks(data, level, block=32768):
    """Bytes of zlib at `level` over independent sync-flushed blocks of `block` bytes: the kernels' framing."""
    total = 0
    for i in range(0, len(data), block):
        c = zlib.compressobj(level, zlib.DEFLATED, -15)
        total += len(c.compress(data[i:i + block]) + c.flush(zlib.Z_SYNC_FLUSH))
    return total


@gpu
def test_lz_small_and_odd_inputs_decode_with_zlib():
    rng = np.random.RandomState(1)
    text = b"".join(b"%d %d %d\n" % (g, c, v) for c in range(1, 40) for g, v in
                    zip(np.sort(rng.choice(20000, 300, replace=False)) + 1, rng.randint(1, 30, 300)))
    assert _lz(b"") == (b"", 0)
    for data in (b"\x05", b"ab", b"abc", b"abcabcabc", text[:5], text[:7], text[:13], text[:1001], text[:32767],
                 text[:32768], text[:32769], text[:100003]):
        for offset in (0, 1, 3, 7):                                  # unaligned input pointers
            _check(data, offset=offset)
    # the length from device memory, count x scale, clamped to max_bytes
    data = text[:80000]
    comp, crc = _lz(data, count=1001, scale=8, max_bytes=80000)
    assert zlib.decompress(comp + b"\x03\x00", -15) == data[:8008] and crc == zlib.crc32(data[:8008])
    comp, crc = _lz(data[:50000], count=10 ** 9, scale=8, max_bytes=50000)
    assert zlib.decompress(comp + b"\x03\x00", -15) == data[:50000] and crc == zlib.crc32(data[:50000])
    comp, crc = _lz(data, count=0, scale=8, max_bytes=80000)
    assert comp == b"" and crc == 0
    # outputs concatenate
    a, _ = _lz(data[:16384])
    b, _ = _lz(data[16384:])
    assert zlib.decompress(a + b + b"\x03\x00", -15) == data


@gpu
def test_lz_every_block_size():
    rng = np.random.RandomState(2)
    counts = np.minimum(rng.negative_binomial(0.5, 0.1, size=30000), 70000).astype(np.int64).tobytes()
    text = b"".join(b"%d %d %d\n" % (g, g // 7 + 1, v) for g, v in zip(range(1, 12000), rng.randint(1, 9, 12000)))
    for block in range(1024, 32769, 1024):
        for data in (counts[:100000], text[:70001]):
            comp = _check(data, block=block)
            for kind, lit, dist, toks, raw in _blocks(comp):
                if kind == "dynamic":
                    assert all(isinstance(t, int) or t[1] <= block for t in toks)


@gpu
def test_lz_random_bytes_are_stored_and_zeros_use_258_at_distance_1():
    rng = np.random.RandomState(3)
    data = rng.bytes(3 * 32768 + 11)
    for block in (32768, 1024):
        comp = _check(data, block=block)
        assert len(comp) == len(data) + 5 * ((len(data) + block - 1) // block)
    zeros = bytes(100000)
    comp = _check(zeros)
    assert len(comp) < 2000
    toks = [t for b in _blocks(comp) for t in b[3]]
    assert (258, 1) in toks and all(t == 0 or t[1] == 1 for t in toks)


@gpu
def test_lz_every_length_and_distance_code():
    rng = np.random.RandomState(4)
    # per block random bytes, then a copy of each of their slices, each followed by a random byte: matches of
    # every length 3..258.  Each copy has a source of its own, so its nearest earlier occurrence is its whole length.
    data = b""
    for group in (list(range(3, 11)) * 4 + list(range(11, 151)), range(151, 211), list(range(211, 258)) + [258] * 6):
        pre = rng.bytes(sum(group))
        blk, at = bytearray(pre), 0
        for length in group:
            blk += pre[at:at + length] + rng.bytes(1)
            at += length
        data += bytes(blk) + rng.bytes(32768 - len(blk))
    comp = _check(data)
    lcodes = {_len_code(t[0]) for b in _blocks(comp) for t in b[3] if isinstance(t, tuple)}
    assert lcodes == set(range(29))
    # per block: a random period of d bytes repeated, for distances at the base of every code
    for block in (32768, 4096):
        seen = set()
        for d in [x for x in DIST_BASE if x < block] + [block - 1]:
            r = rng.bytes(d)
            blk = (r * (block // d + 2))[:block]
            comp = _check(blk, block=block)
            seen |= {_dist_code(t[1]) for b in _blocks(comp) for t in b[3] if isinstance(t, tuple)}
        assert seen == {c for c, x in enumerate(DIST_BASE) if x < block}, block


def _fibonacci_bytes(n, rng):
    f = [1, 2]
    while sum(f) + f[-1] + f[-2] <= n:
        f.append(f[-1] + f[-2])
    vals = np.concatenate([np.full(c, 7 * i % 256, np.uint8) for i, c in enumerate(f)])
    vals = np.concatenate([vals, np.full(n - len(vals), 7 * (len(f) - 1) % 256, np.uint8)])
    return rng.permutation(vals).tobytes()


@gpu
def test_lz_code_lengths_stay_within_15_bits():
    """Skewed histograms of literals, lengths and distances: both codes of every block are at most 15 bits."""
    rng = np.random.RandomState(5)
    fib = [1, 1]
    while len(fib) < 18:
        fib.append(fib[-1] + fib[-2])
    pre = rng.bytes(1024)
    lengths = bytearray(pre)                                        # Fibonacci counts over the length codes
    for length in rng.permutation(np.repeat(LEN_BASE[:16], fib[:16][::-1])):
        o = rng.randint(0, 1024 - length)
        lengths += pre[o:o + length]
    dists = bytearray(pre)                                          # and over the distance codes
    for d in rng.permutation(np.repeat(DIST_BASE[:17], fib[:17][::-1])):
        for _ in range(4):
            dists.append(dists[-int(d)])
        dists.append(rng.randint(256))
    for data in (_fibonacci_bytes(32768, rng) * 2, bytes(lengths), bytes(dists[:32768])):
        comp = _check(data)
        for kind, lit, dist, toks, raw in _blocks(comp):
            if kind == "dynamic":
                assert max(lit) <= 15 and max(dist) <= 15
                assert len(lit) <= 286 and len(dist) <= 30


@gpu
def test_lz_is_deterministic():
    rng = np.random.RandomState(6)
    text = b"".join(b"%d %d %d\n" % (g, c, v) for c in range(1, 300) for g, v in
                    zip(np.sort(rng.choice(20000, 200, replace=False)) + 1, rng.randint(1, 30, 200)))
    a = _lz(text)
    for _ in range(2):
        assert _lz(text) == a


def _sampler_streams(m):
    """The mtx text and the int32 / int64 CSR members of the sampler's counts at depth m (one chunk's worth)."""
    t, alpha, beta = _lineage_tree(2, 50, 10, 2000, seed=5)
    X = sim.sample_density(t, 4000, alpha=alpha, beta=beta, seed=8, device=DEV, scale_mean=m, out="csr")[0]
    text = b"".join(b"%d %d %d\n" % (g + 1, c + 1, v) for c in range(X.shape[0])
                    for g, v in zip(X.indices[X.indptr[c]:X.indptr[c + 1]], X.data[X.indptr[c]:X.indptr[c + 1]]))
    return {"mtx": text, "indices32": X.indices.astype(np.int32).tobytes(),
            "indices64": X.indices.astype(np.int64).tobytes(), "data32": X.data.astype(np.int32).tobytes(),
            "data64": X.data.astype(np.int64).tobytes()}


@gpu
def test_lz_ratio_against_huffman_only_and_zlib():
    ratios = {}
    for m in (-2.0, 0.0):
        for name, data in _sampler_streams(m).items():
            lz = len(_check(data))
            ratios[(m, name)] = (lz / len(_run("pst_deflate_blocks", data)[0]), lz / _zlib_blocks(data, 1))
    print(ratios)                                                    # lz77 / Huffman-only, lz77 / zlib level 1
    # int32 counts are small numbers whose Huffman-only form is already short: on one B200 zlib level 1 itself reached
    # only 0.97 of Huffman-only on them at m = 0 (this kernel 0.90), so that stream is held to 0.92, the rest to 0.85
    for key, (over_huffman, over_zlib1) in ratios.items():
        bound = 0.92 if key[1] == "data32" else 0.85
        assert over_huffman <= bound and over_zlib1 <= 1.15, (key, over_huffman, over_zlib1)


# ------------------------------------------------------------------ end to end
@pytest.fixture(scope="module")
def lineage_tree():
    return _lineage_tree(2, 20, 6, 1000, seed=3)


def _gunzip(path):
    return gzip.decompress(open(path, "rb").read())


def _same_mtx(got, want, path, want_path):
    """An lz77 out="mtx" call against the Huffman-only call of the same arguments."""
    rec, ref = got[0], want[0]
    assert isinstance(rec, formats.MtxRecord) and rec.path == path and rec.shape == ref.shape and rec.nnz == ref.nnz
    assert rec.nbytes == os.path.getsize(os.path.join(path, "matrix.mtx.gz"))
    for a, b in zip(got[1:], want[1:]):
        assert list(a) == list(b)
    assert sorted(os.listdir(path)) == FILES
    for f in FILES:
        assert _gunzip(os.path.join(path, f)) == _gunzip(os.path.join(want_path, f)), f
    mat = os.path.join(path, "matrix.mtx.gz")
    if ref.nnz:
        assert rec.nbytes < ref.nbytes
        L = sp.csr_matrix(scipy.io.mmread(mat, spmatrix=False).T)
        assert (L != ref.load()).nnz == 0
    if shutil.which("gzip"):
        r = subprocess.run(["gzip", "-t"] + [os.path.join(path, f) for f in FILES], capture_output=True)
        assert r.returncode == 0, r.stderr


def _members(path):
    with zipfile.ZipFile(path) as z:
        assert z.testzip() is None
        assert all(i.compress_type == zipfile.ZIP_DEFLATED for i in z.infolist())
        return {n: z.read(n) for n in z.namelist()}


def _same_npz(got, want, path, want_path):
    rec, ref = got[0], want[0]
    assert isinstance(rec, formats.CompressedCsr) and rec.path == path and rec.nbytes == os.path.getsize(path)
    assert (rec.shape, rec.nnz, rec.dtype, rec.index_dtype) == (ref.shape, ref.nnz, ref.dtype, ref.index_dtype)
    assert _members(path) == _members(want_path)
    A, B = sp.load_npz(path), sp.load_npz(want_path)
    for name in ("indptr", "indices", "data"):
        assert np.array_equal(getattr(A, name), getattr(B, name)) and getattr(A, name).dtype == getattr(B, name).dtype
    if ref.nnz:
        assert rec.nbytes < ref.nbytes
    for a, b in zip(got[1:], want[1:]):
        assert list(a) == list(b)


@gpu
@pytest.mark.parametrize("sampler", SAMPLERS)
def test_every_entry_point_writes_the_huffman_content(sampler, lineage_tree, tmp_path):
    t, alpha, beta = lineage_tree
    kw = dict(alpha=alpha, beta=beta, seed=12, device=DEV, sampler=sampler)
    calls = [
        lambda **o: sim.sample_density(t, 1500, **kw, **o),
        lambda **o: sim.sample_whole_tree(t, 7, **kw, **o),
        lambda **o: sim.sample_pseudotime_series(t, [300, 400], [5, 30], 4.0, **kw, **o),
        lambda **o: sim._sample_data_at_times(t, np.arange(0, 60), **kw, **o),
    ]
    for c, call in enumerate(calls):
        p, q = str(tmp_path / ("m%d" % c)), str(tmp_path / ("h%d" % c))
        _same_mtx(call(out="mtx", path=p, compression="lz77"), call(out="mtx", path=q), p, q)
        for dt in (np.int64, np.int32):
            p, q = str(tmp_path / ("m%d_%s.npz" % (c, np.dtype(dt).name))), str(tmp_path / ("h%d_%s.npz" % (c, dt.__name__)))
            _same_npz(call(out="csr", dtype=dt, path=p, compress=True, compression="lz77"),
                      call(out="csr", dtype=dt, path=q, compress=True), p, q)
    X, pt, br, sc = sim.sample_density(t, 800, alpha=alpha, beta=beta, seed=3, device=DEV)
    dkw = dict(seed=4, device=DEV, sampler=sampler, first=5000)
    p, q = str(tmp_path / "d"), str(tmp_path / "dh")
    got = sim.draw_counts(t, pt, br, sc, alpha, beta, out="mtx", path=p, compression="lz77", **dkw)
    want = sim.draw_counts(t, pt, br, sc, alpha, beta, out="mtx", path=q, **dkw)
    _same_mtx((got, pt, br, sc), (want, pt, br, sc), p, q)
    p, q = str(tmp_path / "d.npz"), str(tmp_path / "dh.npz")
    got = sim.draw_counts(t, pt, br, sc, alpha, beta, out="csr", path=p, compress=True, compression="lz77", **dkw)
    want = sim.draw_counts(t, pt, br, sc, alpha, beta, out="csr", path=q, compress=True, **dkw)
    _same_npz((got, pt, br, sc), (want, pt, br, sc), p, q)
    from prosstt_b200 import tree as ptree
    for out, o in (("mtx", {}), ("csr", dict(compress=True))):
        p, q = str(tmp_path / ("r_" + out)), str(tmp_path / ("rh_" + out))
        np.random.seed(92)
        got = sim.sample_whole_tree_restricted(ptree.Tree(), seed=6, device=DEV, sampler=sampler, out=out, path=p,
                                               compression="lz77", **o)
        np.random.seed(92)
        want = sim.sample_whole_tree_restricted(ptree.Tree(), seed=6, device=DEV, sampler=sampler, out=out, path=q,
                                                **o)
        (_same_mtx if out == "mtx" else _same_npz)(got, want, p, q)


def _stream_text(eng, rows, sc, seed, cell0, **kw):
    parts, bounds = [], []

    def consume(lo, hi, compressed, crc, text_len, nnz):
        raw = zlib.decompress(bytes(compressed) + b"\x03\x00", -15)
        assert len(raw) == text_len and zlib.crc32(raw) == crc and raw.count(b"\n") == nnz
        parts.append(raw)
        bounds.append((lo, hi))

    eng.stream_csr(rows, sc, seed, cell0, consume, mtx=True, compression="lz77", **kw)
    return b"".join(parts), bounds


@gpu
def test_chunking_repeats_and_forced_reformat(lineage_tree, tmp_path, monkeypatch):
    t, alpha, beta = lineage_tree
    n, chunk = 1000, 97
    eng, rows, sc = _engine(t, alpha, beta, n)
    want = _stream_text(eng, rows, sc, 5, 77, chunk_cells=n)[0]
    for c in (1, chunk, 5 * n):
        assert _stream_text(eng, rows, sc, 5, 77, chunk_cells=c)[0] == want, c
    ref, ref_bounds = _stream_text(eng, rows, sc, 5, 0, chunk_cells=chunk)
    calls = []
    real = CountEngine.draw

    def spy(self, *a, **k):
        calls.append(1)
        return real(self, *a, **k)

    monkeypatch.setattr(CountEngine, "draw", spy)
    monkeypatch.setattr(pdev, "_mtx_slot_bytes", lambda G, n: 1)    # every chunk formatted again, never redrawn
    got, bounds = _stream_text(eng, rows, sc, 5, 0, chunk_cells=chunk)
    assert got == ref and bounds == ref_bounds and len(calls) == len(bounds) == 11
    monkeypatch.undo()
    eng.check()
    kw = dict(alpha=alpha, beta=beta, seed=31, device=DEV, compression="lz77")
    for out, o, name in (("mtx", {}, "x"), ("csr", dict(compress=True), "x.npz")):
        a, b, s = (str(tmp_path / (p + name)) for p in ("big", "again", "small"))
        sim.sample_density(t, 3001, out=out, path=a, **o, **kw)
        sim.sample_density(t, 3001, out=out, path=b, **o, **kw)
        if out == "mtx":
            for f in FILES:
                assert open(os.path.join(a, f), "rb").read() == open(os.path.join(b, f), "rb").read(), f
        else:
            assert open(a, "rb").read() == open(b, "rb").read()
        monkeypatch.setattr(pdev, "_STAGE_BYTES", 2 * 16 * t.G * 200)
        sim.sample_density(t, 3001, out=out, path=s, **o, **kw)
        monkeypatch.undo()
        if out == "mtx":
            assert _gunzip(os.path.join(a, "matrix.mtx.gz")) == _gunzip(os.path.join(s, "matrix.mtx.gz"))
        else:
            assert _members(a) == _members(s)


@gpu
def test_rank_outputs_stack_to_the_whole(lineage_tree, tmp_path):
    t, alpha, beta = lineage_tree
    world = 3
    kw = dict(alpha=alpha, beta=beta, seed=17, device=DEV, compression="lz77")
    whole = sim.sample_density(t, 1001, alpha=alpha, beta=beta, seed=17, device=DEV, out="csr")[0]
    stem = str(tmp_path / "sim")
    dirs = [formats.shard_path(stem, r, world, suffix="") for r in range(world)]
    files = [formats.shard_path(stem, r, world, suffix=".npz") for r in range(world)]
    for r in range(world):
        sim.sample_density(t, 1001, shard=(r, world), out="mtx", path=dirs[r], **kw)
        sim.sample_density(t, 1001, shard=(r, world), out="csr", path=files[r], compress=True, **kw)
    stacked = sp.csr_matrix(sp.hstack([scipy.io.mmread(os.path.join(p, "matrix.mtx.gz"), spmatrix=False)
                                       for p in dirs]))
    assert stacked.shape == whole.T.shape and (stacked != whole.T).nnz == 0
    stacked = sp.vstack([sp.load_npz(p) for p in files], format="csr")
    assert (stacked != whole).nnz == 0


@gpu
def test_errors_leave_nothing(lineage_tree, tmp_path):
    t, alpha, beta = _random_tree(16, seed=4)
    means = {b: np.array(t.means[b]) for b in t.branches}
    for b in t.branches:
        means[b][-1, 3] = 0.0
    t.add_genes(means)
    t.invalidate_device_cache()
    eng, rows, sc = _engine(t, alpha, beta, 5000)
    rows = torch.full((5000,), 5, dtype=torch.int32, device=DEV)
    rows[4000:] = TreeTables(t, torch.device(DEV)).P - 1
    with pytest.raises(ValueError):                                  # a domain error in a later chunk
        with formats.MtxWriter(str(tmp_path / "domain"), (5000, t.G), *_cells(5000)) as w:
            eng.stream_csr(rows, sc, 1, 0, lambda lo, hi, *a: w.append(hi - lo, a[3], *a[:3]), mtx=True,
                           chunk_cells=100, compression="lz77")
    eng.flags.zero_()
    with pytest.raises(ValueError):
        with formats.CsrNpzWriter(str(tmp_path / "domain.npz"), (5000, t.G), *_cells(5000)) as w:
            eng.stream_csr(rows, sc, 1, 0, lambda lo, hi, parts: [w.append(*q) for q in parts], w.index_dtype,
                           np.int64, chunk_cells=100, compress=True, compression="lz77")
    eng.flags.zero_()
    t2, alpha2, beta2 = lineage_tree
    kw = dict(seed=1, device=DEV, compression="lz77")
    with pytest.raises(IndexError):                                  # a pseudotime outside the tree
        sim._sample_data_at_times(t2, [0, 5, 10 ** 6], alpha=alpha2, beta=beta2, out="mtx",
                                  path=str(tmp_path / "badpt"), **kw)
    with pytest.raises(ValueError):
        sim.sample_density(t2, 50, alpha2, beta2, out="csr", path=str(tmp_path / "plain"), **kw)
    for out, o, name in (("mtx", {}, "twice"), ("csr", dict(compress=True), "twice.npz")):
        p = str(tmp_path / name)
        sim.sample_density(t2, 50, alpha2, beta2, out=out, path=p, **o, **kw)
        with pytest.raises(FileExistsError):
            sim.sample_density(t2, 50, alpha2, beta2, out=out, path=p, **o, **kw)
    assert sorted(os.listdir(tmp_path)) == ["twice", "twice.npz"]
