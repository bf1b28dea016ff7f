"""Compact exchange formats for the count matrix (SURVEY.md 8f row 3).

The reference writes `<job>_simulation.txt`, a dense TSV (prosstt/tree_utils.py:113-146); that
writer is kept byte-compatible in `tree_utils.save_matrices` for small runs.  At the sizes this
package samples (10^10 counts and up) the text dump would take hours, so two binary forms are
added, both readable without this package:

* CSR, built on the device (`to_csr`, pst_csr_fill) and stored in SciPy's `save_npz` layout
  (`save_sparse_npz`): `scipy.sparse.load_npz(path)` / AnnData read it directly.  About 44 % of
  the counts are zero at default parameters and far more at low depth.
* dense int32 `.npy` shards written chunk by chunk from the pinned host buffers the samplers
  stream into (`NpyShardWriter`): `np.load(path, mmap_mode="r")` reads them.
* CSR shards streamed to disk chunk by chunk (`CsrShardWriter`, written by the samplers'
  `out="csr", path=...` through CountEngine.stream_csr), for matrices no host memory holds whole.
  A shard is a directory of plain `.npy` files: the members of `scipy.sparse.save_npz` for a csr
  matrix (`format`, `shape`, `indptr`, `indices`, `data`) and the cell annotations (`pseudotime`
  int64, `branches`, `scalings` float64).  `np.load(..., mmap_mode="r")` reads every member, and
  the CSR members zipped uncompressed (ZIP_STORED) form a file `scipy.sparse.load_npz` reads.
  `load_csr_shard` maps it back without a copy.
* compressed CSR files (`CsrNpzWriter`, written by `out="csr", path=..., compress=True`): one zip64
  `.npz` whose members are the same `.npy` files, each DEFLATE-compressed (the format
  `np.savez_compressed` writes), so `scipy.sparse.load_npz(path)` and `np.load(path)` read it.  The
  GPU compresses each chunk's indptr, indices and data (pst_deflate_blocks: Huffman-only blocks ended by
  a sync-flush marker, concatenated), so only compressed bytes cross PCIe and reach the disk.  The file
  cannot be memory-mapped: the call returns a `CompressedCsr` record, and `load_csr_shard` decompresses
  it into memory.
* 10x directories (`MtxWriter`, written by `out="mtx", path=...`): the gzipped Matrix Market matrix, features
  and barcodes that Seurat::Read10X, DropletUtils::read10xCounts, Matrix::readMM and scanpy.read_10x_mtx read,
  plus the cells' parameters.  The GPU formats each chunk as text (pst_mtx_format) and compresses it
  (pst_deflate_blocks), so only compressed text crosses PCIe and reaches the disk.  The call returns an
  `MtxRecord`.
"""
import collections
import concurrent.futures
import errno
import io
import os
import shutil
import struct
import zlib

import numpy as np
import torch

from prosstt_b200 import _native as nat
from prosstt_b200 import stats as pstats


def to_csr(X, stats=None):
    """Device CSR of a device count matrix.  X: (n, G) int32 CUDA tensor.  Returns
    (indptr int64 (n+1,), indices int32 (nnz,), data int32 (nnz,)) CUDA tensors, columns
    ascending inside each row.  `stats` may pass a count_stats(X) result to skip that pass."""
    X = pstats._check_counts(X, "to_csr")
    n, G = X.shape
    dev = X.device
    if stats is None:
        stats = pstats.count_stats(X)
    indptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    if n:
        torch.cumsum(G - stats["cell_zeros"].to(torch.int64), dim=0, out=indptr[1:])
    nnz = int(indptr[-1].item())
    indices = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
    data = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
    flags = torch.zeros(1, dtype=torch.int32, device=dev)
    nat.call("pst_csr_fill", X.data_ptr(), n, G, X.stride(0) if n else G, indptr, indices, data, flags,
             nat.stream_ptr(dev))
    if int(flags.item()) != 0:
        raise RuntimeError("row pointer does not match the matrix (was X modified after count_stats?)")
    return indptr, indices[:nnz], data[:nnz]


def save_sparse_npz(path, X, compressed=False):
    """Write X (device int32 matrix, or a (indptr, indices, data, shape) tuple from to_csr) in the
    layout of scipy.sparse.save_npz for a csr_matrix."""
    if isinstance(X, torch.Tensor):
        shape = tuple(X.shape)
        indptr, indices, data = to_csr(X)
    else:
        indptr, indices, data, shape = X
    arrays = dict(indices=indices.cpu().numpy(), indptr=indptr.cpu().numpy(), format=np.array("csr".encode("ascii")),
                  shape=np.asarray(shape, dtype=np.int64), data=data.cpu().numpy())
    if not str(path).endswith(".npz"):
        path = str(path) + ".npz"
    with open(path, "wb") as fh:
        (np.savez_compressed if compressed else np.savez)(fh, **arrays)
    return path


def load_sparse_npz(path):
    """(indptr, indices, data, shape) NumPy arrays of a file written by save_sparse_npz (or by
    scipy.sparse.save_npz for a csr matrix)."""
    with np.load(path) as z:
        fmt = z["format"].item()
        fmt = fmt.decode("ascii") if isinstance(fmt, bytes) else str(fmt)
        if fmt != "csr":
            raise ValueError("expected a csr matrix, found %r" % fmt)
        return z["indptr"], z["indices"], z["data"], tuple(int(v) for v in z["shape"])


def csr_to_dense(indptr, indices, data, shape):
    """Dense NumPy matrix of a CSR triple (small matrices / tests)."""
    out = np.zeros(shape, dtype=np.asarray(data).dtype)
    rows = np.repeat(np.arange(shape[0]), np.diff(np.asarray(indptr)))
    out[rows, np.asarray(indices)] = np.asarray(data)
    return out


def widen(Xn, overflow):
    """Exact int32 matrix from a narrow transfer format: Xn (n, G) uint8 or uint16 with saturated
    elements reading 255 / 65535, overflow = (flat index, value) arrays or the dict filled by
    `sample_density(host_out=(..., dict))`."""
    if isinstance(overflow, dict):
        overflow = (overflow["index"], overflow["value"])
    Xn = np.asarray(Xn)
    if Xn.dtype not in (np.dtype(np.uint8), np.dtype(np.uint16)):
        raise TypeError("expected a uint8 or uint16 matrix")
    out = Xn.astype(np.int32)
    index, value = np.asarray(overflow[0]), np.asarray(overflow[1])
    saturated = np.flatnonzero(Xn.reshape(-1) == np.iinfo(Xn.dtype).max)
    if not np.array_equal(saturated, index):
        raise ValueError("overflow list does not match the saturated elements of the matrix")
    out.reshape(-1)[index] = value
    return out


class NpyShardWriter(object):
    """Append-only writer of one dense (n_cells, G) `.npy` file, filled in row blocks.

    The header is written up front for the final shape, so the file is a valid `.npy` once every
    row has been appended; blocks come straight from the pinned host buffers of
    `sample_density(..., host_out=...)` / `DensitySession.step_to_host`.  One writer per rank
    gives one shard per GPU (`<stem>.rank<k>.npy`)."""

    def __init__(self, path, n_cells, G, dtype=np.int32):
        self.path = str(path)
        self.shape = (int(n_cells), int(G))
        self.dtype = np.dtype(dtype)
        self.rows = 0
        self._fh = open(self.path, "wb")
        np.lib.format.write_array_header_2_0(
            self._fh, {"descr": np.lib.format.dtype_to_descr(self.dtype), "fortran_order": False,
                       "shape": self.shape})

    def append(self, block):
        block = np.ascontiguousarray(block, dtype=self.dtype)
        if block.ndim != 2 or block.shape[1] != self.shape[1]:
            raise ValueError("block must have shape (rows, %d)" % self.shape[1])
        if self.rows + block.shape[0] > self.shape[0]:
            raise ValueError("more rows than announced (%d)" % self.shape[0])
        self._fh.write(memoryview(block).cast("B"))
        self.rows += block.shape[0]

    def close(self):
        if self._fh is None:
            return
        self._fh.close()
        self._fh = None
        if self.rows != self.shape[0]:
            raise ValueError("%s: %d of %d rows written" % (self.path, self.rows, self.shape[0]))

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc, tb):
        if exc_type is None:
            self.close()
        elif self._fh is not None:
            self._fh.close()
            self._fh = None
        return False


def shard_path(stem, rank, world, suffix=".npy"):
    """`<stem><suffix>` for one rank, `<stem>.rank<k>of<w><suffix>` otherwise (suffix ".csr" for CSR shards,
    ".npz" for compressed CSR files)."""
    return "%s%s" % (stem, suffix) if world == 1 else "%s.rank%dof%d%s" % (stem, rank, world, suffix)


def _csr_matrix(indptr, indices, data, shape):
    """scipy.sparse.csr_matrix over the given arrays without a copy or a scan: the constructor would check
    every column index and copy int64 index arrays whose contents fit int32.  The arrays are already in
    canonical form (columns ascending in every row, no explicit zeros, no duplicates)."""
    import scipy.sparse as sp
    m = sp.csr_matrix(shape, dtype=data.dtype)
    m.indptr, m.indices, m.data = indptr, indices, data
    m.has_sorted_indices = True
    m.has_canonical_format = True
    return m


def _csr_cells(n, pseudotime, branches, scalings):
    """The cell annotations of a CSR shard or file, checked to hold one value per cell."""
    branches = np.asarray(branches)
    if branches.dtype.kind == "O":                       # readable without pickle
        branches = branches.astype(str)
    cells = dict(pseudotime=np.asarray(pseudotime, dtype=np.int64), branches=branches,
                 scalings=np.asarray(scalings, dtype=np.float64))
    for name, a in cells.items():
        if a.shape != (n,):
            raise ValueError("%s must hold one value per cell (%d), not shape %s" % (name, n, a.shape))
    return cells


def _csr_dtypes(shape, dtype):
    """(index dtype, data dtype) of a CSR shard or file: int32 indices when n_cells x G < 2^31."""
    dtype = np.dtype(dtype)
    if dtype not in (np.dtype(np.int32), np.dtype(np.int64)):
        raise ValueError("CSR data must be int32 or int64, not %s" % dtype)
    n, G = shape
    return (np.dtype(np.int32) if n * G < (1 << 31) else np.dtype(np.int64)), dtype


class CsrShardWriter(object):
    """Writer of one CSR shard (the directory format of the module docstring), appended chunk by chunk.

    indptr and indices are int32 when n_cells x G < 2^31 and int64 otherwise: nnz is not known when the
    files are opened and n_cells x G bounds it, so scipy never has to convert them.  data is `dtype`, int64
    or int32.  Chunks are appended with write(), not through a memory map, so the page cache they pass
    through is not counted against the process; the `.npy` headers of indices and data get their length at
    close(), in the space numpy's header reserves for it.  Everything goes into `<path>.partial`, which
    becomes `<path>` only when close() finds every row written: a short shard, an exception inside `with`
    or abort() leaves nothing at `<path>` (nor at `<path>.partial`).  An existing `<path>` raises
    FileExistsError."""

    def __init__(self, path, shape, pseudotime, branches, scalings, dtype=np.int64):
        self.path = os.fspath(path)
        if os.path.lexists(self.path):
            raise FileExistsError(errno.EEXIST, "the CSR shard exists already", self.path)
        n, G = (int(v) for v in shape)
        self.shape = (n, G)
        self.index_dtype, self.dtype = _csr_dtypes(self.shape, dtype)
        cells = _csr_cells(n, pseudotime, branches, scalings)
        self.rows, self.nnz = 0, 0
        self._dir = self.path + ".partial"
        if os.path.lexists(self._dir):                  # left behind by an interrupted writer
            shutil.rmtree(self._dir)
        os.makedirs(self._dir)
        self._files, self._data_at = {}, {}
        try:
            np.save(self._member("format"), np.array(b"csr"))
            np.save(self._member("shape"), np.array(self.shape, dtype=np.int64))
            for name, a in cells.items():
                np.save(self._member(name), a)
            for name, dt, length in (("indptr", self.index_dtype, n + 1), ("indices", self.index_dtype, 0),
                                     ("data", self.dtype, 0)):
                self._files[name] = open(self._member(name), "wb")
                self._header(name, dt, length)
                self._data_at[name] = self._files[name].tell()
            self._files["indptr"].write(np.zeros(1, dtype=self.index_dtype).tobytes())
        except BaseException:
            self.abort()
            raise

    def _member(self, name):
        return os.path.join(self._dir, name + ".npy")

    def _header(self, name, dtype, length):
        fh = self._files[name]
        fh.seek(0)
        np.lib.format.write_array_header_1_0(fh, {"descr": np.lib.format.dtype_to_descr(dtype),
                                                  "fortran_order": False, "shape": (int(length),)})

    def append(self, indptr, indices, data):
        """Append the next rows: indptr local to them (rows + 1 entries from 0), their nonzeros' columns and
        values."""
        indptr = np.asarray(indptr)
        rows = len(indptr) - 1
        if rows < 0 or indptr[0] != 0:
            raise ValueError("indptr must start at 0")
        m = int(indptr[-1])
        if len(indices) != m or len(data) != m:
            raise ValueError("indices and data must hold indptr[-1] = %d entries" % m)
        if self.rows + rows > self.shape[0]:
            raise ValueError("more rows than announced (%d)" % self.shape[0])
        fh = self._files
        fh["indptr"].write(memoryview((indptr[1:] + self.nnz).astype(self.index_dtype)).cast("B"))
        fh["indices"].write(memoryview(np.ascontiguousarray(indices, dtype=self.index_dtype)).cast("B"))
        fh["data"].write(memoryview(np.ascontiguousarray(data, dtype=self.dtype)).cast("B"))
        self.rows += rows
        self.nnz += m

    def close(self):
        """Finish the shard and move it to `path`; raises (and leaves nothing) when rows are missing."""
        if self._files is None:
            return
        try:
            if self.rows != self.shape[0]:
                raise ValueError("%s: %d of %d rows written" % (self.path, self.rows, self.shape[0]))
            for name, dt in (("indices", self.index_dtype), ("data", self.dtype)):
                self._header(name, dt, self.nnz)
                if self._files[name].tell() != self._data_at[name]:
                    raise RuntimeError("the .npy header of %s outgrew its reserved space" % name)
            for fh in self._files.values():
                fh.close()
            self._files = None
            os.rename(self._dir, self.path)
        except BaseException:
            self.abort()
            raise

    def abort(self):
        """Drop everything written so far."""
        for fh in (self._files or {}).values():
            fh.close()
        self._files = None
        shutil.rmtree(self._dir, ignore_errors=True)

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc, tb):
        if exc_type is None:
            self.close()
        else:
            self.abort()
        return False


def sync_deflate(raw):
    """(bytes, crc32, len) of `raw` compressed as zlib's non-final, sync-flushed raw DEFLATE blocks: the unit
    CsrNpzWriter.append takes (what pst_deflate_blocks makes on the device)."""
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    raw = bytes(raw)
    return c.compress(raw) + c.flush(zlib.Z_SYNC_FLUSH), zlib.crc32(raw), len(raw)


class CompressedCsr(collections.namedtuple("CompressedCsr", "path shape nnz dtype index_dtype nbytes")):
    """The X of a `compress=True` call: a compressed CSR file on disk, not loaded (it cannot be memory-mapped).
    nbytes is the file's size; load() decompresses it (scipy.sparse.load_npz)."""
    __slots__ = ()

    def load(self):
        import scipy.sparse as sp
        return sp.load_npz(self.path)


_ZIP_DATE, _ZIP_TIME = (0 << 9) | (1 << 5) | 1, 0       # fixed timestamp 1980-01-01 00:00: identical files
_ZIP64 = 45                                            # version needed to extract zip64 entries
_NPY_STORED = 5                                        # stored-block header in front of a member's .npy header
_FINAL_BLOCK = b"\x03\x00"                            # empty final block (fixed Huffman, end-of-block)


def _npy_header(dtype, length):
    buf = io.BytesIO()
    np.lib.format.write_array_header_1_0(buf, {"descr": np.lib.format.dtype_to_descr(np.dtype(dtype)),
                                               "fortran_order": False, "shape": (int(length),)})
    return buf.getvalue()


def _npy_bytes(a):
    buf = io.BytesIO()
    np.save(buf, a, allow_pickle=False)
    return buf.getvalue()


class CsrNpzWriter(object):
    """Writer of one compressed CSR file (the `.npz` of the module docstring), appended chunk by chunk.

    The constructor is CsrShardWriter's, with the same dtypes: indptr and indices int32 when n_cells x G < 2^31
    and int64 otherwise, data `dtype`.  append(member, compressed, crc, raw_len) takes the next bytes of
    "indptr", "indices" or "data" as raw DEFLATE blocks that are not final and end on a byte boundary
    (pst_deflate_blocks' output, or sync_deflate's), with the CRC-32 and length of the bytes they decompress
    to.  indptr's leading 0 is the writer's: the appended indptr holds the row ends, offset by the nonzeros
    before them.  The small members are compressed here with zlib.

    Every member is a zip64 entry (local and central zip64 fields, also when small): the .npy header as a
    stored block, the body, the final block 03 00; its CRC combines the header's with the body's.  Zip
    members are contiguous and the three streams grow together, so indices, the largest, goes straight into
    the file and indptr and data into temporaries beside it, which close() appends (copied_at_close: their
    bytes).  As CsrShardWriter: everything goes to `<path>.partial`, renamed to `<path>` only by a complete
    close(); an exception inside `with` or abort() leaves nothing behind; an existing `<path>` raises
    FileExistsError.  The same appends give the same file, byte for byte."""

    def __init__(self, path, shape, pseudotime, branches, scalings, dtype=np.int64):
        self.path = os.fspath(path)
        if os.path.lexists(self.path):
            raise FileExistsError(errno.EEXIST, "the compressed CSR file exists already", self.path)
        n, G = (int(v) for v in shape)
        self.shape = (n, G)
        self.index_dtype, self.dtype = _csr_dtypes(self.shape, dtype)
        cells = _csr_cells(n, pseudotime, branches, scalings)
        self.nnz, self.copied_at_close = 0, 0
        self._partial = self.path + ".partial"
        self._temps = {m: "%s.%s" % (self._partial, m) for m in ("indptr", "data")}
        self._central = []
        self._fh, self._sinks = None, {}
        self._dtypes = {"indptr": self.index_dtype, "indices": self.index_dtype, "data": self.dtype}
        self._crc = dict.fromkeys(self._dtypes, 0)
        self._raw = dict.fromkeys(self._dtypes, 0)
        self._packed = dict.fromkeys(self._dtypes, 0)
        try:
            for p in [self._partial] + list(self._temps.values()):
                if os.path.lexists(p):                  # left behind by an interrupted writer
                    os.remove(p)
            self._fh = open(self._partial, "wb")
            small = dict(format=np.array(b"csr"), shape=np.array(self.shape, dtype=np.int64), **cells)
            for name, a in small.items():
                raw = _npy_bytes(a)
                c = zlib.compressobj(6, zlib.DEFLATED, -15)
                self._entry(name, c.compress(raw) + c.flush(), zlib.crc32(raw), len(raw))
            self._indices_at = self._fh.tell()
            self._local_header("indices", 0, 0, 0)
            self._indices_body = self._fh.tell()
            self._reserved = _NPY_STORED + len(_npy_header(self.index_dtype, 0))
            self._fh.write(bytes(self._reserved))      # its header block, filled in by close()
            self._sinks = {"indices": self._fh}
            for m, p in self._temps.items():
                self._sinks[m] = open(p, "wb")
            self.append("indptr", *sync_deflate(np.zeros(1, self.index_dtype).tobytes()))
        except BaseException:
            self.abort()
            raise

    def _local_header(self, name, crc, packed, raw):
        fname = (name + ".npy").encode("ascii")
        self._fh.write(struct.pack("<IHHHHHIIIHH", 0x04034B50, _ZIP64, 0, 8, _ZIP_TIME, _ZIP_DATE, crc,
                                   0xFFFFFFFF, 0xFFFFFFFF, len(fname), 20) + fname
                       + struct.pack("<HHQQ", 1, 16, raw, packed))

    def _entry(self, name, packed_bytes, crc, raw):
        """One whole member: its local header and its compressed bytes."""
        at = self._fh.tell()
        self._local_header(name, crc, len(packed_bytes), raw)
        self._fh.write(packed_bytes)
        self._central.append((name, crc, len(packed_bytes), raw, at))

    def append(self, member, compressed, crc, raw_len):
        """The next raw_len bytes of member "indptr", "indices" or "data", as non-final DEFLATE blocks."""
        dt = self._dtypes.get(member)
        if dt is None:
            raise ValueError("member must be 'indptr', 'indices' or 'data', not %r" % (member,))
        if raw_len % dt.itemsize:
            raise ValueError("%s takes whole %s values, not %d bytes" % (member, dt, raw_len))
        compressed = memoryview(compressed).cast("B")
        self._sinks[member].write(compressed)
        self._crc[member] = int(nat.load().pst_host_crc32_combine(self._crc[member], int(crc) & 0xFFFFFFFF,
                                                                   int(raw_len)))
        self._raw[member] += int(raw_len)
        self._packed[member] += len(compressed)

    def _header_block(self, member):
        header = _npy_header(self._dtypes[member], self._raw[member] // self._dtypes[member].itemsize)
        return (struct.pack("<BHH", 0, len(header), len(header) ^ 0xFFFF) + header,
                zlib.crc32(header), len(header))

    def _finish(self, member, header):
        """(crc, packed, raw) of a member whose body has been written: header block + body + final block."""
        block, hcrc, hlen = header
        crc = int(nat.load().pst_host_crc32_combine(hcrc, self._crc[member], self._raw[member]))
        return crc, len(block) + self._packed[member] + len(_FINAL_BLOCK), hlen + self._raw[member]

    def close(self):
        """Finish the file and move it to `path`; raises (and leaves nothing) when rows are missing or the
        members disagree."""
        if self._fh is None:
            return
        try:
            n = self.shape[0]
            rows = self._raw["indptr"] // self.index_dtype.itemsize - 1
            if rows != n:
                raise ValueError("%s: %d of %d rows written" % (self.path, rows, n))
            self.nnz = self._raw["indices"] // self.index_dtype.itemsize
            if self._raw["data"] // self.dtype.itemsize != self.nnz:
                raise ValueError("%s: %d column indices but %d values" % (self.path, self.nnz,
                                                                          self._raw["data"] // self.dtype.itemsize))
            fh = self._fh
            for m in self._temps:
                self._sinks[m].close()
            # indices: the final block, then its header block and local header in the space kept for them
            fh.write(_FINAL_BLOCK)
            end = fh.tell()
            head = self._header_block("indices")
            if len(head[0]) != self._reserved:
                raise RuntimeError("the .npy header of indices outgrew its reserved space")
            crc, packed, raw = self._finish("indices", head)
            fh.seek(self._indices_at)
            self._local_header("indices", crc, packed, raw)
            fh.write(head[0])
            fh.seek(end)
            self._central.append(("indices", crc, packed, raw, self._indices_at))
            # indptr and data: whole members, their bodies copied from the temporaries
            for m, p in self._temps.items():
                head = self._header_block(m)
                crc, packed, raw = self._finish(m, head)
                at = fh.tell()
                self._local_header(m, crc, packed, raw)
                fh.write(head[0])
                with open(p, "rb") as src:
                    shutil.copyfileobj(src, fh, 16 << 20)
                fh.write(_FINAL_BLOCK)
                self.copied_at_close += self._packed[m]
                self._central.append((m, crc, packed, raw, at))
                os.remove(p)
            self._central_directory()
            fh.close()
            self._fh = None
            os.rename(self._partial, self.path)
        except BaseException:
            self.abort()
            raise

    def _central_directory(self):
        fh = self._fh
        cd_at = fh.tell()
        for name, crc, packed, raw, at in self._central:
            fname = (name + ".npy").encode("ascii")
            fh.write(struct.pack("<IHHHHHHIIIHHHHHII", 0x02014B50, _ZIP64, _ZIP64, 0, 8, _ZIP_TIME, _ZIP_DATE, crc,
                                 0xFFFFFFFF, 0xFFFFFFFF, len(fname), 28, 0, 0, 0, 0, 0xFFFFFFFF) + fname
                     + struct.pack("<HHQQQ", 1, 24, raw, packed, at))
        cd_size, k = fh.tell() - cd_at, len(self._central)
        eocd64 = fh.tell()
        fh.write(struct.pack("<IQHHIIQQQQ", 0x06064B50, 44, _ZIP64, _ZIP64, 0, 0, k, k, cd_size, cd_at))
        fh.write(struct.pack("<IIQI", 0x07064B50, 0, eocd64, 1))
        fh.write(struct.pack("<IHHHHIIH", 0x06054B50, 0, 0, min(k, 0xFFFF), min(k, 0xFFFF),
                             min(cd_size, 0xFFFFFFFF), min(cd_at, 0xFFFFFFFF), 0))

    def record(self):
        """The CompressedCsr of the closed file."""
        return CompressedCsr(self.path, self.shape, self.nnz, self.dtype, self.index_dtype,
                             os.path.getsize(self.path))

    def abort(self):
        """Drop everything written so far."""
        for f in [self._fh] + list(self._sinks.values()):
            if f is not None:
                f.close()
        self._fh, self._sinks = None, {}
        for p in [self._partial] + list(self._temps.values()):
            try:
                os.remove(p)
            except OSError:
                pass

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc, tb):
        if exc_type is None:
            self.close()
        else:
            self.abort()
        return False


_GZIP_HEADER = b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff"   # DEFLATE, no flags, MTIME 0, XFL 0, OS 255 (unknown)
MTX_HEADER_BYTES = 128                                        # the three header lines of matrix.mtx.gz together
_MTX_BANNER = b"%%MatrixMarket matrix coordinate integer general\n"


def gzip_member(raw, level=6):
    """`raw` as one gzip member (RFC 1952) with the fixed header of every .gz of a 10x directory."""
    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    return _GZIP_HEADER + c.compress(raw) + c.flush() + struct.pack("<II", zlib.crc32(raw), len(raw) & 0xFFFFFFFF)


def mtx_header(G, n, nnz):
    """The first MTX_HEADER_BYTES bytes of the text of matrix.mtx.gz: the banner, a comment line of spaces that
    takes up the slack (so the size line can be rewritten in place once nnz is known) and "<G> <n> <nnz>"."""
    size = b"%d %d %d\n" % (G, n, nnz)
    pad = MTX_HEADER_BYTES - len(_MTX_BANNER) - len(size) - 2
    if pad < 0:
        raise ValueError("the Matrix Market size line %r does not fit the header" % size)
    return _MTX_BANNER + b"%" + b" " * pad + b"\n" + size


def mtx_barcodes(first, n):
    """barcodes.tsv text: cell_<i> for the global cell indices first ... first + n - 1."""
    return "".join("cell_%d\n" % i for i in range(first, first + n)).encode("ascii")


def mtx_features(G):
    """features.tsv text: gene_<j>, gene_<j>, Gene Expression for j = 0 ... G - 1 (the column names of the
    reference's _simulation.txt)."""
    return "".join("gene_%d\tgene_%d\tGene Expression\n" % (j, j) for j in range(G)).encode("ascii")


def mtx_cell_params(first, pseudotime, branches, scalings):
    """cellparams.tsv text: the reference's _cellparams.txt (tree_utils.save_cell_params) indexed by the
    barcodes."""
    from prosstt_b200 import tree_utils
    names = ["cell_%d" % i for i in range(first, first + len(pseudotime))]
    return tree_utils.cell_params_frame(pseudotime, branches, scalings, index=names).to_csv(sep="\t").encode("utf-8")


class MtxRecord(collections.namedtuple("MtxRecord", "path shape nnz nbytes")):
    """The X of an out="mtx" call: a 10x directory on disk.  shape is (cells, genes); nbytes is the size of
    matrix.mtx.gz; load() reads it back (scipy.io.mmread) as the cells x genes int64 csr_matrix."""
    __slots__ = ()

    def load(self):
        import scipy.io
        import scipy.sparse as sp
        m = scipy.io.mmread(os.path.join(self.path, "matrix.mtx.gz"), spmatrix=False)
        return sp.csr_matrix(m.T, dtype=np.int64)


class MtxWriter(object):
    """Writer of one 10x directory (Cell Ranger v3 layout), the matrix appended chunk by chunk:
      matrix.mtx.gz     genes x cells Matrix Market coordinate text, cell-major, genes ascending in a cell;
      features.tsv.gz   gene_<j> \\t gene_<j> \\t Gene Expression;
      barcodes.tsv.gz   cell_<i>, i the global cell index (first + local index);
      cellparams.tsv.gz the reference's _cellparams.txt for these cells, indexed by the barcodes.
    Every .gz is one gzip member with MTIME 0, XFL 0 and OS 255, so the same appends give the same bytes.

    append(rows, nnz, compressed, crc, raw_len) takes the text of the next `rows` cells (their `nnz` lines)
    as raw DEFLATE blocks that are not final and end on a byte boundary (pst_deflate_blocks' output over
    pst_mtx_format's text, or sync_deflate's), with the CRC-32 and length of the text.  The first
    MTX_HEADER_BYTES of the text, whose nnz is not known before close(), are a stored block written at once
    and rewritten in place at close() with the same length; the member's CRC combines the header's with the
    body's.  The three small files are built on a worker thread while the matrix streams.  As CsrShardWriter:
    everything goes to `<path>.partial`, renamed to `<path>` only by a complete close(); an exception inside
    `with` or abort() leaves nothing behind; an existing `<path>` raises FileExistsError."""

    def __init__(self, path, shape, pseudotime, branches, scalings, first=0):
        self.path = os.fspath(path)
        if os.path.lexists(self.path):
            raise FileExistsError(errno.EEXIST, "the 10x directory exists already", self.path)
        n, G = (int(v) for v in shape)
        self.shape, self.first = (n, G), int(first)
        cells = _csr_cells(n, pseudotime, branches, scalings)
        self.rows, self.nnz = 0, 0
        self._crc, self._raw = 0, 0
        self._dir = self.path + ".partial"
        self._fh, self._small = None, None
        if os.path.lexists(self._dir):                  # left behind by an interrupted writer
            shutil.rmtree(self._dir)
        os.makedirs(self._dir)
        try:
            self._fh = open(os.path.join(self._dir, "matrix.mtx.gz"), "wb")
            self._fh.write(_GZIP_HEADER)
            self._header_at = self._fh.tell()
            self._fh.write(self._header_block(0))
            pool = concurrent.futures.ThreadPoolExecutor(max_workers=1)
            self._small = pool.submit(self._write_small, (cells["pseudotime"], cells["branches"], cells["scalings"]))
            pool.shutdown(wait=False)
        except BaseException:
            self.abort()
            raise

    def _header_block(self, nnz):
        header = mtx_header(self.shape[1], self.shape[0], nnz)
        return struct.pack("<BHH", 0, len(header), len(header) ^ 0xFFFF) + header

    def _write_small(self, cells):
        n, G = self.shape
        for name, text in (("features", lambda: mtx_features(G)), ("barcodes", lambda: mtx_barcodes(self.first, n)),
                           ("cellparams", lambda: mtx_cell_params(self.first, *cells))):
            with open(os.path.join(self._dir, name + ".tsv.gz"), "wb") as fh:
                fh.write(gzip_member(text()))

    def append(self, rows, nnz, compressed, crc, raw_len):
        """The text of the next `rows` cells, `nnz` lines of raw_len bytes, as non-final DEFLATE blocks."""
        if self.rows + int(rows) > self.shape[0]:
            raise ValueError("more rows than announced (%d)" % self.shape[0])
        compressed = memoryview(compressed).cast("B")
        self._fh.write(compressed)
        self._crc = int(nat.load().pst_host_crc32_combine(self._crc, int(crc) & 0xFFFFFFFF, int(raw_len)))
        self._raw += int(raw_len)
        self.rows += int(rows)
        self.nnz += int(nnz)

    def close(self):
        """Finish the directory and move it to `path`; raises (and leaves nothing) when rows are missing."""
        if self._fh is None:
            return
        try:
            if self.rows != self.shape[0]:
                raise ValueError("%s: %d of %d rows written" % (self.path, self.rows, self.shape[0]))
            fh = self._fh
            block = self._header_block(self.nnz)
            header = block[5:]
            crc = int(nat.load().pst_host_crc32_combine(zlib.crc32(header), self._crc, self._raw))
            fh.write(_FINAL_BLOCK + struct.pack("<II", crc, (len(header) + self._raw) & 0xFFFFFFFF))
            fh.flush()
            if os.pwrite(fh.fileno(), block, self._header_at) != len(block):
                raise OSError("short write of the matrix.mtx.gz header")
            fh.close()
            self._fh = None
            self._small.result()
            os.rename(self._dir, self.path)
        except BaseException:
            self.abort()
            raise

    def record(self):
        """The MtxRecord of the closed directory."""
        return MtxRecord(self.path, self.shape, self.nnz, os.path.getsize(os.path.join(self.path, "matrix.mtx.gz")))

    def abort(self):
        """Drop everything written so far."""
        if self._fh is not None:
            self._fh.close()
        self._fh = None
        if self._small is not None:
            concurrent.futures.wait([self._small])      # it writes into the directory removed below
        shutil.rmtree(self._dir, ignore_errors=True)

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc, tb):
        if exc_type is None:
            self.close()
        else:
            self.abort()
        return False


def load_csr_shard(path):
    """(X, pseudotime, branches, scalings) of a shard written by CsrShardWriter: X is a canonical
    scipy.sparse.csr_matrix over read-only memory maps of indptr, indices and data (no copy).  A compressed
    file written by CsrNpzWriter gives the same tuple, with X decompressed into memory."""
    if os.path.isfile(path):
        with np.load(path, allow_pickle=False) as z:
            fmt = z["format"].item()
            fmt = fmt.decode("ascii") if isinstance(fmt, bytes) else str(fmt)
            if fmt != "csr":
                raise ValueError("expected a csr matrix, found %r" % fmt)
            shape = tuple(int(v) for v in z["shape"])
            X = _csr_matrix(z["indptr"], z["indices"], z["data"], shape)
            return X, z["pseudotime"], z["branches"], z["scalings"]

    def member(name, mmap_mode=None):
        return np.load(os.path.join(os.fspath(path), name + ".npy"), mmap_mode=mmap_mode, allow_pickle=False)

    fmt = member("format").item()
    fmt = fmt.decode("ascii") if isinstance(fmt, bytes) else str(fmt)
    if fmt != "csr":
        raise ValueError("expected a csr matrix, found %r" % fmt)
    shape = tuple(int(v) for v in member("shape"))
    X = _csr_matrix(member("indptr", "r"), member("indices", "r"), member("data", "r"), shape)
    return X, member("pseudotime"), member("branches"), member("scalings")
