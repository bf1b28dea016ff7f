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
* the reference's own `_simulation.txt` (`TsvWriter`, written by `out="tsv", path=...`): the dense tab-separated
  table of `tree_utils.save_matrices`, byte for byte, that `pd.read_csv(path, sep="\t", index_col=0)` reads;
  with `compress=True` one gzip member of it.  The GPU formats each chunk's rows (pst_tsv_format) and, for the
  gzipped file, compresses them, so only the file's bytes cross PCIe.  The call returns a `TsvRecord`.
* Parquet directories (`ParquetWriter`, written by `out="parquet", path=...`): counts.parquet, one row per nonzero
  (cell, gene, count), read by pandas, pyarrow, polars, DuckDB, Spark and R's arrow, and cells.parquet.  The GPU
  encodes each chunk's columns as DELTA_BINARY_PACKED pages (pst_delta_sizes, pst_delta_write) and, with
  compress=True, gzips them, so only the pages cross PCIe.  The writer serializes the Parquet metadata itself (no
  pyarrow).  The call returns a `ParquetRecord`.
* AnnData Zarr stores (`ZarrWriter`, written by `out="zarr", path=...`): a Zarr v2 directory in AnnData's on-disk
  layout, X as a csr_matrix group and obs as the reference's _cellparams.txt, that `anndata.read_zarr`, zarr-python,
  dask and AnnData's lazy readers open.  The GPU cuts each array into Zarr chunks of `ZARR_CHUNK` elements
  (pst_zarr_cut) and, with compress=True, compresses every chunk into one zlib stream (pst_deflate_segments), so
  only the chunks' bytes cross PCIe.  The call returns a `ZarrRecord`.
"""
import collections
import concurrent.futures
import errno
import io
import json
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


_STORED_MAX = 65535                                           # bytes of one stored DEFLATE block


def _stored_blocks(raw):
    """`raw` as non-final stored DEFLATE blocks (RFC 1951 3.2.4), at most _STORED_MAX bytes each."""
    out = []
    for at in range(0, len(raw), _STORED_MAX):
        piece = raw[at:at + _STORED_MAX]
        out.append(struct.pack("<BHH", 0, len(piece), len(piece) ^ 0xFFFF) + piece)
    return b"".join(out)


def tsv_header(G):
    """The header line of the reference's _simulation.txt: "\tgene_0\tgene_1 ... \n"; pandas writes '""' for a
    frame without columns."""
    if G == 0:
        return b'""\n'
    return ("".join("\tgene_%d" % j for j in range(G)) + "\n").encode("ascii")


class TsvRecord(collections.namedtuple("TsvRecord", "path shape nbytes compressed")):
    """The X of an out="tsv" call: the reference's _simulation.txt on disk, gzipped when `compressed`.  shape is
    (cells, genes); nbytes is the file's size; load() reads it back as the reference's readers do, a
    pandas.DataFrame indexed by the cell names."""
    __slots__ = ()

    def load(self):
        import pandas as pd
        return pd.read_csv(self.path, sep="\t", index_col=0, compression="gzip" if self.compressed else None)


class TsvWriter(object):
    """Writer of one dense tab-separated count table (the reference's _simulation.txt), appended chunk by chunk:
    the header line "\tgene_0 ... \tgene_<G-1>", then one line "cell_<i>\t<count> ... \t<count>" per cell, i the
    global cell index (first + local index).  With compress=True the file is one gzip member with MTIME 0, XFL 0
    and OS 255: the header line as stored blocks, the appended blocks, the final block 03 00, then the CRC-32 (the
    header's combined with the appended text's) and ISIZE.

    append(rows, data, crc, raw_len) takes the text of the next `rows` cells, raw_len bytes: the text itself
    (crc is not used), or with compress=True raw DEFLATE blocks that are not final and end on a byte boundary
    (pst_deflate_blocks' output over pst_tsv_format's text, or sync_deflate's) with the CRC-32 of the text.  As
    CsrShardWriter: everything goes to `<path>.partial`, renamed to `<path>` only by a complete close(); an
    exception inside `with` or abort() leaves nothing behind; an existing `<path>` raises FileExistsError.  The
    same appends give the same bytes."""

    def __init__(self, path, shape, first=0, compress=False):
        self.path = os.fspath(path)
        if os.path.lexists(self.path):
            raise FileExistsError(errno.EEXIST, "the count table exists already", self.path)
        n, G = (int(v) for v in shape)
        self.shape, self.first, self.compress = (n, G), int(first), bool(compress)
        self.rows = 0
        self._partial = self.path + ".partial"
        self._fh = None
        if os.path.lexists(self._partial):              # left behind by an interrupted writer
            os.remove(self._partial)
        try:
            self._fh = open(self._partial, "wb")
            header = tsv_header(G)
            if self.compress:
                self._fh.write(_GZIP_HEADER + _stored_blocks(header))
                self._crc, self._raw = zlib.crc32(header), len(header)
            else:
                self._fh.write(header)
        except BaseException:
            self.abort()
            raise

    def append(self, rows, data, crc, raw_len):
        """The text of the next `rows` cells, raw_len bytes: plain, or as non-final DEFLATE blocks."""
        if self.rows + int(rows) > self.shape[0]:
            raise ValueError("more rows than announced (%d)" % self.shape[0])
        data = memoryview(data).cast("B")
        if not self.compress and len(data) != int(raw_len):
            raise ValueError("%d bytes of text, %d announced" % (len(data), raw_len))
        self._fh.write(data)
        if self.compress:
            self._crc = int(nat.load().pst_host_crc32_combine(self._crc, int(crc) & 0xFFFFFFFF, int(raw_len)))
            self._raw += int(raw_len)
        self.rows += int(rows)

    def close(self):
        """Finish the file and move it to `path`; raises (and leaves nothing) when rows are missing."""
        if self._fh is None:
            return
        try:
            if self.rows != self.shape[0]:
                raise ValueError("%s: %d of %d rows written" % (self.path, self.rows, self.shape[0]))
            if self.compress:
                self._fh.write(_FINAL_BLOCK + struct.pack("<II", self._crc, self._raw & 0xFFFFFFFF))
            self._fh.close()
            self._fh = None
            os.rename(self._partial, self.path)
        except BaseException:
            self.abort()
            raise

    def record(self):
        """The TsvRecord of the closed file."""
        return TsvRecord(self.path, self.shape, os.path.getsize(self.path), self.compress)

    def abort(self):
        """Drop everything written so far."""
        if self._fh is not None:
            self._fh.close()
        self._fh = None
        try:
            os.remove(self._partial)
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


# ---- Parquet (parquet-format's parquet.thrift, serialized with Thrift's compact protocol)
_PQ_MAGIC = b"PAR1"
_PQ_BOOLEAN, _PQ_INT32, _PQ_INT64, _PQ_DOUBLE, _PQ_BYTE_ARRAY = 0, 1, 2, 5, 6      # physical types
_PQ_PLAIN, _PQ_RLE, _PQ_DELTA_BINARY_PACKED = 0, 3, 5                               # encodings
_PQ_UNCOMPRESSED, _PQ_GZIP = 0, 2                                                   # codecs
_PQ_REQUIRED, _PQ_UTF8, _PQ_DATA_PAGE = 0, 0, 0
_PQ_STATS = {_PQ_INT32: "<i", _PQ_INT64: "<q"}                # PLAIN encoding of a min / max statistic
# compact protocol field types
_T_TRUE, _T_I16, _T_I32, _T_I64, _T_BINARY, _T_LIST, _T_STRUCT = 1, 4, 5, 6, 8, 9, 12


def _uleb(v):
    out = bytearray()
    while v >= 0x80:
        out.append((v & 0x7F) | 0x80)
        v >>= 7
    out.append(v)
    return bytes(out)


def _thrift_value(ttype, v):
    if ttype in (_T_I16, _T_I32, _T_I64):
        return _uleb((v << 1) ^ (v >> 63))                 # zigzag
    if ttype == _T_BINARY:
        v = v.encode("utf-8") if isinstance(v, str) else bytes(v)
        return _uleb(len(v)) + v
    if ttype == _T_STRUCT:
        return v                                         # serialized by _thrift_struct
    if ttype == _T_LIST:
        etype, items = v
        head = bytes([(len(items) << 4) | etype]) if len(items) < 15 else bytes([0xF0 | etype]) + _uleb(len(items))
        return head + b"".join(_thrift_value(etype, x) for x in items)
    raise ValueError("thrift type %d is not used here" % ttype)


def _thrift_struct(fields):
    """A struct in Thrift's compact protocol: fields = [(id, type, value)] in ascending id; None values are left
    out (optional fields)."""
    out, last = [], 0
    for fid, ttype, v in fields:
        if v is None:
            continue
        delta = fid - last
        out.append(bytes([(delta << 4) | ttype]) if 0 < delta <= 15 else bytes([ttype]) + _thrift_value(_T_I16, fid))
        out.append(_thrift_value(ttype, v))
        last = fid
    return b"".join(out) + b"\x00"


_EMPTY_STRUCT = _thrift_struct([])


def _pq_page_header(num_values, body_len, page_len, encoding):
    """PageHeader of a V1 data page of a REQUIRED column: no levels, so the page holds the values only."""
    data = _thrift_struct([(1, _T_I32, num_values), (2, _T_I32, encoding), (3, _T_I32, _PQ_RLE), (4, _T_I32, _PQ_RLE)])
    return _thrift_struct([(1, _T_I32, _PQ_DATA_PAGE), (2, _T_I32, body_len), (3, _T_I32, page_len),
                           (5, _T_STRUCT, data)])


def _pq_schema_element(name, ptype=None, string=False, children=None):
    return _thrift_struct([(1, _T_I32, ptype), (3, _T_I32, None if ptype is None else _PQ_REQUIRED),
                           (4, _T_BINARY, name), (5, _T_I32, children), (6, _T_I32, _PQ_UTF8 if string else None),
                           (10, _T_STRUCT, _thrift_struct([(1, _T_STRUCT, _EMPTY_STRUCT)]) if string else None)])


class _ParquetFile(object):
    """One Parquet file written front to back: the magic, row groups of REQUIRED columns with one V1 data page per
    column chunk, then the footer (FileMetaData, its length, the magic) in finish().  columns: [(name, physical
    type, is_string)]; a page comes as its body's pieces (plain, or one gzip member with codec GZIP)."""

    def __init__(self, fh, columns, codec, key_value=()):
        self.fh, self.columns, self.codec, self.key_value = fh, list(columns), codec, list(key_value)
        self.row_groups, self.num_rows = [], 0
        fh.write(_PQ_MAGIC)

    def row_group(self, num_rows, pages):
        """pages: per column (encoding, pieces, body_len, stats), stats None or (min, max) of its values."""
        chunks, start, raw_total, packed_total = [], self.fh.tell(), 0, 0
        for (name, ptype, _), (encoding, pieces, body_len, stats) in zip(self.columns, pages):
            page_len = sum(len(memoryview(p).cast("B")) for p in pieces)
            header = _pq_page_header(num_rows, body_len, page_len, encoding)
            at = self.fh.tell()
            self.fh.write(header)
            for p in pieces:
                self.fh.write(memoryview(p).cast("B"))
            fmt = _PQ_STATS.get(ptype)
            st = None if stats is None else _thrift_struct([
                (3, _T_I64, 0), (5, _T_BINARY, struct.pack(fmt, stats[1])), (6, _T_BINARY, struct.pack(fmt, stats[0]))])
            meta = _thrift_struct([(1, _T_I32, ptype), (2, _T_LIST, (_T_I32, [encoding])), (3, _T_LIST, (_T_BINARY, [name])),
                                   (4, _T_I32, self.codec), (5, _T_I64, num_rows), (6, _T_I64, len(header) + body_len),
                                   (7, _T_I64, len(header) + page_len), (9, _T_I64, at), (12, _T_STRUCT, st)])
            chunks.append(_thrift_struct([(2, _T_I64, at), (3, _T_STRUCT, meta)]))
            raw_total += len(header) + body_len
            packed_total += len(header) + page_len
        self.row_groups.append(_thrift_struct([(1, _T_LIST, (_T_STRUCT, chunks)), (2, _T_I64, raw_total),
                                               (3, _T_I64, num_rows), (5, _T_I64, start), (6, _T_I64, packed_total)]))
        self.num_rows += num_rows

    def finish(self):
        from prosstt_b200 import __version__
        schema = [_pq_schema_element("schema", children=len(self.columns))]
        schema += [_pq_schema_element(name, ptype, string) for name, ptype, string in self.columns]
        kv = [_thrift_struct([(1, _T_BINARY, k), (2, _T_BINARY, v)]) for k, v in self.key_value]
        orders = [_thrift_struct([(1, _T_STRUCT, _EMPTY_STRUCT)])] * len(self.columns)   # TypeDefinedOrder
        footer = _thrift_struct([(1, _T_I32, 2), (2, _T_LIST, (_T_STRUCT, schema)), (3, _T_I64, self.num_rows),
                                 (4, _T_LIST, (_T_STRUCT, self.row_groups)), (5, _T_LIST, (_T_STRUCT, kv) if kv else None),
                                 (6, _T_BINARY, "prosstt_b200 version %s" % __version__),
                                 (7, _T_LIST, (_T_STRUCT, orders))])
        self.fh.write(footer + struct.pack("<I", len(footer)) + _PQ_MAGIC)


def parquet_cells(first, pseudotime, branches, scalings):
    """(columns, [(encoding, body)]) of cells.parquet: the reference's _cellparams.txt as PLAIN columns cell,
    pseudotime, branch (the string form of mtx_cell_params) and scaling."""
    n = len(pseudotime)
    names = np.asarray(branches).astype(str)
    uniq, inv = np.unique(names, return_inverse=True)
    coded = [struct.pack("<I", len(b)) + b for b in (u.encode("utf-8") for u in uniq)]
    columns = [("cell", _PQ_INT64, False), ("pseudotime", _PQ_INT64, False), ("branch", _PQ_BYTE_ARRAY, True),
               ("scaling", _PQ_DOUBLE, False)]
    bodies = [np.arange(first, first + n, dtype="<i8").tobytes(), np.asarray(pseudotime, dtype="<i8").tobytes(),
              b"".join([coded[i] for i in inv.reshape(-1).tolist()]), np.asarray(scalings, dtype="<f8").tobytes()]
    return columns, bodies


class ParquetRecord(collections.namedtuple("ParquetRecord", "path shape nnz nbytes compressed")):
    """The X of an out="parquet" call: a directory with counts.parquet (one row per nonzero count: cell, gene,
    count) and cells.parquet.  shape is (cells, genes) of the call; nbytes is the size of counts.parquet; load()
    reads it back with pyarrow as the cells x genes csr_matrix, with the dtype of its count column."""
    __slots__ = ()

    def load(self):
        import pyarrow.parquet as pq
        counts = pq.ParquetFile(os.path.join(self.path, "counts.parquet"))
        first = int(counts.metadata.metadata[b"prosstt_b200.first_cell"])
        table = counts.read()
        cell, gene, count = (np.array(table.column(c).to_numpy()) for c in ("cell", "gene", "count"))
        n, G = self.shape
        idx = np.int32 if len(cell) < (1 << 31) else np.int64
        indptr = np.zeros(n + 1, dtype=idx)
        np.cumsum(np.bincount(cell - first, minlength=n), out=indptr[1:])
        return _csr_matrix(indptr, gene.astype(idx), count, (n, G))


class ParquetWriter(object):
    """Writer of one Parquet directory, the counts appended chunk by chunk:
      counts.parquet  one row per nonzero count, cell-major, genes ascending in a cell: REQUIRED columns cell INT64
                      (the global cell index first + local index), gene INT32 and count INT64 or INT32 (`dtype`);
                      one row group per appended chunk with nonzeros, each column chunk one V1 DELTA_BINARY_PACKED
                      data page with null_count 0 and its min and max as statistics (TypeDefinedOrder);
                      key-value metadata prosstt_b200.shape "[cells, genes]" and prosstt_b200.first_cell;
      cells.parquet   the reference's _cellparams.txt for these cells as PLAIN columns (parquet_cells).
    compress=True gives every page codec GZIP: one gzip member with MTIME 0, XFL 0 and OS 255.

    append(rows, nnz, pages) takes the next `rows` cells and their `nnz` nonzeros as the pages of the three columns,
    pages = [(data, body_len, crc, min, max)] for cell, gene and count: `data` is the page body of body_len bytes
    (pst_delta_write's), or with compress=True raw DEFLATE blocks that are not final and end on a byte boundary
    (pst_deflate_blocks' output over it, or sync_deflate's) with its CRC-32.  nnz == 0 writes no row group.  As
    CsrShardWriter: everything goes to `<path>.partial`, renamed to `<path>` only by a complete close(); an
    exception inside `with` or abort() leaves nothing behind; an existing `<path>` raises FileExistsError.  The same
    appends give the same bytes."""

    def __init__(self, path, shape, pseudotime, branches, scalings, first=0, dtype=np.int64, compress=False):
        self.path = os.fspath(path)
        if os.path.lexists(self.path):
            raise FileExistsError(errno.EEXIST, "the Parquet directory exists already", self.path)
        n, G = (int(v) for v in shape)
        self.shape, self.first, self.compress = (n, G), int(first), bool(compress)
        self.dtype = np.dtype(dtype)
        if self.dtype not in (np.dtype(np.int32), np.dtype(np.int64)):
            raise ValueError("the count column is int32 or int64, not %s" % self.dtype)
        cells = _csr_cells(n, pseudotime, branches, scalings)
        self.rows, self.nnz = 0, 0
        self._dir = self.path + ".partial"
        self._fh, self._file = None, None
        if os.path.lexists(self._dir):                  # left behind by an interrupted writer
            shutil.rmtree(self._dir)
        os.makedirs(self._dir)
        codec = _PQ_GZIP if self.compress else _PQ_UNCOMPRESSED
        try:
            columns, bodies = parquet_cells(self.first, cells["pseudotime"], cells["branches"], cells["scalings"])
            with open(os.path.join(self._dir, "cells.parquet"), "wb") as fh:
                table = _ParquetFile(fh, columns, codec)
                if n:
                    table.row_group(n, [(_PQ_PLAIN, [gzip_member(b) if self.compress else b], len(b), None)
                                        for b in bodies])
                table.finish()
            self._fh = open(os.path.join(self._dir, "counts.parquet"), "wb")
            count_type = _PQ_INT64 if self.dtype == np.dtype(np.int64) else _PQ_INT32
            self._file = _ParquetFile(self._fh, [("cell", _PQ_INT64, False), ("gene", _PQ_INT32, False),
                                                 ("count", count_type, False)], codec,
                                      [("prosstt_b200.shape", "[%d, %d]" % (n, G)),
                                       ("prosstt_b200.first_cell", "%d" % self.first)])
        except BaseException:
            self.abort()
            raise

    def append(self, rows, nnz, pages=()):
        """The next `rows` cells with their `nnz` nonzeros as the pages of cell, gene and count."""
        if self.rows + int(rows) > self.shape[0]:
            raise ValueError("more rows than announced (%d)" % self.shape[0])
        nnz = int(nnz)
        if nnz:
            if len(pages) != 3:
                raise ValueError("a chunk with nonzeros needs the pages of cell, gene and count")
            out = []
            for data, body_len, crc, vmin, vmax in pages:
                if self.compress:
                    pieces = [_GZIP_HEADER, data, _FINAL_BLOCK + struct.pack("<II", int(crc) & 0xFFFFFFFF,
                                                                             int(body_len) & 0xFFFFFFFF)]
                else:
                    pieces = [data]
                    if len(memoryview(data).cast("B")) != int(body_len):
                        raise ValueError("a page of %d bytes, %d announced" % (len(memoryview(data).cast("B")),
                                                                              body_len))
                out.append((_PQ_DELTA_BINARY_PACKED, pieces, int(body_len), (int(vmin), int(vmax))))
            self._file.row_group(nnz, out)
        self.rows += int(rows)
        self.nnz += nnz

    def close(self):
        """Finish the directory and move it to `path`; raises (and leaves nothing) when rows are missing."""
        if self._fh is None:
            return
        try:
            if self.rows != self.shape[0]:
                raise ValueError("%s: %d of %d rows written" % (self.path, self.rows, self.shape[0]))
            self._file.finish()
            self._fh.close()
            self._fh = None
            os.rename(self._dir, self.path)
        except BaseException:
            self.abort()
            raise

    def record(self):
        """The ParquetRecord of the closed directory."""
        return ParquetRecord(self.path, self.shape, self.nnz,
                             os.path.getsize(os.path.join(self.path, "counts.parquet")), self.compress)

    def abort(self):
        """Drop everything written so far."""
        if self._fh is not None:
            self._fh.close()
        self._fh = None
        shutil.rmtree(self._dir, ignore_errors=True)

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc, tb):
        if exc_type is None:
            self.close()
        else:
            self.abort()
        return False


# ---------------------------------------------------------------------------------------------- AnnData Zarr store
ZARR_CHUNK = 1 << 20            # elements per chunk of every array of a store: 4 or 8 MiB, whole 32 KiB DEFLATE blocks
_ZLIB_HEADER = b"\x78\x01"      # CM 8 (DEFLATE), 32 KiB window, FLEVEL 0, no dictionary
_ZARR_COMPRESSOR = {"id": "zlib", "level": 1}
_ZARR_X = (("indptr", np.dtype("<i8")), ("indices", np.dtype("<i4")), ("data", None))
_ZARR_DICTS = ("obsm", "varm", "obsp", "varp", "layers", "uns")


def _zarr_json(obj):
    return json.dumps(obj, indent=4, sort_keys=True, ensure_ascii=True).encode("ascii")


def zarr_chunks(raw, chunk_bytes, compress):
    """The chunks of an array's raw bytes as ZarrWriter.append takes them, the last zero-padded to chunk_bytes: raw
    bytes, or with compress (raw DEFLATE blocks that are not final, Adler-32, chunk_bytes) made by zlib."""
    raw = bytes(raw)
    out = []
    for at in range(0, len(raw), chunk_bytes):
        piece = raw[at:at + chunk_bytes].ljust(chunk_bytes, b"\0")
        if compress:
            c = zlib.compressobj(1, zlib.DEFLATED, -15)
            piece = (c.compress(piece) + c.flush(zlib.Z_SYNC_FLUSH), zlib.adler32(piece), chunk_bytes)
        out.append(piece)
    return out


def _vlen_utf8(items, size):
    """numcodecs' VLenUTF8 encoding of `items` padded with empty strings to `size` items: the item count, then each
    item's byte length and UTF-8 bytes (little-endian uint32s).  Assembled with NumPy: a chunk holds 2^20 items."""
    coded = [v.encode("utf-8") for v in items]
    lens = np.fromiter(map(len, coded), np.int64, len(coded))
    before = np.cumsum(lens) - lens                          # payload bytes of the items before each one
    out = np.zeros(4 + 4 * size + int(lens.sum()), np.uint8)  # the padding items are zero lengths
    out[:4] = np.frombuffer(struct.pack("<I", size), np.uint8)
    at = 4 + 4 * np.arange(len(coded)) + before              # each item's length field
    for k in range(4):
        out[at + k] = (lens >> (8 * k)) & 0xFF
    out[np.repeat(at + 4 - before, lens) + np.arange(int(lens.sum()))] = np.frombuffer(b"".join(coded), np.uint8)
    return out.tobytes()


def _codes_dtype(categories):
    """pandas' rule for the codes of a categorical: the smallest signed integer type below whose maximum the number
    of categories stays."""
    for dt in (np.int8, np.int16, np.int32):
        if categories < np.iinfo(dt).max:
            return np.dtype(dt)
    return np.dtype(np.int64)


class ZarrRecord(collections.namedtuple("ZarrRecord", "path shape nnz nbytes compressed")):
    """The X of an out="zarr" call: an AnnData Zarr store on disk.  shape is (cells, genes) of the call; nbytes is
    the size of the chunk files of X; load() reads X back as the cells x genes csr_matrix with json, zlib and NumPy
    (anndata.read_zarr(path) reads the whole AnnData)."""
    __slots__ = ()

    def load(self):
        def array(name):
            folder = os.path.join(self.path, "X", name)
            with open(os.path.join(folder, ".zarray")) as fh:
                meta = json.load(fh)
            (length,), (chunk,), dt = meta["shape"], meta["chunks"], np.dtype(meta["dtype"])
            out = np.empty(length, dt)
            for c, at in enumerate(range(0, length, chunk)):
                with open(os.path.join(folder, str(c)), "rb") as fh:
                    raw = fh.read()
                if meta["compressor"] is not None:
                    raw = zlib.decompress(raw)
                piece = np.frombuffer(raw, dt)
                out[at:at + chunk] = piece[:min(chunk, length - at)]
            return out

        indptr, indices, data = (array(name) for name, _ in _ZARR_X)
        idx = np.int32 if len(indices) < (1 << 31) else np.int64
        return _csr_matrix(indptr.astype(idx), indices.astype(idx), data, tuple(self.shape))


class ZarrWriter(object):
    """Writer of one AnnData store in Zarr v2 format (anndata's on-disk specification), X appended chunk by chunk:
      X         csr_matrix group (shape [cells, genes]): indptr int64 (cells + 1 values from 0), indices int32 (genes
                ascending in a cell) and data (`dtype`, int64 or int32);
      obs       dataframe of the reference's _cellparams.txt (tree_utils.cell_params_frame): index cell_<first + i>,
                pseudotime int64, branches categorical (categories the sorted names, codes pandas' smallest type),
                scalings float64;
      var       dataframe with index gene_<j> and no columns;
      obsm, varm, obsp, varp, layers, uns   empty dicts;
      .zmetadata  the consolidated metadata: every .zgroup, .zattrs and .zarray by its key.
    Every array has chunks of ZARR_CHUNK elements (as it was when the writer was made) named 0, 1, ...; the last one
    is stored at full size, zero-padded (empty strings for string arrays).  compress=True gives every array the zlib
    compressor: each chunk file is one zlib stream.  The host writes obs, var and the metadata.

    append(rows, nnz, parts) takes the next `rows` cells and their `nnz` nonzeros as the complete chunks they fill
    (the tail that does not fill a chunk comes with a later append; the last append pads it to a whole chunk), parts =
    [indptr chunks, indices chunks, data chunks]: each chunk is its raw bytes, or with compress=True a tuple (raw
    DEFLATE blocks that are not final and end on a byte boundary, Adler-32 of the raw chunk, raw length), as
    pst_deflate_segments or zarr_chunks make them.  As ParquetWriter: everything goes to `<path>.partial`, renamed to
    `<path>` only by a complete close(), which checks that every array has ceil(length / chunk) chunks; an exception
    inside `with` or abort() leaves nothing behind; an existing `<path>` raises FileExistsError; the same appends
    give the same bytes."""

    def __init__(self, path, shape, pseudotime, branches, scalings, first=0, dtype=np.int64, compress=False):
        self.path = os.fspath(path)
        if os.path.lexists(self.path):
            raise FileExistsError(errno.EEXIST, "the Zarr store exists already", self.path)
        n, G = (int(v) for v in shape)
        self.shape, self.first, self.compress = (n, G), int(first), bool(compress)
        self.dtype = np.dtype(dtype)
        if self.dtype not in (np.dtype(np.int32), np.dtype(np.int64)):
            raise ValueError("X/data is int32 or int64, not %s" % self.dtype)
        self.chunk = int(ZARR_CHUNK)
        self.cells = _csr_cells(n, pseudotime, branches, scalings)
        self.dtypes = [dt or self.dtype.newbyteorder("<") for _, dt in _ZARR_X]
        self.rows, self.nnz, self.chunks = 0, 0, [0, 0, 0]
        self.meta = {}
        self._dir = self.path + ".partial"
        self._open = True
        if os.path.lexists(self._dir):                  # left behind by an interrupted writer
            shutil.rmtree(self._dir)
        try:
            for name, _ in _ZARR_X:
                os.makedirs(os.path.join(self._dir, "X", name))
            if n == 0:                                   # no chunk of cells comes: indptr is [0]
                self.append(0, 0, [zarr_chunks(bytes(8), 8 * self.chunk, self.compress), [], []])
        except BaseException:
            self.abort()
            raise

    def append(self, rows, nnz, parts):
        """The next `rows` cells with their `nnz` nonzeros, as the complete chunks of indptr, indices and data."""
        if self.rows + int(rows) > self.shape[0]:
            raise ValueError("more rows than announced (%d)" % self.shape[0])
        if len(parts) != 3:
            raise ValueError("a chunk needs the chunk lists of indptr, indices and data")
        for j, chunks in enumerate(parts):
            want = self.chunk * self.dtypes[j].itemsize
            for piece in chunks:
                if self.compress:
                    blocks, adler, raw_len = piece
                    if int(raw_len) != want:
                        raise ValueError("a chunk of %d bytes, %d expected" % (raw_len, want))
                    pieces = [_ZLIB_HEADER, blocks, _FINAL_BLOCK, struct.pack(">I", int(adler) & 0xFFFFFFFF)]
                else:
                    if len(memoryview(piece).cast("B")) != want:
                        raise ValueError("a chunk of %d bytes, %d expected" % (len(memoryview(piece).cast("B")), want))
                    pieces = [piece]
                with open(os.path.join(self._dir, "X", _ZARR_X[j][0], str(self.chunks[j])), "wb") as fh:
                    for p in pieces:
                        fh.write(p)
                self.chunks[j] += 1
        self.rows += int(rows)
        self.nnz += int(nnz)

    def _group(self, key, attrs):
        self.meta[key + ".zgroup"] = {"zarr_format": 2}
        self.meta[key + ".zattrs"] = attrs

    def _array(self, key, length, dtype, attrs=None, strings=False):
        self.meta[key + "/.zarray"] = {
            "chunks": [self.chunk], "compressor": _ZARR_COMPRESSOR if self.compress else None,
            "dtype": "|O" if strings else dtype.str, "fill_value": None if strings else (0.0 if dtype.kind == "f" else 0),
            "filters": [{"id": "vlen-utf8"}] if strings else None, "order": "C", "shape": [int(length)],
            "zarr_format": 2}
        if attrs is not None:
            self.meta[key + "/.zattrs"] = attrs

    def _host_array(self, key, values, attrs):
        """A small array the host writes whole: a numeric NumPy array or a list of strings."""
        strings = isinstance(values, list)
        dtype = None if strings else values.dtype.newbyteorder("<")
        self._array(key, len(values), dtype, attrs, strings)
        os.makedirs(os.path.join(self._dir, key), exist_ok=True)
        for c, at in enumerate(range(0, len(values), self.chunk)):
            if strings:
                raw = _vlen_utf8(values[at:at + self.chunk], self.chunk)
            else:
                raw = zarr_chunks(values[at:at + self.chunk].astype(dtype).tobytes(), self.chunk * dtype.itemsize,
                                  False)[0]
            with open(os.path.join(self._dir, key, str(c)), "wb") as fh:
                fh.write(zlib.compress(raw, 1) if self.compress else raw)

    def close(self):
        """Write obs, var and the metadata and move the store to `path`; raises (and leaves nothing) when rows or
        chunks are missing."""
        if not self._open:
            return
        try:
            n, G = self.shape
            if self.rows != n:
                raise ValueError("%s: %d of %d rows written" % (self.path, self.rows, n))
            for j, length in enumerate((n + 1, self.nnz, self.nnz)):
                if self.chunks[j] != -(-length // self.chunk):
                    raise ValueError("%s: X/%s has %d chunks, %d values need %d" % (
                        self.path, _ZARR_X[j][0], self.chunks[j], length, -(-length // self.chunk)))
            array, string_array = ({"encoding-type": e, "encoding-version": "0.2.0"} for e in ("array", "string-array"))
            self._group("", {"encoding-type": "anndata", "encoding-version": "0.1.0"})
            self._group("X/", {"encoding-type": "csr_matrix", "encoding-version": "0.1.0", "shape": [n, G]})
            for j, length in enumerate((n + 1, self.nnz, self.nnz)):
                self._array("X/" + _ZARR_X[j][0], length, self.dtypes[j])
            cells = self.cells
            self._group("obs/", {"_index": "_index", "column-order": ["pseudotime", "branches", "scalings"],
                                 "encoding-type": "dataframe", "encoding-version": "0.2.0"})
            self._host_array("obs/_index", ["cell_%d" % i for i in range(self.first, self.first + n)], string_array)
            self._host_array("obs/pseudotime", cells["pseudotime"], array)
            categories, codes = np.unique(np.asarray(cells["branches"]).astype(str), return_inverse=True)
            self._group("obs/branches/", {"encoding-type": "categorical", "encoding-version": "0.2.0",
                                          "ordered": False})
            self._host_array("obs/branches/categories", [str(c) for c in categories], string_array)
            self._host_array("obs/branches/codes", codes.reshape(-1).astype(_codes_dtype(len(categories))), array)
            self._host_array("obs/scalings", cells["scalings"], array)
            self._group("var/", {"_index": "_index", "column-order": [], "encoding-type": "dataframe",
                                 "encoding-version": "0.2.0"})
            self._host_array("var/_index", ["gene_%d" % j for j in range(G)], string_array)
            for name in _ZARR_DICTS:
                self._group(name + "/", {"encoding-type": "dict", "encoding-version": "0.1.0"})
            for key, value in self.meta.items():
                os.makedirs(os.path.dirname(os.path.join(self._dir, key)), exist_ok=True)
                with open(os.path.join(self._dir, key), "wb") as fh:
                    fh.write(_zarr_json(value))
            with open(os.path.join(self._dir, ".zmetadata"), "wb") as fh:
                fh.write(_zarr_json({"metadata": self.meta, "zarr_consolidated_format": 1}))
            self._open = False
            os.rename(self._dir, self.path)
        except BaseException:
            self.abort()
            raise

    def record(self):
        """The ZarrRecord of the closed store."""
        nbytes = 0
        for name, _ in _ZARR_X:
            folder = os.path.join(self.path, "X", name)
            nbytes += sum(os.path.getsize(os.path.join(folder, f)) for f in os.listdir(folder) if f[0] != ".")
        return ZarrRecord(self.path, self.shape, self.nnz, nbytes, self.compress)

    def abort(self):
        """Drop everything written so far."""
        self._open = False
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
