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
"""
import errno
import os
import shutil

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
    """`<stem><suffix>` for one rank, `<stem>.rank<k>of<w><suffix>` otherwise (suffix ".csr" for CSR shards)."""
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
        self.dtype = np.dtype(dtype)
        if self.dtype not in (np.dtype(np.int32), np.dtype(np.int64)):
            raise ValueError("CSR data must be int32 or int64, not %s" % self.dtype)
        self.index_dtype = np.dtype(np.int32) if n * G < (1 << 31) else np.dtype(np.int64)
        branches = np.asarray(branches)
        if branches.dtype.kind == "O":                   # readable without pickle
            branches = branches.astype(str)
        cells = dict(pseudotime=np.asarray(pseudotime, dtype=np.int64), branches=branches,
                     scalings=np.asarray(scalings, dtype=np.float64))
        for name, a in cells.items():
            if a.shape != (n,):
                raise ValueError("%s must hold one value per cell (%d), not shape %s" % (name, n, a.shape))
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


def load_csr_shard(path):
    """(X, pseudotime, branches, scalings) of a shard written by CsrShardWriter: X is a canonical
    scipy.sparse.csr_matrix over read-only memory maps of indptr, indices and data (no copy)."""
    def member(name, mmap_mode=None):
        return np.load(os.path.join(os.fspath(path), name + ".npy"), mmap_mode=mmap_mode, allow_pickle=False)

    fmt = member("format").item()
    fmt = fmt.decode("ascii") if isinstance(fmt, bytes) else str(fmt)
    if fmt != "csr":
        raise ValueError("expected a csr matrix, found %r" % fmt)
    shape = tuple(int(v) for v in member("shape"))
    X = _csr_matrix(member("indptr", "r"), member("indices", "r"), member("data", "r"), shape)
    return X, member("pseudotime"), member("branches"), member("scalings")
