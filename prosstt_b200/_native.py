"""ctypes binding of libprosstt_b200.so (include/prosstt_b200.h).

There is no CPU fallback: if the library is missing or no CUDA device is present
every compute entry point raises.  PyTorch is used only for device memory and
streams; the signatures carry raw pointers and sizes."""
import ctypes as C
import os

import numpy as np
import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PST_LIB", os.path.join(_PKG, "libprosstt_b200.so"))   # PST_LIB: developer override

# flag bits (include/prosstt_b200.h)
FLAG_DOMAIN, FLAG_ROW, FLAG_CLAMPED, FLAG_NOZONE, FLAG_SCRATCH = 1, 2, 4, 8, 16
SAMPLER_GAMMA_POISSON, SAMPLER_HYBRID = 0, 1
SAMPLERS = {"gamma_poisson": SAMPLER_GAMMA_POISSON, "hybrid": SAMPLER_HYBRID}

# user-visible stream tags (third Philox counter word); < 0x100 by convention
TAG_DENSITY_U, TAG_SERIES_Z, TAG_PICK_U, TAG_SCALING_Z, TAG_BASE_Z = 1, 2, 3, 4, 5

_p, _i32, _i64, _u32, _u64, _f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_double

_SIGNATURES = {
    "pst_abi_version": (C.c_int, []),
    "pst_last_error": (C.c_char_p, []),
    "pst_launch_count": (_u64, []),
    "pst_uniform_f64": (C.c_int, [_u64, _u32, _i64, _i64, _p, _p]),
    "pst_normal_f64": (C.c_int, [_u64, _u32, _i64, _i64, C.c_double, C.c_double, _p, _p, _p, _p]),
    "pst_philox_words": (C.c_int, [_u64, _u32, _i64, _i64, _p, _p]),
    "pst_walk_draws": (C.c_int, [_u64, _i32, _i32, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "pst_walk_scan": (C.c_int, [_i32, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "pst_walk_carry": (C.c_int, [_i32, _i32, _p, _p, _p, _p, _p]),
    "pst_rel_means": (C.c_int, [_p, _p, _p, _i64, _i64, _i32, _i64, _p, _p, _p, _p, _p]),
    "pst_pearson_anticorr": (C.c_int, [_p, _p, _i64, _i64, _p, _p]),
    "pst_lineage_checks": (C.c_int, [_p, _i64, _i32, _p, _p, _i32, _p, _p, _p, _p, _p, _p]),
    "pst_f64_to_f32": (C.c_int, [_p, _i64, C.c_double, _p, _p]),
    "pst_density_index": (C.c_int, [_p, _i32, _p, _i64, _p, _p, _p, _p, _p, _p]),
    "pst_times_from_normals": (C.c_int, [_p, _i64, _i32, _p, _p]),
    "pst_pick_branch": (C.c_int, [_p, _p, _i64, _i32, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p, _p, _p]),
    "pst_rows_from_branch": (C.c_int, [_p, _p, _i64, _i32, _p, _p, _p, _p, _p, _p]),
    "pst_whole_tree_index": (C.c_int, [_p, _p, _p, _i64, _i64, _i64, _i64, _p, _p, _p, _p]),
    "pst_scalings": (C.c_int, [_p, _i64, _p, _p, _p]),
    "pst_base_gene_exp": (C.c_int, [_u64, _u32, _p, _i64, _f64, _f64, _f64, _i32, _p, _p, _p, _p]),
    "pst_nb_params": (C.c_int, [_p, _p, _p, _i64, _i64, _p, _p, _p]),
    "pst_nb_params_f32": (C.c_int, [_p, _p, _p, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _p]),
    "pst_draw_scratch_words": (_i64, [_i64, _i64, _i64]),
    "pst_draw_scratch_layout": (C.c_int, [_i64, _i64, _i64, _p]),
    "pst_draw_counts": (C.c_int, [_p, _i64, _i64, _p, _p, _p, _p, _u64, _i64, _i64, _p, _i64, _p, _i32, _p, _i64,
                                  _p, _p, _p, _p]),
    "pst_count_stats": (C.c_int, [_p, _i64, _i64, _i64, _p, _p, _p, _p, _p, _p]),
    "pst_transform_counts": (C.c_int, [_p, _i64, _i64, _i64, _p, _i32, _p, _i64, _p]),
    "pst_csr_fill": (C.c_int, [_p, _i64, _i64, _i64, _p, _p, _p, _p, _p]),
    "pst_csr_row_counts": (C.c_int, [_p, _i64, _i64, _i64, _p, _p, _p]),
    "pst_csr_row_offsets": (C.c_int, [_p, _i64, _p, _p]),
    "pst_csr_pack": (C.c_int, [_p, _i64, _i64, _i64, _p, _i64, _p, _i32, _p, _i32, _p, _p, _i64, _p, _p, _p]),
    "pst_store_fill": (C.c_int, [_p, _i64, _i32, _p]),
    "pst_host_widen": (C.c_int, [_p, _i32, _p, _i32, _i64, _i32]),
    "pst_host_widen_stream": (C.c_int, [_p, _i32, _p, _i32, _i64, _i32]),
    "pst_host_stream_stores": (C.c_int, []),
    "pst_host_prepare": (C.c_int, [_p, _i64]),
    "pst_host_apply_overflow": (C.c_int, [_p, _i32, _i64, _i64, _p, _p, _i64]),
    "pst_host_checksum": (_u64, [_p, _i64, _i32]),
    "pst_csr_indptr_bytes": (C.c_int, [_p, _i64, _p, _p, _i32, _p]),
    "pst_mtx_row_bytes": (C.c_int, [_p, _i64, _i64, _i64, _i64, _p, _p]),
    "pst_mtx_format": (C.c_int, [_p, _i64, _i64, _i64, _i64, _p, _i64, _p, _p]),
    "pst_tsv_row_bytes": (C.c_int, [_p, _i64, _i64, _i64, _i64, _p, _p]),
    "pst_tsv_format": (C.c_int, [_p, _i64, _i64, _i64, _i64, _p, _i64, _p, _p]),
    "pst_deflate_bound": (_i64, [_i64, _i32]),
    "pst_deflate_workspace_bytes": (_i64, [_i64, _i32]),
    "pst_deflate_blocks": (C.c_int, [_p, _p, _i64, _i64, _i32, _p, _p, _p, _p, _i64, _p]),
    "pst_deflate_lz_workspace_bytes": (_i64, [_i64, _i32]),
    "pst_deflate_lz_blocks": (C.c_int, [_p, _p, _i64, _i64, _i32, _p, _p, _p, _p, _i64, _p]),
    "pst_crc32": (C.c_int, [_p, _i64, _p, _p]),
    "pst_host_crc32_combine": (_u32, [_u32, _u32, _i64]),
    "pst_narrow_counts": (C.c_int, [_p, _i64, _i64, _i64, _p, _i64, _i32, _i64, _p, _p, _i64, _p, _p]),
}

_lib = None


class NativeError(RuntimeError):
    pass


def load():
    """Load the shared library (no device needed) and bind every declared symbol."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            "prosstt_b200: %s is missing - build it with `python -m prosstt_b200.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    if lib.pst_abi_version() != 2:
        raise NativeError("prosstt_b200: ABI version mismatch")
    _lib = lib
    return lib


def declared_symbols():
    return sorted(_SIGNATURES)


def require_cuda():
    if not torch.cuda.is_available():
        raise NativeError("prosstt_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")


def device(dev=None):
    require_cuda()
    if dev is None:
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device(dev)


class _StreamHandle(int):
    """cudaStream_t as an integer that remembers its device: call() makes that device current
    for the launch (the library launches on the CUDA runtime's current device)."""
    dev = None


def stream_ptr(dev):
    h = _StreamHandle(torch.cuda.current_stream(dev).cuda_stream)
    h.dev = torch.device(dev)
    return h


def ptr(t):
    """Device pointer of a tensor (or None)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "device-contiguous tensor expected"
    return t.data_ptr()


def call(name, *args):
    """Call a C-ABI entry point.  Tensor arguments are passed by device pointer and stay
    referenced until the launch has been issued (never take ptr() of a temporary: the
    caching allocator would hand its block to the next allocation).

    The library launches on the CUDA runtime's current device, so the call runs with the
    device of its stream argument (stream_ptr(dev)) made current, and tensor arguments must
    live on that device: a `device="cuda:1"` request works whatever device the caller's
    thread has selected."""
    lib = load()
    raw, dev = [], None
    for a in args:
        if isinstance(a, _StreamHandle):
            dev = a.dev
    for a in args:
        if isinstance(a, torch.Tensor):
            if dev is None:
                dev = a.device
            elif a.device != dev:
                raise ValueError("%s: a tensor argument lives on %s but the call runs on %s" % (name, a.device, dev))
            raw.append(ptr(a))
        else:
            raw.append(a)
    if dev is not None and dev.index is not None and dev.index != torch.cuda.current_device():
        with torch.cuda.device(dev):
            rc = getattr(lib, name)(*raw)
    else:
        rc = getattr(lib, name)(*raw)
    if rc != 0:
        msg = lib.pst_last_error().decode("utf-8", "replace")
        if rc < 0:
            raise ValueError(msg)
        raise NativeError(msg)


def launch_count():
    return int(load().pst_launch_count())


def to_dev(a, dtype, dev):
    """Host array-like -> contiguous device tensor of the given torch dtype.  The upload goes through a
    pinned buffer of torch's caching host allocator and is asynchronous: a copy straight from pageable
    memory would make the host wait for everything queued on the stream before it (the previous call's
    draw kernel), which serialises host set-up and device work of back-to-back sampler calls."""
    if isinstance(a, torch.Tensor):
        return a.to(device=dev, dtype=dtype).contiguous()
    np_dtype = {torch.float64: np.float64, torch.float32: np.float32, torch.int32: np.int32,
                torch.int64: np.int64}[dtype]
    host = np.ascontiguousarray(np.asarray(a, dtype=np_dtype))
    if host.nbytes == 0 or host.nbytes > (256 << 20):
        return torch.from_numpy(host).to(dev)
    staged = torch.empty(host.shape, dtype=dtype, pin_memory=True)
    staged.numpy()[...] = host
    return staged.to(dev, non_blocking=True)


def split_seed(seed):
    """None -> 64 fresh bits from the global legacy numpy stream (so np.random.seed()
    at the top of a script makes a run reproducible, as with the reference)."""
    if seed is None:
        lo, hi = np.random.randint(0, 2 ** 32, size=2, dtype=np.uint64)
        return int(lo) | (int(hi) << 32)
    return int(seed) & 0xFFFFFFFFFFFFFFFF


def derive_seed(seed, salt):
    """A distinct 64-bit key per purpose (splitmix64 step) so that independent stages
    seeded from one user seed never share a Philox key."""
    z = (int(seed) + 0x9E3779B97F4A7C15 * (int(salt) + 1)) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
    return z ^ (z >> 31)
