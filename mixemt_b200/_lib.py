"""ctypes binding of libmixemt_b200.so (the C-ABI declared in include/mixemt_b200.h).

There is no CPU fallback: if the shared library has not been built the import
fails loudly, and every compute entry point raises when no CUDA device is
visible.
"""
import ctypes
import os
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libmixemt_b200.so")

MXB_OK, MXB_ERR_CUDA, MXB_ERR_ARG, MXB_ERR_VALUE, MXB_ERR_KEY, MXB_ERR_NOMEM, \
    MXB_ERR_RANGE = range(7)
MXB_EM_SHARDED = 1
MXB_EM_RAW = 2

c_void_pp = ctypes.POINTER(ctypes.c_void_p)
c_i64 = ctypes.c_int64
c_i32 = ctypes.c_int32
c_dbl = ctypes.c_double
P = ctypes.c_void_p  # every buffer / handle crosses the ABI as a plain pointer


class LibraryMissing(ImportError):
    pass


def _load():
    if not os.path.isfile(LIB_PATH):
        raise LibraryMissing(
            "%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C mixemt_b200/csrc` (there is no CPU fallback)" % LIB_PATH)
    # Let the dlopen("libnccl.so.2") inside the library find torch's bundled NCCL.
    if "MXB_NCCL_LIB" not in os.environ:
        try:
            import nvidia.nccl  # type: ignore
            for base in nvidia.nccl.__path__:
                cand = os.path.join(base, "lib", "libnccl.so.2")
                if os.path.isfile(cand):
                    os.environ["MXB_NCCL_LIB"] = cand
                    break
        except Exception:  # pragma: no cover - NCCL is optional for 1 GPU
            pass
    return ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)


lib = _load()

# name -> (restype, argtypes); mirrors include/mixemt_b200.h one to one.
_PROTOS = {
    "mxb_abi_version": (ctypes.c_int, []),
    "mxb_last_error": (ctypes.c_char_p, []),
    "mxb_device_count": (ctypes.c_int, []),
    "mxb_ctx_create": (ctypes.c_int, [ctypes.c_int, c_void_pp]),
    "mxb_ctx_destroy": (ctypes.c_int, [P]),
    "mxb_ctx_set_stream": (ctypes.c_int, [P, P]),
    "mxb_ctx_synchronize": (ctypes.c_int, [P]),
    "mxb_ctx_trim": (ctypes.c_int, [P]),
    "mxb_ctx_mem_stats": (ctypes.c_int, [P, ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)]),
    "mxb_ctx_launch_count": (c_i64, [P]),
    "mxb_host_alloc": (ctypes.c_int, [ctypes.c_size_t, ctypes.c_int, c_void_pp]),
    "mxb_host_free": (ctypes.c_int, [P]),
    "mxb_host_reserve": (ctypes.c_int, [ctypes.c_size_t, ctypes.c_int]),
    "mxb_host_trim": (ctypes.c_int, []),
    "mxb_stage_timing": (ctypes.c_int, [ctypes.c_int]),
    "mxb_stage_times": (ctypes.c_int, [P, ctypes.c_int]),
    "mxb_comm_unique_id": (ctypes.c_int, [P]),
    "mxb_comm_init": (ctypes.c_int, [P, P, ctypes.c_int, ctypes.c_int]),
    "mxb_comm_destroy": (ctypes.c_int, [P]),
    "mxb_comm_p2p_enabled": (ctypes.c_int, [P]),
    "mxb_comm_allreduce_host": (ctypes.c_int, [P, P, c_i64, ctypes.c_int]),
    "mxb_sig_count": (ctypes.c_int, [P, P, c_i64, P]),
    "mxb_sig_parse": (ctypes.c_int, [P, P, c_i64, P, c_i64, P, P, P, P,
                                     ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)]),
    "mxb_reduce_reads": (ctypes.c_int, [P, P, P, c_i64, c_void_pp]),
    "mxb_sigset_sizes": (ctypes.c_int, [P, ctypes.POINTER(c_i64), ctypes.POINTER(c_i64),
                                        ctypes.POINTER(c_i64)]),
    "mxb_sigset_export": (ctypes.c_int, [P, P, P, P, P, P, P, P, P, P]),
    "mxb_sigset_destroy": (ctypes.c_int, [P]),
    "mxb_phylo_pack": (ctypes.c_int, [P, c_i32, c_i32, c_i32, P, P, P, P, P, P, c_void_pp]),
    "mxb_phylo_destroy": (ctypes.c_int, [P]),
    "mxb_build_matrix": (ctypes.c_int, [P, P, c_i64, P, P, P, P, P, P, c_void_pp,
                                        ctypes.POINTER(ctypes.c_float)]),
    "mxb_matrix_alloc": (ctypes.c_int, [P, c_i64, c_i64, c_void_pp]),
    "mxb_matrix_upload": (ctypes.c_int, [P, P, c_i64, c_i64, c_void_pp]),
    "mxb_matrix_download": (ctypes.c_int, [P, P, P]),
    "mxb_matrix_shape": (ctypes.c_int, [P, ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)]),
    "mxb_matrix_data": (P, [P]),
    "mxb_matrix_argmax_rows": (ctypes.c_int, [P, P, P]),
    "mxb_matrix_destroy": (ctypes.c_int, [P]),
    "mxb_matrix_gather_cols": (ctypes.c_int, [P, P, P, c_i64, c_void_pp]),
    "mxb_matrix_vote_count": (ctypes.c_int, [P, P, P, P, P]),
    "mxb_matrix_vote_first": (ctypes.c_int, [P, P, P, c_i64, P, P]),
    "mxb_assign_reads": (ctypes.c_int, [P, P, P, P, c_i32, c_dbl, P]),
    "mxb_matrix_download_rows": (ctypes.c_int, [P, P, c_i64, c_i64, P]),
    "mxb_matrix_upload_rows": (ctypes.c_int, [P, P, c_i64, c_i64, P]),
    "mxb_matrix_fold_ranks": (ctypes.c_int, [P, P, c_dbl]),
    "mxb_em_create": (ctypes.c_int, [P, P, P, ctypes.c_int, c_void_pp]),
    "mxb_em_destroy": (ctypes.c_int, [P]),
    "mxb_em_set_lnprops": (ctypes.c_int, [P, P]),
    "mxb_em_iterate": (ctypes.c_int, [P, c_i64, c_dbl, ctypes.POINTER(c_i64),
                                      ctypes.POINTER(c_i32)]),
    "mxb_em_pass_bytes": (ctypes.c_int, [P, ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)]),
    "mxb_tile_plan": (ctypes.c_int, [P, c_i64, c_i64, c_i32, P, c_i64, P, P, P, P, P]),
    "mxb_em_iterate_fixed": (ctypes.c_int, [P, c_i64, ctypes.POINTER(ctypes.c_float),
                                            ctypes.POINTER(ctypes.c_float)]),
    "mxb_em_profile": (ctypes.c_int, [P, c_i64, ctypes.POINTER(ctypes.c_float)]),
    "mxb_em_get_lnprops": (ctypes.c_int, [P, ctypes.c_int, P]),
    "mxb_em_read_mix": (ctypes.c_int, [P, P, ctypes.c_int, c_dbl]),
    "mxb_run_em": (ctypes.c_int, [P, P, P, c_i64, c_i64, P, c_i32, c_i64, c_dbl, c_i32,
                                  P, P, P, P]),
    "mxb_run_em_dev": (ctypes.c_int, [P, P, P, P, c_i32, c_i64, c_dbl, c_i32, P, P,
                                      c_void_pp, P, P]),
    "mxb_em_step": (ctypes.c_int, [P, P, P, P, c_i64, c_i64, P, P]),
    "mxb_boot_counts": (ctypes.c_int, [P, P, c_i64, ctypes.c_uint64, c_i64, c_i64, P]),
    "mxb_em_bootstrap": (ctypes.c_int, [P, P, P, P, c_i64, c_i64, ctypes.c_uint64, c_i64, c_dbl,
                                        P, P, P, ctypes.POINTER(c_i32)]),
    "mxb_boot_slots": (ctypes.c_int, [P, c_i64, c_i64, c_i32, c_dbl, c_dbl,
                                      ctypes.POINTER(c_i32)]),
}

EXPORTED_SYMBOLS = tuple(sorted(_PROTOS))

for _name, (_res, _args) in _PROTOS.items():
    _fn = getattr(lib, _name)
    _fn.restype = _res
    _fn.argtypes = _args


class MixemtB200Error(RuntimeError):
    """CUDA / NCCL / argument failure inside the native library."""


class NumericRangeError(MixemtB200Error, ArithmeticError):
    pass


def last_error():
    msg = lib.mxb_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc, what=""):
    """Turn a non-zero status into the exception the reference would raise
    (ValueError / KeyError, SURVEY.md 8b) or a MixemtB200Error."""
    if rc == MXB_OK:
        return
    msg = last_error() or what
    if rc == MXB_ERR_VALUE:
        raise ValueError(msg)
    if rc == MXB_ERR_KEY:
        raise KeyError(msg)
    if rc == MXB_ERR_NOMEM:
        raise MemoryError(msg)
    if rc == MXB_ERR_RANGE:
        raise NumericRangeError(msg)
    raise MixemtB200Error("%s (status %d)" % (msg, rc))


def ptr(arr):
    """Host pointer of a C-contiguous numpy array (None -> NULL)."""
    if arr is None:
        return None
    assert arr.flags["C_CONTIGUOUS"], "array must be C-contiguous"
    return ctypes.c_void_p(arr.ctypes.data)


def as_f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


# ---- results in pooled pinned host memory (mxb_host_alloc) -----------------------------
_PIN_MIN_BYTES = 32 << 20


def pinned_mode():
    """``MIXEMT_B200_PINNED``: ``0`` results are plain numpy arrays; ``1`` every
    matrix-sized result lives in a pooled pinned block (the first one of a size
    pays for the pinning, about a second per 6 GB); default ``auto``: pinned
    when the pool holds a block that fits (``reserve_pinned`` or an earlier
    pinned result put it there), pageable otherwise."""
    return os.environ.get("MIXEMT_B200_PINNED", "auto")


def result_empty(shape, dtype=np.float64):
    """An uninitialised C-contiguous result array, in pooled pinned host memory
    when the mode allows it (see :func:`pinned_mode`), else ``np.empty``.
    The block goes back to the pool when the array (and every view of it) dies."""
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    mode = pinned_mode()
    if mode != "0" and nbytes >= _PIN_MIN_BYTES:
        out = ctypes.c_void_p()
        check(lib.mxb_host_alloc(nbytes, 0 if mode == "1" else 1, ctypes.byref(out)))
        if out.value:
            buf = (ctypes.c_char * nbytes).from_address(out.value)
            weakref.finalize(buf, lib.mxb_host_free, ctypes.c_void_p(out.value))
            return np.frombuffer(buf, dtype=dtype).reshape(shape)
    return np.empty(shape, dtype=dtype)


def reserve_pinned(nbytes, count=1):
    """Pin ``count`` blocks of ``nbytes`` ahead of time and leave them in the
    pool (what a long-running service does once; results of that size are then
    downloaded by plain DMA from the first call on)."""
    check(lib.mxb_host_reserve(int(nbytes), int(count)))


def trim_pinned():
    check(lib.mxb_host_trim())
