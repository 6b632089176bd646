"""Device context, device-resident matrices and multi-GPU plumbing.

One process drives one GPU.  ``torch.distributed`` (when the process was
launched by torchrun) is only used to hand the NCCL unique id from rank 0 to
the other ranks; the per-iteration all-reduce itself is issued by the native
library on its own stream (mixemt_b200/csrc/em.cu).
"""
import ctypes
import os
import weakref

import numpy as np

from . import _lib
from ._lib import lib, check, ptr


class Context(object):
    """Owns an ``mxb_ctx`` (device, stream, optional NCCL communicator)."""

    def __init__(self, device=None):
        if lib.mxb_device_count() <= 0:
            raise _lib.MixemtB200Error(
                "mixemt_b200 needs a CUDA device (B200); none is visible and "
                "there is no CPU fallback")
        if device is None:
            device = int(os.environ.get("MIXEMT_B200_DEVICE",
                                        os.environ.get("LOCAL_RANK", "0")))
        self.device = device
        handle = ctypes.c_void_p()
        check(lib.mxb_ctx_create(device, ctypes.byref(handle)))
        self.handle = handle
        self.rank = 0
        self.world = 1

    # -- multi GPU ---------------------------------------------------------
    def init_comm(self, rank, world, uid):
        check(lib.mxb_comm_init(self.handle, ptr(uid), rank, world))
        self.rank, self.world = rank, world

    def init_comm_from_torch(self):
        """Create the NCCL communicator using torch.distributed for rendezvous."""
        import torch
        import torch.distributed as dist
        if not dist.is_initialized():
            backend = "nccl" if torch.cuda.is_available() else "gloo"
            if backend == "nccl":
                torch.cuda.set_device(self.device)
            dist.init_process_group(backend=backend)
        rank, world = dist.get_rank(), dist.get_world_size()
        if world == 1 or self.world > 1:
            return self
        uid = np.zeros(128, dtype=np.uint8)
        if rank == 0:
            check(lib.mxb_comm_unique_id(ptr(uid)))
        box = [uid.tobytes()]
        dist.broadcast_object_list(box, src=0)
        uid = np.frombuffer(box[0], dtype=np.uint8).copy()
        self.init_comm(rank, world, uid)
        return self

    def allreduce_host(self, arr, op="sum"):
        assert arr.dtype == np.float64 and arr.flags["C_CONTIGUOUS"]
        check(lib.mxb_comm_allreduce_host(self.handle, ptr(arr), arr.size,
                                          1 if op == "max" else 0))
        return arr

    # -- misc ----------------------------------------------------------------
    def set_stream(self, cuda_stream):
        check(lib.mxb_ctx_set_stream(self.handle, ctypes.c_void_p(int(cuda_stream))))

    def synchronize(self):
        check(lib.mxb_ctx_synchronize(self.handle))

    def trim(self):
        """Give cached device blocks back to the driver (see mxb_ctx_trim)."""
        check(lib.mxb_ctx_trim(self.handle))

    @property
    def launch_count(self):
        return int(lib.mxb_ctx_launch_count(self.handle))

    def close(self):
        if self.handle:
            lib.mxb_ctx_destroy(self.handle)
            self.handle = None


_default_ctx = None


def get_context():
    """Process-wide default context (created on first use)."""
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context()
    return _default_ctx


def set_context(ctx):
    global _default_ctx
    _default_ctx = ctx


class RowShard(object):
    """Marks a ``DeviceMatrix`` as this rank's contiguous slice of the rows of one
    matrix split over the ranks (``args.b200_shard = "rows"``).  ``lo`` (the slice's
    first global row) and ``n_total`` (rows of all slices) stay ``None`` until a
    consumer needs them; it then computes them once with ``sharding.shard_offsets``."""

    def __init__(self, lo=None, n_total=None):
        self.lo, self.n_total = lo, n_total


class DeviceMatrix(object):
    """A row-major fp64 matrix resident in HBM (``mxb_matrix``).  ``row_shard`` is
    ``None`` for a whole matrix, a :class:`RowShard` for a rows-mode shard."""

    def __init__(self, ctx, handle):
        self.ctx = ctx
        self.handle = handle
        self.row_shard = None
        n, h = ctypes.c_int64(), ctypes.c_int64()
        check(lib.mxb_matrix_shape(handle, ctypes.byref(n), ctypes.byref(h)))
        self.shape = (n.value, h.value)

    @classmethod
    def from_host(cls, ctx, arr):
        arr = _lib.as_f64(arr)
        assert arr.ndim == 2
        handle = ctypes.c_void_p()
        check(lib.mxb_matrix_upload(ctx.handle, ptr(arr), arr.shape[0], arr.shape[1],
                                    ctypes.byref(handle)))
        return cls(ctx, handle)

    @classmethod
    def empty(cls, ctx, n_rows, n_cols):
        handle = ctypes.c_void_p()
        check(lib.mxb_matrix_alloc(ctx.handle, n_rows, n_cols, ctypes.byref(handle)))
        return cls(ctx, handle)

    def to_host(self, out=None):
        if out is None:
            out = _lib.result_empty(self.shape)
        assert out.shape == self.shape and out.dtype == np.float64
        check(lib.mxb_matrix_download(self.ctx.handle, self.handle, ptr(out)))
        return out

    def argmax_rows(self):
        out = np.empty(self.shape[0], dtype=np.int64)
        check(lib.mxb_matrix_argmax_rows(self.ctx.handle, self.handle, ptr(out)))
        return out

    @property
    def data_ptr(self):
        return lib.mxb_matrix_data(self.handle)

    def fold_ranks(self, sub_log=0.0):
        check(lib.mxb_matrix_fold_ranks(self.ctx.handle, self.handle, float(sub_log)))

    def free(self):
        if self.handle:
            lib.mxb_matrix_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


# Device copies of matrices that build_em_matrix handed to the caller as
# read-only ndarrays: run_em on the very same (still read-only) array skips the
# host->device copy.  Keyed by id(); the weakref drops the entry (and the HBM)
# when the host array dies.
_resident = {}


def resident_mode(args=None):
    """Opt-in residency (``args.b200_resident`` or ``MIXEMT_B200_RESIDENT=1``):
    matrices handed to the caller keep their HBM copy and are read-only."""
    return bool(getattr(args, "b200_resident", False)) or \
        os.environ.get("MIXEMT_B200_RESIDENT", "0") == "1"


def remember_resident(host_arr, dev):
    key = id(host_arr)

    def _drop(_ref, key=key):
        ent = _resident.pop(key, None)
        if ent is not None:
            ent[1].free()

    _resident[key] = (weakref.ref(host_arr, _drop), dev)


def lookup_resident(host_arr):
    ent = _resident.get(id(host_arr))
    if ent is None or ent[0]() is not host_arr:
        return None
    if host_arr.flags.writeable:  # caller unlocked it: contents may have changed
        _resident.pop(id(host_arr), None)
        ent[1].free()
        return None
    dev = ent[1]
    return dev if dev.handle and dev.shape == host_arr.shape else None
