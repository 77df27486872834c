"""ctypes binding of libfrcfrc_cuda (include/frcfrc_cuda.h).

This is the Python face of the drop-in boundary: `unifrac()` mirrors the
reference's `unifrac(abnd, tree, weighted)` (frcfrc/unifrac.go:97) over a
flattened tree and CSR abundances, and yields the flat lower-triangle vector in
IterPairs order (common/common.go:21-31).  There is no CPU path: if the CUDA
library is missing or no sm_100 device is present this raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_build", "libfrcfrc_cuda.so")

UNWEIGHTED, WEIGHTED = 0, 1
PATH_AUTO, PATH_FAST, PATH_EXACT = -1, 0, 1
FLAG_NO_D2H = 1
FLAG_UW_BF16 = 2
FLAG_SHARD_EMBED = 4
FLAG_UW_BITS = 8
FLAG_L_TILES = 16  # normalize=0 (-l as coded) may run the key-matched FP32 tiles (within 1e-5, not bit-exact)
FLAG_PRUNE = 32    # run on the subtree the table observes (exact path: the same bytes; fast paths: within 1e-5)
COMM_ID_BYTES = 128

NORM_L_AS_CODED, NORM_DEFAULT, NORM_L_DOCUMENTED = 0, 1, 2  # frc_opts_t.normalize

EXPORTS = ["frc_abi_version", "frc_ctx_create", "frc_ctx_create_multi", "frc_ctx_destroy", "frc_create",
           "frc_create_cross", "frc_next",
           "frc_next_f32", "frc_chunk_exceptions", "frc_restart", "frc_job_info", "frc_destroy", "frc_last_error",
           "frc_plan_bands", "frc_comm_unique_id", "frc_ctx_comm_init"]


class FrcError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libfrcfrc_cuda error {code}: {msg}")
        self.code = code


class _Tree(C.Structure):
    _fields_ = [("n_nodes", C.c_int32), ("parent", C.c_void_p), ("length", C.c_void_p)]


class _Csr(C.Structure):
    _fields_ = [("n_samples", C.c_int64), ("row_ptr", C.c_void_p), ("col", C.c_void_p),
                ("val", C.c_void_p)]


class _Opts(C.Structure):
    _fields_ = [("mode", C.c_int32), ("normalize", C.c_int32), ("path", C.c_int32),
                ("device", C.c_int32), ("rank", C.c_int32), ("world", C.c_int32),
                ("band_rows", C.c_int64), ("flags", C.c_uint32), ("n_devices", C.c_int32),
                ("devices", C.c_void_p)]


class _Info(C.Structure):
    _fields_ = [("path_taken", C.c_int32), ("n_bands_total", C.c_int32), ("n_bands_mine", C.c_int32),
                ("tree_height", C.c_int32), ("n_pairs_total", C.c_int64), ("n_pairs_mine", C.c_int64),
                ("n_nodes_padded", C.c_int64), ("kernel_launches", C.c_int64), ("h2d_ms", C.c_double),
                ("embed_ms", C.c_double), ("pairs_ms", C.c_double), ("fixup_ms", C.c_double),
                ("run_ms", C.c_double), ("h2d_bytes", C.c_int64),
                ("d2h_bytes", C.c_int64), ("embed_bytes", C.c_int64), ("flagged_pairs", C.c_int64),
                ("operand_kind", C.c_int64), ("gather_bytes", C.c_int64), ("n_devices", C.c_int32),
                ("value_bytes", C.c_int32), ("exceptions", C.c_int64), ("create_ms", C.c_double)]


@dataclass
class JobInfo:
    path_taken: int
    n_bands_total: int
    n_bands_mine: int
    tree_height: int
    n_pairs_total: int
    n_pairs_mine: int
    n_nodes_padded: int
    kernel_launches: int
    h2d_ms: float
    embed_ms: float
    pairs_ms: float
    fixup_ms: float
    run_ms: float
    h2d_bytes: int
    d2h_bytes: int
    embed_bytes: int
    flagged_pairs: int
    operand_kind: int
    gather_bytes: int
    n_devices: int
    value_bytes: int
    exceptions: int
    create_ms: float


_lib = None


def lib():
    """Loads the CUDA library; fails loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FrcError(-1, f"{LIB_PATH} is missing: build it with `python -m frackyfrac_b200.build` "
                               "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.frc_abi_version.restype = C.c_int
        L.frc_ctx_create.argtypes = [C.c_int32, C.POINTER(C.c_void_p)]
        L.frc_ctx_create_multi.argtypes = [C.c_int32, C.c_void_p, C.POINTER(C.c_void_p)]
        L.frc_ctx_destroy.argtypes = [C.c_void_p]
        L.frc_ctx_destroy.restype = None
        L.frc_create.argtypes = [C.c_void_p, C.POINTER(_Tree), C.POINTER(_Csr), C.POINTER(_Opts),
                                 C.POINTER(C.c_void_p)]
        L.frc_create_cross.argtypes = [C.c_void_p, C.POINTER(_Tree), C.POINTER(_Csr), C.POINTER(_Csr),
                                       C.POINTER(_Opts), C.POINTER(C.c_void_p)]
        L.frc_next.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.frc_next_f32.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.frc_chunk_exceptions.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]
        L.frc_restart.argtypes = [C.c_void_p]
        L.frc_job_info.argtypes = [C.c_void_p, C.POINTER(_Info)]
        L.frc_destroy.argtypes = [C.c_void_p]
        L.frc_destroy.restype = None
        L.frc_last_error.argtypes = [C.c_void_p]
        L.frc_last_error.restype = C.c_char_p
        L.frc_plan_bands.argtypes = [C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p,
                                     C.c_int64]
        L.frc_plan_bands.restype = C.c_int64
        L.frc_comm_unique_id.argtypes = [C.c_char_p]
        L.frc_ctx_comm_init.argtypes = [C.c_void_p, C.c_char_p, C.c_int32, C.c_int32]
        _lib = L
    return _lib


class Context:
    """Reusable context (streams + memory pools) over one GPU, or over several GPUs of this process
    (`devices`: a list of ordinals, or -1 for every visible sm_100 device)."""

    def __init__(self, device: int = -1, devices=None):
        # several ranks on one host (torchrun): split the host cores between their worker pools (a context over
        # several devices is the only worker of its process group while it runs: it keeps the library's default)
        local_world = int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1)
        saved = os.environ.get("FRC_HOST_THREADS")
        if saved is None and local_world > 1 and devices is None:
            cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
            os.environ["FRC_HOST_THREADS"] = str(max(2, min(16, cores // local_world)))
        h = C.c_void_p()
        try:
            if devices is None:
                rc = lib().frc_ctx_create(device, C.byref(h))
            elif devices == -1:
                rc = lib().frc_ctx_create_multi(-1, None, C.byref(h))
            else:
                ids = np.ascontiguousarray(devices, np.int32)
                rc = lib().frc_ctx_create_multi(len(ids), ids.ctypes.data, C.byref(h))
        finally:
            if saved is None:
                os.environ.pop("FRC_HOST_THREADS", None)
        if rc:
            raise FrcError(rc, lib().frc_last_error(None).decode())
        self.h = h

    def comm_init(self, comm_id: bytes, rank: int, world: int):
        """Collective over the ranks: binds an NCCL communicator to this context."""
        rc = lib().frc_ctx_comm_init(self.h, comm_id, rank, world)
        if rc:
            raise FrcError(rc, lib().frc_last_error(None).decode())

    def close(self):
        if self.h:
            lib().frc_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def comm_unique_id() -> bytes:
    """The 128-byte NCCL id (call on one rank, hand the bytes to the others)."""
    buf = C.create_string_buffer(COMM_ID_BYTES)
    rc = lib().frc_comm_unique_id(buf)
    if rc:
        raise FrcError(rc, lib().frc_last_error(None).decode())
    return buf.raw


def _csr(keep, row_ptr, col, val):
    """A _Csr over contiguous copies of the arrays (appended to `keep` so that they outlive the call)."""
    rp, c, v = (np.ascontiguousarray(row_ptr, np.int64), np.ascontiguousarray(col, np.int32),
                np.ascontiguousarray(val, np.float64))
    if len(c) != len(v) or (len(rp) and rp[-1] != len(c)):
        raise ValueError("CSR arrays are inconsistent")
    keep += [rp, c, v]
    return _Csr(max(len(rp) - 1, 0), rp.ctypes.data if len(rp) else None, c.ctypes.data, v.ctypes.data)


class Job:
    """One unifrac() call.  Iterate `chunks()` for (first_index, ndarray) runs."""

    def __init__(self, parent, length, row_ptr, col, val, *, weighted: bool, normalize=True,
                 path: int = PATH_AUTO, ctx: Context | None = None, device: int = -1, rank: int = 0,
                 world: int = 1, band_rows: int = 0, flags: int = 0, devices=None, query=None):
        """normalize: True / 1 = default; False / 0 = flag -l as CODED in the reference (unsorted merge-join:
        the bit-exact list walk, or with flags=FLAG_L_TILES the key-matched FP32 tiles wherever `path` picks the
        fast kernels); 2 = flag -l as documented.  devices: None = one GPU (`device` or the context's);
        a list of ordinals or -1 (all) = this process drives several GPUs, one ordered stream.
        query: (row_ptr, col, val) of a second table = frc_create_cross: the table above is the reference and the
        stream is the query-major n_q x n_ref block, flat index q * n_ref + r (band_rows counts query rows)."""
        self._keep = [np.ascontiguousarray(parent, np.int32), np.ascontiguousarray(length, np.float64)]
        p, l = self._keep
        if len(p) != len(l):
            raise ValueError("parent and length differ in size")
        t = _Tree(len(p), p.ctypes.data, l.ctypes.data)
        a = _csr(self._keep, row_ptr, col, val)
        q = None if query is None else _csr(self._keep, *query)
        norm = int(normalize) if not isinstance(normalize, bool) else (1 if normalize else 0)
        ids = None
        if devices is None:
            nd, dp = 0, None
        elif devices == -1:
            nd, dp = -1, None
        else:
            ids = np.ascontiguousarray(devices, np.int32)
            nd, dp = len(ids), ids.ctypes.data
        o = _Opts(WEIGHTED if weighted else UNWEIGHTED, norm, path, device, rank, world, band_rows, flags, nd, dp)
        self.h = C.c_void_p()
        self.flags = flags
        self.ctx = ctx
        if q is None:
            rc = lib().frc_create(ctx.h if ctx else None, C.byref(t), C.byref(a), C.byref(o), C.byref(self.h))
        else:
            rc = lib().frc_create_cross(ctx.h if ctx else None, C.byref(t), C.byref(a), C.byref(q), C.byref(o),
                                        C.byref(self.h))
        if rc:
            self.h = None
            raise FrcError(rc, lib().frc_last_error(None).decode())
        self._keep = None  # inputs were copied

    def next_raw(self):
        """(address, first_index, count) of the next float64 chunk; count == 0 at the end."""
        d, f, n = C.c_void_p(), C.c_int64(), C.c_int64()
        rc = lib().frc_next(self.h, C.byref(d), C.byref(f), C.byref(n))
        if rc:
            raise FrcError(rc, lib().frc_last_error(self.h).decode())
        return d.value, f.value, n.value

    def next_raw_f32(self):
        """(address, first_index, count) of the next float32 band (fast paths); count == 0 at the end."""
        d, f, n = C.c_void_p(), C.c_int64(), C.c_int64()
        rc = lib().frc_next_f32(self.h, C.byref(d), C.byref(f), C.byref(n))
        if rc:
            raise FrcError(rc, lib().frc_last_error(self.h).decode())
        return d.value, f.value, n.value

    def exceptions(self):
        """(flat indices, float64 values) of the last float32 band that fp32 could not carry."""
        i, v, n = C.c_void_p(), C.c_void_p(), C.c_int64()
        rc = lib().frc_chunk_exceptions(self.h, C.byref(i), C.byref(v), C.byref(n))
        if rc:
            raise FrcError(rc, lib().frc_last_error(self.h).decode())
        if n.value == 0:
            return np.zeros(0, np.int64), np.zeros(0, np.float64)
        return (np.ctypeslib.as_array(C.cast(i, C.POINTER(C.c_int64)), shape=(n.value,)).copy(),
                np.ctypeslib.as_array(C.cast(v, C.POINTER(C.c_double)), shape=(n.value,)).copy())

    def chunks(self, copy: bool = True):
        if self.flags & FLAG_NO_D2H:
            raise RuntimeError("chunks() needs host output; this job keeps distances in HBM")
        while True:
            addr, first, n = self.next_raw()
            if n == 0:
                return
            a = np.ctypeslib.as_array(C.cast(addr, C.POINTER(C.c_double)), shape=(n,))
            yield first, (a.copy() if copy else a)

    def chunks_f32(self, copy: bool = True):
        """Float32 bands of a fast-path job straight from the pinned ring (no host widening pass)."""
        if self.flags & FLAG_NO_D2H:
            raise RuntimeError("chunks_f32() needs host output; this job keeps distances in HBM")
        while True:
            addr, first, n = self.next_raw_f32()
            if n == 0:
                return
            a = np.ctypeslib.as_array(C.cast(addr, C.POINTER(C.c_float)), shape=(n,))
            yield first, (a.copy() if copy else a)

    def drain(self, f32=None) -> int:
        """Runs the stream to its end without touching the data; returns pairs seen.  f32: which call
        to drain with (default: the job's native format: float32 on the fast paths)."""
        if f32 is None:
            f32 = self.info().value_bytes == 4
        nxt = self.next_raw_f32 if f32 else self.next_raw
        total = 0
        while True:
            _, _, n = nxt()
            if n == 0:
                return total
            total += n

    def restart(self):
        rc = lib().frc_restart(self.h)
        if rc:
            raise FrcError(rc, lib().frc_last_error(self.h).decode())

    def info(self) -> JobInfo:
        i = _Info()
        lib().frc_job_info(self.h, C.byref(i))
        return JobInfo(*[getattr(i, f[0]) for f in _Info._fields_])

    def close(self):
        if self.h:
            lib().frc_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def plan_bands(n_samples: int, rank: int = 0, world: int = 1, band_rows: int = 0, flags: int = 0):
    """(first_index, count) of the bands `rank` yields, in stream order (host-only helper)."""
    n = lib().frc_plan_bands(n_samples, band_rows, rank, world, flags, None, None, 0)
    if n < 0:
        raise FrcError(-n, "bad band plan arguments")
    first = np.zeros(n, np.int64)
    count = np.zeros(n, np.int64)
    lib().frc_plan_bands(n_samples, band_rows, rank, world, flags, first.ctypes.data, count.ctypes.data, n)
    return first, count


def unifrac(parent, length, row_ptr, col, val, weighted: bool, normalize=True, **kw) -> np.ndarray:
    """All n(n-1)/2 distances (this rank's bands; zeros elsewhere when world > 1)."""
    n = max(len(row_ptr) - 1, 0)
    out = np.zeros(n * (n - 1) // 2 if n >= 2 else 0, np.float64)
    with Job(parent, length, row_ptr, col, val, weighted=weighted, normalize=normalize, **kw) as job:
        for first, a in job.chunks(copy=False):
            out[first:first + len(a)] = a
    return out


def unifrac_cross(parent, length, ref, query, weighted: bool, normalize=True, **kw) -> np.ndarray:
    """The (n_q, n_ref) distances between every query sample and every reference sample (frc_create_cross);
    ref and query are (row_ptr, col, val) tables over the same tree."""
    n_ref, n_q = max(len(ref[0]) - 1, 0), max(len(query[0]) - 1, 0)
    out = np.zeros(n_q * n_ref, np.float64)
    with Job(parent, length, *ref, weighted=weighted, normalize=normalize, query=query, **kw) as job:
        for first, a in job.chunks(copy=False):
            out[first:first + len(a)] = a
    return out.reshape(n_q, n_ref)
