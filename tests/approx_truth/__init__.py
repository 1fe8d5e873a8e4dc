"""Ground truth of approximate search for the tests (approx_truth.c, a scan of every window): compiled with the host C
compiler into a per-user temporary directory on first use, so the test tree itself is never written."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "approx_truth.c")
_lib = None
_u8p, _u32p, _u64p = C.POINTER(C.c_uint8), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        with open(_SRC, "rb") as f:
            tag = hashlib.sha256(f.read()).hexdigest()[:16]
        d = os.path.join(tempfile.gettempdir(), f"kmer_b200_approx_truth_{os.getuid()}")
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, f"libapprox_truth_{tag}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            subprocess.run([os.environ.get("CC", "gcc"), "-O3", "-march=native", "-fPIC", "-std=c11", "-Wall", "-shared",
                            "-o", tmp, _SRC, "-lpthread"], check=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.approx_truth_batch.restype = C.c_int
        L.approx_truth_batch.argtypes = [_u8p, C.c_uint64, _u8p, _u64p, C.c_uint64, C.c_uint32, C.c_uint32, _u64p,
                                         C.POINTER(_u32p), _u64p]
        L.approx_truth_free.argtypes = [C.c_void_p]
        _lib = L
    return _lib


def truth_approx(text, q_ranks, q_offsets, e: int, n_threads: int = 0):
    """(offsets, positions, status) of approximate search by scanning every window: per query, the ascending p with
    p + m <= n and at most e mismatching symbols in T[p, p+m). Status is 2 (undefined) for an empty query, else 0."""
    L = lib()
    t = np.ascontiguousarray(np.asarray(text, dtype=np.uint8))
    q = np.ascontiguousarray(np.asarray(q_ranks, dtype=np.uint8))
    off = np.ascontiguousarray(np.asarray(q_offsets, dtype=np.uint64))
    Q = off.size - 1
    counts = np.zeros(Q, dtype=np.uint64)
    pos = _u32p()
    total = C.c_uint64(0)
    L.approx_truth_batch(t.ctypes.data_as(_u8p), t.size, q.ctypes.data_as(_u8p), off.ctypes.data_as(_u64p), Q, int(e),
                         n_threads or (os.cpu_count() or 1), counts.ctypes.data_as(_u64p), C.byref(pos), C.byref(total))
    offsets = np.zeros(Q + 1, dtype=np.uint64)
    np.cumsum(counts, out=offsets[1:])
    positions = np.ctypeslib.as_array(pos, shape=(total.value,)).copy() if total.value else np.zeros(0, np.uint32)
    L.approx_truth_free(C.cast(pos, C.c_void_p))
    status = np.where(off[1:] == off[:-1], 2, 0).astype(np.uint8)
    return offsets, positions, status
