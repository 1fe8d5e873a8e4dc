"""TEST INFRASTRUCTURE ONLY: ctypes bindings for the two CPU checkers.

* ``Oracle``     -> oracle/libkmer_oracle.so   (oracle/kmer_oracle.c, our C restatement)
* ``Reference``  -> oracle/_ref/libkmer_ref.so (the reference itself, oracle/ref_driver.cpp)

Both expose the same batch contract: ``search(q_ranks, q_offsets) -> (offsets, positions, status)``
with ``status`` 0 = OK, 1 = the reference threw std::invalid_argument, 2 = undefined/other.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(_HERE, "libkmer_oracle.so")
REF_SO = os.path.join(_HERE, "_ref", "libkmer_ref.so")

_u8p = C.POINTER(C.c_uint8)
_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)


def build(quiet: bool = True) -> None:
    """Compile the checkers (gcc/g++ only). Building the checker is not using it."""
    subprocess.run(["make", "-C", _HERE, "all"], check=True,
                   stdout=subprocess.DEVNULL if quiet else None)


def have_reference() -> bool:
    return os.path.exists(REF_SO)


def hit_digests(offsets, positions) -> np.ndarray:
    """One 64-bit digest per query of its CSR hit list (positions and their order): what the stored reference answers
    of tests/golden/live/ keep instead of the lists, which would not fit there."""
    offsets = np.asarray(offsets, dtype=np.uint64)
    counts = np.diff(offsets).astype(np.int64)
    out = np.zeros(counts.size, dtype=np.uint64)
    if positions.size == 0:
        return out
    rank = np.arange(positions.size, dtype=np.uint64) - np.repeat(offsets[:-1], counts)
    with np.errstate(over="ignore"):
        w = (np.asarray(positions, dtype=np.uint64) + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15) + \
            (rank + np.uint64(1)) * np.uint64(0xC2B2AE3D27D4EB4F)
        w ^= w >> np.uint64(29)
        w *= np.uint64(0xBF58476D1CE4E5B9)
        w ^= w >> np.uint64(32)
        nz = counts > 0
        out[nz] = np.add.reduceat(w, offsets[:-1][nz].astype(np.int64))
    return out


def _ptr(a: np.ndarray, t):
    return a.ctypes.data_as(t)


def _as_u8(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.uint8))


def _as_u64(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.uint64))


class _Base:
    _prefix = ""
    _lib = None

    def __init__(self):
        self._h = None

    def close(self):
        if self._h:
            getattr(self._lib, self._prefix + "_destroy")(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def scheme(self, m: int):
        out = np.zeros(4096, dtype=np.uint32)
        use_multi = C.c_int(0)
        n = getattr(self._lib, self._prefix + "_scheme")(self._h, m, _ptr(out, _u32p), out.size, C.byref(use_multi))
        return [int(x) for x in out[:n]], bool(use_multi.value)


def _finish(counts, status, pos_ptr, total, free_fn, keep):
    offsets = np.zeros(counts.size + 1, dtype=np.uint64)
    np.cumsum(counts, out=offsets[1:])
    if keep and total:
        positions = np.ctypeslib.as_array(pos_ptr, shape=(total,)).copy()
    else:
        positions = np.zeros(0, dtype=np.uint32)
    if pos_ptr:
        free_fn(pos_ptr)
    return offsets, positions, status


class Oracle(_Base):
    """The C restatement (oracle/kmer_oracle.c)."""
    _prefix = "ko"

    @classmethod
    def lib(cls):
        if cls._lib is None:
            if not os.path.exists(ORACLE_SO):
                build()
            L = C.CDLL(ORACLE_SO)
            L.ko_create.restype = C.c_void_p
            L.ko_create.argtypes = [_u8p, C.c_uint64, C.c_uint32, _u32p, C.c_uint32]
            L.ko_create_restricted.restype = C.c_void_p
            L.ko_create_restricted.argtypes = [_u8p, C.c_uint64, C.c_uint32, _u32p, C.c_uint32, _u8p, _u64p, C.c_uint64,
                                               C.c_uint32]
            L.ko_restricted_misses.restype = C.c_uint64
            L.ko_destroy.argtypes = [C.c_void_p]
            L.ko_search_batch.restype = C.c_int
            L.ko_search_batch.argtypes = [C.c_void_p, _u8p, _u64p, C.c_uint64, C.c_uint32, _u64p, _u8p,
                                          C.POINTER(_u32p), _u64p, C.c_int]
            L.ko_free.argtypes = [C.c_void_p]
            L.ko_scheme.restype = C.c_uint64
            L.ko_scheme.argtypes = [C.c_void_p, C.c_uint64, _u32p, C.c_uint64, C.POINTER(C.c_int)]
            L.ko_fast_pow.restype = C.c_uint64
            L.ko_fast_pow.argtypes = [C.c_uint64, C.c_uint8]
            L.ko_hash.restype = C.c_uint64
            L.ko_hash.argtypes = [_u8p, C.c_uint32, C.c_uint32]
            L.ko_element_size.restype = C.c_uint64
            L.ko_element_size.argtypes = [C.c_void_p, C.c_uint32]
            L.ko_element_positions.restype = _u32p
            L.ko_element_positions.argtypes = [C.c_void_p, C.c_uint32]
            L.ko_element_hashes.restype = _u64p
            L.ko_element_hashes.argtypes = [C.c_void_p, C.c_uint32]
            L.ko_truth_search_batch.restype = C.c_int
            L.ko_truth_search_batch.argtypes = [_u8p, C.c_uint64, _u8p, _u64p, C.c_uint64, _u64p,
                                                C.POINTER(_u32p), _u64p]
            L.ko_choose_best_k.restype = C.c_uint64
            L.ko_choose_best_k.argtypes = [_u64p, C.c_uint64, C.c_uint64, _u64p]
            cls._lib = L
        return cls._lib

    def __init__(self, text, sigma: int, ks, restrict_to=None, n_threads: int = 0):
        """restrict_to=(q_ranks, q_offsets): hold only the buckets that batch can ask for (ko_create_restricted) --
        same answers for that batch, a fraction of the memory; `restricted_misses()` must stay 0."""
        super().__init__()
        L = self.lib()
        self.text = _as_u8(text)
        self.sigma = int(sigma)
        self.ks = [int(k) for k in ks]
        ks_a = np.asarray(self.ks, dtype=np.uint32)
        if restrict_to is None:
            self._h = L.ko_create(_ptr(self.text, _u8p), self.text.size, self.sigma, _ptr(ks_a, _u32p), ks_a.size)
        else:
            q, off = _as_u8(restrict_to[0]), _as_u64(restrict_to[1])
            self._h = L.ko_create_restricted(_ptr(self.text, _u8p), self.text.size, self.sigma, _ptr(ks_a, _u32p),
                                             ks_a.size, _ptr(q, _u8p), _ptr(off, _u64p), off.size - 1,
                                             n_threads or (os.cpu_count() or 1))
        if not self._h:
            raise ValueError(f"oracle: illegal index sigma={sigma} ks={ks} n={self.text.size}")

    def search(self, q_ranks, q_offsets, n_threads: int = 0, keep_positions: bool = True):
        L = self.lib()
        q = _as_u8(q_ranks)
        off = _as_u64(q_offsets)
        Q = off.size - 1
        counts = np.zeros(Q, dtype=np.uint64)
        status = np.zeros(Q, dtype=np.uint8)
        pos = _u32p()
        total = C.c_uint64(0)
        L.ko_search_batch(self._h, _ptr(q, _u8p), _ptr(off, _u64p), Q, n_threads or (os.cpu_count() or 1),
                          _ptr(counts, _u64p), _ptr(status, _u8p), C.byref(pos), C.byref(total),
                          1 if keep_positions else 0)
        self.last_ub = (status & 0x80) != 0     # queries on which the reference dereferences end() (UB)
        status &= 0x7F
        return _finish(counts, status, pos, total.value, L.ko_free, keep_positions)

    @classmethod
    def restricted_misses(cls) -> int:
        """Lookups (process-wide) that asked a restricted index for a bucket it does not hold; must be 0."""
        return int(cls.lib().ko_restricted_misses())

    def element(self, i: int):
        """(sorted hashes, positions stably sorted by hash) of element i (template order)."""
        L = self.lib()
        n = L.ko_element_size(self._h, i)
        h = np.ctypeslib.as_array(L.ko_element_hashes(self._h, i), shape=(n,)).copy()
        p = np.ctypeslib.as_array(L.ko_element_positions(self._h, i), shape=(n,)).copy()
        return h, p

    @classmethod
    def fast_pow(cls, base: int, exp: int) -> int:
        return int(cls.lib().ko_fast_pow(base, exp))

    @classmethod
    def hash(cls, ranks, sigma: int) -> int:
        r = _as_u8(ranks)
        return int(cls.lib().ko_hash(_ptr(r, _u8p), r.size, sigma))

    @classmethod
    def truth(cls, text, q_ranks, q_offsets):
        """Ground truth occ(q) by plain scan (NOT the reference's behaviour)."""
        L = cls.lib()
        t = _as_u8(text)
        q = _as_u8(q_ranks)
        off = _as_u64(q_offsets)
        Q = off.size - 1
        counts = np.zeros(Q, dtype=np.uint64)
        pos = _u32p()
        total = C.c_uint64(0)
        L.ko_truth_search_batch(_ptr(t, _u8p), t.size, _ptr(q, _u8p), _ptr(off, _u64p), Q, _ptr(counts, _u64p),
                                C.byref(pos), C.byref(total))
        return _finish(counts, np.zeros(Q, dtype=np.uint8), pos, total.value, L.ko_free, True)

    @classmethod
    def choose_best_k(cls, lens, n_k: int = 4):
        a = _as_u64(lens)
        out = np.zeros(16, dtype=np.uint64)
        n = cls.lib().ko_choose_best_k(_ptr(a, _u64p), a.size, n_k, _ptr(out, _u64p))
        return [int(x) for x in out[:n]]


class Reference(_Base):
    """The reference itself (kmer::kmer_index of Clemapfel/kmer_index), compiled into oracle/_ref/."""
    _prefix = "kref"

    @classmethod
    def lib(cls):
        if cls._lib is None:
            if not os.path.exists(REF_SO):
                raise FileNotFoundError(f"{REF_SO} not built (make -C oracle REF=<kmer_index checkout>)")
            L = C.CDLL(REF_SO)
            L.kref_supported.restype = C.c_int
            L.kref_supported.argtypes = [C.c_uint32, _u32p, C.c_uint32]
            L.kref_create.restype = C.c_void_p
            L.kref_create.argtypes = [C.c_uint32, _u32p, C.c_uint32, _u8p, C.c_uint64, C.c_uint32,
                                      C.POINTER(C.c_double)]
            L.kref_destroy.argtypes = [C.c_void_p]
            L.kref_search_batch.restype = C.c_int
            L.kref_search_batch.argtypes = [C.c_void_p, _u8p, _u64p, C.c_uint64, C.c_uint32, _u64p, _u8p,
                                            C.POINTER(_u32p), _u64p, C.POINTER(C.c_double), C.c_int]
            L.kref_free.argtypes = [C.c_void_p]
            L.kref_scheme.restype = C.c_uint64
            L.kref_scheme.argtypes = [C.c_void_p, C.c_uint64, _u32p, C.c_uint64, C.POINTER(C.c_int)]
            L.kref_fast_pow.restype = C.c_uint64
            L.kref_fast_pow.argtypes = [C.c_uint64, C.c_uint8]
            L.kref_choose_best_k.restype = C.c_uint64
            L.kref_choose_best_k.argtypes = [_u64p, C.c_uint64, C.c_uint64, _u64p]
            L.kref_hardware_concurrency.restype = C.c_uint32
            cls._lib = L
        return cls._lib

    @classmethod
    def supported(cls, sigma: int, ks) -> bool:
        ks_a = np.asarray(list(ks), dtype=np.uint32)
        return bool(cls.lib().kref_supported(sigma, _ptr(ks_a, _u32p), ks_a.size))

    def __init__(self, text, sigma: int, ks, n_threads: int = 0):
        super().__init__()
        L = self.lib()
        t = _as_u8(text)
        ks_a = np.asarray([int(k) for k in ks], dtype=np.uint32)
        secs = C.c_double(0)
        self._h = L.kref_create(sigma, _ptr(ks_a, _u32p), ks_a.size, _ptr(t, _u8p), t.size,
                                n_threads or (os.cpu_count() or 1), C.byref(secs))
        if not self._h:
            raise ValueError(f"reference driver has no instantiation for sigma={sigma} ks={list(ks)}")
        self.build_seconds = secs.value
        self.search_seconds = 0.0

    def search(self, q_ranks, q_offsets, n_threads: int = 0, keep_positions: bool = True):
        L = self.lib()
        q = _as_u8(q_ranks)
        off = _as_u64(q_offsets)
        Q = off.size - 1
        counts = np.zeros(Q, dtype=np.uint64)
        status = np.zeros(Q, dtype=np.uint8)
        pos = _u32p()
        total = C.c_uint64(0)
        secs = C.c_double(0)
        L.kref_search_batch(self._h, _ptr(q, _u8p), _ptr(off, _u64p), Q, n_threads or (os.cpu_count() or 1),
                            _ptr(counts, _u64p), _ptr(status, _u8p), C.byref(pos), C.byref(total),
                            C.byref(secs), 1 if keep_positions else 0)
        self.search_seconds = secs.value
        return _finish(counts, status, pos, total.value, L.kref_free, keep_positions)

    @classmethod
    def fast_pow(cls, base: int, exp: int) -> int:
        return int(cls.lib().kref_fast_pow(base, exp))

    @classmethod
    def choose_best_k(cls, lens, n_k: int = 4):
        a = _as_u64(lens)
        out = np.zeros(16, dtype=np.uint64)
        n = cls.lib().kref_choose_best_k(_ptr(a, _u64p), a.size, n_k, _ptr(out, _u64p))
        return [int(x) for x in out[:n]]

    @classmethod
    def hardware_concurrency(cls) -> int:
        return int(cls.lib().kref_hardware_concurrency())
