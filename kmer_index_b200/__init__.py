"""kmer_index_b200: B200-native k-mer index (build + batched search) behind the reference's API.

This package is the thin Python host layer over libkmer_b200.so (hand-written sm_100a kernels behind
the C ABI in include/kmer_b200.h). It mirrors kmer::kmer_index / make_kmer_index of the reference
(kmer_index.hpp:350-579): build from a text of symbol ranks, ``search`` returns sorted positions.
There is no CPU fallback: without the CUDA library every operation raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Iterable, Sequence

import numpy as np

from . import _capi
from ._capi import (MODE_CORRECT, MODE_DEFAULT, MODE_REFERENCE_EXACT, QUERY_OK, QUERY_THROW_INVALID_ARGUMENT,
                    QUERY_TOO_LONG_FOR_SHARD, QUERY_UNDEFINED, KmerB200Error)

__all__ = ["KmerIndex", "make_kmer_index", "BatchResult", "Records", "parse_sequences", "fast_pow", "kmer_hash", "kmer_from_hash", "Spectrum", "choose_best_k", "scheme_for_ks",
           "char_lut", "ALPHABET_CHARS",
           "MODE_REFERENCE_EXACT", "MODE_CORRECT", "KmerB200Error", "ALPHABETS"]

# alphabet sizes of the seqan3 alphabets the reference is used with
ALPHABETS = {"dna4": 4, "dna5": 5, "dna15": 15, "aa27": 27}
# their characters in rank order (seqan3's rank order is the alphabetical order of the character set)
ALPHABET_CHARS = {"dna4": "ACGT", "dna5": "ACGNT", "dna15": "ABCDGHKMNRSTVWY", "aa27": "ABCDEFGHIJKLMNOPQRSTUVWXYZ*"}


def char_lut(alphabet: str) -> np.ndarray:
    """256-entry character -> rank table for kmer_b200_create_from_text / search_batch_text; characters outside
    the alphabet map to 255 (rejected as an invalid rank). Case-insensitive."""
    chars = ALPHABET_CHARS.get(alphabet, alphabet)
    lut = np.full(256, 255, dtype=np.uint8)
    for r, c in enumerate(chars):
        lut[ord(c.upper())] = r
        lut[ord(c.lower())] = r
    return lut


def fast_pow(base: int, exp: int) -> int:
    """kmer::detail::fast_pow (fast_pow.hpp:46-93)."""
    return int(_capi.lib().kmer_b200_fast_pow(base, exp))


def kmer_hash(ranks, sigma: int) -> int:
    """The k-mer hash of `ranks` (kmer_index.hpp:56-73)."""
    r = np.ascontiguousarray(np.asarray(ranks, dtype=np.uint8))
    return int(_capi.lib().kmer_b200_hash(r.ctypes.data_as(_capi.u8p), r.size, sigma))


def kmer_from_hash(h: int, k: int, sigma: int) -> np.ndarray:
    """The k ranks whose kmer_hash is h (first symbol most significant): the inverse of kmer_hash, for printing the
    k-mers of KmerIndex.frequent_kmers."""
    h, k, sigma = int(h), int(k), int(sigma)
    if k < 1 or not 0 <= h < sigma ** k:
        raise ValueError(f"hash {h} is not the hash of a {k}-mer over {sigma} symbols")
    out = np.zeros(k, dtype=np.uint8)
    for i in range(k - 1, -1, -1):
        h, out[i] = divmod(h, sigma)
    return out


class Spectrum:
    """The k-mer spectrum of one element (KmerIndex.spectrum): hist[c] = distinct k-mers occurring c times for
    1 <= c < len(hist) - 1, hist[-1] = those occurring len(hist) - 1 times or more, hist[0] = sigma^k - distinct; total
    = counted windows, distinct = k-mers occurring at least once, max_count = the largest count (0 when none)."""

    def __init__(self, hist: np.ndarray, info):
        self.hist = hist
        self.total = int(info.total)
        self.distinct = int(info.distinct)
        self.max_count = int(info.max_count)
        self.key_space = int(info.key_space)

    def __repr__(self):
        return f"Spectrum(total={self.total}, distinct={self.distinct}, max_count={self.max_count}, bins={self.hist.size})"


def choose_best_k(query_lengths: Iterable[int], n_k: int = 4) -> list[int]:
    """choose_best_k (choose_best_k.hpp:12-60)."""
    a = np.ascontiguousarray(np.asarray(list(query_lengths), dtype=np.uint64))
    out = np.zeros(16, dtype=np.uint64)
    n = _capi.lib().kmer_b200_choose_best_k(a.ctypes.data_as(_capi.u64p), a.size, n_k, out.ctypes.data_as(_capi.u64p))
    return [int(x) for x in out[:n]]


def scheme_for_ks(ks: Sequence[int], m: int):
    """Row m of the scheme table the reference builds in choose_search_scheme (kmer_index.hpp:407-476):
    (_optimal_nk_sum[m], _use_multi_search_scheme[m]). Host-only."""
    ks_a = np.asarray(list(ks), dtype=np.uint32)
    out = np.zeros(4096, dtype=np.uint32)
    multi = C.c_int(0)
    n = _capi.lib().kmer_b200_scheme_for_ks(ks_a.ctypes.data_as(_capi.u32p), ks_a.size, m,
                                            out.ctypes.data_as(_capi.u32p), out.size, C.byref(multi))
    return [int(x) for x in out[:n]], bool(multi.value)


def gather_probe(table_bytes: int = 16 << 30, n_gathers: int = 1 << 30, stream: int | None = None) -> float:
    """Random-gather ceiling of the device in sectors/s (independent 8-byte reads from a table >> L2)."""
    ms = C.c_double(0)
    _capi.check(_capi.lib().kmer_b200_gather_probe(table_bytes, n_gathers, stream, C.byref(ms)))
    return n_gathers / (ms.value * 1e-3)


APPROX_HITS = {"all": _capi.HITS_ALL, "all_best": _capi.HITS_ALL_BEST, "single_best": _capi.HITS_SINGLE_BEST,
               "strata": _capi.HITS_STRATA}


def approx_options(max_mismatches: int, hits: str = "all", strata: int = 0, distances: bool = False) -> _capi.ApproxOptions:
    """kmer_b200_approx_options of a search_approx call (hits: a key of APPROX_HITS)."""
    if hits not in APPROX_HITS:
        raise ValueError(f"hits must be one of {sorted(APPROX_HITS)}, not {hits!r}")
    return _capi.ApproxOptions(int(max_mismatches), APPROX_HITS[hits], int(strata),
                               _capi.APPROX_DISTANCES if distances else 0)


class BatchResult:
    """CSR result of a batch: offsets[Q+1], positions (ascending per query), status[Q]. Approximate search with a hit
    strategy also fills `distances` (uint8 per position: its Hamming distance, with distances=True) and `best_distance`
    (uint8 per query: d_min, 0xFF without a hit; every strategy but "all"); both are None otherwise. Seeding (KmerIndex.seeds) fills
    `seed_offsets` (uint32 per position: the query offset j of its k-mer) and `kmer_counts` (uint32 per k-mer of the batch);
    both are None for other searches. Record votes (KmerIndex.record_votes) hold record ids where the others hold
    positions (`records` names them), `votes` (uint32 per entry) and `kmer_hits` (uint32 per read: its counted k-mers);
    `records`, `votes` and `kmer_hits` are None for other results."""

    def __init__(self, offsets: np.ndarray, positions: np.ndarray, status: np.ndarray, _owner=None,
                 distances: np.ndarray | None = None, best_distance: np.ndarray | None = None,
                 seed_offsets: np.ndarray | None = None, kmer_counts: np.ndarray | None = None,
                 votes: np.ndarray | None = None, kmer_hits: np.ndarray | None = None):
        self.offsets = offsets
        self.positions = positions
        self.status = status
        self.distances = distances
        self.best_distance = best_distance
        self.seed_offsets = seed_offsets
        self.kmer_counts = kmer_counts
        self.votes = votes
        self.kmer_hits = kmer_hits
        self._owner = _owner   # (lib, C result handle) when the arrays are views of the pinned C result

    def free(self):
        """Release the C result (only needed for copy=False results; the arrays become invalid)."""
        if self._owner is not None:
            L, r = self._owner
            self._owner = None
            self.offsets = self.positions = self.status = self.distances = self.best_distance = None
            self.seed_offsets = self.kmer_counts = self.votes = self.kmer_hits = None
            L.kmer_b200_result_free(r)

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def __len__(self) -> int:
        return int(self.status.size)

    def to_vector(self, i: int) -> np.ndarray:
        """kmer_index_result::to_vector() of query i (kmer_index_result.hpp:244-260)."""
        if self.status[i] == QUERY_THROW_INVALID_ARGUMENT:
            raise ValueError("the reference throws std::invalid_argument for this query")
        return self.positions[int(self.offsets[i]):int(self.offsets[i + 1])]

    def as_tuple(self):
        return self.offsets, self.positions, self.status

    @property
    def records(self) -> np.ndarray | None:
        """Record votes: the record id of each entry (the positions array), else None."""
        return self.positions if self.votes is not None else None

    def best(self):
        """Record votes: per read, (record or -1, its votes, the runner-up's votes) as int64 arrays. The runner-up's votes
        are 0 when there is none; a tie shows as equal votes (the record is then the lower id)."""
        if self.votes is None:
            raise ValueError("best() needs a record-vote result")
        Q = self.status.size
        lens = np.diff(self.offsets.astype(np.int64))
        first = self.offsets[:-1].astype(np.int64)
        has1, has2 = lens >= 1, lens >= 2
        rec = np.full(Q, -1, np.int64)
        v1 = np.zeros(Q, np.int64)
        v2 = np.zeros(Q, np.int64)
        rec[has1] = self.positions[first[has1]]
        v1[has1] = self.votes[first[has1]]
        v2[has2] = self.votes[first[has2] + 1]
        return rec, v1, v2


class Records:
    """Sequences parsed from FASTA / FASTQ bytes on the device (kmer_b200_parse_sequences): one concatenated rank text in
    HBM plus the record table. `index(ks)` builds a KmerIndex over it; `locate` maps hit positions to (record, offset)."""

    def __init__(self, handle, data: bytes, sigma: int):
        L = _capi.lib()
        self._L, self._h, self._data, self.sigma = L, handle, data, sigma
        n = int(L.kmer_b200_records_count(handle))
        self.n_symbols = int(L.kmer_b200_records_symbols(handle))
        self.starts = np.ctypeslib.as_array(L.kmer_b200_records_starts(handle), shape=(n + 1,)).copy()
        self.header_offsets = (np.ctypeslib.as_array(L.kmer_b200_records_header_offsets(handle), shape=(n,)).copy()
                               if n else np.zeros(0, np.uint64))

    def __len__(self) -> int:
        return int(self.header_offsets.size)

    def name(self, i: int) -> str:
        """The header line of record i without its marker ('' for a headerless first record)."""
        o = int(self.header_offsets[i])
        if o == 0xFFFFFFFFFFFFFFFF:
            return ""
        end = self._data.find(b"\n", o)
        return self._data[o + 1:end if end >= 0 else len(self._data)].rstrip(b"\r").decode(errors="replace")

    def index(self, ks: Sequence[int], collection: bool = False, **kw) -> "KmerIndex":
        """KmerIndex over the concatenated records. collection=True: a collection index (KmerIndex.attach_records with
        these starts, built in MODE_CORRECT): no hit spans two records, KmerIndex.locate gives (record, offset)."""
        if collection:
            kw["mode"] = MODE_CORRECT
        ix = KmerIndex(None, self.sigma, ks, text_device_ptr=int(self._L.kmer_b200_records_ranks_device(self._h)),
                       n=self.n_symbols, **kw)
        if collection:
            ix.attach_records(self.starts)
        return ix

    def locate(self, positions, query_len: int = 0):
        """(record, offset) of each position; record == 0xFFFFFFFF where a match of query_len symbols would run over the
        end of its record (an artefact of concatenating the records)."""
        p = np.ascontiguousarray(np.asarray(positions, dtype=np.uint32))
        rec = np.zeros(p.size, dtype=np.uint32)
        off = np.zeros(p.size, dtype=np.uint32)
        _capi.check(self._L.kmer_b200_records_locate(self._h, p.ctypes.data_as(_capi.u32p), p.size, query_len,
                                                     rec.ctypes.data_as(_capi.u32p), off.ctypes.data_as(_capi.u32p)))
        return rec, off

    def close(self):
        if getattr(self, "_h", None):
            self._L.kmer_b200_records_free(self._h)
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


def parse_sequences(data, alphabet: str = "dna4", fmt: int = 0, device: int = -1, stream: int | None = None) -> Records:
    """FASTA / FASTQ bytes -> Records (parsed on the device). fmt: 0 = by the first byte, 1 = FASTA, 2 = FASTQ."""
    L = _capi.lib()
    raw = data.encode() if isinstance(data, str) else bytes(data)
    sigma = ALPHABETS[alphabet]
    lut = np.ascontiguousarray(char_lut(alphabet))
    cfg = _capi.Config()
    L.kmer_b200_config_default(C.byref(cfg))
    cfg.device, cfg.stream = device, stream
    h = C.c_void_p()
    _capi.check(L.kmer_b200_parse_sequences(raw, len(raw), lut.ctypes.data_as(_capi.u8p), sigma, fmt, C.byref(cfg), C.byref(h)))
    return Records(h, raw, sigma)


class _DevArray:
    """Zero-copy view of device memory for torch.as_tensor / cupy via __cuda_array_interface__."""

    def __init__(self, ptr: int, n: int, typestr: str, owner):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}
        self._owner = owner


class DeviceResult:
    """Result of a device-resident batch; the buffers live in HBM until free()."""

    def __init__(self, L, handle, Q: int):
        self._L, self._r, self.n_queries = L, handle, Q
        self.n_positions = int(L.kmer_b200_result_n_positions(handle))
        self.offsets_ptr = L.kmer_b200_result_offsets(handle) or 0
        self.positions_ptr = L.kmer_b200_result_positions(handle) or 0
        self.status_ptr = L.kmer_b200_result_status(handle) or 0

    def offsets(self):      # int64 view of the uint64 offsets (values < 2^63)
        return _DevArray(self.offsets_ptr, self.n_queries + 1, "<i8", self)

    def positions(self):    # int32 view of the uint32 positions (reinterpret for positions >= 2^31)
        return _DevArray(self.positions_ptr, self.n_positions, "<i4", self)

    def status(self):
        return _DevArray(self.status_ptr, self.n_queries, "|u1", self)

    def distances(self):
        """uint8 view of d(p) per position (approximate search with distances=True), or None."""
        ptr = self._L.kmer_b200_result_distances(self._r) or 0
        return _DevArray(ptr, self.n_positions, "|u1", self) if ptr else None

    def best_distances(self):
        """uint8 view of d_min per query (approximate search with a hit strategy other than "all"), or None."""
        ptr = self._L.kmer_b200_result_best_distances(self._r) or 0
        return _DevArray(ptr, self.n_queries, "|u1", self) if ptr else None

    def seed_offsets(self):
        """int32 view of the query offset j of each position (seeding, not count-only), or None."""
        ptr = self._L.kmer_b200_result_seed_offsets(self._r) or 0
        return _DevArray(ptr, self.n_positions, "<i4", self) if ptr else None

    def kmer_counts(self):
        """int32 view of the occurrence count of each k-mer of the batch (seeding), or None."""
        ptr = self._L.kmer_b200_result_kmer_counts(self._r) or 0
        return _DevArray(ptr, int(self._L.kmer_b200_result_n_kmers(self._r)), "<i4", self) if ptr else None

    def votes(self):
        """int32 view of the votes of each entry (record votes; positions() then holds record ids), or None."""
        ptr = self._L.kmer_b200_result_votes(self._r) or 0
        return _DevArray(ptr, self.n_positions, "<i4", self) if ptr else None

    def kmer_hits(self):
        """int32 view of the counted k-mers of each read (record votes), or None."""
        ptr = self._L.kmer_b200_result_kmer_hits(self._r) or 0
        return _DevArray(ptr, self.n_queries, "<i4", self) if ptr else None

    def hit_queries(self):
        """int32 view of [n, id_1 .. id_n, ...]: the queries the count pass found hits for (unordered), or None."""
        ptr = self._L.kmer_b200_result_hit_queries(self._r) or 0
        return _DevArray(ptr, self.n_queries + 1, "<i4", self) if ptr else None

    def free(self):
        if self._r:
            self._L.kmer_b200_result_free(self._r)
            self._r = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class KmerIndex:
    """kmer::kmer_index<alphabet, uint32_t, ks...> (kmer_index.hpp:350-566) on one B200."""

    def __init__(self, text, sigma: int, ks: Sequence[int], *, mode: int = MODE_REFERENCE_EXACT, device: int = -1,
                 stream: int | None = None, profile: bool = False, shard_begin: int = 0, n_total: int = 0,
                 halo: int = 0, directory_bits: int = 0, text_device_ptr: int | None = None, n: int | None = None,
                 aux_elements: bool = True, lut: np.ndarray | None = None, key_part: int = 0, key_parts: int = 0,
                 devices: Sequence[int] | None = None, shared_positions: bool = False):
        L = _capi.lib()
        self._L = L
        self._h = C.c_void_p()
        self.sigma = int(sigma)
        self.ks = [int(k) for k in ks]
        cfg = _capi.Config()
        L.kmer_b200_config_default(C.byref(cfg))
        cfg.device = device
        cfg.mode = mode
        cfg.stream = stream
        self.stream = stream          # None: the library made a private stream for this index
        cfg.profile = int(profile)   # 1: per-kernel CUDA-event times; 2: also count gathered sectors per search
        cfg.shard_begin = shard_begin
        cfg.n_total = n_total
        cfg.halo = halo
        cfg.directory_bits = directory_bits
        # bit 0: no auxiliary k' = m elements for sub-k lengths; bit 1: ONE position array (the largest k's) serves every k
        cfg.reserved = (0 if aux_elements else 1) | (2 if shared_positions else 0)
        cfg.key_part, cfg.key_parts = key_part, key_parts   # key-range part of a multi-GPU build (sharded.build_replicated)
        self._adopted = []                                   # arrays handed over with adopt_element: kept alive here
        if devices is not None and len(devices) > 1:         # several GPUs behind this one handle (host batches only)
            self._device_ids = (C.c_int32 * len(devices))(*[int(d) for d in devices])
            cfg.device_ids = C.cast(self._device_ids, C.POINTER(C.c_int32))
            cfg.n_devices = len(devices)
        ks_a = np.asarray(self.ks, dtype=np.uint32)
        if text_device_ptr is not None:
            self.n = int(n)
            _capi.check(L.kmer_b200_create_from_device(C.c_void_p(text_device_ptr), self.n, self.sigma,
                                                       ks_a.ctypes.data_as(_capi.u32p), ks_a.size, C.byref(cfg),
                                                       C.byref(self._h)))
        elif lut is not None:    # `text` is characters (bytes / str / uint8 array of character codes)
            raw = text.encode() if isinstance(text, str) else bytes(text) if isinstance(text, (bytes, bytearray)) else None
            t = np.frombuffer(raw, dtype=np.uint8) if raw is not None else np.ascontiguousarray(np.asarray(text, dtype=np.uint8))
            lut = np.ascontiguousarray(np.asarray(lut, dtype=np.uint8))
            self.n = int(t.size)
            self._lut = lut
            _capi.check(L.kmer_b200_create_from_text(t.ctypes.data_as(C.c_char_p), t.size, lut.ctypes.data_as(_capi.u8p),
                                                     self.sigma, ks_a.ctypes.data_as(_capi.u32p), ks_a.size,
                                                     C.byref(cfg), C.byref(self._h)))
        else:
            t = np.ascontiguousarray(np.asarray(text, dtype=np.uint8))
            self.n = int(t.size)
            _capi.check(L.kmer_b200_create(t.ctypes.data_as(_capi.u8p), t.size, self.sigma,
                                           ks_a.ctypes.data_as(_capi.u32p), ks_a.size, C.byref(cfg), C.byref(self._h)))

    # -- serialization (construct once, load later)
    def save(self, path: str) -> None:
        _capi.check(self._L.kmer_b200_save(self._h, str(path).encode()))

    @classmethod
    def load(cls, path: str, *, mode: int | None = None, device: int = -1, stream: int | None = None,
             profile: int = 0) -> "KmerIndex":
        L = _capi.lib()
        self = cls.__new__(cls)
        self._L = L
        self._adopted = []
        self._h = C.c_void_p()
        cfg = _capi.Config()
        L.kmer_b200_config_default(C.byref(cfg))
        cfg.device, cfg.stream, cfg.profile = device, stream, int(profile)
        cfg.mode = MODE_REFERENCE_EXACT if mode is None else mode
        _capi.check(L.kmer_b200_load(str(path).encode(), C.byref(cfg), C.byref(self._h)))
        n_el = L.kmer_b200_n_elements(self._h)
        self.ks = [int(self.element_info(e).k) for e in range(n_el)]
        self.sigma = None
        self.n = int(self.element_info(0).n_kmers) + self.ks[0] - 1
        return self

    # -- sequence collections
    def attach_records(self, starts) -> None:
        """Make this a collection index (kmer_b200_attach_records): starts[0..R] with starts[0] = 0, non-decreasing,
        starts[R] = n. Every search then reports only windows inside one record; exact search runs in MODE_CORRECT."""
        s = np.ascontiguousarray(np.asarray(starts, dtype=np.uint64))
        if s.size < 2:
            raise ValueError("starts needs at least two entries (one record)")
        _capi.check(self._L.kmer_b200_attach_records(self._h, s.ctypes.data_as(_capi.u64p), s.size - 1))

    @property
    def records(self) -> np.ndarray | None:
        """The record table starts[0..R] of a collection index (uint64), or None."""
        n = C.c_uint64(0)
        p = self._L.kmer_b200_index_records(self._h, C.byref(n))
        return np.ctypeslib.as_array(p, shape=(n.value + 1,)).copy() if p else None

    def locate(self, positions):
        """(record, offset) of each hit position of a collection index: record = the last r with starts[r] <= p, offset =
        p - starts[r] (0xFFFFFFFF, 0 for p >= n). A numpy array (or list) is located on the host and gives uint32 numpy
        arrays; a torch tensor or device view (int32 / uint32) is located by a kernel and gives int32 tensors on its
        device."""
        if hasattr(positions, "__cuda_array_interface__") or type(positions).__module__.startswith("torch"):
            import torch
            t = torch.as_tensor(positions, device="cuda") if not isinstance(positions, torch.Tensor) else positions
            if t.dtype not in (torch.int32, torch.uint32) or not t.is_cuda:
                raise TypeError("device positions must be an int32 / uint32 CUDA tensor or view")
            t = t.contiguous()
            rec = torch.empty(t.numel(), dtype=torch.int32, device=t.device)
            off = torch.empty(t.numel(), dtype=torch.int32, device=t.device)
            torch.cuda.current_stream(t.device).synchronize()
            _capi.check(self._L.kmer_b200_locate_device(self._h, C.c_void_p(t.data_ptr()), t.numel(), C.c_void_p(rec.data_ptr()),
                                                        C.c_void_p(off.data_ptr())))
            torch.cuda.synchronize(t.device)   # the kernel ran on the index's stream
            return rec, off
        p = np.ascontiguousarray(np.asarray(positions, dtype=np.uint32))
        rec = np.zeros(p.size, dtype=np.uint32)
        off = np.zeros(p.size, dtype=np.uint32)
        _capi.check(self._L.kmer_b200_locate(self._h, p.ctypes.data_as(_capi.u32p), p.size, rec.ctypes.data_as(_capi.u32p),
                                             off.ctypes.data_as(_capi.u32p)))
        return rec, off

    # -- lifetime
    def close(self):
        if getattr(self, "_h", None):
            self._L.kmer_b200_destroy(self._h)
            self._h = None
            self._adopted = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def handle(self):
        return self._h

    # -- search
    def search_batch(self, q_ranks, q_offsets, mode: int = MODE_DEFAULT, copy: bool = True) -> BatchResult:
        """Batch of queries in host memory -> host CSR result (kmer_index::search + to_vector per query).
        copy=False returns views of the library's pinned result buffers (valid until BatchResult.free())."""
        q = np.ascontiguousarray(np.asarray(q_ranks, dtype=np.uint8))
        off = np.ascontiguousarray(np.asarray(q_offsets, dtype=np.uint64))
        r = C.c_void_p()
        _capi.check(self._L.kmer_b200_search_batch(self._h, q.ctypes.data, off.ctypes.data, off.size - 1, mode, C.byref(r)))
        return self._host_result(r, off.size - 1, copy)

    def search_batch_text(self, queries, lut: np.ndarray | None = None, mode: int = MODE_DEFAULT) -> BatchResult:
        """Batch of character queries (list of str/bytes); translated to ranks on the device."""
        lut = np.ascontiguousarray(np.asarray(lut if lut is not None else self._lut, dtype=np.uint8))
        raw = [x.encode() if isinstance(x, str) else bytes(x) for x in queries]
        off = np.zeros(len(raw) + 1, dtype=np.uint64)
        np.cumsum([len(x) for x in raw], out=off[1:])
        q = np.frombuffer(b"".join(raw), dtype=np.uint8)
        r = C.c_void_p()
        _capi.check(self._L.kmer_b200_search_batch_text(self._h, q.ctypes.data_as(C.c_char_p), off.ctypes.data, len(raw),
                                                        lut.ctypes.data_as(_capi.u8p), mode, C.byref(r)))
        return self._host_result(r, len(raw), True)

    def search_approx(self, q_ranks, q_offsets, max_mismatches: int, copy: bool = True, *, hits: str = "all",
                      strata: int = 0, distances: bool = False) -> BatchResult:
        """Approximate search of a host batch (kmer_b200_search_approx_batch_ex): per query, every position p, ascending,
        where the text window T[p, p+m) differs from the query in at most max_mismatches (<= 8) symbols. Substitutions
        only; max_mismatches=0 is exact search in MODE_CORRECT. copy=False: views of the library's pinned buffers (valid
        until BatchResult.free()).
        hits: "all", "all_best" (the hits at the smallest distance d_min), "single_best" (the lowest such position) or
        "strata" (distance <= d_min + strata); every choice but "all" sets BatchResult.best_distance. distances=True
        sets BatchResult.distances."""
        q = np.ascontiguousarray(np.asarray(q_ranks, dtype=np.uint8))
        off = np.ascontiguousarray(np.asarray(q_offsets, dtype=np.uint64))
        r = C.c_void_p()
        opt = approx_options(max_mismatches, hits, strata, distances)
        _capi.check(self._L.kmer_b200_search_approx_batch_ex(self._h, q.ctypes.data, off.ctypes.data, off.size - 1, C.byref(opt),
                                                             C.byref(r)))
        return self._host_result(r, off.size - 1, copy)

    def _seed_k(self, k: int | None) -> int:
        if k is None:
            if len(self.ks) != 1:
                raise ValueError("seeding an index with several ks needs k")
            return self.ks[0]
        return int(k)

    # -- k-mer spectrum
    def spectrum(self, k: int | None = None, bins: int = 10001) -> Spectrum:
        """Occurrence histogram of the k-mers of element k (kmer_b200_spectrum); k defaults to the index's only k. On a
        collection index only windows inside one record count (the counts seeding reports)."""
        hist = np.zeros(int(bins), dtype=np.uint64)
        info = _capi.SpectrumInfo()
        _capi.check(self._L.kmer_b200_spectrum(self._h, self._seed_k(k), hist.ctypes.data_as(_capi.u64p), hist.size,
                                               C.byref(info)))
        return Spectrum(hist, info)

    def frequent_kmers(self, k: int | None = None, min_count: int = 2, limit: int | None = None):
        """(hashes, counts) as uint64 arrays: every k-mer occurring at least min_count times, by count descending then hash
        ascending, the first `limit` of them (None: all). kmer_from_hash turns a hash back into ranks."""
        k = self._seed_k(k)
        n = C.c_uint64(0)
        if limit is None:
            _capi.check(self._L.kmer_b200_frequent_kmers(self._h, k, int(min_count), None, None, 0, C.byref(n)))
            limit = n.value
        hashes = np.zeros(int(limit), dtype=np.uint64)
        counts = np.zeros(int(limit), dtype=np.uint64)
        _capi.check(self._L.kmer_b200_frequent_kmers(self._h, k, int(min_count), hashes.ctypes.data_as(_capi.u64p),
                                                     counts.ctypes.data_as(_capi.u64p), hashes.size, C.byref(n)))
        m = min(n.value, hashes.size)
        return hashes[:m], counts[:m]

    def occurrence_cutoff(self, fraction: float, k: int | None = None) -> int:
        """The repeat cap that ignores the most frequent `fraction` of the distinct k-mers (kmer_b200_occurrence_cutoff):
        the smallest c >= 1 with #{count > c} <= floor(fraction * distinct), 0 for an empty spectrum. seeds(...,
        max_occ=cutoff) then drops exactly the k-mers above it."""
        c = C.c_uint64(0)
        _capi.check(self._L.kmer_b200_occurrence_cutoff(self._h, self._seed_k(k), float(fraction), C.byref(c)))
        return int(c.value)

    def seeds(self, q_ranks, q_offsets, k: int | None = None, max_occ: int = 0, copy: bool = True) -> BatchResult:
        """k-mer seeding of a host batch (kmer_b200_seed_batch): per query, for every offset j in [0, m - k], every text
        position p with T[p, p+k) = q[j, j+k), ordered by (j, p); BatchResult.seed_offsets holds each hit's j and
        BatchResult.kmer_counts each k-mer's occurrence count (query order, then j order). k defaults to the index's only
        k. max_occ > 0: k-mers with more than max_occ occurrences give no hits and report max_occ + 1. On a collection
        index only windows inside one record count."""
        q = np.ascontiguousarray(np.asarray(q_ranks, dtype=np.uint8))
        off = np.ascontiguousarray(np.asarray(q_offsets, dtype=np.uint64))
        r = C.c_void_p()
        _capi.check(self._L.kmer_b200_seed_batch(self._h, q.ctypes.data, off.ctypes.data, off.size - 1, self._seed_k(k),
                                                 int(max_occ), C.byref(r)))
        return self._host_result(r, off.size - 1, copy)

    def seeds_batch_device(self, q_ptr: int, off_ptr: int, Q: int, max_len: int, k: int | None = None, max_occ: int = 0):
        """Seeding (see seeds) of a device-resident batch; the result stays on the device."""
        return self._device_call(self._L.kmer_b200_seed_batch_device, q_ptr, off_ptr, Q, max_len, self._seed_k(k), int(max_occ))

    def count_seeds_batch_device(self, q_ptr: int, off_ptr: int, Q: int, max_len: int, k: int | None = None, max_occ: int = 0):
        """Count-only seeding of a device-resident batch: offsets, status and kmer_counts(), no positions."""
        return self._device_call(self._L.kmer_b200_count_seeds_batch_device, q_ptr, off_ptr, Q, max_len, self._seed_k(k),
                                 int(max_occ))

    def record_votes(self, q_ranks, q_offsets, k: int | None = None, max_occ: int = 0, min_votes: int = 1,
                     copy: bool = True) -> BatchResult:
        """Which records of a collection index each read comes from (kmer_b200_record_votes): per read, every record r
        with votes(q, r) >= min_votes, by votes descending then record ascending, where votes(q, r) is the number of the
        read's counted k-mers (1 <= in-record occurrences, <= max_occ when max_occ > 0) that occur in r. BatchResult.records
        holds the record ids, .votes their votes, .kmer_hits each read's counted k-mers; best() gives the top record."""
        q = np.ascontiguousarray(np.asarray(q_ranks, dtype=np.uint8))
        off = np.ascontiguousarray(np.asarray(q_offsets, dtype=np.uint64))
        r = C.c_void_p()
        _capi.check(self._L.kmer_b200_record_votes(self._h, q.ctypes.data, off.ctypes.data, off.size - 1, self._seed_k(k),
                                                   int(max_occ), int(min_votes), C.byref(r)))
        return self._host_result(r, off.size - 1, copy)

    def record_votes_batch_device(self, q_ptr: int, off_ptr: int, Q: int, max_len: int, k: int | None = None, max_occ: int = 0,
                                  min_votes: int = 1):
        """Record votes (see record_votes) of a device-resident batch; the result stays on the device: positions() holds
        the record ids, votes() and kmer_hits() the rest."""
        return self._device_call(self._L.kmer_b200_record_votes_device, q_ptr, off_ptr, Q, max_len, self._seed_k(k), int(max_occ),
                                 int(min_votes))

    def _host_result(self, r, Q: int, copy: bool) -> BatchResult:
        L = self._L
        total = L.kmer_b200_result_n_positions(r)
        offsets = np.ctypeslib.as_array(C.cast(L.kmer_b200_result_offsets(r), _capi.u64p), shape=(Q + 1,))
        status = (np.ctypeslib.as_array(C.cast(L.kmer_b200_result_status(r), _capi.u8p), shape=(Q,))
                  if Q else np.zeros(0, dtype=np.uint8))
        positions = (np.ctypeslib.as_array(C.cast(L.kmer_b200_result_positions(r), _capi.u32p), shape=(total,))
                     if total else np.zeros(0, dtype=np.uint32))
        d_ptr, b_ptr = L.kmer_b200_result_distances(r), L.kmer_b200_result_best_distances(r)
        dist = (np.ctypeslib.as_array(C.cast(d_ptr, _capi.u8p), shape=(total,)) if total else np.zeros(0, np.uint8)) if d_ptr else None
        best = (np.ctypeslib.as_array(C.cast(b_ptr, _capi.u8p), shape=(Q,)) if Q else np.zeros(0, np.uint8)) if b_ptr else None
        s_ptr, c_ptr, n_kmers = L.kmer_b200_result_seed_offsets(r), L.kmer_b200_result_kmer_counts(r), L.kmer_b200_result_n_kmers(r)
        seed = (np.ctypeslib.as_array(C.cast(s_ptr, _capi.u32p), shape=(total,)) if total else np.zeros(0, np.uint32)) if s_ptr else None
        kc = (np.ctypeslib.as_array(C.cast(c_ptr, _capi.u32p), shape=(n_kmers,)) if n_kmers else np.zeros(0, np.uint32)) if c_ptr else None
        v_ptr, h_ptr = L.kmer_b200_result_votes(r), L.kmer_b200_result_kmer_hits(r)
        votes = (np.ctypeslib.as_array(C.cast(v_ptr, _capi.u32p), shape=(total,)) if total else np.zeros(0, np.uint32)) if v_ptr else None
        hits = (np.ctypeslib.as_array(C.cast(h_ptr, _capi.u32p), shape=(Q,)) if Q else np.zeros(0, np.uint32)) if h_ptr else None
        if not copy:
            return BatchResult(offsets, positions, status, _owner=(L, r), distances=dist, best_distance=best, seed_offsets=seed,
                               kmer_counts=kc, votes=votes, kmer_hits=hits)
        out = BatchResult(offsets.copy(), positions.copy(), status.copy(), distances=None if dist is None else dist.copy(),
                          best_distance=None if best is None else best.copy(), seed_offsets=None if seed is None else seed.copy(),
                          kmer_counts=None if kc is None else kc.copy(), votes=None if votes is None else votes.copy(),
                          kmer_hits=None if hits is None else hits.copy())
        L.kmer_b200_result_free(r)
        return out

    def search(self, query, mode: int = MODE_DEFAULT) -> np.ndarray:
        """kmer_index::search(query).to_vector() for one query; raises ValueError where the reference throws
        std::invalid_argument (kmer_index.hpp:121,508). A batch of one: correct but latency-bound."""
        q = np.ascontiguousarray(np.asarray(query, dtype=np.uint8))
        res = self.search_batch(q, np.array([0, q.size], dtype=np.uint64), mode)
        if res.status[0] == QUERY_THROW_INVALID_ARGUMENT:
            if q.size > 10000:
                raise ValueError("query size exceed the maximum size 10000 specified")
            raise ValueError("query size too low for specified k")
        if res.status[0] == QUERY_UNDEFINED:
            raise ValueError("query length 0 or 10000: undefined in the reference")
        return res.positions

    # -- device-resident batches (inputs and result stay in HBM)
    def _device_call(self, fn, q_ptr: int, off_ptr: int, Q: int, max_len: int, mode: int, *extra) -> "DeviceResult":
        r = C.c_void_p()
        _capi.check(fn(self._h, C.c_void_p(q_ptr), C.c_void_p(off_ptr), Q, max_len, mode, *extra, C.byref(r)))
        return DeviceResult(self._L, r, Q)

    def search_batch_device(self, q_ptr: int, off_ptr: int, Q: int, max_len: int, mode: int = MODE_DEFAULT):
        return self._device_call(self._L.kmer_b200_search_batch_device, q_ptr, off_ptr, Q, max_len, mode)

    def count_batch_device(self, q_ptr: int, off_ptr: int, Q: int, max_len: int, mode: int = MODE_DEFAULT):
        return self._device_call(self._L.kmer_b200_count_batch_device, q_ptr, off_ptr, Q, max_len, mode)

    def search_approx_batch_device(self, q_ptr: int, off_ptr: int, Q: int, max_len: int, max_mismatches: int, *,
                                   hits: str = "all", strata: int = 0, distances: bool = False):
        """Approximate search (see search_approx, including hits / strata / distances) of a device-resident batch; the
        result stays on the device."""
        opt = approx_options(max_mismatches, hits, strata, distances)
        return self._device_call(self._L.kmer_b200_search_approx_batch_device_ex, q_ptr, off_ptr, Q, max_len, C.byref(opt))

    def count_approx_batch_device(self, q_ptr: int, off_ptr: int, Q: int, max_len: int, max_mismatches: int, *,
                                  hits: str = "all", strata: int = 0, distances: bool = False):
        """Count-only approximate search of a device-resident batch: offsets and status (and best_distances() for a hit
        strategy other than "all"), no positions."""
        opt = approx_options(max_mismatches, hits, strata, distances)
        return self._device_call(self._L.kmer_b200_count_approx_batch_device_ex, q_ptr, off_ptr, Q, max_len, C.byref(opt))

    def presence_batch_device(self, q_ptr: int, off_ptr: int, Q: int, max_len: int, present_ptr: int,
                              mode: int = MODE_DEFAULT, fmt: int = 0) -> None:
        """fmt 0: uint64 bit mask per query (OR across shards); fmt 1: uint32 nibble flags (SUM across shards)."""
        _capi.check(self._L.kmer_b200_presence_batch_device(self._h, C.c_void_p(q_ptr), C.c_void_p(off_ptr), Q,
                                                            max_len, mode, C.c_void_p(present_ptr), fmt))

    def search_batch_device_global(self, q_ptr: int, off_ptr: int, Q: int, max_len: int, present_global_ptr: int,
                                   mode: int = MODE_DEFAULT, fmt: int = 0):
        return self._device_call(self._L.kmer_b200_search_batch_device_global, q_ptr, off_ptr, Q, max_len, mode,
                                 C.c_void_p(present_global_ptr), fmt)

    def search_sharded_begin(self, q_ptr: int, off_ptr: int, Q: int, max_len: int, present4_ptr: int,
                             mode: int = MODE_DEFAULT):
        """Count pass of a sharded search; this shard's presence flags (uint32 nibble format) go to present4_ptr.
        Returns the pending handle for search_sharded_finish()."""
        h = C.c_void_p()
        _capi.check(self._L.kmer_b200_search_sharded_begin(self._h, C.c_void_p(q_ptr), C.c_void_p(off_ptr), Q, max_len,
                                                           mode, C.c_void_p(present4_ptr), C.byref(h)))
        return h

    def search_sharded_finish(self, pending, present4_global_ptr: int, Q: int) -> "DeviceResult":
        r = C.c_void_p()
        _capi.check(self._L.kmer_b200_search_sharded_finish(pending, C.c_void_p(present4_global_ptr), C.byref(r)))
        return DeviceResult(self._L, r, Q)

    def search_sharded_abort(self, pending) -> None:
        """Releases a pending sharded search that will not be finished."""
        self._L.kmer_b200_search_sharded_abort(pending)

    def search_sharded_peek(self, pending, present4_global_ptr: int, Q: int):
        """(counts, hit list) of a pending sharded search as device array views: int64[Q] per-query counts with the
        whole-text rule applied, int32[1 + Q] hit list ([0] = n). Valid until search_sharded_finish."""
        c, h = C.c_void_p(), C.c_void_p()
        _capi.check(self._L.kmer_b200_search_sharded_peek(pending, C.c_void_p(present4_global_ptr), C.byref(c), C.byref(h)))
        return _DevArray(c.value, Q, "<i8", self), _DevArray(h.value, Q + 1, "<i4", self)

    def search_sharded_add_counts(self, pending, present4_global_ptr: int, ids_ptr: int, counts_ptr: int, n: int,
                                  within_ptr: int) -> None:
        """Between begin and finish on the merging shard: counts[ids] += counts of another shard (int64 device
        arrays); within receives the previous counts. Raises KmerB200Error(code -5) when the batch needs the
        segment sort (then merge after finish instead)."""
        _capi.check(self._L.kmer_b200_search_sharded_add_counts(pending, C.c_void_p(present4_global_ptr), C.c_void_p(ids_ptr),
                                                                C.c_void_p(counts_ptr), n, C.c_void_p(within_ptr)))

    # -- key-range parts (multi-GPU build of a replicated index)
    def element_part(self, e: int) -> _capi.Part:
        part = _capi.Part()
        _capi.check(self._L.kmer_b200_element_part(self._h, e, C.byref(part)))
        return part

    def export_directory(self, e: int, base: int, n: int, dst_ptr: int) -> None:
        """dst[j] = part directory[j] + base for j < n (device pointer), on the index's stream."""
        _capi.check(self._L.kmer_b200_export_directory(self._h, e, base, n, C.c_void_p(dst_ptr)))

    def export_bucket_sizes(self, e: int, sizes_ptr: int) -> int:
        """The part's directory as one byte per bucket (device pointer, key_hi - key_lo bytes); returns the number of
        buckets too large for a byte (> 0: ship the directory itself)."""
        n_large = C.c_uint64(0)
        _capi.check(self._L.kmer_b200_export_bucket_sizes(self._h, e, C.c_void_p(sizes_ptr), C.byref(n_large)))
        return int(n_large.value)

    def directory_from_sizes(self, sizes_ptr: int, n_keys: int, directory_ptr: int) -> None:
        _capi.check(self._L.kmer_b200_directory_from_sizes(self._h, C.c_void_p(sizes_ptr), n_keys, C.c_void_p(directory_ptr)))

    def adopt_element(self, e: int, positions, directory) -> None:
        """Hand the assembled whole element (device tensors: int32 positions[n - k + 1], directory[sigma^k + 1]) to
        the index; the tensors are kept alive by this object."""
        _capi.check(self._L.kmer_b200_adopt_element(self._h, e, C.c_void_p(positions.data_ptr()), positions.numel(),
                                                    C.c_void_p(directory.data_ptr()), directory.numel()))
        self._adopted.append((positions, directory))

    def adopt_element_parts(self, e: int, parts, part_first, directory) -> None:
        """Peer-positions index: `parts` = one int32 device tensor -- or raw device pointer -- per key-range part (this
        GPU's own or another GPU's memory mapped into this process with peer_buffer_open), part_first = n_parts + 1
        ascending CSR indices, directory = the whole directory on this GPU. Tensors passed are kept alive by this
        object; raw pointers must outlive the index."""
        ptrs = (C.c_void_p * len(parts))(*[C.c_void_p(int(t) if isinstance(t, int) else (t.data_ptr() if t is not None else 0))
                                            for t in parts])
        first = np.asarray(part_first, dtype=np.uint64)
        _capi.check(self._L.kmer_b200_adopt_element_parts(self._h, e, ptrs, first.ctypes.data_as(_capi.u64p), len(parts),
                                                          C.c_void_p(directory.data_ptr()), directory.numel()))
        self._adopted.append((list(parts), directory))

    # -- key-range multi-GPU search: routing (sharded.search_routed drives these)
    def route_plan(self, n_queries: int, max_len: int, n_parts: int, slack: float = 0.0) -> _capi.RoutePlan:
        plan = _capi.RoutePlan()
        _capi.check(self._L.kmer_b200_route_plan_make(self._h, n_queries, max_len, n_parts, slack, C.byref(plan)))
        return plan

    def route_queries(self, q_ptr: int, off_ptr: int, Q: int, plan, send_ptr: int, status_ptr: int, mode: int = MODE_DEFAULT):
        counts = (C.c_uint32 * plan.n_parts)()
        _capi.check(self._L.kmer_b200_route_queries_device(self._h, C.c_void_p(q_ptr), C.c_void_p(off_ptr), Q, mode, C.byref(plan),
                                                           C.c_void_p(send_ptr), C.c_void_p(status_ptr), counts))
        return [int(x) for x in counts]

    def search_routed(self, recv_ptr: int, plan, return_ptr: int, mode: int = MODE_DEFAULT):
        splits = (C.c_uint64 * plan.n_parts)()
        r = C.c_void_p()
        _capi.check(self._L.kmer_b200_search_routed_device(self._h, C.c_void_p(recv_ptr), C.byref(plan), mode, C.c_void_p(return_ptr),
                                                           splits, C.byref(r)))
        total = sum(int(x) for x in splits)
        res = DeviceResult(self._L, r, 0)
        res.n_positions = total
        return res, [int(x) for x in splits]

    def unroute(self, send_ptr: int, ret_ptr: int, plan, sent_counts, recv_pos_ptr: int, recv_splits, Q: int, status_ptr: int):
        sc = (C.c_uint32 * plan.n_parts)(*sent_counts)
        rs = (C.c_uint64 * plan.n_parts)(*recv_splits)
        r = C.c_void_p()
        _capi.check(self._L.kmer_b200_unroute_device(self._h, C.c_void_p(send_ptr), C.c_void_p(ret_ptr), C.byref(plan), sc,
                                                     C.c_void_p(recv_pos_ptr), rs, Q, C.c_void_p(status_ptr), C.byref(r)))
        return DeviceResult(self._L, r, Q)

    def presence_words(self, e: int) -> int:
        return int(self._L.kmer_b200_presence_words(self._h, e))

    def presence_export(self, e: int, bitmap_ptr: int) -> None:
        _capi.check(self._L.kmer_b200_presence_export(self._h, e, C.c_void_p(bitmap_ptr)))

    def presence_attach(self, e: int, bitmap) -> None:
        """bitmap: int64 device tensor of presence_words(e) words (kept alive by this object), or None to detach."""
        _capi.check(self._L.kmer_b200_presence_attach(self._h, e, C.c_void_p(bitmap.data_ptr() if bitmap is not None else 0)))
        self._adopted.append(bitmap)

    # -- introspection
    def element_info(self, e: int) -> _capi.ElementInfo:
        info = _capi.ElementInfo()
        _capi.check(self._L.kmer_b200_element_info_get(self._h, e, C.byref(info)))
        return info

    def element_arrays(self, e: int):
        """(sorted hashes, positions stably sorted by hash) of element e."""
        info = self.element_info(e)
        h = np.zeros(info.n_kmers, dtype=np.uint64)
        p = np.zeros(info.n_kmers, dtype=np.uint32)
        _capi.check(self._L.kmer_b200_element_hashes(self._h, e, h.ctypes.data_as(_capi.u64p), h.size))
        _capi.check(self._L.kmer_b200_element_positions(self._h, e, p.ctypes.data_as(_capi.u32p), p.size))
        return h, p

    def scheme(self, m: int):
        out = np.zeros(4096, dtype=np.uint32)
        multi = C.c_int(0)
        n = self._L.kmer_b200_scheme(self._h, m, out.ctypes.data_as(_capi.u32p), out.size, C.byref(multi))
        return [int(x) for x in out[:n]], bool(multi.value)

    PLAN_KINDS = ("exact bucket", "prefix slab", "contiguous verify", "reference :314 plan", "reference multi-k sum plan", "throws")

    def plan_table(self, m_lo: int, m_hi: int, mode: int = MODE_DEFAULT) -> list[dict]:
        """The plan per query length (kmer_b200_plan_table): kind, seed k, lookups, expected candidates / sectors from
        the bucket statistics measured on this index."""
        rows = (_capi.PlanRow * (m_hi - m_lo + 1))()
        _capi.check(self._L.kmer_b200_plan_table(self._h, mode, m_lo, m_hi, rows))
        return [{"m": int(r.m), "kind": self.PLAN_KINDS[r.kind], "seed_k": int(r.seed_k), "lookups": int(r.n_lookups),
                 "candidates": float(r.expected_candidates), "sectors": float(r.expected_sectors)} for r in rows]

    def stats(self) -> dict:
        arr = (_capi.KernelStat * 32)()
        n = self._L.kmer_b200_stats(self._h, arr, 32)
        return {arr[i].name.decode(): {"launches": int(arr[i].launches), "device_ms": float(arr[i].device_ms),
                                       "algorithmic_bytes": float(arr[i].algorithmic_bytes)} for i in range(n)}

    def stats_reset(self):
        self._L.kmer_b200_stats_reset(self._h)

    def last_search_transfer(self) -> tuple[int, int]:
        """(host-to-device, device-to-host) bytes the last host-buffer search on this handle moved over PCIe."""
        a, b = C.c_uint64(0), C.c_uint64(0)
        self._L.kmer_b200_last_search_transfer(self._h, C.byref(a), C.byref(b))
        return int(a.value), int(b.value)

    def build_transfer(self) -> int:
        """Bytes the text took over PCIe when this index was built from a host buffer (kmer_b200_build_transfer)."""
        return int(self._L.kmer_b200_build_transfer(self._h))

    def last_search_host_path(self) -> dict:
        """Which host pipeline the last host-buffer search took (kmer_b200_last_search_host_path)."""
        a, b, r = C.c_uint32(0), C.c_uint32(0), C.c_double(0)
        self._L.kmer_b200_last_search_host_path(self._h, C.byref(a), C.byref(b), C.byref(r))
        names = {0: "single copy", 3: "streaming host pack + raw chunks"}
        return {"pipeline": names.get(int(a.value), str(a.value)), "raw_chunk_pct": int(b.value), "host_pack_gbs": float(r.value)}

    @property
    def last_search_gathers(self) -> int:
        """profile=2: 32-byte sectors the last search gathered at data-dependent addresses."""
        return int(self._L.kmer_b200_last_search_gathers(self._h))

    @property
    def device_bytes(self) -> int:
        return int(self._L.kmer_b200_device_bytes(self._h))


def gather_probe_at(ptr: int, table_bytes: int, n_gathers: int = 1 << 26, stream: int | None = None) -> float:
    """Independent 8-byte reads per second from the given device table (local memory or a mapped peer buffer)."""
    ms = C.c_double(0)
    _capi.check(_capi.lib().kmer_b200_gather_probe_at(C.c_void_p(ptr), table_bytes, n_gathers, C.c_void_p(stream), C.byref(ms)))
    return n_gathers / (ms.value * 1e-3)


def peer_buffer_create(device: int, n_bytes: int) -> tuple[int, bytes]:
    """A device buffer other processes can map: (device pointer, 64-byte CUDA IPC handle)."""
    p = C.c_void_p()
    h = C.create_string_buffer(64)
    _capi.check(_capi.lib().kmer_b200_peer_buffer_create(device, n_bytes, C.byref(p), h))
    return int(p.value), h.raw


def peer_buffer_open(device: int, handle: bytes) -> int:
    """Map a buffer another process made with peer_buffer_create; kernels on `device` can read it (NVLink)."""
    p = C.c_void_p()
    _capi.check(_capi.lib().kmer_b200_peer_buffer_open(device, handle, C.byref(p)))
    return int(p.value)


def peer_buffer_release(device: int, ptr: int, opened: bool) -> None:
    _capi.check(_capi.lib().kmer_b200_peer_buffer_release(device, C.c_void_p(ptr), 1 if opened else 0))


def host_pack_stream(ranks, sigma: int) -> np.ndarray:
    """1-byte ranks -> the device's b-bit MSB-first words (query boundaries ignored), packed by the library's host
    thread pool: what a large host batch is turned into before it crosses PCIe. Needs no device."""
    r = np.ascontiguousarray(np.asarray(ranks, dtype=np.uint8))
    L = _capi.lib()
    words = np.empty(int(L.kmer_b200_host_pack_stream_words(r.size, sigma)), dtype=np.uint64)
    _capi.check(L.kmer_b200_host_pack_stream(r.ctypes.data_as(_capi.u8p), r.size, sigma, words.ctypes.data_as(_capi.u64p)))
    return words


def guard_violations() -> int:
    """KMER_B200_GUARD=1 (set before the library is loaded): stores seen just outside a device buffer so far."""
    return int(_capi.lib().kmer_b200_debug_guard_violations())


def guard_selftest() -> None:
    _capi.check(_capi.lib().kmer_b200_debug_guard_selftest())


def make_kmer_index(text, sigma: int, *ks: int, **kw) -> KmerIndex:
    """kmer::make_kmer_index<ks...>(text) (kmer_index.hpp:569-579); position type is uint32."""
    return KmerIndex(text, sigma, ks, **kw)
