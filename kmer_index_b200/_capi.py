"""ctypes binding of libkmer_b200.so (include/kmer_b200.h). No fallback: a missing library is an error."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("KMER_B200_LIB") or os.path.join(HERE, "libkmer_b200.so")   # KMER_B200_LIB: a tuning build

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)

OK = 0
MODE_REFERENCE_EXACT = 0
MODE_CORRECT = 1
MODE_DEFAULT = 0xFFFFFFFF

QUERY_OK = 0
QUERY_THROW_INVALID_ARGUMENT = 1
QUERY_UNDEFINED = 2
QUERY_TOO_LONG_FOR_SHARD = 3


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("mode", C.c_uint32), ("stream", C.c_void_p), ("shard_begin", C.c_uint64),
                ("n_total", C.c_uint64), ("halo", C.c_uint32), ("directory_bits", C.c_uint32),
                ("profile", C.c_uint32), ("reserved", C.c_uint32), ("key_part", C.c_uint32), ("key_parts", C.c_uint32),
                ("device_ids", C.POINTER(C.c_int32)), ("n_devices", C.c_uint32)]


HITS_ALL = 0
HITS_ALL_BEST = 1
HITS_SINGLE_BEST = 2
HITS_STRATA = 3
APPROX_DISTANCES = 1


class ApproxOptions(C.Structure):
    """kmer_b200_approx_options"""
    _fields_ = [("max_mismatches", C.c_uint32), ("hits", C.c_uint32), ("strata", C.c_uint32), ("flags", C.c_uint32)]


class ElementInfo(C.Structure):
    _fields_ = [("k", C.c_uint32), ("key_bits", C.c_uint32), ("directory_shift", C.c_uint32),
                ("sort_passes", C.c_uint32), ("n_kmers", C.c_uint64), ("directory_entries", C.c_uint64),
                ("device_bytes", C.c_uint64)]


class Part(C.Structure):
    _fields_ = [("key_lo", C.c_uint64), ("key_hi", C.c_uint64), ("n_kmers", C.c_uint64), ("directory_entries", C.c_uint64),
                ("d_positions", C.c_void_p), ("d_directory", C.c_void_p)]


class RoutePlan(C.Structure):
    _fields_ = [("n_parts", C.c_uint32), ("stride", C.c_uint32), ("capacity", C.c_uint32), ("reserved", C.c_uint32),
                ("block_bytes", C.c_uint64), ("return_block_bytes", C.c_uint64)]


class PlanRow(C.Structure):
    _fields_ = [("m", C.c_uint32), ("kind", C.c_uint32), ("seed_k", C.c_uint32), ("n_lookups", C.c_uint32),
                ("expected_candidates", C.c_double), ("expected_sectors", C.c_double)]


class SpectrumInfo(C.Structure):
    _fields_ = [("total", C.c_uint64), ("distinct", C.c_uint64), ("max_count", C.c_uint64), ("key_space", C.c_uint64)]


class KernelStat(C.Structure):
    _fields_ = [("name", C.c_char_p), ("launches", C.c_uint64), ("device_ms", C.c_double),
                ("algorithmic_bytes", C.c_double)]


# every symbol include/kmer_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "kmer_b200_config_default": (None, [C.POINTER(Config)]),
    "kmer_b200_abi_version": (C.c_int, []),
    "kmer_b200_last_error": (C.c_char_p, []),
    "kmer_b200_create": (C.c_int, [u8p, C.c_uint64, C.c_uint32, u32p, C.c_uint32, C.POINTER(Config),
                                   C.POINTER(C.c_void_p)]),
    "kmer_b200_create_from_device": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, u32p, C.c_uint32,
                                               C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "kmer_b200_create_from_text": (C.c_int, [C.c_char_p, C.c_uint64, u8p, C.c_uint32, u32p, C.c_uint32,
                                             C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "kmer_b200_search_batch_text": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_uint64, u8p, C.c_uint32,
                                              C.POINTER(C.c_void_p)]),
    "kmer_b200_parse_sequences": (C.c_int, [C.c_char_p, C.c_uint64, u8p, C.c_uint32, C.c_uint32, C.POINTER(Config),
                                            C.POINTER(C.c_void_p)]),
    "kmer_b200_records_count": (C.c_uint64, [C.c_void_p]),
    "kmer_b200_records_symbols": (C.c_uint64, [C.c_void_p]),
    "kmer_b200_records_starts": (u64p, [C.c_void_p]),
    "kmer_b200_records_header_offsets": (u64p, [C.c_void_p]),
    "kmer_b200_records_ranks_device": (C.c_void_p, [C.c_void_p]),
    "kmer_b200_records_locate": (C.c_int, [C.c_void_p, u32p, C.c_uint64, C.c_uint64, u32p, u32p]),
    "kmer_b200_records_free": (None, [C.c_void_p]),
    "kmer_b200_attach_records": (C.c_int, [C.c_void_p, u64p, C.c_uint64]),
    "kmer_b200_index_records": (u64p, [C.c_void_p, u64p]),
    "kmer_b200_locate": (C.c_int, [C.c_void_p, u32p, C.c_uint64, u32p, u32p]),
    "kmer_b200_locate_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "kmer_b200_destroy": (None, [C.c_void_p]),
    "kmer_b200_save": (C.c_int, [C.c_void_p, C.c_char_p]),
    "kmer_b200_load": (C.c_int, [C.c_char_p, C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "kmer_b200_search_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                                         C.POINTER(C.c_void_p)]),
    "kmer_b200_search_batch_ptrs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                                              C.POINTER(C.c_void_p)]),
    "kmer_b200_search_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                                C.c_uint32, C.POINTER(C.c_void_p)]),
    "kmer_b200_count_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                               C.c_uint32, C.POINTER(C.c_void_p)]),
    "kmer_b200_search_approx_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                                                C.POINTER(C.c_void_p)]),
    "kmer_b200_search_approx_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                                       C.c_uint32, C.POINTER(C.c_void_p)]),
    "kmer_b200_count_approx_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                                      C.c_uint32, C.POINTER(C.c_void_p)]),
    "kmer_b200_search_approx_batch_ex": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(ApproxOptions),
                                                   C.POINTER(C.c_void_p)]),
    "kmer_b200_search_approx_batch_device_ex": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                                          C.POINTER(ApproxOptions), C.POINTER(C.c_void_p)]),
    "kmer_b200_count_approx_batch_device_ex": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                                         C.POINTER(ApproxOptions), C.POINTER(C.c_void_p)]),
    "kmer_b200_seed_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32,
                                       C.POINTER(C.c_void_p)]),
    "kmer_b200_seed_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32,
                                              C.c_uint32, C.POINTER(C.c_void_p)]),
    "kmer_b200_count_seeds_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32,
                                                     C.c_uint32, C.POINTER(C.c_void_p)]),
    "kmer_b200_record_votes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32,
                                         C.POINTER(C.c_void_p)]),
    "kmer_b200_record_votes_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32,
                                                C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]),
    "kmer_b200_spectrum": (C.c_int, [C.c_void_p, C.c_uint32, u64p, C.c_uint64, C.POINTER(SpectrumInfo)]),
    "kmer_b200_frequent_kmers": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64, u64p, u64p, C.c_uint64, u64p]),
    "kmer_b200_occurrence_cutoff": (C.c_int, [C.c_void_p, C.c_uint32, C.c_double, u64p]),
    "kmer_b200_result_n_queries": (C.c_uint64, [C.c_void_p]),
    "kmer_b200_result_n_positions": (C.c_uint64, [C.c_void_p]),
    "kmer_b200_result_on_device": (C.c_int, [C.c_void_p]),
    "kmer_b200_result_hit_queries": (C.c_void_p, [C.c_void_p]),
    "kmer_b200_result_offsets": (C.c_void_p, [C.c_void_p]),
    "kmer_b200_result_positions": (C.c_void_p, [C.c_void_p]),
    "kmer_b200_result_status": (C.c_void_p, [C.c_void_p]),
    "kmer_b200_result_distances": (C.c_void_p, [C.c_void_p]),
    "kmer_b200_result_best_distances": (C.c_void_p, [C.c_void_p]),
    "kmer_b200_result_seed_offsets": (C.c_void_p, [C.c_void_p]),
    "kmer_b200_result_kmer_counts": (C.c_void_p, [C.c_void_p]),
    "kmer_b200_result_n_kmers": (C.c_uint64, [C.c_void_p]),
    "kmer_b200_result_votes": (C.c_void_p, [C.c_void_p]),
    "kmer_b200_result_kmer_hits": (C.c_void_p, [C.c_void_p]),
    "kmer_b200_result_free": (None, [C.c_void_p]),
    "kmer_b200_presence_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                                  C.c_uint32, C.c_void_p, C.c_uint32]),
    "kmer_b200_search_batch_device_global": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                                       C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]),
    "kmer_b200_search_sharded_begin": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                                 C.c_uint32, C.c_void_p, C.POINTER(C.c_void_p)]),
    "kmer_b200_search_sharded_finish": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "kmer_b200_search_sharded_abort": (None, [C.c_void_p]),
    "kmer_b200_search_sharded_peek": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "kmer_b200_search_sharded_add_counts": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "kmer_b200_element_part": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(Part)]),
    "kmer_b200_export_directory": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64, C.c_void_p]),
    "kmer_b200_export_bucket_sizes": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, u64p]),
    "kmer_b200_directory_from_sizes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "kmer_b200_adopt_element": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64]),
    "kmer_b200_peer_buffer_create": (C.c_int, [C.c_int, C.c_uint64, C.POINTER(C.c_void_p), C.c_char_p]),
    "kmer_b200_peer_buffer_open": (C.c_int, [C.c_int, C.c_char_p, C.POINTER(C.c_void_p)]),
    "kmer_b200_peer_buffer_release": (C.c_int, [C.c_int, C.c_void_p, C.c_int]),
    "kmer_b200_adopt_element_parts": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p), u64p, C.c_uint32, C.c_void_p,
                                                C.c_uint64]),
    "kmer_b200_route_plan_make": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_double, C.POINTER(RoutePlan)]),
    "kmer_b200_route_queries_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(RoutePlan),
                                                 C.c_void_p, C.c_void_p, u32p]),
    "kmer_b200_search_routed_device": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(RoutePlan), C.c_uint32, C.c_void_p, u64p,
                                                 C.POINTER(C.c_void_p)]),
    "kmer_b200_unroute_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(RoutePlan), u32p, C.c_void_p, u64p,
                                           C.c_uint64, C.c_void_p, C.POINTER(C.c_void_p)]),
    "kmer_b200_presence_words": (C.c_uint64, [C.c_void_p, C.c_uint32]),
    "kmer_b200_presence_export": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p]),
    "kmer_b200_presence_attach": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p]),
    "kmer_b200_n_elements": (C.c_uint32, [C.c_void_p]),
    "kmer_b200_element_info_get": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(ElementInfo)]),
    "kmer_b200_element_positions": (C.c_int, [C.c_void_p, C.c_uint32, u32p, C.c_uint64]),
    "kmer_b200_element_hashes": (C.c_int, [C.c_void_p, C.c_uint32, u64p, C.c_uint64]),
    "kmer_b200_scheme": (C.c_uint64, [C.c_void_p, C.c_uint64, u32p, C.c_uint64, C.POINTER(C.c_int)]),
    "kmer_b200_plan_table": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(PlanRow)]),
    "kmer_b200_scheme_for_ks": (C.c_uint64, [u32p, C.c_uint32, C.c_uint64, u32p, C.c_uint64, C.POINTER(C.c_int)]),
    "kmer_b200_stats": (C.c_uint32, [C.c_void_p, C.POINTER(KernelStat), C.c_uint32]),
    "kmer_b200_stats_reset": (None, [C.c_void_p]),
    "kmer_b200_device_bytes": (C.c_uint64, [C.c_void_p]),
    "kmer_b200_debug_guard_violations": (C.c_uint64, []),
    "kmer_b200_debug_guard_selftest": (C.c_int, []),
    "kmer_b200_last_search_gathers": (C.c_uint64, [C.c_void_p]),
    "kmer_b200_last_search_transfer": (None, [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "kmer_b200_build_transfer": (C.c_uint64, [C.c_void_p]),
    "kmer_b200_last_search_host_path": (None, [C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_double)]),
    "kmer_b200_gather_probe": (C.c_int, [C.c_uint64, C.c_uint64, C.c_void_p, C.POINTER(C.c_double)]),
    "kmer_b200_gather_probe_at": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.POINTER(C.c_double)]),
    "kmer_b200_host_pack_stream_words": (C.c_uint64, [C.c_uint64, C.c_uint32]),
    "kmer_b200_host_pack_stream": (C.c_int, [u8p, C.c_uint64, C.c_uint32, u64p]),
    "kmer_b200_fast_pow": (C.c_uint64, [C.c_uint64, C.c_uint8]),
    "kmer_b200_hash": (C.c_uint64, [u8p, C.c_uint32, C.c_uint32]),
    "kmer_b200_choose_best_k": (C.c_uint64, [u64p, C.c_uint64, C.c_uint64, u64p]),
    "kmer_b200_synth_ranks_device": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint64,
                                               C.c_void_p]),
}

_lib = None


def lib() -> C.CDLL:
    """Load libkmer_b200.so. Raises (never falls back) when the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -m kmer_index_b200.build` "
                               "(there is no CPU or PyTorch fallback for the k-mer index)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        if L.kmer_b200_abi_version() != 2:
            raise RuntimeError("libkmer_b200.so ABI version mismatch")
        _lib = L
    return _lib


class KmerB200Error(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"kmer_b200 error {code}: {message}")
        self.code = code


def check(code: int) -> None:
    if code != OK:
        raise KmerB200Error(code, (lib().kmer_b200_last_error() or b"").decode())
