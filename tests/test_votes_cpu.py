"""The numpy ground truth of record votes (tests/votes_truth.py) against a naive per-window dict tally, on small
collections with empty, 1-symbol, exactly-k and adjacent records, caps at, below and above the counts and min_votes 1, 2
and above every vote; plus the ctypes prototypes against the C header. Needs no device."""
import ctypes
import os

import numpy as np
import pytest

from test_seeds_cpu import low_entropy_text, small_batch
from votes_truth import assert_votes_equal, votes_naive, votes_truth


def repeated_collection(sigma, k, rng):
    """Records of every size (empty, 1 symbol, k - 1, k, adjacent short ones) around copies of one block, so that k-mers
    occur in several records and several times in one."""
    block = low_entropy_text(60, sigma, rng)
    parts, lens = [], [0, 1, k - 1, k, 0, 0, 2, 1, k + 1]
    for ln in lens:
        parts.append(rng.integers(0, sigma, ln).astype(np.uint8))
    for _ in range(4):
        parts.append(np.concatenate([block, block[:20]]))   # a record holding some k-mers twice
        parts.append(rng.integers(0, sigma, 30).astype(np.uint8))
    lens = [p.size for p in parts]
    starts = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    return np.concatenate(parts).astype(np.uint8), starts


@pytest.mark.parametrize("max_occ", [0, 1, 3, 8, 1000])
@pytest.mark.parametrize("min_votes", [1, 2, 1000])
def test_truth_matches_naive_tally(max_occ, min_votes):
    rng = np.random.default_rng(11 + max_occ * 7 + min_votes)
    for sigma, k in ((4, 5), (4, 8), (27, 3)):
        text, starts = repeated_collection(sigma, k, rng)
        q, off = small_batch(text, sigma, k, rng, Q=40)
        want = votes_naive(text, k, q, off, starts, max_occ, min_votes)
        assert_votes_equal(votes_truth(text, sigma, k, q, off, starts, max_occ, min_votes), want,
                           label=f"sigma={sigma} k={k} max_occ={max_occ} min_votes={min_votes}")
        if min_votes == 1000:
            assert want[1].size == 0
        if max_occ == 0 and min_votes == 1:
            assert want[1].size and np.any(np.diff(want[0].astype(np.int64)) > 1)   # reads with several records


def test_votes_rules():
    """A k-mer occurring twice in one record is one vote; the same k-mer at two offsets of a read is two; empty records
    get none; a read shorter than k has no entries and no k-mer hits."""
    k = 4
    a = np.array([0, 1, 2, 3, 0, 1, 2, 3], np.uint8)      # record 0: 0123 twice
    text = np.concatenate([a, np.array([3, 3, 3, 3], np.uint8), np.array([0, 1, 2, 3], np.uint8)])
    starts = np.array([0, 8, 8, 12, 16], np.uint64)           # record 1 empty
    q = np.concatenate([np.array([0, 1, 2, 3, 0, 1, 2, 3], np.uint8), np.array([0, 1, 2], np.uint8)])
    off = np.array([0, 8, 11], np.uint64)
    offsets, records, votes, hits, status = votes_truth(text, 4, k, q, off, starts)
    # read 0: 0123 at j = 0 and j = 4 (records 0 and 3), 1230 / 2301 / 3012 in record 0 only
    assert records[:2].tolist() == [0, 3] and votes[:2].tolist() == [5, 2]
    assert offsets.tolist() == [0, 2, 2] and hits.tolist() == [5, 0] and not status.any()
    assert_votes_equal((offsets, records, votes, hits, status), votes_naive(text, k, q, off, starts))


def test_prototypes_match_header():
    from conftest import ROOT
    from kmer_index_b200 import _capi
    P = ctypes.POINTER(ctypes.c_void_p)
    assert _capi.SYMBOLS["kmer_b200_record_votes"] == (ctypes.c_int, [ctypes.c_void_p] * 3 + [ctypes.c_uint64] + [ctypes.c_uint32] * 3 + [P])
    assert _capi.SYMBOLS["kmer_b200_record_votes_device"] == (ctypes.c_int, [ctypes.c_void_p] * 3 + [ctypes.c_uint64] * 2 +
                                                              [ctypes.c_uint32] * 3 + [P])
    header = open(os.path.join(ROOT, "include", "kmer_b200.h")).read()
    for name in ("kmer_b200_record_votes(", "kmer_b200_record_votes_device(", "kmer_b200_result_votes(", "kmer_b200_result_kmer_hits("):
        assert name in header and name[:-1] in _capi.SYMBOLS
