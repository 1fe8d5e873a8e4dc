"""The numpy ground truth of the k-mer spectrum (tests/spectrum_truth.py) against a plain dict count, the cutoff
definition on hand-made count sets, kmer_from_hash, and the ctypes declarations. No GPU needed."""
import ctypes

import numpy as np
import pytest

from collection_truth import random_starts
from spectrum_truth import counts_naive, counts_truth, cutoff, frequent, histogram


@pytest.mark.parametrize("sigma,k,n,records", [(4, 1, 50, 0), (4, 3, 300, 0), (4, 5, 400, 7), (5, 4, 350, 12), (27, 2, 500, 30),
                                              (4, 6, 40, 15), (4, 3, 3, 1)])
def test_truth_matches_dict_count(sigma, k, n, records):
    rng = np.random.default_rng(sigma * 1000 + k * 10 + n)
    text = rng.integers(0, sigma, n).astype(np.uint8)
    starts = random_starts(n, records, rng, short=records // 2) if records else None
    h, c = counts_truth(text, sigma, k, starts)
    want = counts_naive(text, sigma, k, starts)
    assert dict(zip(h.tolist(), c.tolist())) == want


def test_truth_with_empty_and_adjacent_records():
    text = np.array([0, 1, 2, 3, 0, 1, 2, 3, 3, 3, 3, 2], dtype=np.uint8)
    starts = np.array([0, 0, 3, 3, 4, 9, 12, 12], dtype=np.uint64)   # empty records, a 1-symbol record, adjacent starts
    for k in (1, 2, 3, 4, 5):
        h, c = counts_truth(text, 4, k, starts)
        assert dict(zip(h.tolist(), c.tolist())) == counts_naive(text, 4, k, starts)


def test_histogram_bins():
    counts = np.array([1, 1, 2, 3, 7, 70000], dtype=np.uint64)
    assert histogram(counts, 2, 16).tolist() == [10, 6]
    assert histogram(counts, 4, 16).tolist() == [10, 2, 1, 3]
    assert histogram(counts, 10, 2 ** 64).tolist() == [2 ** 64 - 1 - 5, 2, 1, 1, 0, 0, 0, 1, 0, 1]


def test_cutoff_definition():
    assert cutoff([], 0.1) == 0
    assert cutoff([5], 0.0) == 5
    assert cutoff([1, 1, 1], 0.0) == 1
    assert cutoff([1, 2, 3, 4], 0.0) == 4          # f = 0: the largest count
    assert cutoff([1, 2, 3, 4], 0.25) == 3         # one k-mer may lie above
    assert cutoff([1, 2, 3, 4], 0.49) == 3         # floor(0.49 * 4) = 1
    assert cutoff([1, 2, 3, 4], 0.5) == 2
    assert cutoff([1, 4, 4, 4, 9], 0.2) == 4       # ties at 4: one above (9) is allowed
    assert cutoff([1, 4, 4, 4, 9], 0.39) == 4
    assert cutoff([1, 4, 4, 4, 9], 0.4) == 4       # two allowed, but 4 leaves only 9 above
    assert cutoff([1, 4, 4, 4, 9], 0.8) == 1       # floor(4.0) = 4: only the three 4s and 9 above 1
    assert cutoff([2, 2], 0.99) == 2               # floor(1.98) = 1: c = 1 leaves two above, c = 2 none
    # the cutoff is the (floor(f * distinct) + 1)-th largest count, at least 1
    rng = np.random.default_rng(3)
    for _ in range(200):
        c = rng.integers(1, 30, int(rng.integers(1, 40)))
        f = float(rng.random())
        assert cutoff(c, f) == max(1, int(np.sort(c)[::-1][int(np.floor(f * c.size))]))


def test_frequent_order():
    h = np.array([5, 1, 9, 3, 7], dtype=np.uint64)
    c = np.array([2, 4, 2, 4, 1], dtype=np.uint64)
    fh, fc, n = frequent(h, c, 2)
    assert fh.tolist() == [1, 3, 5, 9] and fc.tolist() == [4, 4, 2, 2] and n == 4
    fh, fc, n = frequent(h, c, 1, cap=3)
    assert fh.tolist() == [1, 3, 5] and n == 5


@pytest.mark.parametrize("sigma,k", [(4, 1), (4, 16), (4, 31), (5, 17), (27, 7), (27, 13), (15, 9)])
def test_kmer_from_hash_round_trip(sigma, k):
    import kmer_index_b200 as kb
    rng = np.random.default_rng(sigma + k)
    for _ in range(20):
        r = rng.integers(0, sigma, k).astype(np.uint8)
        h = kb.kmer_hash(r, sigma)
        assert np.array_equal(kb.kmer_from_hash(h, k, sigma), r)
    assert kb.kmer_from_hash(0, k, sigma).tolist() == [0] * k
    assert kb.kmer_from_hash(sigma ** k - 1, k, sigma).tolist() == [sigma - 1] * k
    with pytest.raises(ValueError):
        kb.kmer_from_hash(sigma ** k, k, sigma)


def test_spectrum_symbols_declared():
    from kmer_index_b200 import _capi
    u64p = ctypes.POINTER(ctypes.c_uint64)
    assert _capi.SYMBOLS["kmer_b200_spectrum"][1][:4] == [ctypes.c_void_p, ctypes.c_uint32, u64p, ctypes.c_uint64]
    assert _capi.SYMBOLS["kmer_b200_frequent_kmers"] == (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64, u64p, u64p,
                                                                      ctypes.c_uint64, u64p])
    assert _capi.SYMBOLS["kmer_b200_occurrence_cutoff"] == (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_double, u64p])
    assert [f for f, _ in _capi.SpectrumInfo._fields_] == ["total", "distinct", "max_count", "key_space"]
