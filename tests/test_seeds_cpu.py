"""The numpy ground truth of k-mer seeding (tests/seeds_truth.py) against a naive per-window scan, and the ctypes
prototypes of the seeding entry points against the C header. Needs no device."""
import ctypes

import numpy as np
import pytest

from seeds_truth import assert_seeds_equal, seeds_naive, seeds_truth

# the index shapes of tests/test_gpu_approx.py: (sigma, ks)
SHAPES = {"dna4_k12": (4, [12]), "dna4_k16": (4, [16]), "dna4_multi": (4, [5, 7, 9, 11, 13]), "dna15_k8": (15, [8]),
          "aa27_k5": (27, [5]), "dna5_k20": (5, [20]), "dna4_k31": (4, [31])}


def small_batch(text, sigma, k, rng, Q=40):
    """Text windows (at 0, at the end, anywhere; some repeated k-mers), random reads, and queries of 0 .. k - 1 symbols."""
    n = text.size
    qs = []
    for i in range(Q):
        m = int(rng.integers(0, 3 * k + 8))
        kind = i % 5
        if kind == 0:
            qs.append(text[:min(m, n)])
        elif kind == 1:
            qs.append(text[max(n - m, 0):])
        elif kind == 2 and m <= n:
            s = int(rng.integers(0, n - m + 1))
            qs.append(text[s:s + m])
        elif kind == 3:
            qs.append(rng.integers(0, sigma, m).astype(np.uint8))
        else:
            qs.append(rng.integers(0, sigma, int(rng.integers(0, k))).astype(np.uint8))
    off = np.zeros(len(qs) + 1, dtype=np.uint64)
    np.cumsum([x.size for x in qs], out=off[1:])
    return (np.concatenate(qs).astype(np.uint8) if off[-1] else np.zeros(0, np.uint8)), off


def low_entropy_text(n, sigma, rng):
    """Random text with runs of one symbol and a repeated motif: buckets of many positions."""
    t = rng.integers(0, sigma, n).astype(np.uint8)
    t[n // 4:n // 4 + n // 8] = 0
    motif = rng.integers(0, sigma, 7).astype(np.uint8)
    for s in range(n // 2, n // 2 + n // 8, 7):
        t[s:s + 7] = motif[:max(0, min(7, n - s))]
    return t


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("max_occ", [0, 1, 3])
def test_truth_matches_naive_scan(shape, max_occ):
    sigma, ks = SHAPES[shape]
    rng = np.random.default_rng(sum(map(ord, shape)) + max_occ)
    text = low_entropy_text(600, sigma, rng)
    for k in ks:
        q, off = small_batch(text, sigma, k, rng)
        assert_seeds_equal(seeds_truth(text, sigma, k, q, off, max_occ), seeds_naive(text, k, q, off, max_occ),
                           label=f"{shape} k={k} max_occ={max_occ}")


@pytest.mark.parametrize("max_occ", [0, 1, 3])
def test_truth_matches_naive_scan_on_collections(max_occ):
    """Records of every size: empty, shorter than k, about k, long; k-mers across a junction count only inside one."""
    rng = np.random.default_rng(7 + max_occ)
    for sigma, k in ((4, 5), (4, 12), (27, 3), (5, 20)):
        lens = [0, 3, k - 1, k, k + 1, 0, 0, 40, 1, 250, 2 * k, 0]
        starts = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
        text = low_entropy_text(int(starts[-1]), sigma, rng)
        q, off = small_batch(text, sigma, k, rng, Q=60)
        got = seeds_truth(text, sigma, k, q, off, max_occ, starts=starts)
        assert_seeds_equal(got, seeds_naive(text, k, q, off, max_occ, starts=starts), label=f"sigma={sigma} k={k}")
        # no reported window spans a record start
        s = starts.astype(np.int64)
        for p in got[1].astype(np.int64):
            assert not np.any((s > p) & (s < p + k))


def test_short_and_empty_queries():
    rng = np.random.default_rng(3)
    text = rng.integers(0, 4, 300).astype(np.uint8)
    q = np.concatenate([text[:5], text[10:26], text[40:41]])
    off = np.array([0, 0, 5, 5, 21, 22, 22], dtype=np.uint64)
    offsets, positions, status, seed_offsets, counts = seeds_truth(text, 4, 16, q, off)
    assert counts.size == 1 and counts[0] >= 1          # the one 16-mer of the batch, a window of the text
    assert list(np.diff(offsets.astype(np.int64))) == [0, 0, 0, int(counts[0]), 0, 0]
    assert 10 in positions.tolist() and set(seed_offsets.tolist()) == {0}
    assert not status.any()


def test_prototypes_match_header():
    from kmer_index_b200 import _capi
    dev = [ctypes.c_void_p] * 3 + [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32,
                                   ctypes.POINTER(ctypes.c_void_p)]
    assert _capi.SYMBOLS["kmer_b200_seed_batch"] == (ctypes.c_int, [ctypes.c_void_p] * 3 + [ctypes.c_uint64, ctypes.c_uint32,
                                                                                             ctypes.c_uint32,
                                                                                             ctypes.POINTER(ctypes.c_void_p)])
    assert _capi.SYMBOLS["kmer_b200_seed_batch_device"] == (ctypes.c_int, dev)
    assert _capi.SYMBOLS["kmer_b200_count_seeds_batch_device"] == (ctypes.c_int, dev)
    assert _capi.SYMBOLS["kmer_b200_result_n_kmers"] == (ctypes.c_uint64, [ctypes.c_void_p])
    import os
    from conftest import ROOT
    header = open(os.path.join(ROOT, "include", "kmer_b200.h")).read()
    for name in ("kmer_b200_seed_batch(", "kmer_b200_seed_batch_device(", "kmer_b200_count_seeds_batch_device(",
                 "kmer_b200_result_seed_offsets(", "kmer_b200_result_kmer_counts(", "kmer_b200_result_n_kmers("):
        assert name in header
