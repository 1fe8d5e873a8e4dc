"""CPU checks of the collection surface: the two derivations of the collection ground truth (tests/collection_truth.py)
agree on random collections with empty, 1-symbol and short records, the hit-strategy truth follows from them, and the
ctypes prototypes of the collection entry points match the C header (compiled with the host C compiler)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from approx_hits_truth import hit_distances
from collection_truth import hits_truth, random_starts, truth_filtered, truth_per_record
from conftest import ROOT


def random_batch(text, starts, rng, Q=160, m_hi=24):
    """random queries, record windows and windows across record starts, 0..40 symbols"""
    sigma = int(text.max()) + 1
    qs = []
    inner = [int(s) for s in starts[1:-1]]
    for i in range(Q):
        m = int(rng.integers(0, m_hi + 1))
        kind = i % 3
        if kind == 0 or m > text.size:
            x = rng.integers(0, sigma, m).astype(np.uint8)
        elif kind == 1:
            p = int(rng.integers(0, text.size - m + 1))
            x = text[p:p + m].copy()
        else:
            s = inner[int(rng.integers(0, len(inner)))] if inner else 0
            p = min(max(0, s - m // 2), text.size - m)
            x = text[p:p + m].copy()
        if x.size > 2 and i % 5 == 0:
            x[int(rng.integers(0, x.size))] = (x[0] + 1) % sigma
        qs.append(x)
    off = np.zeros(Q + 1, np.uint64)
    np.cumsum([x.size for x in qs], out=off[1:])
    return np.concatenate(qs).astype(np.uint8), off


@pytest.mark.parametrize("sigma,n,R", [(2, 400, 30), (4, 3000, 60), (4, 500, 1), (5, 800, 120)])
def test_two_derivations_agree(sigma, n, R):
    rng = np.random.default_rng(sigma * 1000 + R)
    text = rng.integers(0, sigma, n).astype(np.uint8)
    text[n // 3:n // 3 + n // 10] = 0                    # a constant run across records
    starts = random_starts(n, R, rng, short=R // 3)
    assert starts[0] == 0 and starts[-1] == n and np.all(np.diff(starts.astype(np.int64)) >= 0)
    q, off = random_batch(text, starts, rng)
    for e in (0, 1, 2, 4, 8):
        a = truth_per_record(text, starts, q, off, e)
        b = truth_filtered(text, starts, q, off, e)
        for x, y in zip(a, b):
            assert np.array_equal(x, y), (sigma, R, e)
        if R > 1 and e == 0:
            # windows across a record start exist in the concatenation and are not hits of the collection
            plain = truth_filtered(text, np.array([0, n], np.uint64), q, off, e)
            assert plain[1].size >= a[1].size


def test_hit_strategies_follow_from_per_record_truth():
    rng = np.random.default_rng(5)
    text = rng.integers(0, 4, 1500).astype(np.uint8)
    starts = random_starts(text.size, 25, rng, short=8)
    q, off = random_batch(text, starts, rng, Q=90)
    strategies = [("all", 0), ("all_best", 0), ("strata", 1), ("single_best", 0)]
    for e in (0, 2, 5):
        got = hits_truth(text, starts, q, off, e, strategies)
        a_off, a_pos, _ = truth_per_record(text, starts, q, off, e)
        assert np.array_equal(got[("all", 0)][0], a_off) and np.array_equal(got[("all", 0)][1], a_pos)
        d = hit_distances(text, q, off, a_off, a_pos)
        assert np.all(d <= e)
        best = got[("single_best", 0)]
        for i in range(off.size - 1):
            seg = d[int(a_off[i]):int(a_off[i + 1])]
            if seg.size:
                assert best[4][i] == seg.min()
                assert best[1][int(best[0][i])] == a_pos[int(a_off[i]) + int(np.argmin(seg))]


PROTOTYPES = {
    "kmer_b200_attach_records": "int (*)(kmer_b200_index *, const uint64_t *, uint64_t)",
    "kmer_b200_index_records": "const uint64_t *(*)(const kmer_b200_index *, uint64_t *)",
    "kmer_b200_locate": "int (*)(kmer_b200_index *, const uint32_t *, uint64_t, uint32_t *, uint32_t *)",
    "kmer_b200_locate_device": "int (*)(kmer_b200_index *, const uint32_t *, uint64_t, uint32_t *, uint32_t *)",
}


def test_prototypes_match_header(tmp_path):
    from kmer_index_b200 import _capi
    checks = "".join(f'_Static_assert(__builtin_types_compatible_p(__typeof__(&{name}), {proto}), "{name}");\n'
                     for name, proto in PROTOTYPES.items())
    src = tmp_path / "protos.c"
    src.write_text('#include "kmer_b200.h"\n' + checks + "int main(void) { return 0; }\n")
    subprocess.run([os.environ.get("CC", "gcc"), "-std=gnu11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                    "-o", str(tmp_path / "protos")], check=True)
    u64p, u32p = _capi.u64p, _capi.u32p
    assert _capi.SYMBOLS["kmer_b200_attach_records"] == (ctypes.c_int, [ctypes.c_void_p, u64p, ctypes.c_uint64])
    assert _capi.SYMBOLS["kmer_b200_index_records"] == (u64p, [ctypes.c_void_p, u64p])
    assert _capi.SYMBOLS["kmer_b200_locate"] == (ctypes.c_int, [ctypes.c_void_p, u32p, ctypes.c_uint64, u32p, u32p])
    assert _capi.SYMBOLS["kmer_b200_locate_device"] == (ctypes.c_int, [ctypes.c_void_p] * 2 + [ctypes.c_uint64] + [ctypes.c_void_p] * 2)
