"""CPU checks of the hit-strategy surface: the ctypes mirror of kmer_b200_approx_options against the C header (compiled
with the host C compiler), and the numpy derivation of the expected results (tests/approx_hits_truth.py) against a brute
force over every window."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from approx_hits_truth import NO_HIT, hits_truth
from conftest import ROOT


def test_options_struct_matches_header(tmp_path):
    from kmer_index_b200 import _capi
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "kmer_b200.h"\n'
                   "int main(void) { printf(\"%zu %zu %zu %zu %zu %d %d %d %d %d\\n\", sizeof(kmer_b200_approx_options),"
                   " offsetof(kmer_b200_approx_options, max_mismatches), offsetof(kmer_b200_approx_options, hits),"
                   " offsetof(kmer_b200_approx_options, strata), offsetof(kmer_b200_approx_options, flags),"
                   " KMER_B200_HITS_ALL, KMER_B200_HITS_ALL_BEST, KMER_B200_HITS_SINGLE_BEST, KMER_B200_HITS_STRATA,"
                   " KMER_B200_APPROX_DISTANCES); return 0; }\n")
    exe = str(tmp_path / "layout")
    subprocess.run([os.environ.get("CC", "gcc"), "-std=c11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                    str(src), "-o", exe], check=True)
    got = [int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    S = _capi.ApproxOptions
    assert got[:5] == [ctypes.sizeof(S), S.max_mismatches.offset, S.hits.offset, S.strata.offset, S.flags.offset]
    assert got[5:] == [_capi.HITS_ALL, _capi.HITS_ALL_BEST, _capi.HITS_SINGLE_BEST, _capi.HITS_STRATA,
                       _capi.APPROX_DISTANCES]


def brute(text, q, off, e, hits, s):
    """every window, every query: the strategy's definition written out directly"""
    n = text.size
    pos, dist, best, counts = [], [], [], []
    for i in range(off.size - 1):
        qi = q[int(off[i]):int(off[i + 1])]
        m = qi.size
        ds = [int((text[p:p + m] != qi).sum()) for p in range(n - m + 1)] if 0 < m <= n else []
        H = [(d, p) for p, d in enumerate(ds) if d <= e]
        if not H:
            best.append(NO_HIT)
            counts.append(0)
            continue
        dm = min(d for d, _ in H)
        best.append(dm)
        lim = {"all": e, "all_best": dm, "strata": min(e, dm + s)}.get(hits)
        sel = [min(H)] if hits == "single_best" else [(d, p) for d, p in H if d <= lim]
        sel.sort(key=lambda t: t[1])
        pos += [p for _, p in sel]
        dist += [d for d, _ in sel]
        counts.append(len(sel))
    o = np.zeros(len(counts) + 1, np.uint64)
    np.cumsum(counts, out=o[1:])
    return o, np.array(pos, np.uint32), np.array(dist, np.uint8), np.array(best, np.uint8)


@pytest.mark.parametrize("sigma", [2, 4, 5])
def test_derivation_equals_brute_force(sigma):
    rng = np.random.default_rng(11 + sigma)
    text = rng.integers(0, sigma, 300).astype(np.uint8)
    text[40:90] = 0
    lens = rng.integers(0, 14, 60)
    lens[:3] = [0, 301, 300]
    qs = [rng.integers(0, sigma, m).astype(np.uint8) if i % 2 else text[(p := int(rng.integers(0, max(1, 300 - m)))):p + m].copy()
          for i, m in enumerate(lens)]
    for j, x in enumerate(qs):
        if j % 2 == 0 and x.size > 3:
            x[int(rng.integers(0, x.size))] = (x[0] + 1) % sigma
    q = np.concatenate(qs).astype(np.uint8)
    off = np.zeros(len(qs) + 1, np.uint64)
    np.cumsum([x.size for x in qs], out=off[1:])
    strategies = [("all", 0), ("all_best", 0), ("strata", 1), ("strata", 2), ("strata", 9), ("single_best", 0)]
    for e in (0, 1, 3, 8):
        got = hits_truth(text, q, off, e, strategies)
        for h, s in strategies:
            w_off, w_pos, w_dist, w_best = brute(text, q, off, e, h, s)
            g_off, g_pos, g_st, g_dist, g_best = got[(h, s)]
            label = (e, h, s)
            assert np.array_equal(g_off, w_off) and np.array_equal(g_pos, w_pos), label
            assert np.array_equal(g_dist, w_dist), label
            assert (g_best is None) if h == "all" else np.array_equal(g_best, w_best), label
            assert np.array_equal(g_st, np.where(np.diff(off) == 0, 2, 0).astype(np.uint8)), label
        assert np.array_equal(got[("strata", 9)][0], got[("all", 0)][0])
