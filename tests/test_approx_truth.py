"""The approximate-search ground truth (tests/approx_truth) against a plain numpy brute force: the checker the GPU
tests of approximate search rely on. CPU only."""
import numpy as np
import pytest
from numpy.lib.stride_tricks import sliding_window_view

from approx_truth import truth_approx


def brute_approx(text, q, off, e):
    """(offsets, positions, status) of every window within e mismatches, from sliding windows and a count of !=."""
    text = np.asarray(text, dtype=np.uint8)
    counts, pos, status = [], [], []
    for i in range(off.size - 1):
        qq = q[int(off[i]):int(off[i + 1])]
        m = qq.size
        status.append(2 if m == 0 else 0)
        if m == 0 or m > text.size:
            counts.append(0)
            continue
        d = (sliding_window_view(text, m) != qq).sum(axis=1)
        hits = np.flatnonzero(d <= e).astype(np.uint32)
        counts.append(hits.size)
        pos.append(hits)
    offsets = np.zeros(len(counts) + 1, dtype=np.uint64)
    np.cumsum(counts, out=offsets[1:])
    positions = np.concatenate(pos) if pos else np.zeros(0, np.uint32)
    return offsets, positions.astype(np.uint32), np.array(status, dtype=np.uint8)


def plant(text, Q, m_lo, m_hi, d_max, sigma, seed):
    """Q text windows with exactly d substitutions each, d cycling through 0..d_max (capped at the window length); the
    windows include ones at position 0 and ones ending at n. Returns (ranks, offsets, origins, d per query)."""
    rng = np.random.default_rng(seed)
    n = text.size
    lens = rng.integers(m_lo, m_hi + 1, Q)
    lens = np.minimum(lens, n)
    off = np.zeros(Q + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    ranks = np.empty(int(off[-1]), dtype=np.uint8)
    origins = np.empty(Q, dtype=np.int64)
    ds = np.empty(Q, dtype=np.int64)
    for i in range(Q):
        m = int(lens[i])
        start = 0 if i % 7 == 0 else (n - m if i % 7 == 1 else int(rng.integers(0, n - m + 1)))
        w = text[start:start + m].copy()
        d = min(i % (d_max + 1), m)
        if sigma > 1:
            for j in rng.choice(m, size=d, replace=False):
                w[j] = (int(w[j]) + int(rng.integers(1, sigma))) % sigma
        ranks[int(off[i]):int(off[i + 1])] = w
        origins[i] = start
        ds[i] = d
    return ranks, off, origins, ds


@pytest.mark.parametrize("sigma", [4, 15, 27])
@pytest.mark.parametrize("e", [0, 1, 2, 4])
def test_truth_approx_matches_brute_force(sigma, e):
    from kmer_index_b200 import synth
    text = synth.random_text(3000, sigma, 11 + sigma)
    if sigma == 4:
        text[1000:1400] = 0                                    # long runs: many near-identical windows
    q_r, q_off = synth.stress_queries(text, 150, 1, 40, sigma, 5 + e)
    p_r, p_off, _, _ = plant(text, 150, 1, 60, e + 1, sigma, 7 + e)
    # queries shorter than e + 1, longer than the text, empty, windows ending exactly at n
    extra = [np.zeros(0, np.uint8), text[:e].copy(), text[-(e + 1):].copy(), text[-25:].copy(),
             synth.random_text(3001, sigma, 3), text.copy()]
    parts = [q_r, p_r] + extra
    lens = np.concatenate([np.diff(q_off), np.diff(p_off), [x.size for x in extra]]).astype(np.uint64)
    off = np.zeros(lens.size + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    q = np.concatenate(parts).astype(np.uint8)
    got = truth_approx(text, q, off, e)
    want = brute_approx(text, q, off, e)
    for g, w in zip(got, want):
        assert np.array_equal(g, w)


def test_truth_approx_planted_and_threads():
    from kmer_index_b200 import synth
    text = synth.random_text(5000, 4, 2)
    q, off, origins, ds = plant(text, 200, 20, 80, 3, 4, 9)
    off_a, pos_a, _ = truth_approx(text, q, off, 2, n_threads=1)
    off_b, pos_b, _ = truth_approx(text, q, off, 2, n_threads=7)
    assert np.array_equal(off_a, off_b) and np.array_equal(pos_a, pos_b)
    for i in range(200):
        hits = pos_a[int(off_a[i]):int(off_a[i + 1])]
        assert (origins[i] in hits) == (ds[i] <= 2), i


def test_truth_approx_zero_is_exact_truth(oracle_mod):
    from kmer_index_b200 import synth
    for sigma in (4, 15, 27):
        text = synth.random_text(4000, sigma, 21)
        q, off = synth.stress_queries(text, 300, 1, 30, sigma, 22)
        got = truth_approx(text, q, off, 0)
        want = oracle_mod.Oracle.truth(text, q, off)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
