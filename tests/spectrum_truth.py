"""Ground truth of the k-mer spectrum (KmerIndex.spectrum / frequent_kmers / occurrence_cutoff) in numpy, and a plain
dict count to check it against.

count(h) is the number of windows p in [0, n - k] with hash h; on a collection index only windows that cross no record
start count (no start s with p < s < p + k)."""
import math
from collections import Counter

import numpy as np

from seeds_truth import in_record, window_hashes


def counts_truth(text, sigma, k, starts=None):
    """(hashes ascending, counts) of every k-mer that occurs: hash every window, drop the record-crossing ones, np.unique."""
    h = window_hashes(text, k, sigma)
    h = h[in_record(len(text), k, starts)]
    u, c = np.unique(h, return_counts=True)
    return u.astype(np.uint64), c.astype(np.uint64)


def counts_naive(text, sigma, k, starts=None):
    """The same as a dict, one window at a time."""
    starts = set(int(s) for s in (starts if starts is not None else []))
    out = Counter()
    for p in range(len(text) - k + 1):
        if any(p < s < p + k for s in starts):
            continue
        h = 0
        for x in text[p:p + k]:
            h = h * sigma + int(x)
        out[h] += 1
    return dict(out)


def histogram(counts, bins, key_space):
    """hist[c] for 1 <= c < bins - 1, the overflow bin hist[bins - 1], hist[0] = key_space - distinct (saturated)."""
    hist = np.zeros(bins, dtype=np.uint64)
    c = np.minimum(np.asarray(counts, dtype=np.int64), bins - 1)
    np.add.at(hist, c, 1)
    hist[0] = min(key_space - len(counts), 2 ** 64 - 1)
    return hist


def frequent(hashes, counts, min_count, cap=None):
    """(hashes, counts) with count >= min_count, count descending then hash ascending; N = how many exist."""
    sel = counts >= min_count
    h, c = hashes[sel], counts[sel]
    order = np.lexsort((h, -c.astype(np.int64)))
    n = order.size
    order = order[:cap] if cap is not None else order
    return h[order], c[order], n


def cutoff(counts, fraction):
    """The smallest c >= 1 with #{count > c} <= floor(fraction * distinct); 0 when nothing is counted."""
    counts = np.asarray(counts, dtype=np.int64)
    if counts.size == 0:
        return 0
    allowed = math.floor(fraction * counts.size)
    c = 1
    srt = np.sort(counts)
    while srt.size - np.searchsorted(srt, c, side="right") > allowed:
        c += 1
    return c
