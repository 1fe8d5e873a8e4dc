"""Expected results of the hit strategies of approximate search, derived with numpy from the every-window ground truth
(tests/approx_truth): d(p) of each truth hit, d_min per query, then the filter of the strategy."""
from __future__ import annotations

import numpy as np

from approx_truth import truth_approx

NO_HIT = 0xFF


def hit_distances(text, q_ranks, q_offsets, res_offsets, res_positions) -> np.ndarray:
    """uint8 Hamming distance between each listed window T[p, p+m) and its query"""
    text = np.asarray(text, dtype=np.uint8)
    out = np.zeros(res_positions.size, dtype=np.uint8)
    for i in range(res_offsets.size - 1):
        a, b = int(res_offsets[i]), int(res_offsets[i + 1])
        if a == b:
            continue
        qi = np.asarray(q_ranks[int(q_offsets[i]):int(q_offsets[i + 1])], dtype=np.uint8)
        win = np.lib.stride_tricks.sliding_window_view(text, qi.size)[res_positions[a:b].astype(np.int64)]
        out[a:b] = (win != qi).sum(axis=1)
    return out


def filter_hits(offsets, positions, status, dist, e: int, hits: str, strata: int = 0):
    """(offsets, positions, status, distances, best_distance) of strategy `hits` from the result of "all" with its
    distances. best_distance is None for "all"."""
    Q = status.size
    best = np.full(Q, NO_HIT, dtype=np.uint8)
    keep = np.zeros(positions.size, dtype=bool)
    for i in range(Q):
        a, b = int(offsets[i]), int(offsets[i + 1])
        if a == b or status[i] != 0:
            continue
        d = dist[a:b]
        dm = int(d.min())
        best[i] = dm
        if hits == "all":
            keep[a:b] = True
        elif hits == "all_best":
            keep[a:b] = d == dm
        elif hits == "strata":
            keep[a:b] = d <= min(e, dm + strata)
        elif hits == "single_best":
            keep[a + int(np.argmin(d))] = True   # the first minimum: positions ascend, so the lowest p
        else:
            raise ValueError(hits)
    qid = np.repeat(np.arange(Q), np.diff(offsets).astype(np.int64))
    counts = np.bincount(qid[keep], minlength=Q).astype(np.uint64)
    new_off = np.zeros(Q + 1, dtype=np.uint64)
    np.cumsum(counts, out=new_off[1:])
    return new_off, positions[keep], status.copy(), dist[keep], (None if hits == "all" else best)


def hits_truth(text, q_ranks, q_offsets, e: int, strategies):
    """{(hits, strata): (offsets, positions, status, distances, best_distance)} for each (hits, strata) of strategies"""
    off, pos, st = truth_approx(text, q_ranks, q_offsets, e)
    dist = hit_distances(text, q_ranks, q_offsets, off, pos)
    return {(h, s): filter_hits(off, pos, st, dist, e, h, s) for h, s in strategies}
