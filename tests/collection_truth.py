"""Ground truth of search on a collection index (text = the records back to back, starts[0..R] their starts), derived in
two independent ways from the every-window scan (tests/approx_truth):
  (a) per record: the scan of each record's own text, positions shifted by its start, concatenated per query;
  (b) on the concatenation: the scan of the whole text minus the windows that contain a record start other than their
      own first symbol."""
from __future__ import annotations

import numpy as np

from approx_hits_truth import filter_hits, hit_distances
from approx_truth import truth_approx


def _csr(lists, Q):
    off = np.zeros(Q + 1, dtype=np.uint64)
    np.cumsum([x.size for x in lists], out=off[1:])
    pos = np.concatenate(lists).astype(np.uint32) if lists else np.zeros(0, np.uint32)
    return off, pos


def truth_per_record(text, starts, q_ranks, q_offsets, e: int):
    """(a): (offsets, positions, status)"""
    text = np.asarray(text, dtype=np.uint8)
    off_q = np.asarray(q_offsets, dtype=np.uint64)
    Q = off_q.size - 1
    per_query = [[] for _ in range(Q)]
    for r in range(len(starts) - 1):
        a, b = int(starts[r]), int(starts[r + 1])
        if a == b:
            continue
        o, p, _ = truth_approx(text[a:b], q_ranks, off_q, e)
        for i in np.flatnonzero(np.diff(o)):
            per_query[i].append(p[int(o[i]):int(o[i + 1])].astype(np.int64) + a)
    lists = [np.concatenate(x) if x else np.zeros(0, np.int64) for x in per_query]
    offsets, positions = _csr(lists, Q)
    status = np.where(off_q[1:] == off_q[:-1], 2, 0).astype(np.uint8)
    return offsets, positions, status


def truth_filtered(text, starts, q_ranks, q_offsets, e: int):
    """(b): (offsets, positions, status)"""
    off_q = np.asarray(q_offsets, dtype=np.uint64)
    o, p, st = truth_approx(text, q_ranks, off_q, e)
    m = np.repeat(np.diff(off_q).astype(np.int64), np.diff(o).astype(np.int64))
    s = np.asarray(starts, dtype=np.int64)
    keep = np.searchsorted(s, p.astype(np.int64), "right") == np.searchsorted(s, p.astype(np.int64) + m - 1, "right")
    qid = np.repeat(np.arange(off_q.size - 1), np.diff(o).astype(np.int64))
    counts = np.bincount(qid[keep], minlength=off_q.size - 1)
    offsets = np.zeros(off_q.size, dtype=np.uint64)
    np.cumsum(counts, out=offsets[1:])
    return offsets, p[keep], st


def hits_truth(text, starts, q_ranks, q_offsets, e: int, strategies):
    """{(hits, strata): (offsets, positions, status, distances, best_distance)} of the collection, from (a)"""
    off, pos, st = truth_per_record(text, starts, q_ranks, q_offsets, e)
    dist = hit_distances(text, q_ranks, q_offsets, off, pos)
    return {(h, s): filter_hits(off, pos, st, dist, e, h, s) for h, s in strategies}


def random_starts(n: int, n_records: int, rng, short: int = 0) -> np.ndarray:
    """starts[0..R] of n symbols cut into n_records records: `short` of them empty, 1-symbol or a few symbols long (next
    to each other too), the rest of random lengths"""
    lens = np.zeros(n_records, dtype=np.int64)
    special = rng.choice(n_records, size=min(short, n_records), replace=False)
    lens[special] = rng.choice([0, 0, 1, 1, 2, 3, 5, 7, 11, 15], size=special.size)
    rest = np.setdiff1d(np.arange(n_records), special)
    left = n - int(lens.sum())
    assert left >= rest.size
    if rest.size:
        cuts = np.sort(rng.choice(left - 1, size=rest.size - 1, replace=False) + 1) if rest.size > 1 else np.zeros(0, np.int64)
        lens[rest] = np.diff(np.concatenate([[0], cuts, [left]]))
    else:
        lens[-1] += left
    starts = np.zeros(n_records + 1, dtype=np.uint64)
    np.cumsum(lens, out=starts[1:])
    return starts
