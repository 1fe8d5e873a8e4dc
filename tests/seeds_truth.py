"""Ground truth of k-mer seeding (KmerIndex.seeds) in numpy, and a naive per-window scan to check it against.

The truth follows the index's own layout: a stable argsort of the text's k-mer hashes gives every bucket in ascending
position order; on a collection index the windows that span a record start are dropped from it. A query's hits are the
buckets of its k-mers in j order, so they come out ordered by (j, p)."""
import numpy as np


def window_hashes(ranks, k, sigma):
    """The k-mer hash (kmer_index.hpp:56-73) at every start s <= len - k of `ranks`."""
    r = np.asarray(ranks, dtype=np.uint64)
    n = r.size - k + 1
    if n <= 0:
        return np.zeros(0, dtype=np.uint64)
    h = np.zeros(n, dtype=np.uint64)
    for t in range(k):
        h = h * np.uint64(sigma) + r[t:t + n]
    return h


def in_record(n, k, starts):
    """in_record[p] for p <= n - k: no record start s with p < s < p + k (every window when starts is None)."""
    if starts is None or n < k:
        return np.ones(max(n - k + 1, 0), dtype=bool)
    b = np.zeros(n + 1, dtype=np.int64)
    s = np.asarray(starts, dtype=np.int64)
    b[s[(s > 0) & (s < n)]] = 1
    cs = np.cumsum(b)
    p = np.arange(n - k + 1)
    return cs[p + k - 1] - cs[p] == 0


def query_kmers(q, off, k, sigma):
    """(hash, query id, j) of every k-mer of the batch, in query order then j order."""
    q = np.asarray(q, dtype=np.uint8)
    off = np.asarray(off, dtype=np.int64)
    Q = off.size - 1
    lens = np.diff(off)
    nk = np.maximum(lens - k + 1, 0)
    qid = np.repeat(np.arange(Q), nk)
    base = np.concatenate([[0], np.cumsum(nk)])[:-1]
    j = np.arange(int(nk.sum())) - np.repeat(base, nk)
    starts = off[:-1][qid] + j
    h = window_hashes(q[int(off[0]):], k, sigma) if q.size else np.zeros(0, np.uint64)
    return (h[starts - off[0]] if starts.size else np.zeros(0, np.uint64)), qid, j


def seeds_truth(text, sigma, k, q, off, max_occ=0, starts=None):
    """(offsets, positions, status, seed_offsets, kmer_counts) of seeding the batch (q, off) against text."""
    text = np.asarray(text, dtype=np.uint8)
    off = np.asarray(off, dtype=np.int64)
    Q = off.size - 1
    H = window_hashes(text, k, sigma)
    order = np.argsort(H, kind="stable")
    keep = in_record(text.size, k, starts)[order]
    sorted_h, kept = H[order][keep], order[keep].astype(np.uint32)   # the in-record part of every bucket, in order
    hq, qid, j = query_kmers(q, off, k, sigma)
    lo = np.searchsorted(sorted_h, hq, side="left")
    cnt = np.searchsorted(sorted_h, hq, side="right") - lo
    if max_occ > 0:
        counts = np.minimum(cnt, max_occ + 1)
        contrib = np.where(cnt > max_occ, 0, cnt)
    else:
        counts, contrib = cnt, cnt
    total = int(contrib.sum())
    first = np.concatenate([[0], np.cumsum(contrib)])[:-1]
    idx = np.repeat(lo - first, contrib) + np.arange(total)
    positions = kept[idx] if total else np.zeros(0, np.uint32)
    seed_offsets = np.repeat(j, contrib).astype(np.uint32)
    per_q = np.bincount(qid, weights=contrib, minlength=Q).astype(np.int64) if Q else np.zeros(0, np.int64)
    offsets = np.zeros(Q + 1, dtype=np.uint64)
    np.cumsum(per_q, out=offsets[1:])
    return offsets, positions.astype(np.uint32), np.zeros(Q, np.uint8), seed_offsets, counts.astype(np.uint32)


def seeds_naive(text, k, q, off, max_occ=0, starts=None):
    """The same by comparing every k-mer of every query with every text window (small inputs only)."""
    text = np.asarray(text, dtype=np.uint8)
    n = text.size
    ok = in_record(n, k, starts)
    win = np.lib.stride_tricks.sliding_window_view(text, k) if n >= k else np.zeros((0, k), np.uint8)
    offsets, positions, seed_offsets, counts = [0], [], [], []
    for i in range(len(off) - 1):
        qq = np.asarray(q[int(off[i]):int(off[i + 1])], dtype=np.uint8)
        got = 0
        for jj in range(qq.size - k + 1):
            hits = np.nonzero(np.all(win == qq[jj:jj + k], axis=1) & ok)[0]
            c = hits.size
            counts.append(min(c, max_occ + 1) if max_occ > 0 else c)
            if max_occ > 0 and c > max_occ:
                continue
            positions.extend(hits.tolist())
            seed_offsets.extend([jj] * c)
            got += c
        offsets.append(offsets[-1] + got)
    Q = len(off) - 1
    return (np.array(offsets, np.uint64), np.array(positions, np.uint32), np.zeros(Q, np.uint8),
            np.array(seed_offsets, np.uint32), np.array(counts, np.uint32))


def assert_seeds_equal(got, want, label=""):
    names = ("offsets", "positions", "status", "seed_offsets", "kmer_counts")
    for name, g, w in zip(names, got, want):
        g, w = np.asarray(g), np.asarray(w)
        assert g.shape == w.shape, f"{label}: {name}: shape {g.shape} != {w.shape}"
        if not np.array_equal(g.astype(np.int64), w.astype(np.int64)):
            bad = np.nonzero(g.astype(np.int64) != w.astype(np.int64))[0]
            raise AssertionError(f"{label}: {name} differs at {bad[:8]} ({bad.size} entries): {g[bad[:4]]} != {w[bad[:4]]}")
