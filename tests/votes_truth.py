"""Ground truth of record votes (KmerIndex.record_votes) in numpy, built on the seeding truth, and a naive per-window
dict tally to check it against.

votes(q, r) = the number of counted k-mers of read q (1 <= in-record occurrences, <= max_occ when max_occ > 0) with an
occurrence in record r, where the record of position p is the last r with starts[r] <= p. Per read, every (r, votes) with
votes >= min_votes, by votes descending then record ascending."""
import numpy as np

from seeds_truth import in_record, query_kmers, seeds_truth


def votes_truth(text, sigma, k, q, off, starts, max_occ=0, min_votes=1):
    """(offsets, records, votes, kmer_hits, status) of record votes of the batch (q, off) on the collection (text, starts)."""
    off = np.asarray(off, dtype=np.int64)
    Q = off.size - 1
    s_off, pos, _, j, counts = seeds_truth(text, sigma, k, q, off, max_occ, starts=starts)
    qid = np.repeat(np.arange(Q, dtype=np.int64), np.diff(s_off.astype(np.int64)))
    rec = np.searchsorted(np.asarray(starts, dtype=np.int64), pos.astype(np.int64), side="right") - 1
    # one vote per (read, k-mer offset, record), then the votes per (read, record)
    trip = np.unique(np.stack([qid, j.astype(np.int64), rec]), axis=1) if qid.size else np.zeros((3, 0), np.int64)
    pairs, votes = (np.unique(trip[[0, 2]], axis=1, return_counts=True) if trip.shape[1]
                    else (np.zeros((2, 0), np.int64), np.zeros(0, np.int64)))
    keep = votes >= min_votes
    rq, rr, rv = pairs[0][keep], pairs[1][keep], votes[keep]
    order = np.lexsort((rr, -rv, rq))
    rq, rr, rv = rq[order], rr[order], rv[order]
    offsets = np.zeros(Q + 1, dtype=np.uint64)
    np.cumsum(np.bincount(rq, minlength=Q)[:Q], out=offsets[1:])
    counted = (counts >= 1) & ((counts <= max_occ) if max_occ > 0 else True)
    _, kq, _ = query_kmers(q, off, k, sigma)
    kmer_hits = np.bincount(kq, weights=counted, minlength=Q)[:Q].astype(np.uint32) if Q else np.zeros(0, np.uint32)
    return offsets, rr.astype(np.uint32), rv.astype(np.uint32), kmer_hits, np.zeros(Q, np.uint8)


def votes_naive(text, k, q, off, starts, max_occ=0, min_votes=1):
    """The same by comparing every k-mer of every read with every text window and tallying in a dict (small inputs)."""
    text = np.asarray(text, dtype=np.uint8)
    n = text.size
    ok = in_record(n, k, starts)
    win = np.lib.stride_tricks.sliding_window_view(text, k) if n >= k else np.zeros((0, k), np.uint8)
    st = [int(x) for x in starts]
    offsets, records, votes, hits = [0], [], [], []
    for i in range(len(off) - 1):
        qq = np.asarray(q[int(off[i]):int(off[i + 1])], dtype=np.uint8)
        tally, h = {}, 0
        for jj in range(qq.size - k + 1):
            occ = [int(p) for p in np.nonzero(np.all(win == qq[jj:jj + k], axis=1) & ok)[0]]
            if not occ or (max_occ > 0 and len(occ) > max_occ):
                continue
            h += 1
            recs = set()
            for p in occ:
                r = max(x for x in range(len(st) - 1) if st[x] <= p)
                recs.add(r)
            for r in recs:
                tally[r] = tally.get(r, 0) + 1
        got = sorted(((r, v) for r, v in tally.items() if v >= min_votes), key=lambda rv: (-rv[1], rv[0]))
        records += [r for r, _ in got]
        votes += [v for _, v in got]
        hits.append(h)
        offsets.append(offsets[-1] + len(got))
    Q = len(off) - 1
    return (np.array(offsets, np.uint64), np.array(records, np.uint32), np.array(votes, np.uint32), np.array(hits, np.uint32),
            np.zeros(Q, np.uint8))


def assert_votes_equal(got, want, label=""):
    names = ("offsets", "records", "votes", "kmer_hits", "status")
    for name, g, w in zip(names, got, want):
        g, w = np.asarray(g), np.asarray(w)
        assert g.shape == w.shape, f"{label}: {name}: shape {g.shape} != {w.shape}"
        if not np.array_equal(g.astype(np.int64), w.astype(np.int64)):
            bad = np.nonzero(g.astype(np.int64) != w.astype(np.int64))[0]
            raise AssertionError(f"{label}: {name} differs at {bad[:8]} ({bad.size} entries): {g[bad[:4]]} != {w[bad[:4]]}")
