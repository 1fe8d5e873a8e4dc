"""Record votes on 3 Gbp collections (dna4, k = 16, text generated on the device as bench.py does).

Collections: the synthetic text cut into R = 25 and R = 10^5 records at seeded random places (as collection_bench.py
does), and a strain-like one: 10^3 near-copies of a 3 Mbp genome with 0.1 % substitutions, where every read's k-mers occur
in about 10^3 records, more than a read's shared-memory table holds, so every read takes the overflow path. Reads are
approx_bench.make_batch with e = 0 (--reads of 100 symbols and --reads of 150, 80 % text windows; --strain-reads each on
the strain-like collection, whose workaround materialises about 10^3 hits per k-mer).

Per collection and max_occ (0 and occurrence_cutoff(0.0002)) it records the median device time (CUDA events on the
index's stream) of record_votes_batch_device, of seeds_batch_device (the full seeding call on the same batch), and of the
workaround, alternating: seeds_batch_device + locate + a torch unique / bincount tally, run over chunks of reads so that
its hit lists fit in memory. The votes must equal the workaround's tally. Writes one JSON file (default
profiles/votes_c5.json).

    python profiles/tools/votes_bench.py [--n 3000000000] [--reads 10000000] [--strain-reads 5000] [--reps 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles", "tools"))

import kmer_index_b200 as kb  # noqa: E402
from approx_bench import READ_SEED, TEXT_SEED, card, make_batch  # noqa: E402
from kmer_index_b200 import _capi  # noqa: E402

K = 16
CHUNK = 1 << 20   # reads per workaround chunk


def timed(fn, stream):
    """(ms, result) of fn on `stream`, by CUDA events"""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    r = fn()
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b), r


def workaround(ix, q, off, max_occ, dev, keep=False):
    """seeds + locate + tally per chunk of reads: (pairs sorted by (read, -votes, record) as int64 read << 32 | record,
    votes) when keep, else None"""
    Q = off.numel() - 1
    out_p, out_v = [], []
    for c0 in range(0, Q, CHUNK):
        c1 = min(Q, c0 + CHUNK)
        o = off[c0:c1 + 1]
        s = ix.seeds_batch_device(q.data_ptr(), o.data_ptr(), c1 - c0, 150, max_occ=max_occ)
        n = s.n_positions
        if n:
            pos = torch.as_tensor(s.positions(), device=dev)
            j = torch.as_tensor(s.seed_offsets(), device=dev).to(torch.int64)
            rec, _ = ix.locate(pos)
            so = torch.as_tensor(s.offsets(), device=dev)
            qid = torch.repeat_interleave(torch.arange(c1 - c0, device=dev), torch.diff(so))
            trip = torch.unique((qid << 40) | (j << 32) | rec.to(torch.int64))   # one vote per (read, j, record)
            pairs, votes = torch.unique(trip >> 40 << 32 | (trip & 0xFFFFFFFF), return_counts=True)
            order = torch.sort(-votes, stable=True).indices
            order = order[torch.sort(pairs[order] >> 32, stable=True).indices]
            if keep:
                out_p.append(pairs[order] + ((c0 << 32) if c0 else 0))
                out_v.append(votes[order])
        s.free()
    if not keep:
        return None
    return torch.cat(out_p) if out_p else torch.zeros(0, dtype=torch.int64, device=dev), \
        torch.cat(out_v) if out_v else torch.zeros(0, dtype=torch.int64, device=dev)


def measure(ix, q, off, dev, stream, reps, label):
    Q = off.numel() - 1
    call = (q.data_ptr(), off.data_ptr(), Q, 150)
    rows = []
    for max_occ in (0, ix.occurrence_cutoff(0.0002)):
        ix.stats_reset()
        for _ in range(2):   # warm-up of every shape
            ix.record_votes_batch_device(*call, max_occ=max_occ).free()
            ix.seeds_batch_device(*call, max_occ=max_occ).free()
        workaround(ix, q, off, max_occ, dev)
        torch.cuda.empty_cache()
        overflow_launches = ix.stats().get("votes_overflow", {}).get("launches", 0)
        ts = {"votes": [], "seeds_full": [], "workaround": []}
        for _ in range(reps):   # alternating
            t, r = timed(lambda: ix.record_votes_batch_device(*call, max_occ=max_occ), stream)
            ts["votes"].append(t)
            r.free()
            t, r = timed(lambda: ix.seeds_batch_device(*call, max_occ=max_occ), stream)
            ts["seeds_full"].append(t)
            r.free()
            ts["workaround"].append(timed(lambda: workaround(ix, q, off, max_occ, dev), stream)[0])
        row = {"collection": label, "max_occ": max_occ, "overflow_launches": overflow_launches}
        for name, t in ts.items():
            row[name] = {"median_ms": float(np.median(t)), "ms": t}
        row["votes_over_seeds"] = row["votes"]["median_ms"] / row["seeds_full"]["median_ms"]
        row["workaround_over_votes"] = row["workaround"]["median_ms"] / row["votes"]["median_ms"]
        r = ix.record_votes_batch_device(*call, max_occ=max_occ)
        torch.cuda.synchronize()
        o = torch.as_tensor(r.offsets(), device=dev)
        rec = torch.as_tensor(r.positions(), device=dev).to(torch.int64) if r.n_positions else torch.zeros(0, dtype=torch.int64, device=dev)
        vot = torch.as_tensor(r.votes(), device=dev).to(torch.int64) if r.n_positions else torch.zeros(0, dtype=torch.int64, device=dev)
        hits = torch.as_tensor(r.kmer_hits(), device=dev).to(torch.int64)
        qid = torch.repeat_interleave(torch.arange(Q, device=dev), torch.diff(o))
        wp, wv = workaround(ix, q, off, max_occ, dev, keep=True)
        row["entries"] = int(r.n_positions)
        row["mean_entries_per_read"] = r.n_positions / Q
        row["reads_with_entries"] = int((torch.diff(o) > 0).sum().item())
        row["kmer_hits"] = int(hits.sum().item())
        row["identical_to_workaround"] = bool(torch.equal((qid << 32) | rec, wp) and torch.equal(vot, wv))
        r.free()
        del o, rec, vot, hits, qid, wp, wv
        torch.cuda.empty_cache()   # the workaround's tensors stay in torch's cache, out of reach of the library's pool
        rows.append(row)
        print(json.dumps({k: v for k, v in row.items()})[:600], flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3_000_000_000)
    ap.add_argument("--reads", type=int, default=10_000_000, help="reads per length (100 and 150)")
    ap.add_argument("--strain-reads", type=int, default=5000, help="reads per length on the strain-like collection")
    ap.add_argument("--records", default="25,100000")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "votes_c5.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("votes_bench.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    sptr = stream.cuda_stream
    n = args.n
    out = {"workload": f"dna4 k={K}, {n / 1e9:g} Gbp collections, {args.reads} reads of 100 + {args.reads} of 150 symbols "
                       f"({args.strain_reads} + {args.strain_reads} on the strain-like one), 80 % text windows",
           "card": card(), "reps": args.reps, "rows": []}
    text = torch.empty(n, dtype=torch.uint8, device=dev)
    _capi.check(_capi.lib().kmer_b200_synth_ranks_device(text.data_ptr(), n, 0, 4, TEXT_SEED, sptr))
    torch.cuda.synchronize()
    q, off, _, _, _ = make_batch(text, n, args.reads, 0, READ_SEED, dev)
    rng = np.random.default_rng(5)
    for R in [int(x) for x in args.records.split(",")]:
        starts = np.concatenate([[0], np.sort(rng.choice(n - 1, R - 1, replace=False) + 1), [n]]).astype(np.uint64)
        ix = kb.KmerIndex(None, 4, [K], stream=sptr, device=0, text_device_ptr=text.data_ptr(), n=n, mode=kb.MODE_CORRECT)
        ix.attach_records(starts)
        out["rows"] += measure(ix, q, off, dev, stream, args.reps, f"R={R}")
        ix.close()
    del q, off
    # strain-like: copies of the first G symbols, 0.1 % of each copy's symbols replaced by a random symbol
    G, copies = 3_000_000, n // 3_000_000
    g = torch.Generator(device=dev)
    g.manual_seed(17)
    strain = text[:G * copies].view(copies, G)
    strain[1:] = strain[0]
    n_sub = G // 1000
    for c in range(1, copies):
        at = torch.randint(0, G, (n_sub,), generator=g, device=dev)
        strain[c, at] = torch.randint(0, 4, (n_sub,), generator=g, device=dev, dtype=torch.uint8)
    torch.cuda.synchronize()
    ns = G * copies
    starts = np.arange(0, ns + 1, G, dtype=np.uint64)
    ix = kb.KmerIndex(None, 4, [K], stream=sptr, device=0, text_device_ptr=text.data_ptr(), n=ns, mode=kb.MODE_CORRECT)
    ix.attach_records(starts)
    q, off, _, _, _ = make_batch(text[:ns], ns, args.strain_reads, 0, READ_SEED + 1, dev)
    out["rows"] += measure(ix, q, off, dev, stream, args.reps, f"strain-like {copies} x {G}")
    ix.close()
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k != "rows"}, indent=1))


if __name__ == "__main__":
    main()
