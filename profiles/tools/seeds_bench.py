"""k-mer seeding on the config-5 index (3 Gbp dna4, k = 16, text generated on the device as bench.py does).

The batch: approx_bench.make_batch with e = 0 -- --reads reads of 100 symbols and --reads of 150, 80 % text windows.
For each max_occ it records the median device time (CUDA events on the index's stream) of the count-only and the full
seeding, alternating with the workaround seeding replaces: every read cut into its 16-mers, searched as queries of
their own by CORRECT-mode search_batch_device. Hits must be identical to the workaround's at max_occ = 0. Sectors per
k-mer come from a separate profile = 2 index, gather_probe() is the ceiling, and the host C ABI forms of both (host
buffers in, host result out) are timed once each with their H2D bytes. Writes one JSON file (default
profiles/seeds_c5.json).

    python profiles/tools/seeds_bench.py [--n 3000000000] [--reads 1000000] [--reps 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles", "tools"))

import kmer_index_b200 as kb  # noqa: E402
from approx_bench import READ_SEED, TEXT_SEED, card, make_batch, median_ms  # noqa: E402
from kmer_index_b200 import _capi  # noqa: E402

K = 16


def split_kmers(q, off, dev):
    """every k-mer of every read as a query of its own (the workaround): (ranks, offsets) on the device"""
    lens = off[1:] - off[:-1]
    nk = torch.clamp(lens - K + 1, min=0)
    qid = torch.repeat_interleave(torch.arange(lens.numel(), device=dev), nk)
    first = torch.cumsum(nk, 0) - nk
    j = torch.arange(int(nk.sum().item()), device=dev) - first[qid]
    starts = off[:-1][qid] + j
    kq = torch.empty(starts.numel() * K, dtype=torch.uint8, device=dev)
    for c0 in range(0, starts.numel(), 1 << 24):
        s = starts[c0:c0 + (1 << 24)]
        kq[c0 * K:(c0 + s.numel()) * K] = q[s[:, None] + torch.arange(K, device=dev)].reshape(-1)
    koff = torch.arange(starts.numel() + 1, dtype=torch.int64, device=dev) * K
    return kq, koff


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3_000_000_000)
    ap.add_argument("--reads", type=int, default=1_000_000, help="reads per length (100 and 150)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "seeds_c5.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("seeds_bench.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    sptr = stream.cuda_stream
    n, reads = args.n, args.reads
    out = {"workload": f"dna4 k={K}, {n / 1e9:g} Gbp text, {reads} reads of 100 + {reads} of 150 symbols, 80 % text windows",
           "card": card(), "reps": args.reps, "max_occ": []}
    text = torch.empty(n, dtype=torch.uint8, device=dev)
    _capi.check(_capi.lib().kmer_b200_synth_ranks_device(text.data_ptr(), n, 0, 4, TEXT_SEED, sptr))
    torch.cuda.synchronize()
    ix = kb.KmerIndex(None, 4, [K], stream=sptr, device=0, text_device_ptr=text.data_ptr(), n=n)
    q, off, _, _, _ = make_batch(text, n, reads, 0, READ_SEED, dev)
    kq, koff = split_kmers(q, off, dev)
    torch.cuda.synchronize()
    Q, NK = off.numel() - 1, koff.numel() - 1
    call, kcall = (q.data_ptr(), off.data_ptr(), Q, 150), (kq.data_ptr(), koff.data_ptr(), NK, K)
    out.update(queries=Q, kmers=NK, query_bytes=int(q.numel()), split_query_bytes=int(kq.numel()))
    for max_occ in (0, 100):
        for _ in range(2):   # warm-up of every shape
            ix.count_seeds_batch_device(*call, max_occ=max_occ).free()
            ix.seeds_batch_device(*call, max_occ=max_occ).free()
            ix.search_batch_device(*kcall, kb.MODE_CORRECT).free()
        ts = {"count": [], "full": [], "split_exact_full": []}
        for _ in range(args.reps):   # alternating
            ts["count"] += median_ms(lambda: ix.count_seeds_batch_device(*call, max_occ=max_occ), stream, 1)[1]
            ts["full"] += median_ms(lambda: ix.seeds_batch_device(*call, max_occ=max_occ), stream, 1)[1]
            ts["split_exact_full"] += median_ms(lambda: ix.search_batch_device(*kcall, kb.MODE_CORRECT), stream, 1)[1]
        rec = {"max_occ": max_occ}
        for name, t in ts.items():
            med = float(np.median(t))
            rec[name] = {"median_ms": med, "ms": t, "kmers_per_s": NK / (med * 1e-3)}
        r = ix.seeds_batch_device(*call, max_occ=max_occ)
        w = ix.search_batch_device(*kcall, kb.MODE_CORRECT)
        torch.cuda.synchronize()
        pos = torch.as_tensor(r.positions(), device=dev)
        wpos = torch.as_tensor(w.positions(), device=dev)
        counts = torch.as_tensor(r.kmer_counts(), device=dev)
        rec["hits"] = int(r.n_positions)
        rec["split_exact_hits"] = int(w.n_positions)
        rec["capped_kmers"] = int((counts > max_occ).sum().item()) if max_occ else 0
        if max_occ == 0:
            wcounts = torch.diff(torch.as_tensor(w.offsets(), device=dev))
            rec["identical_to_split_exact"] = bool(torch.equal(pos, wpos) and torch.equal(counts.to(torch.int64), wcounts))
        torch.cuda.synchronize()
        r.free()
        w.free()
        out["max_occ"].append(rec)
        print(json.dumps(rec)[:400], flush=True)

    # sectors per k-mer (profile = 2: every data-dependent 32-byte sector counted) and the gather ceiling
    prof = kb.KmerIndex(None, 4, [K], stream=sptr, device=0, text_device_ptr=text.data_ptr(), n=n, profile=2)
    prof.count_seeds_batch_device(*call).free()
    sectors_count = prof.last_search_gathers
    prof.seeds_batch_device(*call).free()
    sectors_full = prof.last_search_gathers
    prof.close()
    probe = kb.gather_probe()
    c0 = out["max_occ"][0]["count"]["median_ms"]
    out["sectors"] = {"count_pass_per_kmer": sectors_count / NK, "count_plus_write_per_kmer": sectors_full / NK,
                      "gather_probe_sectors_per_s": probe, "count_ceiling_ms": sectors_count / probe * 1e3,
                      "count_ms": c0, "count_share_of_ceiling": sectors_count / probe * 1e3 / c0}

    # the host C ABI: host buffers in, host result out (one call each; the wall time includes both copies)
    hq, hoff = q.cpu().numpy(), off.cpu().numpy().view(np.uint64)
    hkq, hkoff = kq.cpu().numpy(), koff.cpu().numpy().view(np.uint64)
    del kq
    torch.cuda.empty_cache()
    host = {}
    for name, fn in (("seeds", lambda: ix.seeds(hq, hoff, copy=False)),
                     ("split_exact", lambda: ix.search_batch(hkq, hkoff, mode=kb.MODE_CORRECT, copy=False))):
        fn().free()   # warm-up
        t0 = time.perf_counter()
        res = fn()
        dt = time.perf_counter() - t0
        h2d, d2h = ix.last_search_transfer()
        host[name] = {"wall_ms": dt * 1e3, "h2d_bytes": h2d, "d2h_bytes": d2h, "hits": int(res.offsets[-1])}
        res.free()
    host["h2d_ratio_split_over_seeds"] = host["split_exact"]["h2d_bytes"] / host["seeds"]["h2d_bytes"]
    out["host_c_abi"] = host
    ix.close()
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k != "max_occ"}, indent=1))


if __name__ == "__main__":
    main()
