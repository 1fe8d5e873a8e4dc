"""Hit strategies of approximate search on the config-5 index (3 Gbp dna4, k = 16, text generated on the device as
bench.py does) with the reads of approx_bench.make_batch (10^7 of 100 and 10^7 of 150 symbols, 20 % random).

For each e in 0..4 it records the median device time (CUDA events on the index's stream, over --reps repetitions) of
"all", "all" + distances, "all_best", "strata" 1 and "single_best", each as the full and the count-only device search;
one repetition of every (strategy, form) pair per round, rounds alternating the pairs. It checks that every planted
read's best distance is at most its planted d and re-verifies a sample of 10^4 hits of each strategy on the host (the
returned distance equals the window's Hamming distance, within e). The card's name and power limit are read in the
same process. Writes one JSON file (default profiles/approx_hits_c5.json).

    python profiles/tools/approx_hits_bench.py [--n 3000000000] [--reads 10000000] [--reps 5] [--out FILE]
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
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import kmer_index_b200 as kb  # noqa: E402
from approx_bench import READ_SEED, TEXT_SEED, card, make_batch, median_ms  # noqa: E402
from kmer_index_b200 import _capi  # noqa: E402

# name -> (hits, strata, distances)
STRATEGIES = {"all": ("all", 0, False), "all+distances": ("all", 0, True), "all_best": ("all_best", 0, False),
              "strata1": ("strata", 1, False), "single_best": ("single_best", 0, False)}


def to_host(view, dev, dtype=None):
    t = torch.as_tensor(view, device=dev).clone()
    return t if dtype is None else t.to(dtype)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3_000_000_000)
    ap.add_argument("--reads", type=int, default=10_000_000, help="reads per length (100 and 150)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--budgets", default="0,1,2,3,4")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "approx_hits_c5.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("approx_hits_bench.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda", 0)
    info = card()
    stream = torch.cuda.Stream(device=dev)
    sptr = stream.cuda_stream
    n, reads = args.n, args.reads
    text = torch.empty(n, dtype=torch.uint8, device=dev)
    _capi.check(_capi.lib().kmer_b200_synth_ranks_device(text.data_ptr(), n, 0, 4, TEXT_SEED, sptr))
    torch.cuda.synchronize()
    out = {"workload": f"dna4 k=16, {n / 1e9:g} Gbp text, {reads} reads of 100 + {reads} of 150 symbols, 20 % random",
           "card": info, "reps": args.reps, "budgets": []}
    t0 = time.time()
    ix = kb.KmerIndex(None, 4, [16], stream=sptr, device=0, text_device_ptr=text.data_ptr(), n=n)
    torch.cuda.synchronize()
    out["build_s"] = time.time() - t0
    for e in [int(x) for x in args.budgets.split(",")]:
        q, off, origins, planted, d = make_batch(text, n, reads, e, READ_SEED + e, dev)
        torch.cuda.synchronize()
        Q = off.numel() - 1
        call = (q.data_ptr(), off.data_ptr(), Q, 150, e)
        runs = {}
        for name, (h, s, dist) in STRATEGIES.items():
            runs[(name, "full")] = lambda h=h, s=s, dist=dist: ix.search_approx_batch_device(*call, hits=h, strata=s, distances=dist)
            runs[(name, "count")] = lambda h=h, s=s: ix.count_approx_batch_device(*call, hits=h, strata=s)
        for fn in runs.values():   # warm-up of every shape
            fn().free()
        times = {k: [] for k in runs}
        for _ in range(args.reps):  # one repetition of each pair per round: the pairs alternate
            for k, fn in runs.items():
                times[k] += median_ms(fn, stream, 1)[1]
        rec = {"e": e, "queries": Q, "strategies": {}}
        for name, (h, s, dist) in STRATEGIES.items():
            r = ix.search_approx_batch_device(*call, hits=h, strata=s, distances=True)   # the check run: with distances
            torch.cuda.synchronize()
            o = to_host(r.offsets(), dev)
            p = (to_host(r.positions(), dev, torch.int64) & 0xFFFFFFFF) if r.n_positions else torch.empty(0, dtype=torch.int64, device=dev)
            dd = to_host(r.distances(), dev, torch.int64) if r.n_positions else torch.empty(0, dtype=torch.int64, device=dev)
            bd = to_host(r.best_distances(), dev, torch.int64) if r.best_distances() is not None else None
            torch.cuda.synchronize()
            r.free()
            srec = {k2: {"median_ms": float(np.median(times[(name, k2)])), "ms": times[(name, k2)],
                         "queries_per_s": Q / (float(np.median(times[(name, k2)])) * 1e-3)} for k2 in ("full", "count")}
            srec["hits"] = int(o[-1].item())
            if bd is not None:
                ok = (bd[planted] <= d[planted]).all().item()   # a planted read's window is within its d (<= e)
                srec["planted_best_distance_within_d"] = bool(ok)
                srec["queries_with_hits"] = int((bd != 0xFF).sum().item())
            if p.numel():
                g = torch.Generator(device=dev)
                g.manual_seed(11 + e)
                pick = torch.randint(0, p.numel(), (min(10_000, p.numel()),), generator=g, device=dev)
                qid = torch.searchsorted(o[1:], pick, right=True)   # o[qid] <= pick < o[qid + 1]
                bad = 0
                for m in (100, 150):
                    mask = (off[qid + 1] - off[qid]) == m
                    sel, sq = pick[mask], qid[mask]
                    cols = torch.arange(m, device=dev)
                    tw = text[p[sel][:, None] + cols]
                    qw = q[off[sq][:, None] + cols]
                    ham = (tw != qw).sum(dim=1)
                    bad += int(((ham > e) | (ham != dd[sel])).sum().item())
                srec["spot_checked_hits"] = int(pick.numel())
                srec["spot_check_failures"] = bad
            rec["strategies"][name] = srec
        out["budgets"].append(rec)
        print(json.dumps({"e": e, **{k: (v["full"]["median_ms"], v["count"]["median_ms"], v["hits"])
                                     for k, v in rec["strategies"].items()}}), flush=True)
        del q, off, origins, planted, d
        torch.cuda.empty_cache()
    ix.close()
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"out": args.out, "card": info}))


if __name__ == "__main__":
    main()
