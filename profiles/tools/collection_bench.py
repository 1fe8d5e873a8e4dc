"""Collection index against the plain index on the config-5 text (3 Gbp dna4, k = 16, generated on the device as
bench.py does), cut into R = 1, 25 (chromosome-like) and 10^5 (transcript-like) records at seeded random places.

The batch is approx_bench.make_batch: 10^7 reads of 100 and 10^7 of 150 symbols. Per R it records the median device
time (CUDA events on the indexes' stream, alternating plain and collection in the same process) of the count-only and
the full approximate search for e = 0..4, all-best and single-best at e = 2, exact CORRECT-mode search (the collection
answers it through approximate search with e = 0, the plain index through its exact kernels) and kmer_b200_locate_device
over the hits of the e = 2 search; hits of both, the boundary bitmap's bytes and the card. Writes one JSON file (default
profiles/collection_c5.json).

    python profiles/tools/collection_bench.py [--n 3000000000] [--reads 10000000] [--reps 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import kmer_index_b200 as kb  # noqa: E402
from approx_bench import READ_SEED, TEXT_SEED, card, make_batch  # noqa: E402
from kmer_index_b200 import _capi  # noqa: E402


def timed(fn, stream):
    """device ms of one call (events on the index's stream), and its result's hit count"""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    r = fn()
    b.record(stream)
    b.synchronize()
    n = r.n_positions if r.positions_ptr else int(torch.as_tensor(r.offsets(), device="cuda")[-1].item())
    r.free()
    return a.elapsed_time(b), int(n)


def alternate(calls, stream, reps):
    """{name: {median_ms, ms, hits}} with the calls interleaved rep by rep"""
    for fn in calls.values():   # warm-up of every shape
        timed(fn, stream)
    out = {k: {"ms": []} for k in calls}
    for _ in range(reps):
        for k, fn in calls.items():
            t, n = timed(fn, stream)
            out[k]["ms"].append(t)
            out[k]["hits"] = n
    for v in out.values():
        v["median_ms"] = float(np.median(v["ms"]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3_000_000_000)
    ap.add_argument("--reads", type=int, default=10_000_000, help="reads per length (100 and 150)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--records", default="1,25,100000")
    ap.add_argument("--budgets", default="0,1,2,3,4")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "collection_c5.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("collection_bench.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    sptr = stream.cuda_stream
    n, reads = args.n, args.reads
    out = {"workload": f"dna4 k=16, {n / 1e9:g} Gbp text, {reads} reads of 100 + {reads} of 150 symbols, 20 % random",
           "card": card(), "reps": args.reps, "records": []}
    text = torch.empty(n, dtype=torch.uint8, device=dev)
    _capi.check(_capi.lib().kmer_b200_synth_ranks_device(text.data_ptr(), n, 0, 4, TEXT_SEED, sptr))
    torch.cuda.synchronize()
    budgets = [int(x) for x in args.budgets.split(",")]
    batches = {}
    for e in budgets:
        q, off, _, _, _ = make_batch(text, n, reads, e, READ_SEED + e, dev)
        batches[e] = (q, off)
    torch.cuda.synchronize()
    plain = kb.KmerIndex(None, 4, [16], stream=sptr, device=0, text_device_ptr=text.data_ptr(), n=n, mode=kb.MODE_CORRECT)
    L = _capi.lib()
    for R in [int(x) for x in args.records.split(",")]:
        rng = np.random.default_rng(1000 + R)
        starts = np.concatenate([[0], np.sort(rng.choice(n - 1, R - 1, replace=False) + 1), [n]]).astype(np.uint64)
        coll = kb.KmerIndex(None, 4, [16], stream=sptr, device=0, text_device_ptr=text.data_ptr(), n=n, mode=kb.MODE_CORRECT)
        bytes_before = coll.device_bytes
        coll.attach_records(starts)
        rec = {"R": R, "device_bytes_added": coll.device_bytes - bytes_before, "bitmap_bytes": (n // 64 + 1) * 8,
               "budgets": []}
        for e in budgets:
            q, off = batches[e]
            call = (q.data_ptr(), off.data_ptr(), off.numel() - 1, 150)
            calls = {"plain_count": lambda: plain.count_approx_batch_device(*call, e),
                     "collection_count": lambda: coll.count_approx_batch_device(*call, e),
                     "plain_full": lambda: plain.search_approx_batch_device(*call, e),
                     "collection_full": lambda: coll.search_approx_batch_device(*call, e)}
            if e == 2:
                for h in ("all_best", "single_best"):
                    calls[f"plain_{h}"] = lambda h=h: plain.search_approx_batch_device(*call, e, hits=h)
                    calls[f"collection_{h}"] = lambda h=h: coll.search_approx_batch_device(*call, e, hits=h)
            if e == 0:
                calls["plain_exact_correct_full"] = lambda: plain.search_batch_device(*call, kb.MODE_CORRECT)
                calls["collection_exact_correct_full"] = lambda: coll.search_batch_device(*call, kb.MODE_CORRECT)
                calls["plain_exact_correct_count"] = lambda: plain.count_batch_device(*call, kb.MODE_CORRECT)
                calls["collection_exact_correct_count"] = lambda: coll.count_batch_device(*call, kb.MODE_CORRECT)
            r = {"e": e, "queries": call[2], **alternate(calls, stream, args.reps)}
            if e == 2:
                res = coll.search_approx_batch_device(*call, e)
                stream.synchronize()
                hits = res.n_positions
                rec_out = torch.empty(max(hits, 1), dtype=torch.int32, device=dev)
                off_out = torch.empty(max(hits, 1), dtype=torch.int32, device=dev)
                torch.cuda.synchronize()
                ts = []
                for _ in range(args.reps + 1):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(stream)
                    _capi.check(L.kmer_b200_locate_device(coll.handle, C.c_void_p(res.positions_ptr), hits,
                                                          C.c_void_p(rec_out.data_ptr()), C.c_void_p(off_out.data_ptr())))
                    b.record(stream)
                    b.synchronize()
                    ts.append(a.elapsed_time(b))
                ts = ts[1:]
                r["locate_device"] = {"hits": hits, "ms": ts, "median_ms": float(np.median(ts)),
                                      "ns_per_hit": float(np.median(ts)) * 1e6 / max(hits, 1)}
                # spot check against a host binary search
                pos = torch.as_tensor(res.positions(), device=dev)[:100_000].cpu().numpy().view(np.uint32).astype(np.int64)
                want = np.searchsorted(starts.astype(np.int64), pos, "right") - 1
                r["locate_device"]["spot_check_ok"] = bool(np.array_equal(rec_out[:pos.size].cpu().numpy(), want))
                res.free()
            rec["budgets"].append(r)
            print(json.dumps({"R": R, "e": e, **{k: (v["median_ms"], v.get("hits")) for k, v in r.items() if isinstance(v, dict)}}),
                  flush=True)
        coll.close()
        out["records"].append(rec)
    plain.close()
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"out": args.out, "card": out["card"]}))


if __name__ == "__main__":
    main()
