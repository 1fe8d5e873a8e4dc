"""Approximate search on the config-5 index (3 Gbp dna4, k = 16, text generated on the device as bench.py does).

The batch: 10^7 reads of 100 symbols and 10^7 of 150, text windows with 0..e random substitutions, of which 20 % are
replaced by random reads. For each e in 0..4 it records the median device time (CUDA events on the index's stream, over
--reps warm repetitions) of the count-only and the full approximate search, queries/s and hits, and, alternating with
them in the same process, exact CORRECT-mode search of the same batch; sectors/query come from a separate profile=2
index; gather_probe() is the ceiling. It checks that every planted read within e substitutions finds its origin and
re-verifies a sample of hits on the host. Writes one JSON file (default profiles/approx_c5.json).

    python profiles/tools/approx_bench.py [--n 3000000000] [--reads 10000000] [--reps 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import kmer_index_b200 as kb  # noqa: E402
from kmer_index_b200 import _capi  # noqa: E402

TEXT_SEED, READ_SEED = 205, 4242   # the text of bench.py's config 5


def card():
    out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    return {"nvidia_smi": out, "torch_name": torch.cuda.get_device_name(0)}


def make_batch(text, n, reads, e, seed, dev):
    """(q, offsets, origins, planted mask, d) on the device: reads of 100 then of 150 symbols"""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    lens = torch.cat([torch.full((reads,), 100, dtype=torch.int64, device=dev), torch.full((reads,), 150, dtype=torch.int64, device=dev)])
    Q = lens.numel()
    off = torch.zeros(Q + 1, dtype=torch.int64, device=dev)
    torch.cumsum(lens, 0, out=off[1:])
    q = torch.empty(int(off[-1].item()), dtype=torch.uint8, device=dev)
    origins = torch.randint(0, n - 150 + 1, (Q,), generator=g, device=dev, dtype=torch.int64)
    planted = torch.rand(Q, generator=g, device=dev) >= 0.2
    d = torch.randint(0, e + 1, (Q,), generator=g, device=dev, dtype=torch.int64)
    for m, q0 in ((100, 0), (150, reads)):
        for c0 in range(0, reads, 1 << 20):
            c1 = min(reads, c0 + (1 << 20))
            ids = torch.arange(q0 + c0, q0 + c1, device=dev)
            cols = torch.arange(m, device=dev)
            w = text[origins[ids, None] + cols]                           # (chunk, m) text windows
            for s in range(e):                                            # up to e substitutions (d per read)
                j = torch.randint(0, m, (ids.numel(),), generator=g, device=dev)
                delta = torch.randint(1, 4, (ids.numel(),), generator=g, device=dev, dtype=torch.uint8)
                rows = torch.nonzero(d[ids] > s).squeeze(1)
                w[rows, j[rows]] = (w[rows, j[rows]] + delta[rows]) % 4   # a repeated column can undo one: <= d
            rnd = torch.randint(0, 4, w.shape, generator=g, device=dev, dtype=torch.uint8)
            w = torch.where(planted[ids, None], w, rnd)
            q[int(off[q0 + c0].item()):int(off[q0 + c1].item())] = w.reshape(-1)
    return q, off, origins, planted, d


def median_ms(fn, stream, reps):
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        r = fn()
        b.record(stream)
        b.synchronize()
        ts.append(a.elapsed_time(b))
        r.free()
    return float(np.median(ts)), ts


def fetch(r, Q, dev):
    o = torch.as_tensor(r.offsets(), device=dev).clone()
    p = (torch.as_tensor(r.positions(), device=dev).clone() if r.n_positions and r.positions_ptr   # count-only: none
         else torch.empty(0, dtype=torch.int32, device=dev))
    torch.cuda.synchronize()   # the copies run on torch's stream; the result is freed in the index's stream order
    return o, p


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3_000_000_000)
    ap.add_argument("--reads", type=int, default=10_000_000, help="reads per length (100 and 150)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--budgets", default="0,1,2,3,4")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "approx_c5.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("approx_bench.py measures on a CUDA device; none is visible")
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
    budgets = [int(x) for x in args.budgets.split(",")]
    for e in budgets:
        q, off, origins, planted, d = make_batch(text, n, reads, e, READ_SEED + e, dev)
        torch.cuda.synchronize()
        Q = off.numel() - 1
        call = (q.data_ptr(), off.data_ptr(), Q, 150)
        for _ in range(2):    # warm-up of every shape
            ix.count_approx_batch_device(*call, e).free()
            ix.search_approx_batch_device(*call, e).free()
            ix.search_batch_device(*call, kb.MODE_CORRECT).free()
        rec = {"e": e, "queries": Q}
        t_count, t_full, t_exact = [], [], []
        for _ in range(args.reps):   # alternating: approximate count, approximate full, exact CORRECT search
            t_count += median_ms(lambda: ix.count_approx_batch_device(*call, e), stream, 1)[1]
            t_full += median_ms(lambda: ix.search_approx_batch_device(*call, e), stream, 1)[1]
            t_exact += median_ms(lambda: ix.search_batch_device(*call, kb.MODE_CORRECT), stream, 1)[1]
        for name, ts in (("count", t_count), ("full", t_full), ("exact_correct_full", t_exact)):
            med = float(np.median(ts))
            rec[name] = {"median_ms": med, "ms": ts, "queries_per_s": Q / (med * 1e-3)}
        r = ix.search_approx_batch_device(*call, e)
        torch.cuda.synchronize()
        o, p = fetch(r, Q, dev)
        r.free()
        rc = ix.count_approx_batch_device(*call, e)
        torch.cuda.synchronize()
        oc, _ = fetch(rc, Q, dev)
        rc.free()
        rec["hits"] = int(o[-1].item())
        rec["count_only_equals_full"] = bool(torch.equal(o, oc))
        # planted reads within e substitutions (all of them: d <= e by construction) find their origin
        counts = o[1:] - o[:-1]
        qid = torch.repeat_interleave(torch.arange(Q, device=dev), counts)
        pos = p.to(torch.int64) & 0xFFFFFFFF   # uint32 positions held as int32
        at_origin = pos == origins[qid]
        found = torch.zeros(Q, dtype=torch.bool, device=dev)
        found[qid[at_origin]] = True
        rec["planted"] = int(planted.sum().item())
        rec["planted_found_at_origin"] = int((found & planted).sum().item())
        # host re-verification of a sample of hits
        if p.numel():
            g = torch.Generator(device=dev)
            g.manual_seed(7 + e)
            pick = torch.randint(0, p.numel(), (min(10_000, p.numel()),), generator=g, device=dev)
            bad = 0
            for m in (100, 150):
                sel = pick[(off[qid[pick] + 1] - off[qid[pick]]) == m]
                cols = torch.arange(m, device=dev)
                tw = text[pos[sel][:, None] + cols].cpu().numpy()
                qw = q[off[qid[sel]][:, None] + cols].cpu().numpy()
                bad += int(((tw != qw).sum(axis=1) > e).sum())
            rec["spot_checked_hits"] = int(pick.numel())
            rec["spot_check_failures"] = bad
        out["budgets"].append(rec)
        del q, off, origins, planted, d, o, p, oc, qid, counts, at_origin, found
        torch.cuda.empty_cache()
        print(json.dumps({k: v for k, v in rec.items()}), flush=True)
    ix.close()
    # sectors per query: a separate profile=2 index (the accounting pass is not the timed kernel)
    ixp = kb.KmerIndex(None, 4, [16], stream=sptr, device=0, text_device_ptr=text.data_ptr(), n=n, profile=2)
    for rec in out["budgets"]:
        e = rec["e"]
        q, off, _, _, _ = make_batch(text, n, reads, e, READ_SEED + e, dev)
        torch.cuda.synchronize()
        Q = off.numel() - 1
        ixp.count_approx_batch_device(q.data_ptr(), off.data_ptr(), Q, 150, e).free()
        rec["sectors_per_query"] = ixp.last_search_gathers / Q
        ixp.count_batch_device(q.data_ptr(), off.data_ptr(), Q, 150, kb.MODE_CORRECT).free()
        rec["exact_sectors_per_query"] = ixp.last_search_gathers / Q
        del q, off
    ixp.close()
    del text
    torch.cuda.empty_cache()
    probe = kb.gather_probe(16 << 30, 1 << 29, sptr)
    out["gather_probe_sectors_per_s"] = probe
    for rec in out["budgets"]:
        rec["count_sectors_per_s"] = rec["sectors_per_query"] * rec["queries"] / (rec["count"]["median_ms"] * 1e-3)
        rec["count_share_of_gather_ceiling"] = rec["count_sectors_per_s"] / probe
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"out": args.out, "gather_probe": probe, "card": info}))


if __name__ == "__main__":
    main()
