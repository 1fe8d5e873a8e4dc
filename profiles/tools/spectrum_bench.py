"""k-mer spectrum timing (KmerIndex.spectrum / frequent_kmers / occurrence_cutoff).

Config 5: the 3 Gbp dna4 text generated on the device as bench.py does (kmer_b200_synth_ranks_device), k = 16, dense
directory of 4^16 + 1 entries (17.2 GB). Per entry point: the median device ms of --reps calls (CUDA events on the
index's stream around the whole call, allocation and copy back included), after one warm-up call. The dense sweep kernel
alone is timed in a separate torch.profiler pass; the share of the copy peak is the directory bytes over that kernel time
over 6535 GB/s (the device-to-device copy rate measured on a B200, DESIGN.md section 4).

Read set: a synthetic FASTQ of --reads reads of 150 symbols sampled from a --genome-symbol dna4 genome with 1 % random
substitutions, parsed on the device (parse_sequences), indexed as a collection at k = 21 and its spectrum read; reports
the parse, build and spectrum times, the windows the junction correction removes and the histogram's coverage peak.

    python profiles/tools/spectrum_bench.py [--n 3000000000] [--reps 5] [--reads 1000000] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import kmer_index_b200 as kb  # noqa: E402
from approx_bench import TEXT_SEED, card  # noqa: E402
from kmer_index_b200 import _capi  # noqa: E402

COPY_PEAK_GBS = 6535.0


def timed(fn, stream, reps):
    fn()  # warm-up
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        r = fn()
        b.record(stream)
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return {"ms": ms, "median_ms": float(np.median(ms))}, r


def kernel_ms(fn, names):
    """per kernel name (substring match): total device ms and calls in one profiled call of fn"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        for name in names:
            if name in ev.name and ev.device_type.name == "CUDA":
                d = out.setdefault(name, {"ms": 0.0, "calls": 0})
                d["ms"] += ev.device_time / 1000.0
                d["calls"] += 1
    return out


def fastq_reads(genome, reads, length, rng):
    starts = rng.integers(0, genome.size - length + 1, reads)
    seq = genome[starts[:, None] + np.arange(length)]
    err = rng.random(seq.shape) < 0.01
    seq[err] = (seq[err] + rng.integers(1, 4, int(err.sum()))) % 4
    chars = np.frombuffer(b"ACGT", dtype=np.uint8)[seq]
    lines = np.empty((reads, 2 * length + 7), dtype=np.uint8)
    lines[:, 0:2] = np.frombuffer(b"@r", dtype=np.uint8)
    lines[:, 2] = ord("\n")
    lines[:, 3:3 + length] = chars
    lines[:, 3 + length:6 + length] = np.frombuffer(b"\n+\n", dtype=np.uint8)
    lines[:, 6 + length:6 + 2 * length] = ord("I")
    lines[:, 6 + 2 * length] = ord("\n")
    return lines.tobytes()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3_000_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--genome", type=int, default=20_000_000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "spectrum_c5.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("spectrum_bench.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    sptr = stream.cuda_stream
    n = args.n
    out = {"card": card(), "reps": args.reps, "copy_peak_gbs": COPY_PEAK_GBS}

    # ---- config 5
    text = torch.empty(n, dtype=torch.uint8, device=dev)
    _capi.check(_capi.lib().kmer_b200_synth_ranks_device(text.data_ptr(), n, 0, 4, TEXT_SEED, sptr))
    torch.cuda.synchronize()
    ix = kb.KmerIndex(None, 4, [16], stream=sptr, device=0, text_device_ptr=text.data_ptr(), n=n)
    info = ix.element_info(0)
    dir_bytes = int(info.directory_entries) * 4
    c5 = {"workload": f"dna4 k=16, {n / 1e9:g} Gbp synthetic text", "directory_shift": int(info.directory_shift),
          "directory_entries": int(info.directory_entries), "directory_bytes": dir_bytes}
    c5["spectrum"], s = timed(lambda: ix.spectrum(bins=10001), stream, args.reps)
    c5["result"] = {"total": s.total, "distinct": s.distinct, "max_count": s.max_count, "hist_1_8": s.hist[1:9].tolist()}
    c5["frequent_top100"], (fh, fc) = timed(lambda: ix.frequent_kmers(min_count=1, limit=100), stream, args.reps)
    c5["top_counts"] = fc[:10].tolist()
    c5["cutoff_0.0002"], cut = timed(lambda: ix.occurrence_cutoff(0.0002), stream, args.reps)
    c5["cutoff_value"] = cut
    k = kernel_ms(lambda: ix.spectrum(bins=10001), ["spectrum_dense_kernel", "spectrum_sweep_kernel"])
    c5["kernels"] = k
    sweep = k.get("spectrum_dense_kernel", {}).get("ms")
    if sweep:
        c5["dense_sweep_gbs"] = dir_bytes / (sweep * 1e-3) / 1e9
        c5["dense_sweep_share_of_copy_peak"] = c5["dense_sweep_gbs"] / COPY_PEAK_GBS
    c5["whole_call_share_of_copy_peak"] = dir_bytes / (c5["spectrum"]["median_ms"] * 1e-3) / 1e9 / COPY_PEAK_GBS
    ix.close()
    del text
    torch.cuda.empty_cache()
    out["config5"] = c5
    print(json.dumps({"config5": {k: v for k, v in c5.items() if k not in ("kernels",)}}), flush=True)

    # ---- read set: FASTQ -> parse on the device -> collection index -> spectrum
    rng = np.random.default_rng(5)
    genome = rng.integers(0, 4, args.genome).astype(np.uint8)
    data = fastq_reads(genome, args.reads, 150, rng)
    rs = {"workload": f"{args.reads} reads of 150 symbols, 1 % substitutions, from a {args.genome / 1e6:g} Mbp genome, k = 21",
          "fastq_bytes": len(data)}
    t0 = time.perf_counter()
    recs = kb.parse_sequences(data, "dna4", fmt=0)
    torch.cuda.synchronize()
    rs["parse_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    cix = recs.index([21], collection=True)
    torch.cuda.synchronize()
    rs["build_s"] = time.perf_counter() - t0
    pix = recs.index([21])
    rs["records"] = len(recs)
    rs["spectrum"], cs = timed(lambda: cix.spectrum(bins=1001), torch.cuda.current_stream(), args.reps)
    ps = pix.spectrum(bins=1001)
    rs["junction_windows"] = ps.total - cs.total
    rs["junction_bound"] = 20 * (len(recs) - 1)
    rs["total"], rs["distinct"], rs["max_count"] = cs.total, cs.distinct, cs.max_count
    h = cs.hist[:1000].astype(np.int64)
    rs["coverage_peak"] = int(np.argmax(h[3:]) + 3)
    rs["hist_1_40"] = h[1:41].tolist()
    rs["cutoff_0.0002"] = cix.occurrence_cutoff(0.0002)
    cix.close()
    pix.close()
    recs.close()
    out["read_set"] = rs
    out["card_after"] = card()
    print(json.dumps({"read_set": rs}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"out": args.out, "card": out["card"]}))


if __name__ == "__main__":
    main()
