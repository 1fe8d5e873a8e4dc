#!/usr/bin/env python
"""bench.py -- k-mer index build + batched search on B200 (see DESIGN.md "Measurement").

One step = one pass of the hot path over one synthetic batch: build the index from the packed text's raw
ranks (resident in HBM), then answer the whole query batch (resident in HBM, result left in HBM).
    value  = queries / s of the search half of the step (whole job, all ranks)
    build  = text symbols / s of the build half
    e2e    = the same two numbers through the reference-facing C ABI with HOST buffers: H2D of text and
             queries, D2H of offsets + positions + status inside the timed region
N > 1 (torchrun): the text is sharded by position range with a halo, every rank searches all queries on
its shard, presence masks are OR-ed and the per-shard hit lists gathered over NCCL (kmer_index_b200/sharded.py).

`--impl reference` times the reference's own CPU implementation (oracle/_ref, compiled from the reference's source
where oracle/Makefile's REF points; else the oracle port) on a bounded sample of the same workload on the host cores.

`--dump-outputs DIR` (one GPU) writes what the last timed step's search returned for a fixed, seeded sample of the
queries to DIR/*.npy, so that two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs; "c5" is the one the headline metric is quoted on and it fits one B200
    "c1": dict(name="kmer_index<dna4,k=10> 1 Mbp, 1e4 queries len 10", sigma=4, ks=[10], n=1_000_000, Q=10_000, m=(10, 10)),
    "c2": dict(name="kmer_index<dna4,k=12> 100 Mbp, 1e6 queries len 13-100", sigma=4, ks=[12], n=100_000_000,
               Q=1_000_000, m=(13, 100)),
    "c3": dict(name="multi_kmer_index<dna4,{5,7,9,11,13}> 100 Mbp, 1e6 queries len 4-40", sigma=4, ks=[5, 7, 9, 11, 13],
               n=100_000_000, Q=1_000_000, m=(4, 40)),
    "c4a": dict(name="kmer_index<dna15,k=8> 50 M symbols, 1e6 queries len 8", sigma=15, ks=[8], n=50_000_000, Q=1_000_000,
                m=(8, 8)),
    "c4b": dict(name="kmer_index<aa27,k=5> 50 M symbols, 1e6 queries len 5", sigma=27, ks=[5], n=50_000_000, Q=1_000_000,
                m=(5, 5)),
    "c5": dict(name="kmer_index<dna4,k=16> 3 Gbp, 1e8 queries len 16-64", sigma=4, ks=[16], n=3_000_000_000,
               Q=100_000_000, m=(16, 64), ref_Q=1_000_000),
}
TEXT_SEED, QUERY_SEED = 205, 1239


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c5", choices=sorted(WORKLOADS))
    ap.add_argument("--scale", type=float, default=1.0, help="shrink n and Q (development only; invalid as a result)")
    ap.add_argument("--text-symbols", type=int, default=0, help="override the text length only (development only; invalid as a result)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--count-only", action="store_true", help="time search without materialising positions")
    ap.add_argument("--multi", default="replicated", choices=["routed", "replicated", "peer", "position-range"],
                    help="N > 1: 'routed' = every GPU keeps one key-range part of the index, each GPU routes its 1/N of the "
                         "batch to the owners of the queries' first k-mers and gets the results back (three all-to-alls); "
                         "'replicated' = the parts are all-gathered over NVLink into the whole index on every GPU and each GPU "
                         "answers 1/N of the batch locally; 'peer' = only the directory is replicated, the position parts stay "
                         "where they were sorted and are read over NVLink (CUDA IPC mappings); 'position-range' = text shards with halo, every GPU searches the "
                         "whole batch, hit lists merged on rank 0")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's search result for a fixed sample of the queries to "
                         "DIR/{query_ids,offsets,positions,status}.npy, 64 MB at most")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.gpus != 1 or args.impl != "ours"):
        ap.error("--dump-outputs writes the search result of one GPU: it needs --gpus 1 and --impl ours")
    return args


# ------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own CPU implementation on a bounded sample
# ------------------------------------------------------------------------------------------------------------
def cpu_reference_sample(wl, steps: int, warmup: int):
    """Times the reference's build + search on the host cores. The sample keeps the workload's alphabet, ks and
    query-length range; the text is capped at 50 M symbols (the reference's hash map does not fit / finish beyond that on
    a bench budget) and the batch at ref_Q queries per step. The reference index is built ONCE (its build is
    single-threaded per k: ~20 s at 50 Mbp) and every step searches the same batch on it; search value = median."""
    import platform

    from kmer_index_b200 import synth
    from oracle import bindings

    sigma, ks, (m_lo, m_hi) = wl["sigma"], wl["ks"], wl["m"]
    cores = os.cpu_count() or 1
    n = min(wl["n"], 50_000_000)
    # seconds of reference search per step: its rest handling probes up to sigma^(k-rest) buckets per query
    Q = min(wl["Q"], wl.get("ref_Q", 20_000 if m_hi > max(ks) else 1_000_000))
    text = synth.random_text(n, sigma, TEXT_SEED)
    q, off = synth.random_queries(Q, m_lo, m_hi, sigma, QUERY_SEED)
    use_ref = bindings.have_reference() and bindings.Reference.supported(sigma, ks)
    if not use_ref:
        bindings.build()
    if use_ref:
        idx = bindings.Reference(text, sigma, ks, n_threads=cores)  # make_kmer_index<ks...>(text, hw threads)
        tb = idx.build_seconds
    else:
        t0 = time.perf_counter()
        idx = bindings.Oracle(text, sigma, ks)
        tb = time.perf_counter() - t0
    s_times = []
    for it in range(warmup + steps):
        if use_ref:
            idx.search(q, off, n_threads=cores, keep_positions=True)    # striped over the reference thread_pool
            ts = idx.search_seconds
        else:
            t0 = time.perf_counter()
            idx.search(q, off, n_threads=cores)
            ts = time.perf_counter() - t0
        if it >= warmup:
            s_times.append(ts)
    idx.close()
    ts = float(np.median(s_times))
    build_threads = min(len(ks), cores)  # the reference parallelises the build over k only (kmer_index.hpp:487-490)
    cpu_model = ""
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                cpu_model = ln.split(":", 1)[1].strip()
                break
    except OSError:
        cpu_model = platform.processor()
    return {
        "kind": "reference" if use_ref else "port",
        "cores": cores,
        "cpu": cpu_model,
        "search_qps": Q / ts,
        "search_qps_spread": [Q / max(s_times), Q / min(s_times)],
        "build_bases_per_s": n / tb,
        "build_threads": build_threads,
        "ms_per_step": ts * 1e3,
        "sample": f"text {n} of {wl['n']} symbols, {Q} of {wl['Q']} random queries len {m_lo}-{m_hi}; index built once "
                  f"({tb:.1f} s on {build_threads} thread(s), one per k) outside the step loop, every step searches the batch "
                  f"striped over {cores} threads; value = median of {len(s_times)} steps",
    }


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_sample(wl, max(1, args.steps), args.warmup)
    line = {
        "impl": "reference", "metric": "search_queries_per_s", "value": r["search_qps"], "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": wl["name"], "sample": r["sample"]},
        "build": {"metric": "build_gbases_per_s", "value": r["build_bases_per_s"] / 1e9, "unit": "Gbases/s",
                  "threads": r["build_threads"]},
        "cpu_baseline": {"value": r["search_qps"], "unit": "queries/s", "cores": r["cores"], "kind": r["kind"],
                         "sample": r["sample"], "build_gbases_per_s": r["build_bases_per_s"] / 1e9, "cpu": r["cpu"],
                         "search_qps_min_max": r["search_qps_spread"]},
        "e2e": {"value": r["search_qps"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.path = tempfile.mktemp(prefix="clocks_", suffix=".csv")
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={device_index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for ln in open(self.path):
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except OSError:
            pass
        if sm:
            busy = [x for x in sm if x > 0.5 * max(sm)] or sm
            out.update(sm_mhz=float(np.median(busy)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------------------------
# --dump-outputs
# ------------------------------------------------------------------------------------------------------------
DUMP_QUERIES, DUMP_SEED = 1 << 20, 20251
DUMP_BYTES = 64 << 20


def dump_result(out_dir, res, Q: int, dev, count_only: bool):
    """Write a DeviceResult of Q queries as DIR/<name>.npy, DUMP_BYTES at most:
        query_ids  float64 [S]      the sampled queries, ascending: all of them up to DUMP_QUERIES, else a sample
                                    drawn with DUMP_SEED, so it depends on Q alone
        offsets    float64 [S + 1]  CSR offsets of the sampled queries' hit lists in `positions`
        positions  float64 [P]      their positions (empty without hits; not written for a count-only search)
        status     float32 [S]      their status codes
    The hit lists are exact in float64 (positions < 2^32). Should the sampled hit lists not fit, the sample is cut to
    its longest prefix that does."""
    import torch
    S = min(Q, DUMP_QUERIES)
    ids = np.arange(Q) if S == Q else np.sort(np.random.default_rng(DUMP_SEED).choice(Q, S, replace=False))
    d_ids = torch.from_numpy(ids).to(dev)
    off = torch.as_tensor(res.offsets(), device=dev)
    counts = off[d_ids + 1] - off[d_ids]
    if not count_only:
        room = (DUMP_BYTES - 4096 - S * (8 + 8 + 4)) // 8    # 4 KiB for the last offset and the .npy headers
        S = int(torch.searchsorted(torch.cumsum(counts, 0), room, right=True).item())
        d_ids, counts = d_ids[:S], counts[:S]
    s_off = torch.zeros(S + 1, dtype=torch.int64, device=dev)
    torch.cumsum(counts, 0, out=s_off[1:])
    out = {"query_ids": d_ids.double(), "offsets": s_off.double(),
           "status": torch.as_tensor(res.status(), device=dev)[d_ids].float()}
    if not count_only:
        total = int(s_off[-1].item())
        src = torch.repeat_interleave(off[d_ids] - s_off[:-1], counts) + torch.arange(total, device=dev)
        pos = torch.as_tensor(res.positions(), device=dev)[src] if total else torch.empty(0, dtype=torch.int32, device=dev)
        out["positions"] = (pos.to(torch.int64) & 0xFFFFFFFF).double()
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


# ------------------------------------------------------------------------------------------------------------
# ours
# ------------------------------------------------------------------------------------------------------------
def run_ours(args, wl):
    import torch
    import torch.distributed as dist

    import kmer_index_b200 as kb
    from kmer_index_b200 import _capi, sharded

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = _capi.lib()
    # a dedicated non-default stream: the library enqueues everything on it (cfg.stream) and the CUDA events
    # below are recorded on it, so the timed region sees every kernel of the step
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sptr = stream.cuda_stream

    sigma, ks = wl["sigma"], wl["ks"]
    n = max(int(wl["n"] * args.scale), 4 * max(ks))
    if args.text_symbols:
        n = args.text_symbols
    Q = max(int(wl["Q"] * args.scale), 1)
    m_lo, m_hi = wl["m"]
    k_max = max(ks)
    routed = world > 1 and args.multi == "routed" and len(ks) == 1 and m_lo >= ks[0]
    # 'peer': like 'replicated' for the search (each GPU answers 1/N of the batch from a whole directory) but the position
    # array stays in the parts the GPUs sorted, mapped into every rank over NVLink (sharded.assemble_peer)
    peer = world > 1 and args.multi == "peer"
    replicated = world > 1 and (peer or args.multi == "replicated" or (args.multi == "routed" and not routed))
    parted = routed or replicated   # the index is built from key-range parts; every rank holds the whole text and 1/N of the batch

    # ---- the text. position-range: this rank's slice (k-mer/match starts [begin, end) plus a halo of m_hi - 1 symbols);
    # replicated: the whole text on every rank (each rank sorts only its key-range part of it)
    shard = sharded.shard_range(n, 1 if parted else world, 0 if parted else rank, halo=max(m_hi, k_max) - 1)
    n_local = shard.length
    text = torch.empty(n_local, dtype=torch.uint8, device=dev)
    _capi.check(L.kmer_b200_synth_ranks_device(text.data_ptr(), n_local, shard.begin, sigma, TEXT_SEED, sptr))

    # ---- the query batch: Q queries defined by the seeds alone. position-range: every rank holds all of them
    # ("queries are broadcast"); replicated: rank r holds queries [r Q / N, (r + 1) Q / N)
    g = torch.Generator(device=dev)
    g.manual_seed(QUERY_SEED)
    lens = torch.randint(m_lo, m_hi + 1, (Q,), generator=g, device=dev, dtype=torch.int64)
    q_lo, q_hi = (rank * Q // world, (rank + 1) * Q // world) if parted else (0, Q)
    sym_lo = int(lens[:q_lo].sum().item())
    Ql = q_hi - q_lo
    q_off = torch.zeros(Ql + 1, dtype=torch.int64, device=dev)
    torch.cumsum(lens[q_lo:q_hi], 0, out=q_off[1:])
    n_sym = int(q_off[-1].item())
    del lens
    q = torch.empty(n_sym, dtype=torch.uint8, device=dev)
    _capi.check(L.kmer_b200_synth_ranks_device(q.data_ptr(), n_sym, sym_lo, sigma, QUERY_SEED ^ 0xC0FFEE, sptr))
    torch.cuda.synchronize()

    def make_index(profile, text_ptr=None, host_text=None):
        if parted:
            return kb.KmerIndex(host_text, sigma, ks, stream=sptr, profile=profile, device=local_rank,
                                text_device_ptr=text_ptr, n=n_local, key_part=rank, key_parts=world)
        return kb.KmerIndex(host_text, sigma, ks, stream=sptr, profile=profile, device=local_rank,
                            shard_begin=shard.begin, n_total=n if world > 1 else 0, halo=shard.halo,
                            text_device_ptr=text_ptr, n=n_local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    assemble_marks = []   # (label, event) marks of the last replicated assembly
    # shared position buffers of the peer mode: mapped once, like a communicator, reused by every build
    peer_buffers = sharded.PeerPositions(world, rank, dist, dev) if peer else None

    def finish_build(ix):
        """the cross-GPU part of the build: all-gather of the parts (replicated) or of the presence bitmap (routed)"""
        if peer:
            assemble_marks.clear()
            sharded.assemble_peer(ix, world, rank, dist, dev, peer_buffers, timing=assemble_marks)
        elif replicated:
            assemble_marks.clear()
            sharded.assemble_replicated(ix, world, rank, dist, dev, timing=assemble_marks)
        elif routed:
            sharded.share_presence(ix, world, rank, dist, dev)

    def search_resident(ix, count_only):
        if routed:
            res = sharded.search_routed(ix, q.data_ptr(), q_off.data_ptr(), Ql, m_hi, -(-Q // world), world, rank, dist, dev)
            h = res.n_positions
            res.free()
            return h
        if replicated:
            return sharded.search_device(ix, q.data_ptr(), q_off.data_ptr(), Ql, m_hi, 1, dev, count_only=count_only)
        return sharded.search_device(ix, q.data_ptr(), q_off.data_ptr(), Q, m_hi, world, dev, count_only=count_only)

    def device_step(profile, keep=False):
        """build + search with inputs resident in HBM; returns (build_ms, gather_ms, search_ms, hits, stats, kept).
        keep (--dump-outputs, one GPU): the search call sharded.search_device makes, but the index and the result stay
        open and come back as kept = (index, result); otherwise kept is None. That step's search_ms then leaves out the
        result's free, which sharded.search_device enqueues before e[3]: four stream-ordered cudaFreeAsync calls."""
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record(stream)
        ix = make_index(profile, text_ptr=text.data_ptr())
        e[1].record(stream)
        finish_build(ix)   # NCCL: part of the build
        e[2].record(stream)
        if keep:
            res = (ix.count_batch_device if args.count_only else ix.search_batch_device)(q.data_ptr(), q_off.data_ptr(), Q, m_hi)
            hits = res.n_positions
        else:
            hits = search_resident(ix, args.count_only)
        e[3].record(stream)
        torch.cuda.synchronize()
        stats = ix.stats() if profile else None
        times = e[0].elapsed_time(e[2]), e[1].elapsed_time(e[2]), e[2].elapsed_time(e[3])
        if keep:
            return (*times, hits, stats, (ix, res))
        ix.close()
        return (*times, hits, stats, None)

    # ---- warm-up, then exactly K timed steps between barriers
    sampler = ClockSampler(local_rank) if rank == 0 else None   # started early: nvidia-smi needs ~1 s to come up
    for _ in range(args.warmup):
        device_step(False)
    barrier()
    b_ms, g_ms, s_ms, stats_acc, hits = [], [], [], {}, 0
    t_region = time.perf_counter()
    for i in range(args.steps):
        tb, tg, ts, hits, st, kept = device_step(True, keep=bool(args.dump_outputs) and i == args.steps - 1)
        b_ms.append(tb)
        g_ms.append(tg)
        s_ms.append(ts)
        for name, v in st.items():
            a = stats_acc.setdefault(name, {"launches": 0, "device_ms": 0.0, "algorithmic_bytes": 0.0})
            for key in a:
                a[key] += v[key]
    barrier()
    t_region = time.perf_counter() - t_region
    clocks = sampler.stop() if sampler else None
    if kept:
        ix, res = kept
        dump_result(args.dump_outputs, res, Q, dev, args.count_only)
        res.free()
        ix.close()
    # where the cross-GPU part of the last timed build went (rank 0's stream)
    assemble_ms = {}
    for (_, a), (label, b) in zip(assemble_marks, assemble_marks[1:]):
        assemble_ms[label] = assemble_ms.get(label, 0.0) + a.elapsed_time(b)

    # ---- outside the timed region: result fingerprint (hits, status histogram, position checksum -- identical for
    # every N and both multi-GPU modes), algorithmic gathers of the batch (profile = 2 counts the 32-byte sectors the
    # search must fetch at data-dependent addresses) and the device's random-gather ceiling
    gathers = gather_peak = None
    ix = make_index(2, text_ptr=text.data_ptr())
    finish_build(ix)
    search_resident(ix, True)
    gathers = ix.last_search_gathers
    if routed:
        fp = sharded.fingerprint_of(sharded.search_routed(ix, q.data_ptr(), q_off.data_ptr(), Ql, m_hi, -(-Q // world), world, rank,
                                                          dist, dev), Ql, dev, q_lo)
    else:
        fp = sharded.fingerprint(ix, q.data_ptr(), q_off.data_ptr(), Ql if replicated else Q, m_hi,
                                 1 if replicated else world, dev, q_lo)
    ix.close()
    if parted:
        t = torch.tensor([fp["hits"], fp["checksum"]] + fp["status_hist"] + [gathers], dtype=torch.int64, device=dev)
        dist.all_reduce(t)   # int64 sums wrap: the checksum is defined modulo 2^64
        t = [int(x) for x in t.cpu()]
        fp = {"hits": t[0], "checksum": t[1], "status_hist": t[2:6]}
        gathers = t[6]
        hits = fp["hits"]
    if rank == 0:
        try:
            gather_peak = kb.gather_probe(16 << 30, 1 << 29, sptr)
        except kb.KmerB200Error:
            gather_peak = None

    # ---- end to end through the host C ABI (pinned host buffers in, pinned host result out)
    e2e = None
    if not args.no_e2e:
        h_text = text.cpu().pin_memory()
        h_q = q.cpu().pin_memory()
        h_off = q_off.cpu().pin_memory()
        eb, es = [], []
        d2h = 0
        host_path = None
        for it in range(min(args.warmup, 1) + args.steps):
            barrier()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record(stream)
            ix = make_index(False, host_text=h_text.numpy())
            finish_build(ix)
            ev[1].record(stream)
            text_h2d = ix.build_transfer() or n_local   # what the text put on the link (large texts are partly packed on the host)
            if routed:
                res = sharded.search_routed_host(ix, h_q, h_off, -(-Q // world), m_hi, world, rank, dist, dev)
            elif world == 1 or replicated:
                res = sharded.search_host(ix, h_q.numpy(), h_off.numpy().view(np.uint64), 1, dev)
            else:
                res = sharded.search_host(ix, h_q, h_off, world, dev)
            ev[2].record(stream)
            torch.cuda.synchronize()
            d2h = (Ql + 1) * 8 + Ql + 4 * int(res.positions.size)
            if not routed and (world == 1 or replicated):
                # the plain C-ABI host call: the library reports what it actually put on the link (16-bit lengths
                # instead of offsets, packed ranks for pageable input)
                abi_h2d, abi_d2h = ix.last_search_transfer()
                host_path = ix.last_search_host_path()
            res.free()
            ix.close()
            if it >= min(args.warmup, 1):
                eb.append(ev[0].elapsed_time(ev[1]))
                es.append(ev[1].elapsed_time(ev[2]))
        # position-range: every rank uploads 1/world of the query batch (then NCCL all-gather); replicated: its own slice
        h2d_q = (n_sym + (Ql + 1) * 8) // (1 if parted else world)
        if not routed and (world == 1 or replicated):
            h2d_q, d2h = abi_h2d, abi_d2h
        e2e = {"build_ms": float(np.mean(eb)), "search_ms": float(np.mean(es)), "h2d": text_h2d + h2d_q, "d2h": d2h,
               "host_path": host_path}
        del h_text, h_q, h_off

    # ---- max over ranks
    def max_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    build_ms = max_over_ranks(float(np.mean(b_ms)))
    gather_ms = max_over_ranks(float(np.mean(g_ms)))
    search_ms = max_over_ranks(float(np.mean(s_ms)))
    if e2e:
        e2e["build_ms"] = max_over_ranks(e2e["build_ms"])
        e2e["search_ms"] = max_over_ranks(e2e["search_ms"])
        if world > 1:   # bytes per step over all ranks
            t = torch.tensor([e2e["h2d"], e2e["d2h"] if (rank == 0 or parted) else 0], dtype=torch.float64, device=dev)
            dist.all_reduce(t)
            e2e["h2d"], e2e["d2h"] = int(t[0].item()), int(t[1].item())

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except (OSError, ValueError):
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        # dominant kernel = the largest share of device time in the step
        name, st = max(stats_acc.items(), key=lambda kv: kv[1]["device_ms"])
        launches = max(st["launches"], 1)
        achieved = st["algorithmic_bytes"] / (st["device_ms"] * 1e-3) / 1e9 if st["device_ms"] > 0 else 0.0
        kernels = {k: {"launches_per_step": v["launches"] / args.steps, "ms_per_step": v["device_ms"] / args.steps,
                       "algorithmic_gbs": (v["algorithmic_bytes"] / (v["device_ms"] * 1e-3) / 1e9) if v["device_ms"] > 0 and
                       v["algorithmic_bytes"] > 0 else None}
                   for k, v in stats_acc.items() if v["launches"]}
        for v in kernels.values():
            v["frac_of_hbm_peak"] = v["algorithmic_gbs"] / peak if v["algorithmic_gbs"] else None
        sharding = "none"
        if routed:
            sharding = (f"partitioned index x{world}: every GPU keeps one key-range part of the hashes (+ the packed text and a "
                        f"presence bitmap), holds 1/{world} of the batch, routes each query to the owner of its first k-mer and "
                        f"gets the results back (three NCCL all-to-alls inside search_ms)")
        elif peer:
            sharding = (f"peer positions x{world}: every GPU sorts one key-range part of the hashes; the directory is "
                        f"all-gathered (one byte per bucket) and whole on every GPU, the position array stays in the parts, "
                        f"mapped into every rank over NVLink (CUDA IPC); each GPU answers 1/{world} of the batch")
        elif replicated:
            sharding = (f"replicated index x{world}: every GPU sorts one key-range part of the hashes, parts all-gathered "
                        f"over NCCL (inside build_ms), each GPU answers 1/{world} of the batch")
        elif world > 1:
            sharding = f"position range x{world}, halo {shard.halo}, every GPU searches the whole batch, merge on rank 0"
        line = {
            "metric": "search_queries_per_s", "value": Q / (search_ms * 1e-3), "unit": "queries/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": build_ms + search_ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": wl["name"] + (f" (scaled x{args.scale})" if args.scale != 1.0 else "")
                                   + (f" (text overridden to {args.text_symbols} symbols)" if args.text_symbols else ""),
                       "text_symbols": n, "queries": Q, "query_len": [m_lo, m_hi], "sigma": sigma, "ks": ks,
                       "sharding": sharding,
                       "mode": "reference_exact", "count_only": bool(args.count_only),
                       "l2": "inputs larger than L2 (text, index and batch are each >> 126 MB)" if n * 4 > 2e8 else
                             "inputs smaller than L2; step rebuilds the index so no data is reused across steps"},
            "build": {"metric": "build_gbases_per_s", "value": n / (build_ms * 1e-3) / 1e9, "unit": "Gbases/s",
                      "ms": build_ms, "nccl_ms": gather_ms if parted else 0.0,
                      **({"assemble_ms_rank0": assemble_ms} if assemble_ms else {})},
            "search": {"ms": search_ms, "hits": int(hits), "checksum": fp["checksum"], "status_hist": fp["status_hist"]},
            "roofline": {"kernel": name, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                         "avg_launch_ms": st["device_ms"] / launches,
                         "algorithmic_bytes_per_launch": st["algorithmic_bytes"] / launches},
            "kernels": kernels,
            "gpu_launches": int(sum(v["launches"] for v in stats_acc.values())),
            "clocks": clocks,
            "wall_s_timed_region": t_region,
        }
        # whole build against the HBM peak on both byte models of SURVEY.md 8d
        build_keys = ("pack_text", "radix_hist_text", "radix_hist_pairs", "column_scan", "radix_scatter_text",
                      "radix_scatter_pairs", "directory_fill")
        lsd_bytes = sum(stats_acc[k]["algorithmic_bytes"] for k in build_keys if k in stats_acc) / args.steps
        bits = 2 if sigma <= 4 else 4 if sigma <= 16 else 8
        must_move = sum((n_local - k + 1) * (bits / 8.0 + 4.0) + 4.0 * min(sigma ** k, 8 * n_local) for k in ks)
        kernel_build_ms = sum(stats_acc[k]["device_ms"] for k in build_keys if k in stats_acc) / args.steps
        if kernel_build_ms > 0:
            line["roofline_build"] = {
                "ms": kernel_build_ms, "lsd_model_bytes": lsd_bytes, "must_move_bytes": must_move,
                "lsd_model_frac": lsd_bytes / (kernel_build_ms * 1e-3) / 1e9 / peak,
                "must_move_frac": must_move / (kernel_build_ms * 1e-3) / 1e9 / peak,
                "note": "rank 0's kernels; lsd_model = bytes an LSD radix build moves with this pass structure, must_move = "
                        "text in + positions out + directory out"}
        # search roofline: sectors gathered per second against the measured random-gather ceiling
        s_ms = stats_acc.get("search_count", {"device_ms": 0.0})["device_ms"] / args.steps
        if gathers and gather_peak and s_ms > 0:
            g_rank0 = gathers / (world if parted else 1)
            rate = g_rank0 / (s_ms * 1e-3)
            line["roofline_search"] = {"kernel": "search_count", "bound": "hbm", "achieved": rate * 32 / 1e9,
                                       "peak": gather_peak * 32 / 1e9, "unit": "GB/s", "frac": rate / gather_peak,
                                       "frac_of_hbm_peak_32B_sectors": rate * 32 / 1e9 / peak,
                                       "traffic": None, "sectors_per_query": gathers / Q,
                                       "gather_peak_sectors_per_s": gather_peak,
                                       "peak_source": "measured here: kmer_b200_gather_probe, independent 8-byte reads from a "
                                                      "16 GiB table (random-gather ceiling; 32-byte sectors x gathers/s)",
                                       "avg_launch_ms": s_ms, "rank": 0}
            if name.startswith("search"):
                # the step is search-dominated: the dominant kernel's roofline is the gather one
                line["roofline"] = dict(line["roofline_search"])
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            key = f"{args.workload}:{name}"
            if key in traffic and args.scale == 1.0 and not args.text_symbols and world == 1:   # captured on the unsharded workload
                line["roofline"]["traffic"] = traffic[key]["dram_bytes_per_launch"]
                line["roofline"]["traffic_source"] = traffic[key]["source"]
            skey = f"{args.workload}:search_count"
            if "roofline_search" in line and skey in traffic and args.scale == 1.0 and world == 1:
                line["roofline_search"]["traffic"] = traffic[skey]["dram_bytes_per_launch"]
                line["roofline_search"]["traffic_source"] = traffic[skey]["source"]
        except (OSError, ValueError, KeyError):
            pass
        if e2e:
            line["e2e"] = {"value": Q / (e2e["search_ms"] * 1e-3), "unit": "queries/s",
                           "h2d_bytes_per_step": int(e2e["h2d"]), "d2h_bytes_per_step": int(e2e["d2h"]),
                           "search_ms": e2e["search_ms"], "build_ms": e2e["build_ms"],
                           "build_gbases_per_s": n / (e2e["build_ms"] * 1e-3) / 1e9}
            if e2e.get("host_path"):   # which host pipeline kmer_b200_search_batch chose (rank 0's view)
                line["e2e"]["host_path"] = e2e["host_path"]
        if not args.no_cpu_baseline and world == 1:
            r = cpu_reference_sample(wl, 3, 0)
            line["cpu_baseline"] = {"value": r["search_qps"], "unit": "queries/s", "cores": r["cores"], "kind": r["kind"],
                                    "sample": r["sample"], "build_gbases_per_s": r["build_bases_per_s"] / 1e9,
                                    "build_threads": r["build_threads"], "cpu": r["cpu"],
                                    "search_qps_min_max": r["search_qps_spread"]}
        print(json.dumps(line), flush=True)
    if peer_buffers is not None:
        peer_buffers.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
