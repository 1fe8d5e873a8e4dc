"""Generate tests/golden/*.npz from the COMPILED REFERENCE (oracle/_ref/libkmer_ref.so).

Needs a checkout of the reference (Clemapfel/kmer_index) to build oracle/_ref first:

    make -C oracle REF=/path/to/kmer_index && python tests/golden/make_golden.py

Each fixture stores the inputs explicitly (text ranks, query ranks + offsets) next to the
reference's outputs (per-query sorted positions in CSR form + status), so the fixtures do not
depend on the generator. `ub` marks queries on which the reference dereferences an end()
iterator (kmer_index.hpp:317,546): its answer there depends on stale heap bytes, so those
queries pin nothing and parity tests skip them.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

sys.path.insert(0, os.path.join(ROOT, "tests"))
import test_oracle_golden as live  # noqa: E402
from kmer_index_b200 import synth  # noqa: E402
from oracle.bindings import Oracle, Reference, hit_digests  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def case(name, text, sigma, ks, q, off):
    ref = Reference(text, sigma, ks)
    r_off, r_pos, r_status = ref.search(q, off)
    ora = Oracle(text, sigma, ks)
    ora.search(q, off)
    ub = ora.last_ub.copy()
    scheme_m = np.arange(1, 130, dtype=np.uint32)
    rows = [ref.scheme(int(m)) for m in scheme_m]
    scheme_len = np.array([len(r[0]) for r in rows], dtype=np.uint32)
    scheme_flat = np.array([k for r in rows for k in r[0]], dtype=np.uint8)
    scheme_multi = np.array([r[1] for r in rows], dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), text=text, sigma=np.uint32(sigma),
                        ks=np.asarray(ks, dtype=np.uint32), q=q, q_off=off, r_off=r_off, r_pos=r_pos,
                        r_status=r_status, ub=ub, scheme_m=scheme_m, scheme_len=scheme_len,
                        scheme_flat=scheme_flat, scheme_multi=scheme_multi)
    print(f"{name}: n={text.size} Q={off.size - 1} hits={r_pos.size} throws={(r_status == 1).sum()} "
          f"other={(r_status > 1).sum()} ub={ub.sum()}")


def live_case(name, sigma, ks, batches):
    """live/<name>.npz: the reference's answers to the batches of tests/test_oracle_golden.py's live tests, per query the
    hit count, the status, the digest of the hit list (hit_digests: the lists themselves would not fit) and the UB flag."""
    arrays = {}
    for j, (text, q, off) in enumerate(batches):
        r_off, r_pos, r_status = Reference(text, sigma, ks).search(q, off)
        ora = Oracle(text, sigma, ks)
        ora.search(q, off)
        arrays.update({f"counts{j}": np.diff(r_off).astype(np.uint32), f"digests{j}": hit_digests(r_off, r_pos),
                       f"status{j}": r_status, f"ub{j}": ora.last_ub.astype(np.uint8)})
    os.makedirs(live.LIVE_DIR, exist_ok=True)
    np.savez_compressed(os.path.join(live.LIVE_DIR, name + ".npz"), **arrays)
    print(f"live/{name}: {len(batches)} batch(es)")


def main():
    for sigma, ks, mmax in live.LIVE_CASES:
        live_case(live.live_name("live", sigma, ks), sigma, ks, [live.live_batch(sigma, ks, mmax)])
    for sigma, ks in live.REFERENCE_SHAPES:
        live_case(live.live_name("sweep", sigma, ks), sigma, ks, [b[1:] for b in live.sweep_batches(sigma, ks)])
    low = synth.low_entropy_text(7)
    for ks, mmax, Q in [([3], 20, 600), ([5], 32, 800), ([6], 40, 800), ([14], 45, 800), ([16], 70, 800),
                        ([12], 100, 800), ([5, 7, 9, 11, 13], 60, 1200), ([9, 10], 60, 800),
                        ([10, 11, 12], 40, 600)]:
        q, off = synth.stress_queries(low, Q, 1, mmax, 4, 99 + ks[0], low_sigma=2)
        case("low_dna4_k" + "_".join(map(str, ks)), low, 4, ks, q, off)
    # BASELINE config shapes, scaled to fixture size
    t = synth.random_text(20000, 4, 201)
    q, off = synth.stress_queries(t, 500, 10, 10, 4, 1235)
    case("c1_dna4_k10", t, 4, [10], q, off)
    t = synth.random_text(30000, 4, 202)
    q, off = synth.stress_queries(t, 800, 13, 100, 4, 1236)
    case("c2_dna4_k12", t, 4, [12], q, off)
    t = synth.random_text(30000, 4, 203)
    q, off = synth.stress_queries(t, 1200, 4, 40, 4, 1237)
    case("c3_dna4_multi", t, 4, [5, 7, 9, 11, 13], q, off)
    t = synth.random_text(20000, 15, 204)
    q, off = synth.stress_queries(t, 500, 3, 20, 15, 1238)
    case("c4_dna15_k8", t, 15, [8], q, off)
    t = synth.random_text(20000, 27, 205)
    q, off = synth.stress_queries(t, 500, 1, 14, 27, 1239)
    case("c4_aa27_k5", t, 27, [5], q, off)
    t = synth.random_text(30000, 4, 206)
    q, off = synth.stress_queries(t, 800, 16, 64, 4, 1240)
    case("c5_dna4_k16", t, 4, [16], q, off)
    # test_main.cpp:76-78 shapes (dna15, single k and k,k+1,k+2; query lengths k-5 .. 2k-1)
    t = synth.random_text(20000, 15, 207)
    q, off = synth.stress_queries(t, 400, 1, 19, 15, 1241)
    case("tm_dna15_k10", t, 15, [10], q, off)
    case("tm_dna15_k10_11_12", t, 15, [10, 11, 12], q, off)
    q, off = synth.stress_queries(t, 400, 1, 9, 15, 1242)
    case("tm_dna15_k5_6_7", t, 15, [5, 6, 7], q, off)
    # k-mers wider than one 64-bit packed window (aa27 k >= 9, dna5 k >= 17) and hashes wider than 32 bits
    low27 = np.where(low == 0, 3, 26).astype(np.uint8)
    q, off = synth.stress_queries(low27, 500, 5, 40, 27, 1243, low_sigma=2)
    q = np.where(q == 0, 3, np.where(q == 1, 26, q)).astype(np.uint8)
    case("wide_low_aa27_k12", low27, 27, [12], q, off)
    case("wide_low_aa27_k9_10", low27, 27, [9, 10], q, off)
    t = synth.random_text(20000, 27, 208)
    q, off = synth.stress_queries(t, 500, 8, 40, 27, 1244)
    case("wide_aa27_k12", t, 27, [12], q, off)
    case("wide_aa27_k9_10", t, 27, [9, 10], q, off)
    t = synth.random_text(20000, 5, 209)
    q, off = synth.stress_queries(t, 500, 10, 60, 5, 1245)
    case("wide_dna5_k18", t, 5, [18], q, off)
    low5 = np.where(low == 0, 2, 4).astype(np.uint8)
    q, off = synth.stress_queries(low5, 500, 10, 60, 5, 1246, low_sigma=2)
    q = np.where(q == 0, 2, np.where(q == 1, 4, q)).astype(np.uint8)
    case("wide_low_dna5_k18", low5, 5, [18], q, off)
    q, off = synth.stress_queries(low, 500, 9, 70, 4, 1247, low_sigma=2)
    case("wide_low_dna4_k20", low, 4, [20], q, off)
    t = synth.random_text(20000, 15, 210)
    q, off = synth.stress_queries(t, 400, 12, 40, 15, 1248)
    case("wide_dna15_k16", t, 15, [16], q, off)
    # fast_pow (fast_pow.hpp:46-93) and choose_best_k (choose_best_k.hpp:12-60)
    bases = np.array([0, 1, 2, 3, 4, 5, 15, 27, 255, 65537, 2 ** 32 + 1], dtype=np.uint64)
    exps = np.arange(0, 80, dtype=np.uint8)
    fp = np.array([[Reference.fast_pow(int(b), int(e)) for e in exps] for b in bases], dtype=np.uint64)
    intervals = [list(range(20, 41)), list(range(10, 100)), [30, 60, 90], list(range(4, 41)), [16, 32, 48, 64]]
    cbk = [Reference.choose_best_k(iv, 4) for iv in intervals]
    np.savez_compressed(os.path.join(OUT, "scalars.npz"), bases=bases, exps=exps, fast_pow=fp,
                        cbk_intervals=np.array([len(iv) for iv in intervals], dtype=np.uint32),
                        cbk_flat=np.array([x for iv in intervals for x in iv], dtype=np.uint64),
                        cbk_out=np.array(cbk, dtype=np.uint64))
    print("scalars: fast_pow", fp.shape, "choose_best_k", cbk)


if __name__ == "__main__":
    main()
