"""CPU: pin the C restatement (oracle/kmer_oracle.c) against the fixtures generated from the compiled
reference (tests/golden/make_golden.py) and, when oracle/_ref is present, against the reference live."""
import os

import numpy as np
import pytest

from conftest import GOLDEN_DIR, ROOT, assert_results_equal, golden_cases, load_golden

# the reference's answers to the batches of the two live tests below, stored by make_golden.py
LIVE_DIR = os.path.join(GOLDEN_DIR, "live")


def live_name(test, sigma, ks):
    return f"{test}_s{sigma}_k" + "_".join(map(str, ks))


def reference_answers(oracle_mod, name, sigma, ks, batches):
    """The reference's answer to every (text, q, off) of `batches` as (offsets, positions, status, digests, ub): live
    when oracle/_ref is built (ub None), else from LIVE_DIR/<name>.npz, which holds per query the hit count, the status,
    the digest of the hit list (oracle.bindings.hit_digests; positions None) and the oracle's UB flag; else a skip."""
    if oracle_mod.have_reference():
        out = []
        for text, q, off in batches:
            with oracle_mod.Reference(text, sigma, ks) as r:
                o, p, s = r.search(q, off)
            out.append((o, p, s, oracle_mod.hit_digests(o, p), None))
        return out
    path = os.path.join(LIVE_DIR, name + ".npz")
    if not os.path.exists(path):
        pytest.skip(f"neither oracle/_ref nor {os.path.relpath(path, ROOT)} (tests/golden/make_golden.py stores it)")
    g = np.load(path)
    out = []
    for j in range(len(batches)):
        o = np.zeros(g[f"counts{j}"].size + 1, dtype=np.uint64)
        np.cumsum(g[f"counts{j}"], out=o[1:])
        out.append((o, None, g[f"status{j}"], g[f"digests{j}"], g[f"ub{j}"].astype(bool)))
    return out


def compare_with_reference(oracle_mod, got, ub, want, label):
    """Exact on the queries the oracle does not flag UB; returns per query whether the two answers are the same."""
    w_off, w_pos, w_st, w_dig, w_ub = want
    if w_ub is not None:
        assert np.array_equal(ub, w_ub), f"{label}: UB flags differ from the stored ones"
    if w_pos is not None:
        assert_results_equal(got, (w_off, w_pos, w_st), skip=ub, label=label)
    same = (np.diff(got[0]) == np.diff(w_off)) & (got[2] == w_st) & (oracle_mod.hit_digests(got[0], got[1]) == w_dig)
    bad = np.nonzero(~same & ~ub)[0]
    assert bad.size == 0, f"{label}: queries {bad[:8].tolist()} differ from the reference"
    return same


@pytest.mark.parametrize("name", golden_cases())
def test_oracle_matches_golden(oracle_mod, name):
    g = load_golden(name)
    with oracle_mod.Oracle(g["text"], int(g["sigma"]), g["ks"].tolist()) as o:
        got = o.search(g["q"], g["q_off"])
        # the UB mask is a property of the algorithm, so the restatement must reproduce it too
        assert np.array_equal(o.last_ub, g["ub"].astype(bool))
        assert_results_equal(got, (g["r_off"], g["r_pos"], g["r_status"]), skip=g["ub"].astype(bool), label=name)
        flat, o_ = g["scheme_flat"], 0
        for m, ln, multi in zip(g["scheme_m"], g["scheme_len"], g["scheme_multi"]):
            ks, use_multi = o.scheme(int(m))
            assert ks == flat[o_:o_ + ln].tolist() and use_multi == bool(multi), (name, int(m))
            o_ += int(ln)


def test_ub_queries_only_differ_by_reference_out_of_range():
    """On the UB-flagged queries the compiled reference either agrees with the 'not equal' evaluation
    or dies with std::out_of_range (status 2) -- never a silent different answer in the fixtures."""
    n_diff = 0
    for name in golden_cases():
        g = load_golden(name)
        n_diff += int((g["r_status"] > 1).sum())
        assert np.all(g["ub"][g["r_status"] > 1] == 1), name
    assert n_diff >= 1  # the fixtures do contain such a case (low_dna4_k5)


def test_fast_pow_and_choose_best_k(oracle_mod):
    s = load_golden("scalars")
    for bi, b in enumerate(s["bases"]):
        for ei, e in enumerate(s["exps"]):
            assert oracle_mod.Oracle.fast_pow(int(b), int(e)) == int(s["fast_pow"][bi, ei]), (b, e)
    o_ = 0
    for ln, want in zip(s["cbk_intervals"], s["cbk_out"]):
        iv = s["cbk_flat"][o_:o_ + ln]
        o_ += int(ln)
        assert oracle_mod.Oracle.choose_best_k(iv, 4) == want.tolist()


def test_truth_scan_small(oracle_mod):
    text = np.array([0, 1, 0, 1, 0, 2, 0, 1], dtype=np.uint8)
    q = np.array([0, 1, 0, 1, 0, 3], dtype=np.uint8)
    off = np.array([0, 2, 5, 6], dtype=np.uint64)
    o, p, _ = oracle_mod.Oracle.truth(text, q, off)
    assert o.tolist() == [0, 3, 5, 5] and p.tolist() == [0, 2, 6, 0, 2]


LIVE_CASES = [(4, [6], 40), (4, [5, 7, 9, 11, 13], 60), (15, [5, 6, 7], 12), (27, [3], 9), (5, [4], 14)]


def live_batch(sigma, ks, mmax):
    from kmer_index_b200 import synth
    text = synth.low_entropy_text(11, sigma=sigma)
    q, off = synth.stress_queries(text, 1500, 1, mmax, sigma, 4242 + ks[0], low_sigma=2)
    return text, q, off


@pytest.mark.parametrize("sigma,ks,mmax", LIVE_CASES)
def test_oracle_matches_live_reference(oracle_mod, sigma, ks, mmax):
    text, q, off = live_batch(sigma, ks, mmax)
    want, = reference_answers(oracle_mod, live_name("live", sigma, ks), sigma, ks, [(text, q, off)])
    with oracle_mod.Oracle(text, sigma, ks) as o:
        got = o.search(q, off)
        compare_with_reference(oracle_mod, got, np.asarray(o.last_ub).astype(bool), want, f"sigma={sigma} ks={ks}")


@pytest.mark.parametrize("name", golden_cases())
def test_restricted_oracle_equals_full_on_golden(oracle_mod, name):
    """ko_create_restricted (the index holding only the buckets a batch can ask for -- what makes the 3 Gbp
    config-5 check affordable on a CPU) answers every golden batch exactly like the full restatement and like
    the fixture generated from the compiled reference; no lookup may reach a bucket it does not hold."""
    g = load_golden(name)
    sigma, ks = int(g["sigma"]), g["ks"].tolist()
    if any(float(sigma) ** k > 2.0 ** 36 for k in ks):
        with pytest.raises(ValueError):
            oracle_mod.Oracle(g["text"], sigma, ks, restrict_to=(g["q"], g["q_off"]))
        return
    before = oracle_mod.Oracle.restricted_misses()
    with oracle_mod.Oracle(g["text"], sigma, ks, restrict_to=(g["q"], g["q_off"]), n_threads=3) as o:
        got = o.search(g["q"], g["q_off"])
        assert np.array_equal(o.last_ub, g["ub"].astype(bool))
    assert oracle_mod.Oracle.restricted_misses() == before
    assert_results_equal(got, (g["r_off"], g["r_pos"], g["r_status"]), skip=g["ub"].astype(bool), label=name)


def test_restricted_oracle_equals_full_on_random_text(oracle_mod):
    from kmer_index_b200 import synth
    text = synth.random_text(3_000_000, 4, 77)
    q, off = synth.stress_queries(text, 4000, 10, 64, 4, 78)
    with oracle_mod.Oracle(text, 4, [16]) as full, oracle_mod.Oracle(text, 4, [16], restrict_to=(q, off)) as part:
        want = full.search(q, off)
        got = part.search(q, off)
        assert part.element(0)[0].size < full.element(0)[0].size // 50
    assert want[1].size > 1000
    assert_results_equal(got, want, label="restricted vs full")
    assert oracle_mod.Oracle.restricted_misses() == 0


REFERENCE_SHAPES = [(4, [10]), (4, [12]), (4, [5, 7, 9, 11, 13]), (15, [8]), (27, [5]), (4, [16]), (4, [3]), (4, [5]), (4, [6]),
                    (4, [14]), (4, [9, 10]), (4, [10, 11, 12]), (15, [5]), (15, [10]), (15, [5, 6, 7]), (15, [10, 11, 12]),
                    (5, [4]), (27, [3]), (27, [9, 10]), (27, [12]), (5, [18]), (4, [20]), (15, [16])]


def _sweep_texts(sigma, seed):
    from kmer_index_b200 import synth
    yield "low entropy", synth.low_entropy_text(seed, sigma=sigma)
    yield "random", synth.random_text(20000, sigma, seed)
    yield "random over two ranks", synth.random_text(9000, min(sigma, 2), seed + 1)
    rng = np.random.default_rng(seed)
    p = int(rng.integers(1, 9))
    t = np.tile(rng.integers(0, sigma, p, dtype=np.uint8), 5000 // p + 1)[:5000]
    t[rng.integers(0, 5000, 20)] = rng.integers(0, sigma, 20, dtype=np.uint8)
    yield f"period {p} with 20 point changes", t


def sweep_batches(sigma, ks):
    from kmer_index_b200 import synth
    for kind, text in _sweep_texts(sigma, 100 + ks[0]):
        q, off = synth.stress_queries(text, 300, 1, min(6 * max(ks) + 7, 130), sigma, 7000 + ks[0], low_sigma=2)
        yield kind, text, q, off


@pytest.mark.parametrize("sigma,ks", REFERENCE_SHAPES)
def test_oracle_matches_live_reference_sweep(oracle_mod, sigma, ks):
    """Every shape the compiled reference was instantiated for (oracle/ref_driver.cpp), four kinds of text (long buckets,
    periodic stretches: every multi-part plan returns non-empty results), queries of 1 .. 6 k + 7 symbols. Queries on
    which the reference dereferences an end iterator (kmer_index.hpp:317, :546; the oracle flags them) are skipped in the
    exact comparison -- there the reference's answer depends on stale heap bytes -- but must still agree with the
    oracle's defined value almost always."""
    batches = list(sweep_batches(sigma, ks))
    wants = reference_answers(oracle_mod, live_name("sweep", sigma, ks), sigma, ks, [b[1:] for b in batches])
    flagged = agree = 0
    for (kind, text, q, off), want in zip(batches, wants):
        with oracle_mod.Oracle(text, sigma, ks) as o:
            got = o.search(q, off)
            ub = np.asarray(o.last_ub).astype(bool)
        same = compare_with_reference(oracle_mod, got, ub, want, f"sigma={sigma} ks={ks} {kind}")
        flagged += int(ub.sum())
        agree += int(same[ub].sum())
    assert agree >= 0.95 * flagged, (agree, flagged)
