"""Every compiled variant of the search and build kernels against the independent references. The host picks a variant
from the shape of the input (lanes per query G, the lean count kernel and its CTA count, the sorter and its digit width);
each case here forces one through the library's environment overrides, proves with torch.profiler that the intended
kernel instantiation ran, and compares the result bit for bit with the C restatement oracle (REFERENCE_EXACT), the plain
scan (CORRECT), the oracle's CSR (build) or the every-window scan (approximate search, hit strategies, collections)."""
import contextlib
import os
import re
import subprocess
import sys
from collections import Counter

import numpy as np
import pytest

from approx_hits_truth import hits_truth
from collection_truth import hits_truth as collection_hits_truth
from collection_truth import random_starts
from conftest import assert_results_equal
from test_gpu_approx import concat, mixed_batch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GROUPS = [1, 2, 4, 8, 32]
HEAVY_CANDIDATES = 2048          # longer candidate lists go to the warp-per-query launch when G < 32


@pytest.fixture(scope="module")
def kb():
    import kmer_index_b200
    return kmer_index_b200


# ---- the staging rule of search_geometry (csrc/capi.cu) restated: which G a batch keeps

def symbol_bits(sigma):
    return 2 if sigma <= 4 else 4 if sigma <= 16 else 8


def chunks_per_lane(group, bits):
    """cpl of pack_query_group (csrc/query_pack.cuh): a 64-bit word holds 8 / bits chunks of 8 symbols"""
    lpw = 8 // bits
    return lpw // group if lpw > group else 1


def round_symbols(group, bits):
    """symbols packed per round by a group of G lanes (8 * G * cpl)"""
    return 8 * group * chunks_per_lane(group, bits)


def q_words(group, bits, max_len):
    """search_q_words (csrc/search_kernels.cu): shared-memory words staged per query"""
    lpw = 8 // bits
    cpl = chunks_per_lane(group, bits)
    rounds = -(-max(max_len, 1) // round_symbols(group, bits))
    return rounds * (group * cpl // lpw) + 2


def staged_group(group, bits, max_len):
    """G after the 48 KB loop of search_geometry: raised while the 256 / G packed queries of a CTA overflow 48 KB"""
    while group < 32 and q_words(group, bits, max_len) * 8 * (256 // group) > 48 * 1024:
        group = 32 if group == 8 else group * 2
    return group


def lane_limit(group, bits, cap):
    """the longest batch max_len (at most cap) that keeps G"""
    lo, hi = 1, cap
    while lo < hi:
        mid = (lo + hi + 1) // 2
        if staged_group(group, bits, mid) == group:
            lo = mid
        else:
            hi = mid - 1
    return lo


# ---- which kernels ran

@contextlib.contextmanager
def kernels_launched():
    """Counter of the names of the CUDA kernels launched inside the block (torch.profiler, CUDA activities)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    names = Counter()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        yield names
        torch.cuda.synchronize()
    names.update(e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)


def template_args(names, kernel):
    """the template argument lists of the launched instantiations of `kernel` (one entry per distinct instantiation)"""
    pat = re.compile(rf"\b{kernel}<([^<>]*)>")
    return [tuple(a.strip() for a in m.group(1).split(",")) for name in names for m in [pat.search(name)] if m]


def launches(names, kernel):
    return sum(c for name, c in names.items() if re.search(rf"\b{kernel}\b", name))


LANES_ARG = {"search_kernel": 1, "search_listed_write_kernel": 0, "search_approx_kernel": 1, "search_approx_hits_kernel": 1,
             "search_approx_coll_kernel": 1, "approx_distances_kernel": 0}


def lanes(names, kernel):
    """the lanes-per-query argument of every launched instantiation of `kernel`"""
    return {int(a[LANES_ARG[kernel]]) for a in template_args(names, kernel)}


def kernel_summary(names):
    return sorted(n.split("(")[0] for n in names)


# ---- inputs

ZERO_RUN = (20_000, 26_000)      # a constant run: the bucket of 0^k holds ~6000 candidates
ONE_RUN = (30_000, 31_500)       # and one under 2048: ~1500 consecutive hits answered by the G-lane launch
PERIODIC_AT, PERIODIC_LEN = 40_000, 3000


def variant_text(sigma, ks, n=200_000, seed=5):
    """random text with two constant runs and, per k, a stretch of period k (the parts of a query taken from it are equal, so
    the reference's defective plan for P > 2 parts with a rest finds matches)"""
    from kmer_index_b200 import synth
    text = synth.random_text(n, sigma, seed + sigma)
    text[ZERO_RUN[0]:ZERO_RUN[1]] = 0
    text[ONE_RUN[0]:ONE_RUN[1]] = 1
    for j, k in enumerate(ks):
        a = PERIODIC_AT + j * 5000
        text[a:a + PERIODIC_LEN] = np.resize(text[a - k:a], PERIODIC_LEN)
    return text


def query_batch(text, sigma, ks, lens, seed, extra=600):
    """per length: a text window, a window of each constant run, one of each periodic stretch, the window ending at n and a
    random query; then `extra` stress queries of 1..max(lens)"""
    from kmer_index_b200 import synth
    rng = np.random.default_rng(seed)
    n = text.size
    qs = []
    for m in lens:
        s = int(rng.integers(0, n - m + 1))
        qs += [text[s:s + m], np.zeros(m, np.uint8), np.ones(m, np.uint8), text[n - m:], synth.random_text(m, sigma, seed + m)]
        for j in range(len(ks)):
            a = PERIODIC_AT + j * 5000 + int(rng.integers(0, 50))
            if m <= PERIODIC_LEN - 50:
                qs.append(text[a:a + m])
    off = np.zeros(len(qs) + 1, np.uint64)
    np.cumsum([x.size for x in qs], out=off[1:])
    q2, o2 = synth.stress_queries(text, extra, 1, max(lens), sigma, seed + 1)
    return concat((np.concatenate(qs), off), (q2, o2))


def on_device(q, off):
    import torch
    dev = torch.device("cuda", 0)
    d_q = torch.from_numpy(q if q.size else np.zeros(1, np.uint8)).to(dev)
    d_off = torch.from_numpy(off.view(np.int64)).to(dev)
    torch.cuda.synchronize()
    return d_q, d_off


def fetch(r):
    """(offsets, positions, status, distances, best_distances) of a device result as host arrays; frees it"""
    import torch
    dev = torch.device("cuda", 0)
    torch.cuda.synchronize()

    def host(v):
        return torch.as_tensor(v, device=dev).cpu().numpy()
    o = host(r.offsets()).astype(np.uint64)
    st = host(r.status()) if r.n_queries else np.zeros(0, np.uint8)
    p = host(r.positions()).view(np.uint32) if r.n_positions and r.positions_ptr else np.zeros(0, np.uint32)
    d = r.distances()
    d = None if d is None else host(d) if r.n_positions else np.zeros(0, np.uint8)
    b = r.best_distances()
    b = None if b is None else host(b)
    r.free()
    return o, p, st, d, b


# ---- exact search at every G

EXACT_SHAPES = {"dna4_k12": (4, [12]), "dna4_k20": (4, [20]), "dna4_multi": (4, [5, 9, 13]), "dna15_k8": (15, [8]),
                "aa27_k5": (27, [5]), "aa27_k12": (27, [12])}


def exact_lengths(ks, group, bits):
    """1..k, multiples and non-multiples of each k, two to three packing rounds of G and the longest length G keeps
    (up to 1024)"""
    R = round_symbols(group, bits)
    lim = lane_limit(group, bits, 1024)
    lens = set(range(1, max(ks) + 1)) | {lim, 2 * R - 1, 2 * R, 2 * R + 1, 3 * R - 1, 3 * R}
    for k in ks:
        lens |= {2 * k, 3 * k, 4 * k, 2 * k + 1, 3 * k + 2, 4 * k - 1, 5 * k + 3}
    return sorted(m for m in lens if m <= lim)


@pytest.fixture(scope="module")
def exact_refs(oracle_mod):
    """per shape: the text and its oracle, built once"""
    made = {}

    def get(shape):
        if shape not in made:
            sigma, ks = EXACT_SHAPES[shape]
            text = variant_text(sigma, ks)
            made[shape] = (text, oracle_mod.Oracle(text, sigma, ks))
        return made[shape]
    yield get
    for _, o in made.values():
        o.close()


def check_exact(kb, ix, text, q, off, want, truth, label):
    """both modes; host (twice: the second batch finds the auxiliary elements the first one built), device and
    count-only forms"""
    d_q, d_off = on_device(q, off)
    Q, max_len = off.size - 1, int(np.diff(off).max())
    for mode, ref in ((kb.MODE_REFERENCE_EXACT, want), (kb.MODE_CORRECT, truth)):
        lab = f"{label} mode={mode}"
        for attempt in range(2):
            assert_results_equal(ix.search_batch(q, off, mode=mode).as_tuple(), ref, label=f"{lab} host/{attempt}")
        o, p, st, _, _ = fetch(ix.search_batch_device(d_q.data_ptr(), d_off.data_ptr(), Q, max_len, mode))
        assert_results_equal((o, p, st), ref, label=f"{lab} device")
        o, p, st, _, _ = fetch(ix.count_batch_device(d_q.data_ptr(), d_off.data_ptr(), Q, max_len, mode))
        assert np.array_equal(o, ref[0]) and p.size == 0, f"{lab} count-only"
        if mode == kb.MODE_REFERENCE_EXACT:
            assert np.array_equal(st, ref[2]), f"{lab} count-only status"


EXACT_CASES = [pytest.param(s, False, id=s) for s in EXACT_SHAPES] + [pytest.param("dna4_k12", True, id="dna4_k12-no_lean")]


@pytest.mark.parametrize("group", GROUPS)
@pytest.mark.parametrize("shape,no_lean", EXACT_CASES)
def test_exact_search_at_every_group(kb, exact_refs, monkeypatch, shape, no_lean, group):
    """KMER_B200_GROUP = G: every count / write pass of the general kernel runs with G lanes per query; the constant run
    sends long candidate lists to the warp launch. dna4 k = 12 adds a batch of at most 128 symbols, which the lean count
    kernel answers -- or, with KMER_B200_NO_LEAN=1, the general count pass at G."""
    sigma, ks = EXACT_SHAPES[shape]
    bits = symbol_bits(sigma)
    text, o = exact_refs(shape)
    batches = [query_batch(text, sigma, ks, exact_lengths(ks, group, bits), 100 + group)]
    if shape == "dna4_k12":
        batches.append(query_batch(text, sigma, ks, [m for m in exact_lengths(ks, 2, bits) if m <= 128], 200 + group))
    monkeypatch.setenv("KMER_B200_GROUP", str(group))
    if no_lean:
        monkeypatch.setenv("KMER_B200_NO_LEAN", "1")
    refs = []
    for q, off in batches:
        assert staged_group(group, bits, int(np.diff(off).max())) == group
        want = o.search(q, off)
        assert int(np.diff(want[0]).max()) > HEAVY_CANDIDATES and want[1].size > 0
        refs.append((q, off, want, o.truth(text, q, off)))
    # dna4 k = 12 with the dense directory the lean kernel needs (the automatic choice is a sparse one for this text)
    with kernels_launched() as names, kb.KmerIndex(text, sigma, ks, directory_bits=24 if shape == "dna4_k12" else 0) as ix:
        if shape == "dna4_k12":
            assert ix.element_info(0).directory_shift == 0
        for i, (q, off, want, truth) in enumerate(refs):
            check_exact(kb, ix, text, q, off, want, truth, f"{shape} G={group} batch {i}")
    single = "true" if len(ks) == 1 else "false"
    general = template_args(names, "search_kernel")
    assert lanes(names, "search_kernel") == {group} and lanes(names, "search_listed_write_kernel") == {group}, kernel_summary(names)
    assert ("0", str(group), single) in general, kernel_summary(names)
    assert {a[2] for a in general} == {single}
    lean = launches(names, "search_count_lean_kernel") > 0
    assert lean == (shape == "dna4_k12" and not no_lean), kernel_summary(names)
    # the warp launch follows every pass of a G < 32 kernel, and the lean count pass at any G (its listed queries)
    heavy = set(template_args(names, "search_heavy_kernel"))
    if group < 32:
        assert ("0", single) in heavy and ("1", single) in heavy, kernel_summary(names)
    else:
        assert heavy == ({("0", single)} if lean else set()), kernel_summary(names)


# ---- approximate search, hit strategies and collections at every G

APPROX_SHAPES = {"dna4_k12": (4, [12]), "dna15_k8": (15, [8]), "aa27_k5": (27, [5])}
BUDGETS = [0, 1, 3, 8]
STRATEGIES = [("all", 0), ("all_best", 0), ("single_best", 0), ("strata", 1)]


def approx_batch(text, sigma, ks, group, bits, e, seed):
    """mixed_batch of 1..m_hi symbols, then windows of two to three packing rounds of G (and of the longest length G
    keeps) with a few substitutions, and constant queries (candidate lists beyond 2048)"""
    R = round_symbols(group, bits)
    lim = lane_limit(group, bits, 1024)
    m_hi = min(lim, max(3 * R + 1, 150))
    q1, o1, _, _, _ = mixed_batch(text, sigma, e, seed, Q=150, m_hi=m_hi)
    rng = np.random.default_rng(seed)
    qs = []
    for i, m in enumerate(sorted(m for m in {2 * R - 1, 2 * R, 2 * R + 1, 3 * R, lim, ks[0], 2 * ks[0] + 1} if m <= lim)):
        for j in range(3):
            s = int(rng.integers(0, text.size - m + 1))
            w = text[s:s + m].copy()
            for c in rng.choice(m, size=min(m, (i + j) % (e + 2)), replace=False):
                w[c] = (int(w[c]) + 1) % sigma
            qs.append(w)
        qs.append(np.zeros(m, np.uint8))
    off = np.zeros(len(qs) + 1, np.uint64)
    np.cumsum([x.size for x in qs], out=off[1:])
    return concat((q1, o1), (np.concatenate(qs), off))


def check_approx(ix, q, off, e, truth, label):
    """every strategy with distances: host, device and count-only forms"""
    d_q, d_off = on_device(q, off)
    Q, max_len = off.size - 1, int(np.diff(off).max())
    for h, s in STRATEGIES:
        w_off, w_pos, w_st, w_dist, w_best = truth[(h, s)]
        lab = f"{label} e={e} {h}/{s}"
        got = ix.search_approx(q, off, e, hits=h, strata=s, distances=True)
        assert_results_equal(got.as_tuple(), (w_off, w_pos, w_st), label=f"{lab} host")
        assert np.array_equal(got.distances, w_dist), f"{lab} host distances"
        assert (got.best_distance is None) if w_best is None else np.array_equal(got.best_distance, w_best), f"{lab} host best"
        o, p, st, d, b = fetch(ix.search_approx_batch_device(d_q.data_ptr(), d_off.data_ptr(), Q, max_len, e, hits=h, strata=s,
                                                             distances=True))
        assert_results_equal((o, p, st), (w_off, w_pos, w_st), label=f"{lab} device")
        assert np.array_equal(d, w_dist), f"{lab} device distances"
        assert (b is None) if w_best is None else np.array_equal(b, w_best), f"{lab} device best"
        o, p, st, d, b = fetch(ix.count_approx_batch_device(d_q.data_ptr(), d_off.data_ptr(), Q, max_len, e, hits=h, strata=s,
                                                            distances=True))
        assert np.array_equal(o, w_off) and np.array_equal(st, w_st) and p.size == 0 and d is None, f"{lab} count-only"
        assert (b is None) if w_best is None else np.array_equal(b, w_best), f"{lab} count-only best"


@pytest.fixture(scope="module")
def approx_texts():
    made = {}

    def get(shape):
        if shape not in made:
            sigma, ks = APPROX_SHAPES[shape]
            text = variant_text(sigma, ks, n=60_000, seed=9)
            made[shape] = (text, random_starts(text.size, 40, np.random.default_rng(10 + sigma), short=14))
        return made[shape]
    return get


@pytest.mark.parametrize("group", GROUPS)
@pytest.mark.parametrize("collection", [False, True], ids=["plain", "collection"])
@pytest.mark.parametrize("shape", list(APPROX_SHAPES))
def test_approximate_search_at_every_group(kb, approx_texts, monkeypatch, shape, collection, group):
    """KMER_B200_GROUP = G for the approximate count / best / listed / write passes and the distance kernel; on a
    collection index (empty and short records) the record-boundary instantiations"""
    sigma, ks = APPROX_SHAPES[shape]
    bits = symbol_bits(sigma)
    text, starts = approx_texts(shape)
    cases = []
    for e in BUDGETS:
        q, off = approx_batch(text, sigma, ks, group, bits, e, 300 + 10 * group + e)
        assert staged_group(group, bits, int(np.diff(off).max())) == group
        truth = (collection_hits_truth(text, starts, q, off, e, STRATEGIES) if collection
                 else hits_truth(text, q, off, e, STRATEGIES))
        if e == 0 and not collection:
            assert int(np.diff(truth[("all", 0)][0]).max()) > HEAVY_CANDIDATES
        cases.append((e, q, off, truth))
    monkeypatch.setenv("KMER_B200_GROUP", str(group))
    with kernels_launched() as names, kb.KmerIndex(text, sigma, ks) as ix:
        if collection:
            ix.attach_records(starts)
        for e, q, off, truth in cases:
            check_approx(ix, q, off, e, truth, f"{shape} {'collection' if collection else 'plain'} G={group}")
    grid = ["search_approx_coll_kernel"] if collection else ["search_approx_kernel", "search_approx_hits_kernel"]
    for kernel in grid + ["approx_distances_kernel"]:
        assert lanes(names, kernel) == {group}, (kernel, kernel_summary(names))
    other = ["search_approx_kernel", "search_approx_hits_kernel"] if collection else ["search_approx_coll_kernel"]
    assert not any(launches(names, kernel) for kernel in other), kernel_summary(names)
    heavy = ["search_approx_heavy_coll_kernel"] if collection else ["search_approx_heavy_kernel", "search_approx_heavy_hits_kernel"]
    for kernel in heavy:
        assert (launches(names, kernel) > 0) == (group < 32), (kernel, kernel_summary(names))


# ---- the lean count kernel

LEAN_KS = [10, 12, 16]


def lean_lengths(k, m_max):
    """m < k, m = k, P parts with rests 1-4 (the throw rule of k = 16), P > 2 with a rest (the defective plan) and the
    longest length of the batch"""
    lens = set(range(1, k + 1)) | {m_max, m_max - 1}
    for p in range(1, 9):
        lens |= {p * k, *(p * k + r for r in range(1, 5)), p * k + k // 2}
    return sorted(m for m in lens if m <= m_max)


def lean_batch(text, k, m_max, seed):
    return query_batch(text, 4, [k], lean_lengths(k, m_max), seed, extra=2000)


@pytest.fixture(scope="module")
def lean_refs(oracle_mod):
    made = {}

    def get(k):
        if k not in made:
            text = variant_text(4, [k])
            made[k] = (text, oracle_mod.Oracle(text, 4, [k]))
        return made[k]
    yield get
    for _, o in made.values():
        o.close()


@pytest.mark.parametrize("no_lean", [False, True], ids=["lean", "no_lean"])
@pytest.mark.parametrize("m_max", [64, 128], ids=["W2", "W4"])
@pytest.mark.parametrize("k", LEAN_KS)
def test_lean_count_kernel(kb, lean_refs, monkeypatch, k, m_max, no_lean):
    """dna4, one k, dense directory (directory_bits = 2k; the automatic choice is a sparse one for this text): batches of
    at most 64 symbols take the W = 2 instantiation, 65-128 the W = 4 one; the general count pass (KMER_B200_NO_LEAN=1)
    and the oracle must agree with it, in both modes"""
    text, o = lean_refs(k)
    q, off = lean_batch(text, k, m_max, 400 + k + m_max)
    assert int(np.diff(off).max()) == m_max
    want = o.search(q, off)
    lens = np.diff(off).astype(np.int64)
    counts = np.diff(want[0]).astype(np.int64)
    assert counts.max() > HEAVY_CANDIDATES
    assert counts[(lens >= 3 * k) & (lens % k != 0)].sum() > 0                    # the defective plan finds matches
    if k == 16:
        assert (want[2] == kb.QUERY_THROW_INVALID_ARGUMENT).any()                # sigma^(k - rest) > 10^7: the throw rule
    truth = o.truth(text, q, off)
    if no_lean:
        monkeypatch.setenv("KMER_B200_NO_LEAN", "1")
    with kernels_launched() as names, kb.KmerIndex(text, 4, [k], directory_bits=2 * k) as ix:
        assert ix.element_info(0).directory_shift == 0
        check_exact(kb, ix, text, q, off, want, truth, f"lean k={k} m_max={m_max} no_lean={no_lean}")
    lean = template_args(names, "search_count_lean_kernel")
    if no_lean:
        assert not lean and any(a[0] == "0" for a in template_args(names, "search_kernel")), kernel_summary(names)
    else:
        assert lean == [("2", "8") if m_max <= 64 else ("4", "5")], kernel_summary(names)
        assert not any(a[0] == "0" for a in template_args(names, "search_kernel")), kernel_summary(names)


LEAN6_CASE = r"""
import sys
sys.path.insert(0, "tests")
import numpy as np
import kmer_index_b200 as kb
from oracle import bindings
from conftest import assert_results_equal
from test_gpu_variants import kernels_launched, kernel_summary, lean_batch, template_args, variant_text
for k in (10, 12, 16):
    text = variant_text(4, [k])
    q, off = lean_batch(text, k, 64, 500 + k)
    with bindings.Oracle(text, 4, [k]) as o:
        want = o.search(q, off)
    truth = bindings.Oracle.truth(text, q, off)
    with kernels_launched() as names, kb.KmerIndex(text, 4, [k], directory_bits=2 * k) as ix:
        for attempt in range(2):
            assert_results_equal(ix.search_batch(q, off).as_tuple(), want, label=f"k={k}/{attempt}")
        assert_results_equal(ix.search_batch(q, off, mode=kb.MODE_CORRECT).as_tuple(), truth, label=f"k={k} correct")
    assert template_args(names, "search_count_lean_kernel") == [("2", "6")], kernel_summary(names)
print("lean 6 CTAs ok")
"""


def test_lean_count_kernel_six_ctas_per_sm():
    """KMER_B200_LEAN_BLOCKS=6 (the 40-register instantiation) is read once per process: a process of its own"""
    env = dict(os.environ, KMER_B200_LEAN_BLOCKS="6")
    env.pop("KMER_B200_GROUP", None)
    env.pop("KMER_B200_NO_LEAN", None)
    out = subprocess.run([sys.executable, "-c", LEAN6_CASE], capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    assert "lean 6 CTAs ok" in out.stdout


# ---- the build: sorter x digit width x length

SORT_TILE, SCAN_CHUNK_TILES = 8192, 64
DIGITS = [None, 4, 5, 6, 7]
# 32-bit keys: dna4 k = 16 (byte-aligned digits), sigma 16 (4-bit symbols), sigma 5 (31 bits), aa27 k = 6 (8-bit
# symbols); 64-bit keys: sigma 2 k = 40 (k * bits = 80 > 64: two-window hash), dna15 k = 12
DIGIT_SHAPES = [(4, 16), (16, 8), (5, 13), (27, 6), (2, 40), (15, 12)]
LENGTH_SHAPES = [(4, 16), (5, 13)]
LENGTHS = [1, 2, SORT_TILE - 1, SORT_TILE, SORT_TILE + 1, SORT_TILE * SCAN_CHUNK_TILES - 1, SORT_TILE * SCAN_CHUNK_TILES,
           SORT_TILE * SCAN_CHUNK_TILES + 1, 3_000_017]


def key_bits(sigma, k):
    return max(1, (sigma ** k - 1).bit_length())


def onesweep_applies(sigma, k):
    return key_bits(sigma, k) <= 32 and k * symbol_bits(sigma) <= 64


def sort_passes(onesweep, sigma, k, digits):
    """passes of the tiled sorter (equal shares of the key bits) and of onesweep (for a power-of-two alphabet the digit
    rounded to whole symbols, at most 8 bits), as build_element / sort_element_onesweep choose them"""
    kbits, bits = key_bits(sigma, k), symbol_bits(sigma)
    passes = -(-kbits // digits)
    if onesweep and sigma == 1 << bits:
        w = -(-kbits // passes)
        w = -(-w // bits) * bits
        if w > 8:
            w = 8 // bits * bits
        passes = -(-kbits // w)
    return passes


@pytest.fixture(scope="module")
def build_refs(oracle_mod):
    """per (sigma, k, n_kmers): text, the oracle's CSR, a small batch and the oracle's answers"""
    made = {}

    def get(sigma, k, n_kmers):
        key = (sigma, k, n_kmers)
        if key not in made:
            from kmer_index_b200 import synth
            n = n_kmers + k - 1
            text = synth.random_text(n, sigma, 60 + n % 97)
            if n >= 20_000:
                text[n // 4:n // 4 + 3000] = 0                 # a bucket of ~3000 k-mers across tile boundaries
            q, off = synth.stress_queries(text, 300, 1, 48, sigma, 61)
            with oracle_mod.Oracle(text, sigma, [k]) as o:
                made[key] = (text, o.element(0), q, off, o.search(q, off))
        return made[key]
    return get


def check_build(kb, build_refs, monkeypatch, sigma, k, n_kmers, sorter, digits):
    text, (oh, op), q, off, want = build_refs(sigma, k, n_kmers)
    monkeypatch.setenv("KMER_B200_SORT", sorter)
    if digits is None:
        monkeypatch.delenv("KMER_B200_DIGIT_BITS", raising=False)
    else:
        monkeypatch.setenv("KMER_B200_DIGIT_BITS", str(digits))
    onesweep = sorter == "onesweep" and onesweep_applies(sigma, k)
    label = f"sigma={sigma} k={k} n_kmers={n_kmers} {sorter} digits={digits}"
    with kernels_launched() as names:
        ix = kb.KmerIndex(text, sigma, [k])
    try:
        info = ix.element_info(0)
        assert info.n_kmers == n_kmers and info.key_bits == key_bits(sigma, k), label
        assert info.sort_passes == sort_passes(onesweep, sigma, k, digits or 8), (label, info.sort_passes)
        if onesweep:
            assert launches(names, "onesweep_kernel") == info.sort_passes, (label, kernel_summary(names))
            assert launches(names, "radix_scatter_kernel") == 0, (label, kernel_summary(names))
        else:
            assert launches(names, "radix_scatter_kernel") == info.sort_passes, (label, kernel_summary(names))
            assert launches(names, "onesweep_kernel") == 0, (label, kernel_summary(names))
        h, p = ix.element_arrays(0)
        assert np.array_equal(h.astype(np.uint64), oh), f"{label}: hashes"
        assert np.array_equal(p, op), f"{label}: positions"
        for attempt in range(2):     # sub-k queries build auxiliary elements with the same sorter
            assert_results_equal(ix.search_batch(q, off).as_tuple(), want, label=f"{label} search/{attempt}")
    finally:
        ix.close()


@pytest.mark.parametrize("digits", DIGITS, ids=lambda d: f"digits{d or 8}")
@pytest.mark.parametrize("sorter", ["tiled", "onesweep"])
@pytest.mark.parametrize("sigma,k", DIGIT_SHAPES)
def test_build_at_every_digit_width(kb, build_refs, monkeypatch, sigma, k, sorter, digits):
    """KMER_B200_DIGIT_BITS 4-8 under both sorters: narrower digits leave the byte-aligned path and end in a partial last
    digit; where onesweep does not apply (64-bit keys, k * bits > 64) the tiled sorter runs and the CSR is the same"""
    check_build(kb, build_refs, monkeypatch, sigma, k, 200_003, sorter, digits)


@pytest.mark.parametrize("n_kmers", LENGTHS)
@pytest.mark.parametrize("sorter,digits", [("tiled", None), ("tiled", 5), ("onesweep", None), ("onesweep", 5)])
@pytest.mark.parametrize("sigma,k", LENGTH_SHAPES)
def test_build_at_tile_and_chunk_boundaries(kb, build_refs, monkeypatch, sigma, k, sorter, digits, n_kmers):
    """1 and 2 k-mers, one k-mer around the 8192-k-mer sort tile and around the 64-tile scan chunk, and a larger odd size"""
    check_build(kb, build_refs, monkeypatch, sigma, k, n_kmers, sorter, digits)


@pytest.mark.parametrize("digits", [4, 6])
@pytest.mark.parametrize("sigma,ks,parts", [(4, [12], 2), (4, [16], 3), (27, [5], 3), (4, [5, 9, 13], 2)])
def test_key_range_parts_with_narrow_digits(kb, oracle_mod, monkeypatch, sigma, ks, parts, digits):
    """a key-range part sorts its filtered (hash - lo, position) pairs with the tiled sorter whatever KMER_B200_SORT says;
    its positions are the oracle's CSR restricted to [key_lo, key_hi), in the same order"""
    import torch

    from kmer_index_b200 import sharded, synth
    dev = torch.device("cuda", 0)
    text = synth.random_text(300_001, sigma, 71)
    text[1000:4000] = 0
    monkeypatch.setenv("KMER_B200_SORT", "onesweep")
    monkeypatch.setenv("KMER_B200_DIGIT_BITS", str(digits))
    with oracle_mod.Oracle(text, sigma, ks) as o:
        csr = [o.element(e) for e in range(len(ks))]
    stream = torch.cuda.current_stream().cuda_stream
    with kernels_launched() as names:
        idx = [kb.KmerIndex(text, sigma, ks, key_part=r, key_parts=parts, stream=stream or None) for r in range(parts)]
    try:
        assert launches(names, "onesweep_kernel") == 0 and launches(names, "radix_scatter_kernel") > 0, kernel_summary(names)
        for e, k in enumerate(ks):
            oh, op = csr[e]
            for r, ix in enumerate(idx):
                p = ix.element_part(e)
                sel = (oh >= p.key_lo) & (oh < p.key_hi)
                assert p.n_kmers == int(sel.sum()), (ks, e, r)
                got = sharded._dev_view(p.d_positions, p.n_kmers, dev).cpu().numpy().view(np.uint32)
                assert np.array_equal(got, op[sel]), (ks, e, r)
    finally:
        for ix in idx:
            ix.close()
