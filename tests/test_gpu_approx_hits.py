"""Hit strategies of approximate search (all + distances, all best, strata, single best; kmer_b200_*_approx_*_ex) on
the GPU, bit for bit against the numpy derivation from the every-window ground truth (tests/approx_hits_truth.py)."""
import ctypes as C

import numpy as np
import pytest

from approx_hits_truth import NO_HIT, hits_truth
from conftest import assert_results_equal
from test_gpu_approx import BUDGETS, SHAPES, concat, mixed_batch

pytestmark = pytest.mark.gpu

# (hits, strata): ALL (with distances), ALL_BEST, STRATA 1 and 2, SINGLE_BEST
STRATEGIES = [("all", 0), ("all_best", 0), ("strata", 1), ("strata", 2), ("single_best", 0)]


@pytest.fixture(scope="module")
def kb():
    import kmer_index_b200
    return kmer_index_b200


def wants_distances(hits, e):
    """"all" always asks for distances; the other strategies on alternate budgets (both paths are covered)"""
    return hits == "all" or e % 2 == 0


def check(got, want, label, distances=True):
    """got: BatchResult; want: (offsets, positions, status, distances, best_distance)"""
    w_off, w_pos, w_st, w_dist, w_best = want
    assert_results_equal(got.as_tuple(), (w_off, w_pos, w_st), label=label)
    if distances:
        assert got.distances is not None and np.array_equal(got.distances, w_dist), label
    else:
        assert got.distances is None, label
    if w_best is None:
        assert got.best_distance is None, label
    else:
        assert got.best_distance is not None and np.array_equal(got.best_distance, w_best), label


def run_all(ix, text, q, off, e, label):
    """every strategy of STRATEGIES on the host form against the derivation; returns the derivation"""
    want = hits_truth(text, q, off, e, STRATEGIES)
    for h, s in STRATEGIES:
        dist = wants_distances(h, e)
        got = ix.search_approx(q, off, e, hits=h, strata=s, distances=dist)
        check(got, want[(h, s)], f"{label} e={e} {h}/{s}", dist)
    return want


@pytest.mark.parametrize("shape", list(SHAPES))
def test_hits_match_truth(kb, shape):
    """Every budget, random and planted queries of 1..150 symbols; "all" equals search_approx exactly; a planted read
    whose distance at its origin is strictly the smallest is the single best at its origin."""
    from kmer_index_b200 import synth
    sigma, ks = SHAPES[shape]
    text = synth.random_text(60_000, sigma, 31 + sigma)
    with kb.KmerIndex(text, sigma, ks) as ix:
        for e in BUDGETS:
            q, off, Q, origins, ds = mixed_batch(text, sigma, e, 500 + e)
            want = run_all(ix, text, q, off, e, shape)
            plain = ix.search_approx(q, off, e)
            got = ix.search_approx(q, off, e, hits="all", distances=True)
            assert_results_equal(got.as_tuple(), plain.as_tuple(), label=f"{shape} e={e} all vs search_approx")
            single = ix.search_approx(q, off, e, hits="single_best")
            a_off, a_pos, _, a_dist, _ = want[("all", 0)]
            n_strict = 0
            for i in range(origins.size):
                qi = Q + i
                seg_p = a_pos[int(a_off[qi]):int(a_off[qi + 1])]
                seg_d = a_dist[int(a_off[qi]):int(a_off[qi + 1])]
                if ds[i] <= e and np.count_nonzero(seg_d <= ds[i]) == 1:
                    assert single.to_vector(qi).tolist() == [int(origins[i])], (shape, e, i)
                    assert int(seg_p[seg_d <= ds[i]][0]) == int(origins[i])
                    n_strict += 1
            assert n_strict > 0


@pytest.mark.parametrize("shape", ["dna4_k12", "dna4_multi", "aa27_k5"])
def test_device_and_count_only_forms_equal_host(kb, shape):
    import torch

    from kmer_index_b200 import synth
    sigma, ks = SHAPES[shape]
    text = synth.random_text(50_000, sigma, 43)
    dev = torch.device("cuda", 0)
    with kb.KmerIndex(text, sigma, ks) as ix:
        for e in (0, 2, 5):
            q, off, _, _, _ = mixed_batch(text, sigma, e, 600 + e, Q=300)
            d_q = torch.from_numpy(q).to(dev)
            d_off = torch.from_numpy(off.view(np.int64)).to(dev)
            Q, max_len = off.size - 1, int(np.diff(off).max())
            for h, s in STRATEGIES:
                host = ix.search_approx(q, off, e, hits=h, strata=s, distances=True)
                torch.cuda.synchronize()
                for fn in (ix.search_approx_batch_device, ix.count_approx_batch_device):
                    r = fn(d_q.data_ptr(), d_off.data_ptr(), Q, max_len, e, hits=h, strata=s, distances=True)
                    torch.cuda.synchronize()
                    label = f"{shape} e={e} {h}/{s} {fn.__name__}"
                    o = torch.as_tensor(r.offsets(), device=dev).cpu().numpy().astype(np.uint64)
                    st = torch.as_tensor(r.status(), device=dev).cpu().numpy()
                    assert np.array_equal(o, host.offsets) and np.array_equal(st, host.status), label
                    bd = r.best_distances()
                    if h == "all":
                        assert bd is None, label
                    else:
                        assert np.array_equal(torch.as_tensor(bd, device=dev).cpu().numpy(), host.best_distance), label
                    if fn == ix.search_approx_batch_device:
                        p = (torch.as_tensor(r.positions(), device=dev).cpu().numpy().view(np.uint32) if r.n_positions
                             else np.zeros(0, np.uint32))
                        d = (torch.as_tensor(r.distances(), device=dev).cpu().numpy() if r.n_positions
                             else np.zeros(0, np.uint8))
                        assert np.array_equal(p, host.positions) and np.array_equal(d, host.distances), label
                    else:
                        assert r.distances() is None and not r.positions_ptr, label
                    r.free()


def test_edge_cases(kb):
    """empty query, m > n, m <= e, the whole text, and a text without the query's symbol (d_min = m: every window)"""
    from kmer_index_b200 import synth
    text = synth.random_text(5_000, 4, 71)
    n = text.size
    with kb.KmerIndex(text, 4, [10]) as ix:
        empty = ix.search_approx(np.zeros(0, np.uint8), np.zeros(1, np.uint64), 2, hits="all_best", distances=True)
        assert len(empty) == 0 and empty.positions.size == 0 and empty.best_distance.size == 0
        assert empty.distances is not None and empty.distances.size == 0
        none = ix.search_approx(synth.random_text(40, 4, 70), np.array([0, 40], np.uint64), 0, distances=True)
        assert none.positions.size == 0 and none.distances is not None and none.distances.size == 0
        qs = [np.zeros(0, np.uint8), text[:2].copy(), text[:3].copy(), text[-4:].copy(), synth.random_text(n + 1, 4, 72),
              text.copy(), text[-37:].copy(), synth.random_text(3, 4, 73), synth.random_text(8, 4, 74)]
        lens = np.array([x.size for x in qs], dtype=np.uint64)
        off = np.zeros(lens.size + 1, dtype=np.uint64)
        np.cumsum(lens, out=off[1:])
        q = np.concatenate(qs)
        for e in (0, 3, 8):
            want = run_all(ix, text, q, off, e, "edges")
            got = ix.search_approx(q, off, e, hits="single_best", distances=True)
            assert got.status[0] == kb.QUERY_UNDEFINED and got.best_distance[0] == NO_HIT and got.to_vector(0).size == 0
            assert got.best_distance[4] == NO_HIT and got.to_vector(4).size == 0         # m > n
            assert got.best_distance[5] == 0 and got.to_vector(5).tolist() == [0]       # the whole text
            assert want[("all_best", 0)][4][5] == 0
    # a text over {0, 1, 2}: a query of 3s has d = m in every window
    text3 = synth.random_text(4_000, 3, 75)
    with kb.KmerIndex(text3, 4, [8]) as ix:
        qs = [np.full(m, 3, np.uint8) for m in (1, 2, 5, 8)] + [text3[100:140].copy()]
        q, off = concat(*[(x, np.array([0, x.size], np.uint64)) for x in qs])
        for e in (2, 5, 8):
            run_all(ix, text3, q, off, e, "no symbol 3")
            got = ix.search_approx(q, off, e, hits="all_best", distances=True)
            for i, x in enumerate(qs[:4]):
                if x.size <= e:
                    assert got.best_distance[i] == x.size
                    assert np.array_equal(got.to_vector(i), np.arange(text3.size - x.size + 1, dtype=np.uint32))
                else:
                    assert got.best_distance[i] == NO_HIT and got.to_vector(i).size == 0
            single = ix.search_approx(q, off, e, hits="single_best")
            assert [single.to_vector(i).tolist() for i in range(4)] == [[0] if x.size <= e else [] for x in qs[:4]]


def test_invalid_options_and_ranks(kb):
    from kmer_index_b200 import _capi, synth
    text = synth.random_text(5_000, 4, 76)
    q, off = synth.stress_queries(text, 50, 5, 40, 4, 77)
    with kb.KmerIndex(text, 4, [10]) as ix:
        L = _capi.lib()
        r = C.c_void_p()
        assert L.kmer_b200_search_approx_batch_ex(ix.handle, q.ctypes.data, off.ctypes.data, off.size - 1, None,
                                                  C.byref(r)) == -1
        for opt in (_capi.ApproxOptions(9, 0, 0, 0), _capi.ApproxOptions(2, 4, 0, 0), _capi.ApproxOptions(2, 1, 0, 2),
                    _capi.ApproxOptions(2, 2, 0, 0x80000001)):
            assert L.kmer_b200_search_approx_batch_ex(ix.handle, q.ctypes.data, off.ctypes.data, off.size - 1,
                                                      C.byref(opt), C.byref(r)) == -1
        with pytest.raises(ValueError):
            ix.search_approx(q, off, 1, hits="best")
        bad = q.copy()
        bad[3] = 4
        for h in ("all_best", "single_best", "strata"):
            with pytest.raises(kb.KmerB200Error) as err:
                ix.search_approx(bad, off, 1, hits=h, strata=1)
            assert err.value.code == -4
        got = ix.search_approx(q, off, 1, hits="single_best", distances=True)   # the handle is still usable
        check(got, hits_truth(text, q, off, 1, [("single_best", 0)])[("single_best", 0)], "after errors")


@pytest.mark.parametrize("sigma,ks", [(4, [12]), (4, [5, 7, 9, 11, 13]), (15, [8])])
def test_heavy_candidate_lists(kb, sigma, ks):
    """Constant runs make buckets of ~70 000 candidates: the best pass and the re-seeded passes take the warp launch."""
    from kmer_index_b200 import synth
    text = synth.random_text(150_000, sigma, 5)
    text[20_000:90_000] = 0
    text[100_000:100_300] = np.resize(np.array([1, 0, 0], dtype=np.uint8), 300)
    q, off = synth.stress_queries(text, 600, 1, 100, sigma, 6, low_sigma=2)
    lens = np.diff(off).astype(np.int64)
    for i in range(0, 300, 3):
        q[int(off[i]):int(off[i]) + int(lens[i])] = 0
        if lens[i] > 4:
            q[int(off[i]) + int(lens[i]) // 2] = 1               # one substitution in a constant query
    with kb.KmerIndex(text, sigma, ks) as ix:
        for e in (0, 1, 2):
            want = run_all(ix, text, q, off, e, f"heavy {ks}")
            assert int(np.diff(want[("all_best", 0)][0]).max()) > 2048
            assert int(np.diff(want[("strata", 1)][0]).max()) > 2048


def test_auxiliary_elements_sparse_directory_save_load_and_parts(kb, tmp_path):
    import torch

    from kmer_index_b200 import sharded, synth
    # slab seeds before and after auxiliary elements exist
    text = synth.random_text(80_000, 4, 51)
    with kb.KmerIndex(text, 4, [12], mode=kb.MODE_CORRECT) as ix:
        for e in (1, 3, 8):
            q, off, _, _, _ = mixed_batch(text, 4, e, 700 + e, Q=300, m_hi=60)
            run_all(ix, text, q, off, e, "before aux")
            short, s_off = synth.stress_queries(text, 400, 1, 11, 4, 710 + e)
            ix.search_batch(short, s_off)     # builds the auxiliary elements of lengths 1..11
            run_all(ix, text, q, off, e, "after aux")
    sigma, n = 4, 200_000
    text = synth.random_text(n, sigma, 61)
    text[5000:8000] = 0
    q, off, _, _, _ = mixed_batch(text, sigma, 3, 720, Q=300)
    with kb.KmerIndex(text, sigma, [12], directory_bits=12) as ix:
        assert ix.element_info(0).directory_shift > 0
        for e in (0, 3):
            run_all(ix, text, q, off, e, "sparse")
        path = str(tmp_path / "index.kmerb200")
        ix.save(path)
    with kb.KmerIndex.load(path) as ld:
        for e in (0, 3):
            run_all(ld, text, q, off, e, "loaded")
    # peer-positions index emulated on one GPU: the directory whole, the positions left in the key-range parts
    dev = torch.device("cuda", 0)
    for ks, parts in (([12], 4), ([5, 7, 9, 11, 13], 3)):
        stream = torch.cuda.current_stream().cuda_stream
        idx = [kb.KmerIndex(text, sigma, ks, key_part=r, key_parts=parts, stream=stream or None) for r in range(parts)]
        try:
            with pytest.raises(kb.KmerB200Error) as err:
                idx[0].search_approx(q, off, 1, hits="all_best")     # a key-range part that has not been adopted
            assert err.value.code == -5
            for e, k in enumerate(ks):
                ps = [ix.element_part(e) for ix in idx]
                bufs, first = [], [0]
                dir_full = torch.empty(sigma ** k + 1, dtype=torch.int32, device=dev)
                for r, (ix, p) in enumerate(zip(idx, ps)):
                    buf = torch.empty(max(p.n_kmers, 1), dtype=torch.int32, device=dev)
                    if p.n_kmers:
                        buf[:p.n_kmers].copy_(sharded._dev_view(p.d_positions, p.n_kmers, dev))
                    bufs.append(buf)
                    n_dir = p.key_hi - p.key_lo + (1 if r == parts - 1 else 0)
                    ix.export_directory(e, first[-1], n_dir, dir_full.data_ptr() + 4 * p.key_lo)
                    first.append(first[-1] + p.n_kmers)
                torch.cuda.synchronize()
                idx[0].adopt_element_parts(e, bufs, first, dir_full)
            for e in (0, 3):
                run_all(idx[0], text, q, off, e, f"parts {ks}")
        finally:
            for ix in idx:
                ix.close()


def test_refused_handles_stay_usable(kb, oracle_mod):
    from kmer_index_b200 import synth
    n = 200_000
    text = synth.random_text(n, 4, 81)
    q, off = synth.stress_queries(text[:100_000], 200, 10, 40, 4, 82)
    want = oracle_mod.Oracle.truth(text[:100_000], q, off)
    handles = [kb.KmerIndex(text[:100_000], 4, [10, 12], shared_positions=True, mode=kb.MODE_CORRECT),
               kb.KmerIndex(text[:100_063], 4, [12], shard_begin=0, n_total=n, halo=63, mode=kb.MODE_CORRECT)]
    try:
        for ix in handles:
            for h in ("all_best", "single_best", "strata"):
                with pytest.raises(kb.KmerB200Error) as err:
                    ix.search_approx(q, off, 1, hits=h, strata=1, distances=True)
                assert err.value.code == -5
            got = ix.search_batch(q, off).as_tuple()
            if ix is handles[1]:
                assert got[1].size > 0
            else:
                assert_results_equal(got, want, label="after refusal")
    finally:
        for ix in handles:
            ix.close()


def test_multi_device_handle_refuses_and_stays_usable(kb, oracle_mod):
    import torch

    from kmer_index_b200 import synth
    if torch.cuda.device_count() < 2:
        pytest.skip("a multi-device handle needs two GPUs")
    text = synth.random_text(100_000, 4, 83)
    q, off = synth.stress_queries(text, 200, 10, 40, 4, 84)
    with kb.KmerIndex(text, 4, [12], devices=[0, 1], mode=kb.MODE_CORRECT) as ix:
        for h in ("all_best", "single_best", "strata"):
            with pytest.raises(kb.KmerB200Error) as err:
                ix.search_approx(q, off, 1, hits=h, strata=1, distances=True)
            assert err.value.code == -5
        assert_results_equal(ix.search_batch(q, off).as_tuple(), oracle_mod.Oracle.truth(text, q, off),
                             label="multi-device after refusal")


def test_large_planted_reads(kb):
    """50 Mbp dna4, 10^5 reads of 100 symbols with 0..3 substitutions, e = 3: every read's best distance is its planted
    d, its single best is its origin, and its all-best hits include the origin."""
    from kmer_index_b200 import synth
    n, Q, m, e = 50_000_000, 100_000, 100, 3
    text = synth.random_text(n, 4, 93)
    rng = np.random.default_rng(94)
    origins = rng.integers(0, n - m + 1, Q)
    ds = np.arange(Q) % (e + 1)
    reads = text[origins[:, None] + np.arange(m)]
    for i in range(Q):
        cols = rng.choice(m, size=int(ds[i]), replace=False)
        reads[i, cols] = (reads[i, cols] + rng.integers(1, 4, cols.size)) % 4
    q = reads.reshape(-1).astype(np.uint8)
    off = (np.arange(Q + 1, dtype=np.uint64) * m)
    with kb.KmerIndex(text, 4, [16]) as ix:
        single = ix.search_approx(q, off, e, hits="single_best", distances=True)
        assert np.array_equal(single.best_distance, ds.astype(np.uint8))
        assert np.array_equal(np.diff(single.offsets), np.ones(Q, np.uint64))
        assert np.array_equal(single.positions, origins.astype(np.uint32))
        assert np.array_equal(single.distances, ds.astype(np.uint8))
        best = ix.search_approx(q, off, e, hits="all_best", distances=True)
        assert np.array_equal(best.best_distance, single.best_distance)
        counts = np.diff(best.offsets).astype(np.int64)
        qid = np.repeat(np.arange(Q), counts)
        assert np.all(best.distances == ds[qid])
        for i in range(0, Q, 97):
            assert origins[i] in best.to_vector(i), i
        win = text[best.positions.astype(np.int64)[:, None] + np.arange(m)]
        assert np.array_equal((win != reads[qid]).sum(axis=1), best.distances.astype(np.int64))
