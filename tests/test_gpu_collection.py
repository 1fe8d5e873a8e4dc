"""Collection index (kmer_b200_attach_records) on the GPU: every search reports only windows inside one record, bit for
bit equal to searching each record on its own (tests/collection_truth.py, derivation (a))."""
import ctypes as C

import numpy as np
import pytest

from approx_hits_truth import filter_hits, hit_distances
from collection_truth import hits_truth, random_starts, truth_per_record
from conftest import assert_results_equal
from test_gpu_approx import SHAPES, device_results, mixed_batch

pytestmark = pytest.mark.gpu

STRATEGIES = [("all", 0), ("all_best", 0), ("single_best", 0), ("strata", 1), ("strata", 2)]


@pytest.fixture(scope="module")
def kb():
    import kmer_index_b200
    return kmer_index_b200


def collection(n, sigma, seed, R=40, short=14):
    from kmer_index_b200 import synth
    rng = np.random.default_rng(seed)
    text = synth.random_text(n, sigma, seed)
    return text, random_starts(n, R, rng, short=short)


def junction_batch(text, starts, sigma, seed, Q=200, m_hi=150):
    """windows across record starts (exact and with a few substitutions) and short queries taken at record ends"""
    rng = np.random.default_rng(seed)
    inner = [int(s) for s in starts[1:-1] if 0 < int(s) < text.size]
    qs = []
    for i in range(Q):
        m = int(rng.integers(1, m_hi + 1)) if i % 2 else int(rng.integers(1, 12))
        s = inner[int(rng.integers(0, len(inner)))]
        p = min(max(0, s - int(rng.integers(0, m + 1))), text.size - m)
        x = text[p:p + m].copy()
        for j in rng.choice(m, size=min(m, i % 3), replace=False):
            x[j] = (int(x[j]) + 1) % sigma
        qs.append(x)
    off = np.zeros(Q + 1, np.uint64)
    np.cumsum([x.size for x in qs], out=off[1:])
    return np.concatenate(qs), off


def full_batch(text, starts, sigma, e, seed, Q=300):
    from test_gpu_approx import concat
    q1, o1, _, _, _ = mixed_batch(text, sigma, e, seed, Q=Q)
    q2, o2 = junction_batch(text, starts, sigma, seed + 7)
    return concat((q1, o1), (q2, o2))


def host_tuple(r):
    return r.offsets, r.positions, r.status


@pytest.mark.parametrize("shape", list(SHAPES))
def test_collection_matches_per_record_truth(kb, shape):
    """Seven index shapes, budgets 0-8, queries of 1..150 symbols (records shorter than k and than m, empty and 1-symbol
    records); e = 0 equals exact search in CORRECT mode and in the default mode."""
    sigma, ks = SHAPES[shape]
    text, starts = collection(60_000, sigma, 31 + sigma)
    with kb.KmerIndex(text, sigma, ks) as ix:
        ix.attach_records(starts)
        assert np.array_equal(ix.records, starts)
        for e in range(9):
            q, off = full_batch(text, starts, sigma, e, 100 + e)
            want = truth_per_record(text, starts, q, off, e)
            assert_results_equal(ix.search_approx(q, off, e).as_tuple(), want, label=f"{shape} e={e}")
            if e == 0:
                assert_results_equal(ix.search_batch(q, off, mode=kb.MODE_CORRECT).as_tuple(), want, label=f"{shape} exact")
                assert_results_equal(ix.search_batch(q, off).as_tuple(), want, label=f"{shape} exact default mode")


@pytest.mark.parametrize("shape", ["dna4_k12", "dna4_multi", "aa27_k5"])
def test_strategies_and_forms(kb, shape):
    sigma, ks = SHAPES[shape]
    text, starts = collection(50_000, sigma, 41, R=30)
    with kb.KmerIndex(text, sigma, ks) as ix:
        ix.attach_records(starts)
        for e in (0, 2, 5):
            q, off = full_batch(text, starts, sigma, e, 200 + e, Q=200)
            truth = hits_truth(text, starts, q, off, e, STRATEGIES)
            full, count = device_results(kb, ix, q, off, e)
            assert_results_equal(full, truth[("all", 0)][:3], label=f"device {shape} e={e}")
            assert np.array_equal(count[0], truth[("all", 0)][0]) and np.array_equal(count[2], truth[("all", 0)][2])
            for h, s in STRATEGIES:
                w_off, w_pos, w_st, w_dist, w_best = truth[(h, s)]
                for dist in (False, True):
                    got = ix.search_approx(q, off, e, hits=h, strata=s, distances=dist)
                    label = f"{shape} e={e} {h}/{s} distances={dist}"
                    assert_results_equal(host_tuple(got), (w_off, w_pos, w_st), label=label)
                    assert (got.best_distance is None) if h == "all" else np.array_equal(got.best_distance, w_best), label
                    if dist:
                        assert np.array_equal(got.distances, w_dist), label
                dev = device_strategy(kb, ix, q, off, e, h, s)
                assert np.array_equal(dev["offsets"], w_off) and np.array_equal(dev["positions"], w_pos), (shape, e, h, s)
                assert np.array_equal(dev["count_offsets"], w_off), (shape, e, h, s)
                if h != "all":
                    assert np.array_equal(dev["best"], w_best) and np.array_equal(dev["count_best"], w_best), (shape, e, h, s)


def device_strategy(kb, ix, q, off, e, hits, strata):
    import torch
    dev = torch.device("cuda", 0)
    d_q = torch.from_numpy(q).to(dev)
    d_off = torch.from_numpy(off.view(np.int64)).to(dev)
    Q, max_len = off.size - 1, int(np.diff(off).max())
    torch.cuda.synchronize()
    out = {}
    for key, fn in (("", ix.search_approx_batch_device), ("count_", ix.count_approx_batch_device)):
        r = fn(d_q.data_ptr(), d_off.data_ptr(), Q, max_len, e, hits=hits, strata=strata)
        torch.cuda.synchronize()
        out[key + "offsets"] = torch.as_tensor(r.offsets(), device=dev).cpu().numpy().astype(np.uint64)
        if not key:
            out["positions"] = (torch.as_tensor(r.positions(), device=dev).cpu().numpy().view(np.uint32) if r.n_positions
                                else np.zeros(0, np.uint32))
        b = r.best_distances()
        out[key + "best"] = torch.as_tensor(b, device=dev).cpu().numpy() if b is not None else None
        r.free()
    return out


def test_exact_forms_and_modes(kb):
    """CORRECT-mode search_batch, _ptrs, _text, _device and count_batch_device equal the e = 0 truth; REFERENCE_EXACT is
    refused; host batches take the single-copy staging."""
    import torch
    from kmer_index_b200 import _capi
    text, starts = collection(40_000, 4, 51, R=25)
    q, off = full_batch(text, starts, 4, 0, 300, Q=200)
    want = truth_per_record(text, starts, q, off, 0)
    with kb.KmerIndex(text, 4, [5, 7, 9, 11, 13]) as ix:
        ix.attach_records(starts)
        assert_results_equal(ix.search_batch(q, off, mode=kb.MODE_CORRECT).as_tuple(), want, label="search_batch")
        assert ix.last_search_host_path()["pipeline"] == "single copy"
        Q = off.size - 1
        bufs = [np.ascontiguousarray(q[int(off[i]):int(off[i + 1])]) for i in range(Q)]
        ptrs = (C.c_void_p * Q)(*[b.ctypes.data if b.size else None for b in bufs])
        lens = np.diff(off).astype(np.uint64)
        r = C.c_void_p()
        _capi.check(ix._L.kmer_b200_search_batch_ptrs(ix.handle, ptrs, lens.ctypes.data, Q, kb.MODE_CORRECT, C.byref(r)))
        assert_results_equal(host_tuple(ix._host_result(r, Q, True)), want, label="ptrs")
        chars = ["".join("ACGT"[int(c)] for c in b) for b in bufs]
        assert_results_equal(ix.search_batch_text(chars, lut=kb.char_lut("dna4"), mode=kb.MODE_CORRECT).as_tuple(), want,
                             label="text")
        dev = torch.device("cuda", 0)
        d_q, d_off = torch.from_numpy(q).to(dev), torch.from_numpy(off.view(np.int64)).to(dev)
        max_len = int(np.diff(off).max())
        torch.cuda.synchronize()
        for fn in (ix.search_batch_device, ix.count_batch_device):
            for mode in (kb.MODE_CORRECT, kb.MODE_DEFAULT):
                res = fn(d_q.data_ptr(), d_off.data_ptr(), Q, max_len, mode)
                torch.cuda.synchronize()
                o = torch.as_tensor(res.offsets(), device=dev).cpu().numpy().astype(np.uint64)
                assert np.array_equal(o, want[0])
                assert np.array_equal(torch.as_tensor(res.status(), device=dev).cpu().numpy(), want[2])
                if fn == ix.search_batch_device and res.n_positions:
                    assert np.array_equal(torch.as_tensor(res.positions(), device=dev).cpu().numpy().view(np.uint32), want[1])
                res.free()
        for call in (lambda: ix.search_batch(q, off, mode=kb.MODE_REFERENCE_EXACT),
                     lambda: ix.search_batch_device(d_q.data_ptr(), d_off.data_ptr(), Q, max_len, kb.MODE_REFERENCE_EXACT),
                     lambda: ix.count_batch_device(d_q.data_ptr(), d_off.data_ptr(), Q, max_len, kb.MODE_REFERENCE_EXACT)):
            with pytest.raises(kb.KmerB200Error) as err:
                call()
            assert err.value.code == -1
        assert_results_equal(ix.search_batch(q, off).as_tuple(), want, label="still usable")


def test_junction_artefact_and_in_record_hit(kb):
    """A query that occurs exactly only across a junction and with 2 substitutions inside a record: single best returns
    the in-record window at d = 2, count-only counts 1, a plain index returns the junction window."""
    from kmer_index_b200 import synth
    text = synth.random_text(20_000, 4, 61)
    starts = np.array([0, 7_000, 13_000, 20_000], np.uint64)
    m = 40
    q = text[7_000 - 17:7_000 - 17 + m].copy()
    inside = 15_000
    text[inside:inside + m] = q
    text[inside + 5] = (text[inside + 5] + 1) % 4
    text[inside + 30] = (text[inside + 30] + 2) % 4
    off = np.array([0, m], np.uint64)
    with kb.KmerIndex(text, 4, [12]) as plain, kb.KmerIndex(text, 4, [12]) as ix:
        ix.attach_records(starts)
        p = plain.search_approx(q, off, 2, hits="single_best", distances=True)
        assert p.positions.tolist() == [7_000 - 17] and p.distances.tolist() == [0]
        got = ix.search_approx(q, off, 2, hits="single_best", distances=True)
        assert got.positions.tolist() == [inside] and got.distances.tolist() == [2] and got.best_distance.tolist() == [2]
        assert ix.search_approx(q, off, 2).positions.tolist() == [inside]
        assert ix.search_approx(q, off, 1).positions.size == 0
        assert ix.search_batch(q, off).positions.size == 0 and plain.search_batch(q, off, mode=kb.MODE_CORRECT).positions.size == 1
        _, count = device_results(kb, ix, q, off, 2)
        assert count[0].tolist() == [0, 1]
        assert np.array_equal(ix.locate(got.positions)[0], [2]) and np.array_equal(ix.locate(got.positions)[1], [2_000])


def test_single_record_equals_plain_index(kb):
    sigma, ks = 4, [5, 7, 9, 11, 13]
    from kmer_index_b200 import synth
    text = synth.random_text(30_000, sigma, 71)
    with kb.KmerIndex(text, sigma, ks, mode=kb.MODE_CORRECT) as plain, kb.KmerIndex(text, sigma, ks) as ix:
        ix.attach_records([0, text.size])
        for e in (0, 1, 3, 8):
            q, off, _, _, _ = mixed_batch(text, sigma, e, 700 + e, Q=200)
            for h, s in STRATEGIES:
                a = plain.search_approx(q, off, e, hits=h, strata=s, distances=True)
                b = ix.search_approx(q, off, e, hits=h, strata=s, distances=True)
                assert_results_equal(host_tuple(b), host_tuple(a), label=f"e={e} {h}/{s}")
                assert np.array_equal(a.distances, b.distances)
                assert (a.best_distance is None and b.best_distance is None) or np.array_equal(a.best_distance, b.best_distance)
            if e == 0:
                assert_results_equal(ix.search_batch(q, off).as_tuple(), plain.search_batch(q, off).as_tuple(), label="exact")


def test_large_collection(kb):
    """50 Mbp dna4 in 10^4 records, 10^5 reads of 100 symbols with 0..4 substitutions, e = 4: the plain index's hits
    minus those across a record start, every read planted inside a record finds its origin."""
    from kmer_index_b200 import synth
    n, Q, m, e, R = 50_000_000, 100_000, 100, 4, 10_000
    rng = np.random.default_rng(92)
    text = synth.random_text(n, 4, 91)
    starts = random_starts(n, R, rng, short=200)
    origins = rng.integers(0, n - m + 1, Q)
    ds = np.arange(Q) % (e + 1)
    reads = text[origins[:, None] + np.arange(m)]
    for i in range(Q):
        cols = rng.choice(m, size=int(ds[i]), replace=False)
        reads[i, cols] = (reads[i, cols] + rng.integers(1, 4, cols.size)) % 4
    q = reads.reshape(-1).astype(np.uint8)
    off = np.arange(Q + 1, dtype=np.uint64) * m
    with kb.KmerIndex(text, 4, [16]) as ix:
        plain = ix.search_approx(q, off, e)
        ix.attach_records(starts)
        got = ix.search_approx(q, off, e)
        s = starts.astype(np.int64)
        p = plain.positions.astype(np.int64)
        keep = np.searchsorted(s, p, "right") == np.searchsorted(s, p + m - 1, "right")
        qid = np.repeat(np.arange(Q), np.diff(plain.offsets).astype(np.int64))
        w_off = np.zeros(Q + 1, np.uint64)
        np.cumsum(np.bincount(qid[keep], minlength=Q), out=w_off[1:])
        assert np.array_equal(got.offsets, w_off) and np.array_equal(got.positions, plain.positions[keep])
        inside = np.searchsorted(s, origins, "right") == np.searchsorted(s, origins + m - 1, "right")
        assert inside.sum() > Q // 2
        for i in np.flatnonzero(inside)[:5000]:
            assert origins[i] in got.positions[int(got.offsets[i]):int(got.offsets[i + 1])], i
        full, count = device_results(kb, ix, q, off, e, max_len=m)
        assert np.array_equal(count[0], got.offsets) and np.array_equal(full[1], got.positions)
        best = ix.search_approx(q, off, e, hits="single_best")
        w = filter_hits(got.offsets, got.positions, got.status, hit_distances(text, q, off, got.offsets, got.positions), e,
                        "single_best")
        assert np.array_equal(best.positions, w[1]) and np.array_equal(best.best_distance, w[4])


def test_heavy_sparse_auxiliary_and_peer_parts(kb, tmp_path):
    import torch

    from kmer_index_b200 import sharded, synth
    sigma, n = 4, 200_000
    text = synth.random_text(n, sigma, 81)
    text[20_000:90_000] = 0                       # a constant run cut by many records: heavy candidate lists
    rng = np.random.default_rng(82)
    starts = random_starts(n, 60, rng, short=20)
    q, off = full_batch(text, starts, sigma, 2, 800, Q=300)
    qz, oz = synth.stress_queries(text, 300, 1, 100, sigma, 83, low_sigma=2)
    for i in range(0, 300, 3):
        qz[int(oz[i]):int(oz[i + 1])] = 0
    from test_gpu_approx import concat
    q, off = concat((q, off), (qz, oz))
    want = {e: truth_per_record(text, starts, q, off, e) for e in (0, 2)}
    assert int(np.diff(want[0][0]).max()) > 2048
    with kb.KmerIndex(text, sigma, [12], directory_bits=12) as ix:
        ix.attach_records(starts)
        assert ix.element_info(0).directory_shift > 0
        for e in (0, 2):
            assert_results_equal(ix.search_approx(q, off, e).as_tuple(), want[e], label=f"sparse e={e}")
    with kb.KmerIndex(text, sigma, [12], mode=kb.MODE_CORRECT) as ix:
        short, s_off = synth.stress_queries(text, 400, 1, 11, sigma, 84)
        ix.search_batch(short, s_off)             # auxiliary k' = m elements for lengths 1..11, before the records
        ix.attach_records(starts)
        for e in (0, 2):
            assert_results_equal(ix.search_approx(q, off, e).as_tuple(), want[e], label=f"aux e={e}")
    dev = torch.device("cuda", 0)
    for ks, parts in (([12], 4), ([5, 7, 9, 11, 13], 3)):
        stream = torch.cuda.current_stream().cuda_stream
        idx = [kb.KmerIndex(text, sigma, ks, key_part=r, key_parts=parts, stream=stream or None) for r in range(parts)]
        try:
            with pytest.raises(kb.KmerB200Error) as err:
                idx[0].attach_records(starts)     # a key-range part that has not been adopted
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
            idx[0].attach_records(starts)
            for e in (0, 2):
                assert_results_equal(idx[0].search_approx(q, off, e).as_tuple(), want[e], label=f"parts {ks} e={e}")
        finally:
            for ix in idx:
                ix.close()


def test_fasta_records_index(kb):
    from kmer_index_b200 import synth
    rng = np.random.default_rng(91)
    lens = [3_000, 1, 0, 9, 12_000, 40, 7_000]
    seqs = [synth.random_text(L, 4, 100 + i) if L else np.zeros(0, np.uint8) for i, L in enumerate(lens)]
    fasta = "".join(f">rec{i}\n" + "\n".join("".join("ACGT"[int(c)] for c in s[j:j + 60]) for j in range(0, s.size, 60)) + "\n"
                    for i, s in enumerate(seqs))
    text = np.concatenate(seqs)
    with kb.parse_sequences(fasta, "dna4") as recs:
        assert np.array_equal(recs.starts, np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64))
        with recs.index([11], collection=True) as ix:
            assert np.array_equal(ix.records, recs.starts)
            q, off = full_batch(text, recs.starts, 4, 2, 900, Q=150)
            for e in (0, 2):
                assert_results_equal(ix.search_approx(q, off, e).as_tuple(), truth_per_record(text, recs.starts, q, off, e),
                                     label=f"fasta e={e}")
            assert_results_equal(ix.search_batch(q, off).as_tuple(), truth_per_record(text, recs.starts, q, off, 0), label="fasta exact")
            got = ix.search_approx(q, off, 2)
            rec, o = ix.locate(got.positions)
            r2, o2 = recs.locate(got.positions)
            assert np.array_equal(rec, r2) and np.array_equal(o, o2)
        with recs.index([11]) as plain:
            assert plain.records is None


def test_locate_host_and_device(kb):
    import torch
    from kmer_index_b200 import synth
    rng = np.random.default_rng(101)
    n = 1_000_000
    text = synth.random_text(n, 4, 102)
    for R, short in ((1, 0), (25, 5), (100_000, 30_000)):
        starts = random_starts(n, R, rng, short=short)
        pos = np.concatenate([rng.integers(0, n, 200_000), starts[:-1].astype(np.int64)[:1000], [n - 1, n, n + 5]]).astype(np.uint32)
        s = starts.astype(np.int64)
        w_rec = np.searchsorted(s, pos.astype(np.int64), "right") - 1
        valid = pos.astype(np.int64) < n
        w_off = np.where(valid, pos.astype(np.int64) - s[np.minimum(w_rec, R)], 0)
        w_rec = np.where(valid, w_rec, 0xFFFFFFFF)
        with kb.KmerIndex(text, 4, [12]) as ix:
            with pytest.raises(kb.KmerB200Error) as err:
                ix.locate(pos)
            assert err.value.code == -1
            ix.attach_records(starts)
            rec, off = ix.locate(pos)
            assert np.array_equal(rec, w_rec) and np.array_equal(off, w_off), R
            d_rec, d_off = ix.locate(torch.from_numpy(pos.view(np.int32)).cuda())
            assert np.array_equal(d_rec.cpu().numpy().view(np.uint32), w_rec) and np.array_equal(d_off.cpu().numpy().view(np.uint32), w_off)


def test_save_load_version4(kb, tmp_path):
    text, starts = collection(80_000, 4, 111, R=50)
    q, off = full_batch(text, starts, 4, 3, 1000, Q=200)
    want = {e: truth_per_record(text, starts, q, off, e) for e in (0, 3)}
    with kb.KmerIndex(text, 4, [10, 12]) as ix:
        ix.save(str(tmp_path / "plain.kmerb200"))
        plain_bytes = ix.device_bytes
        ix.attach_records(starts)
        assert ix.device_bytes >= plain_bytes + text.size // 8 + 8 * starts.size
        ix.save(str(tmp_path / "coll.kmerb200"))
        with pytest.raises(kb.KmerB200Error) as err:
            ix.attach_records(starts)             # once
        assert err.value.code == -1
    version = lambda p: int(np.fromfile(p, dtype=np.uint32, count=3)[2])
    assert version(tmp_path / "plain.kmerb200") == 3 and version(tmp_path / "coll.kmerb200") == 4
    with kb.KmerIndex.load(str(tmp_path / "coll.kmerb200")) as ld:
        assert np.array_equal(ld.records, starts)
        for e in (0, 3):
            assert_results_equal(ld.search_approx(q, off, e).as_tuple(), want[e], label=f"loaded e={e}")
        assert_results_equal(ld.search_batch(q, off).as_tuple(), want[0], label="loaded exact")
    with kb.KmerIndex.load(str(tmp_path / "plain.kmerb200")) as ld:
        assert ld.records is None


def test_refusals(kb):
    import torch
    from kmer_index_b200 import _capi, synth
    n = 100_000
    text = synth.random_text(n, 4, 121)
    starts = np.array([0, 40_000, n], np.uint64)
    L = _capi.lib()
    with kb.KmerIndex(text, 4, [12]) as ix:
        for bad in ([1, 40_000, n], [0, 50_000, 40_000, n], [0, 40_000, n - 1], [0, 40_000, n + 1]):
            with pytest.raises(kb.KmerB200Error) as err:
                ix.attach_records(bad)
            assert err.value.code == -1, bad
        s = np.ascontiguousarray(starts)
        assert L.kmer_b200_attach_records(ix.handle, s.ctypes.data_as(_capi.u64p), 0) == -1
        assert L.kmer_b200_attach_records(ix.handle, None, 2) == -1
        assert L.kmer_b200_attach_records(ix.handle, s.ctypes.data_as(_capi.u64p), 1 << 32) == -1
        assert ix.records is None
        ix.attach_records(starts)
        dev = torch.device("cuda", 0)
        q, off = synth.stress_queries(text, 100, 12, 30, 4, 122)
        d_q, d_off = torch.from_numpy(q).to(dev), torch.from_numpy(off.view(np.int64)).to(dev)
        scratch = torch.zeros(1000, dtype=torch.int64, device=dev)
        torch.cuda.synchronize()
        Q = off.size - 1
        calls = [lambda: ix.presence_batch_device(d_q.data_ptr(), d_off.data_ptr(), Q, 30, scratch.data_ptr()),
                 lambda: ix.search_batch_device_global(d_q.data_ptr(), d_off.data_ptr(), Q, 30, scratch.data_ptr()),
                 lambda: ix.search_sharded_begin(d_q.data_ptr(), d_off.data_ptr(), Q, 30, scratch.data_ptr()),
                 lambda: ix.route_plan(Q, 30, 2)]
        for call in calls:
            with pytest.raises(kb.KmerB200Error) as err:
                call()
            assert err.value.code == -5
        assert_results_equal(ix.search_batch(q, off).as_tuple(), truth_per_record(text, starts, q, off, 0), label="usable")
    handles = [kb.KmerIndex(text, 4, [10, 12], shared_positions=True, mode=kb.MODE_CORRECT),
               kb.KmerIndex(text[:60_063], 4, [12], shard_begin=0, n_total=n, halo=63, mode=kb.MODE_CORRECT)]
    try:
        for ix in handles:
            with pytest.raises(kb.KmerB200Error) as err:
                ix.attach_records([0, 10, ix.n])
            assert err.value.code == -5
    finally:
        for ix in handles:
            ix.close()
    if torch.cuda.device_count() >= 2:
        with kb.KmerIndex(text, 4, [12], devices=[0, 1]) as multi:
            with pytest.raises(kb.KmerB200Error) as err:
                multi.attach_records(starts)
            assert err.value.code == -5
