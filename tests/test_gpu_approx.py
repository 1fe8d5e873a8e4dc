"""Approximate search (kmer_b200_search_approx_batch and its device forms) on the GPU, bit for bit against the ground
truth of a window-by-window scan (tests/approx_truth)."""
import numpy as np
import pytest

from approx_truth import truth_approx
from conftest import assert_results_equal

pytestmark = pytest.mark.gpu

BUDGETS = [0, 1, 2, 3, 5, 8]
SHAPES = {"dna4_k12": (4, [12]), "dna4_k16": (4, [16]), "dna4_multi": (4, [5, 7, 9, 11, 13]), "dna15_k8": (15, [8]),
          "aa27_k5": (27, [5]), "dna5_k20": (5, [20]), "dna4_k31": (4, [31])}


@pytest.fixture(scope="module")
def kb():
    import kmer_index_b200
    return kmer_index_b200


def plant(text, Q, m_lo, m_hi, d_max, sigma, seed):
    """Q text windows (lengths m_lo..m_hi) with exactly d substitutions each, d cycling through 0..d_max (at most the
    window length); every 7th window starts at 0, every 7th + 1 ends at n. Returns (ranks, offsets, origins, d)."""
    rng = np.random.default_rng(seed)
    n = text.size
    lens = np.minimum(rng.integers(m_lo, m_hi + 1, Q), n)
    off = np.zeros(Q + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    ranks = np.empty(int(off[-1]), dtype=np.uint8)
    origins = np.empty(Q, dtype=np.int64)
    ds = np.empty(Q, dtype=np.int64)
    for i in range(Q):
        m = int(lens[i])
        start = 0 if i % 7 == 0 else (n - m if i % 7 == 1 else int(rng.integers(0, n - m + 1)))
        w = text[start:start + m].copy()
        d = min(i % (d_max + 1), m)
        for j in rng.choice(m, size=d, replace=False):
            w[j] = (int(w[j]) + int(rng.integers(1, sigma))) % sigma
        ranks[int(off[i]):int(off[i + 1])] = w
        origins[i], ds[i] = start, d
    return ranks, off, origins, ds


def concat(*batches):
    """(ranks, offsets) of several batches back to back."""
    qs = [np.asarray(q, dtype=np.uint8) for q, _ in batches]
    lens = np.concatenate([np.diff(np.asarray(o, dtype=np.uint64)) for _, o in batches]).astype(np.uint64)
    off = np.zeros(lens.size + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    return np.concatenate(qs), off


def mixed_batch(text, sigma, e, seed, Q=400, m_hi=150):
    """random / text-sampled / low-period queries of 1..m_hi symbols plus windows with 0..e+1 planted substitutions"""
    from kmer_index_b200 import synth
    q1, o1 = synth.stress_queries(text, Q, 1, m_hi, sigma, seed)
    q2, o2, origins, ds = plant(text, Q, 1, m_hi, e + 1, sigma, seed + 1)
    q, off = concat((q1, o1), (q2, o2))
    return q, off, Q, origins, ds


def check_planted(res, first, origins, ds, e):
    """planted window i (query first + i) is found at its origin exactly when it carries <= e substitutions"""
    offs, pos = res[0], res[1]
    for i in range(origins.size):
        hits = pos[int(offs[first + i]):int(offs[first + i + 1])]
        assert (int(origins[i]) in hits) == (ds[i] <= e), (i, int(ds[i]), e)


def device_results(kb, ix, q, off, e, max_len=None):
    """(full result, count-only result) of the device entry points, as host arrays"""
    import torch
    dev = torch.device("cuda", 0)
    d_q = torch.from_numpy(q if q.size else np.zeros(1, np.uint8)).to(dev)
    d_off = torch.from_numpy(off.view(np.int64)).to(dev)
    Q = off.size - 1
    max_len = max_len if max_len is not None else int(np.diff(off).max(initial=1))
    torch.cuda.synchronize()
    out = []
    for fn in (ix.search_approx_batch_device, ix.count_approx_batch_device):
        r = fn(d_q.data_ptr(), d_off.data_ptr(), Q, max_len, e)
        torch.cuda.synchronize()
        o = torch.as_tensor(r.offsets(), device=dev).cpu().numpy().astype(np.uint64)
        p = (torch.as_tensor(r.positions(), device=dev).cpu().numpy().view(np.uint32) if r.n_positions and r.positions_ptr
             else np.zeros(0, np.uint32))
        st = torch.as_tensor(r.status(), device=dev).cpu().numpy() if Q else np.zeros(0, np.uint8)
        r.free()
        out.append((o, p, st))
    return out


@pytest.mark.parametrize("shape", list(SHAPES))
def test_approx_matches_ground_truth(kb, shape):
    """Every budget, random and planted queries of 1..150 symbols (bucket seeds and prefix-slab seeds, windows at 0 and
    ending at n); e = 0 is CORRECT-mode exact search."""
    from kmer_index_b200 import synth
    sigma, ks = SHAPES[shape]
    text = synth.random_text(60_000, sigma, 31 + sigma)
    with kb.KmerIndex(text, sigma, ks) as ix:
        for e in BUDGETS:
            q, off, Q, origins, ds = mixed_batch(text, sigma, e, 100 + e)
            want = truth_approx(text, q, off, e)
            got = ix.search_approx(q, off, e).as_tuple()
            assert_results_equal(got, want, label=f"{shape} e={e}")
            check_planted(got, Q, origins, ds, e)
            if e == 0:
                assert_results_equal(got, ix.search_batch(q, off, mode=kb.MODE_CORRECT).as_tuple(), label=f"{shape} e=0 vs exact")


@pytest.mark.parametrize("shape", ["dna4_k12", "dna4_multi", "aa27_k5"])
def test_device_entry_points_and_count_only(kb, shape):
    from kmer_index_b200 import synth
    sigma, ks = SHAPES[shape]
    text = synth.random_text(50_000, sigma, 41)
    with kb.KmerIndex(text, sigma, ks) as ix:
        for e in (0, 2, 5):
            q, off, _, _, _ = mixed_batch(text, sigma, e, 200 + e, Q=300)
            host = ix.search_approx(q, off, e).as_tuple()
            full, count = device_results(kb, ix, q, off, e)
            assert_results_equal(full, host, label=f"device {shape} e={e}")
            assert np.array_equal(count[0], host[0]) and np.array_equal(count[2], host[2])
            assert_results_equal(host, truth_approx(text, q, off, e), label=f"host {shape} e={e}")


def test_same_result_once_auxiliary_elements_exist(kb):
    """Exact sub-k searches build auxiliary k' = m elements; approximate seeds then come from them instead of slabs."""
    from kmer_index_b200 import synth
    text = synth.random_text(80_000, 4, 51)
    with kb.KmerIndex(text, 4, [12], mode=kb.MODE_CORRECT) as ix:
        for e in (1, 3, 8):
            q, off, _, _, _ = mixed_batch(text, 4, e, 300 + e, Q=300, m_hi=60)
            want = truth_approx(text, q, off, e)
            assert_results_equal(ix.search_approx(q, off, e).as_tuple(), want, label=f"before aux e={e}")
            short, s_off = synth.stress_queries(text, 400, 1, 11, 4, 310 + e)
            ix.search_batch(short, s_off)     # builds the auxiliary elements of lengths 1..11
            assert_results_equal(ix.search_approx(q, off, e).as_tuple(), want, label=f"after aux e={e}")


@pytest.mark.parametrize("sigma,ks", [(4, [12]), (4, [5, 7, 9, 11, 13]), (15, [8])])
def test_heavy_candidate_lists_take_the_warp_path(kb, sigma, ks):
    """Constant runs make buckets of ~70 000 candidates: those queries go to the warp-per-query launch."""
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
            want = truth_approx(text, q, off, e)
            for attempt in range(2):
                assert_results_equal(ix.search_approx(q, off, e).as_tuple(), want, label=f"heavy {ks} e={e}/{attempt}")
            assert int(np.diff(want[0]).max()) > 2048


def test_sparse_directory_save_load_and_position_parts(kb, tmp_path):
    import torch

    from kmer_index_b200 import sharded, synth
    sigma, n = 4, 200_000
    text = synth.random_text(n, sigma, 61)
    text[5000:8000] = 0
    q, off, _, _, _ = mixed_batch(text, sigma, 3, 400, Q=300)
    want = {e: truth_approx(text, q, off, e) for e in (0, 3)}
    with kb.KmerIndex(text, sigma, [12], directory_bits=12) as ix:
        assert ix.element_info(0).directory_shift > 0
        for e in (0, 3):
            assert_results_equal(ix.search_approx(q, off, e).as_tuple(), want[e], label=f"sparse e={e}")
        path = str(tmp_path / "index.kmerb200")
        ix.save(path)
    with kb.KmerIndex.load(path) as ld:
        for e in (0, 3):
            assert_results_equal(ld.search_approx(q, off, e).as_tuple(), want[e], label=f"loaded e={e}")
    # peer-positions index emulated on one GPU: the directory whole, the positions left in the key-range parts
    dev = torch.device("cuda", 0)
    for ks, parts in (([12], 4), ([5, 7, 9, 11, 13], 3)):
        stream = torch.cuda.current_stream().cuda_stream
        idx = [kb.KmerIndex(text, sigma, ks, key_part=r, key_parts=parts, stream=stream or None) for r in range(parts)]
        try:
            with pytest.raises(kb.KmerB200Error):
                idx[0].search_approx(q, off, 1)                  # a key-range part that has not been adopted
            assert len(idx[0].search_batch(q, off)) == off.size - 1  # still answers exact search (its own part's hits)
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
                assert_results_equal(idx[0].search_approx(q, off, e).as_tuple(), want[e], label=f"parts {ks} e={e}")
        finally:
            for ix in idx:
                ix.close()


def test_edge_cases(kb):
    from kmer_index_b200 import synth
    text = synth.random_text(5_000, 4, 71)
    n = text.size
    with kb.KmerIndex(text, 4, [10]) as ix:
        empty = ix.search_approx(np.zeros(0, np.uint8), np.zeros(1, np.uint64), 2)
        assert len(empty) == 0 and empty.offsets.tolist() == [0] and empty.positions.size == 0
        qs = [np.zeros(0, np.uint8), text[:2].copy(), text[:3].copy(), text[-4:].copy(), synth.random_text(n + 1, 4, 72),
              text.copy(), text[-37:].copy()]
        lens = np.array([x.size for x in qs], dtype=np.uint64)
        off = np.zeros(lens.size + 1, dtype=np.uint64)
        np.cumsum(lens, out=off[1:])
        q = np.concatenate(qs)
        for e in (0, 3, 8):
            got = ix.search_approx(q, off, e)
            assert_results_equal(got.as_tuple(), truth_approx(text, q, off, e), label=f"edges e={e}")
            assert got.status[0] == kb.QUERY_UNDEFINED and got.to_vector(0).size == 0
            for i, x in enumerate(qs[1:4], start=1):            # m <= e: every window 0 .. n - m
                if x.size <= e:
                    assert np.array_equal(got.to_vector(i), np.arange(n - x.size + 1, dtype=np.uint32))
            assert got.to_vector(4).size == 0                  # m > n
            assert got.to_vector(5).tolist() == [0]            # the whole text
        with pytest.raises(kb.KmerB200Error) as err:
            ix.search_approx(q, off, 9)
        assert err.value.code == -1
        bad = q.copy()
        bad[3] = 4
        with pytest.raises(kb.KmerB200Error) as err:
            ix.search_approx(bad, off, 1)
        assert err.value.code == -4
        assert ix.search_approx(q, off, 1).status[0] == kb.QUERY_UNDEFINED   # the handle is still usable


def test_unsupported_handles_refuse_and_stay_usable(kb, oracle_mod):
    from kmer_index_b200 import synth
    n = 200_000
    text = synth.random_text(n, 4, 81)
    q, off = synth.stress_queries(text[:100_000], 200, 10, 40, 4, 82)
    want = oracle_mod.Oracle.truth(text[:100_000], q, off)
    handles = [kb.KmerIndex(text[:100_000], 4, [10, 12], shared_positions=True, mode=kb.MODE_CORRECT),
               kb.KmerIndex(text[:100_063], 4, [12], shard_begin=0, n_total=n, halo=63, mode=kb.MODE_CORRECT)]
    try:
        for ix in handles:
            with pytest.raises(kb.KmerB200Error) as err:
                ix.search_approx(q, off, 1)
            assert err.value.code == -5
            got = ix.search_batch(q, off).as_tuple()
            if ix is handles[0]:
                assert_results_equal(got, want, label="shared positions after refusal")
            else:
                assert got[1].size > 0
    finally:
        for ix in handles:
            ix.close()


def test_large_planted_reads(kb):
    """50 Mbp dna4, 10^5 reads of 100 symbols with 0..3 substitutions, e = 3: every read finds its origin, every hit is
    re-verified on the host, count-only equals the full result."""
    from kmer_index_b200 import synth
    n, Q, m, e = 50_000_000, 100_000, 100, 3
    text = synth.random_text(n, 4, 91)
    rng = np.random.default_rng(92)
    origins = rng.integers(0, n - m + 1, Q)
    ds = np.arange(Q) % (e + 1)
    reads = text[origins[:, None] + np.arange(m)]
    for i in range(Q):
        cols = rng.choice(m, size=int(ds[i]), replace=False)
        reads[i, cols] = (reads[i, cols] + rng.integers(1, 4, cols.size)) % 4
    q = reads.reshape(-1).astype(np.uint8)
    off = (np.arange(Q + 1, dtype=np.uint64) * m)
    with kb.KmerIndex(text, 4, [16]) as ix:
        got = ix.search_approx(q, off, e)
        counts = np.diff(got.offsets).astype(np.int64)
        assert np.all(got.status == 0) and np.all(counts >= 1)
        qid = np.repeat(np.arange(Q), counts)
        for i in range(Q):
            seg = got.positions[int(got.offsets[i]):int(got.offsets[i + 1])]
            assert np.all(seg[1:] > seg[:-1]) and origins[i] in seg, i
        win = text[got.positions.astype(np.int64)[:, None] + np.arange(m)]
        assert np.all((win != reads[qid]).sum(axis=1) <= e)
        full, count = device_results(kb, ix, q, off, e, max_len=m)
        assert np.array_equal(count[0], got.offsets) and np.array_equal(full[1], got.positions)
