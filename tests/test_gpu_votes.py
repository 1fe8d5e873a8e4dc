"""Record votes on the device (KmerIndex.record_votes and record_votes_batch_device) against the numpy ground truth of
tests/votes_truth.py, bit for bit: offsets, records, votes, k-mer hits and status. Covers both sides of the per-read
shared-memory table: reads whose records fit it and reads whose records overflow it into the global-memory path."""
import os
import subprocess
import sys

import numpy as np
import pytest

from collection_truth import random_starts
from conftest import ROOT
from test_gpu_seeds import concat, on_device, seed_batch
from votes_truth import assert_votes_equal, votes_truth

pytestmark = pytest.mark.gpu
CAPACITY = 384   # kVoteCapacity: distinct records a read's shared-memory table holds


@pytest.fixture(scope="module")
def kb():
    import kmer_index_b200
    return kmer_index_b200


def device_arrays(r, Q):
    import torch
    dev = torch.device("cuda", 0)
    torch.cuda.synchronize()
    o = torch.as_tensor(r.offsets(), device=dev).cpu().numpy().astype(np.uint64)
    st = torch.as_tensor(r.status(), device=dev).cpu().numpy() if Q else np.zeros(0, np.uint8)
    h = torch.as_tensor(r.kmer_hits(), device=dev).cpu().numpy().view(np.uint32) if Q else np.zeros(0, np.uint32)
    if r.n_positions:
        rec = torch.as_tensor(r.positions(), device=dev).cpu().numpy().view(np.uint32)
        v = torch.as_tensor(r.votes(), device=dev).cpu().numpy().view(np.uint32)
    else:
        assert r.votes() is not None
        rec = v = np.zeros(0, np.uint32)
    return o, rec, v, h, st


def check_forms(ix, q, off, k, max_occ, min_votes, want, label, device=True):
    r = ix.record_votes(q, off, k=k, max_occ=max_occ, min_votes=min_votes)
    assert_votes_equal((r.offsets, r.records, r.votes, r.kmer_hits, r.status), want, label=f"{label} host")
    if not device:
        return r
    Q = off.size - 1
    d_q, d_off = on_device(q, off)
    max_len = int(np.diff(off.astype(np.int64)).max(initial=1))
    dr = ix.record_votes_batch_device(d_q.data_ptr(), d_off.data_ptr(), Q, max_len, k=k, max_occ=max_occ, min_votes=min_votes)
    assert_votes_equal(device_arrays(dr, Q), want, label=f"{label} device")
    dr.free()
    return r


def junction_reads(text, starts, every=7, half=30):
    s = starts.astype(np.int64)
    js = [int(x) for x in s[1:-1:every] if half < x < text.size - half]
    q = np.concatenate([text[x - half:x + half] for x in js]).astype(np.uint8)
    return q, np.arange(len(js) + 1, dtype=np.uint64) * np.uint64(2 * half)


def overflow_launches(ix):
    return ix.stats().get("votes_overflow", {}).get("launches", 0)


SHAPES = {"dna4_k12": (4, 12, {}), "dna4_k16_sparse": (4, 16, {"directory_bits": 12}), "dna5_k17": (5, 17, {}),
          "aa27_k7": (27, 7, {})}


@pytest.mark.parametrize("shape", list(SHAPES))
def test_votes_match_truth(kb, shape):
    """Dense and sparse directories, 32- and 64-bit keys; random collections with short and empty records, reads planted
    inside records and across junctions, a repeat whose buckets span many records."""
    from kmer_index_b200 import synth
    sigma, k, kw = SHAPES[shape]
    n = 120_000
    text = synth.random_text(n, sigma, 7 + sigma + k)
    rng = np.random.default_rng(k)
    for x in range(30_000, 60_000, 600):               # one block copied into 50 places: k-mers in many records
        text[x:x + 200] = text[10_000:10_200]
    starts = random_starts(n, 400, rng, short=40)
    q, off = concat(seed_batch(text, sigma, k, 3 * k, Q=300), junction_reads(text, starts))
    with kb.KmerIndex(text, sigma, [k], mode=kb.MODE_CORRECT, **kw) as ix:
        if "directory_bits" in kw:
            assert ix.element_info(0).directory_shift > 0
        ix.attach_records(starts)
        for max_occ in (0, 5, 10 ** 6):
            for min_votes in (1, 2):
                want = votes_truth(text, sigma, k, q, off, starts, max_occ, min_votes)
                if max_occ == 0 and min_votes == 1:
                    assert np.diff(want[0].astype(np.int64)).max() > 20
                check_forms(ix, q, off, k, max_occ, min_votes, want, f"{shape} max_occ={max_occ} min_votes={min_votes}",
                            device=min_votes == 1)
        assert overflow_launches(ix) == 0
        other = ix.search_approx(q, off, 1)
        assert other.records is None and other.votes is None and other.kmer_hits is None


def test_overflow_path(kb):
    """3000 copies of one record plus noise: the reads of that record hit more records than the table holds and take the
    global-memory path, interleaved in one batch with reads that do not. Exact either way."""
    from kmer_index_b200 import synth
    sigma, k, L, copies = 4, 14, 80, 3000
    rec = synth.random_text(L, sigma, 5)
    rng = np.random.default_rng(6)
    parts = []
    for c in range(copies):
        parts.append(rec.copy())
        if c % 10 == 0:
            parts.append(rng.integers(0, sigma, int(rng.integers(0, 50))).astype(np.uint8))   # noise records, some empty
    parts.append(synth.random_text(100_000, sigma, 7))
    text = np.concatenate(parts).astype(np.uint8)
    starts = np.concatenate([[0], np.cumsum([p.size for p in parts])]).astype(np.uint64)
    qs = []
    for i in range(60):
        if i % 3 == 0:
            s = int(rng.integers(0, L - 40))
            qs.append(rec[s:s + int(rng.integers(k, L - s + 1))])                # overflows
        elif i % 3 == 1:
            s = int(rng.integers(starts[-2], text.size - 200))
            qs.append(text[s:s + 150])                                          # one record
        else:
            qs.append(np.concatenate([rec[-30:], text[int(starts[-2]):int(starts[-2]) + 40]]))   # both
    off = np.zeros(len(qs) + 1, dtype=np.uint64)
    np.cumsum([x.size for x in qs], out=off[1:])
    q = np.concatenate(qs).astype(np.uint8)
    with kb.KmerIndex(text, sigma, [k], mode=kb.MODE_CORRECT) as ix:
        ix.attach_records(starts)
        for max_occ, min_votes in ((0, 1), (0, 3), (10 ** 5, 1), (2000, 1), (0, 10 ** 6)):
            ix.stats_reset()
            want = votes_truth(text, sigma, k, q, off, starts, max_occ, min_votes)
            r = check_forms(ix, q, off, k, max_occ, min_votes, want, f"overflow max_occ={max_occ} min_votes={min_votes}")
            if max_occ != 2000:
                assert overflow_launches(ix) > 0
                if min_votes == 1:
                    assert np.diff(want[0].astype(np.int64)).max() >= copies > CAPACITY
            else:
                assert overflow_launches(ix) == 0      # the cap drops the repeated k-mers before they vote
        best, v1, v2 = r.best()
        assert np.array_equal(best >= 0, np.diff(r.offsets.astype(np.int64)) > 0)


def test_long_read_and_long_buckets(kb):
    from kmer_index_b200 import synth
    sigma, k, n = 4, 16, 600_000
    text = synth.random_text(n, sigma, 61)
    text[100_000:200_000] = 2                          # a bucket of ~1e5 positions
    rng = np.random.default_rng(63)
    starts = random_starts(n, 500, rng, short=20)
    qs = [text[150_000:150_040], text[5_000:25_000], synth.random_text(10 ** 6, sigma, 64)]
    qs[-1][500_000:500_200] = 2
    qs[-1][700_000:702_000] = text[300_000:302_000]
    q = np.concatenate(qs).astype(np.uint8)
    off = np.zeros(len(qs) + 1, dtype=np.uint64)
    np.cumsum([x.size for x in qs], out=off[1:])
    with kb.KmerIndex(text, sigma, [k], mode=kb.MODE_CORRECT) as ix:
        ix.attach_records(starts)
        cut = ix.occurrence_cutoff(0.0002)
        assert 1 <= cut < 10 ** 5
        for max_occ in (0, 100, cut):
            want = votes_truth(text, sigma, k, q, off, starts, max_occ)
            check_forms(ix, q, off, k, max_occ, 1, want, f"long max_occ={max_occ}")


def test_agrees_with_seeds_and_locate(kb):
    """A larger batch: the votes equal the GPU's own seeds() + locate() tallied in numpy."""
    from kmer_index_b200 import synth
    sigma, k, n = 4, 15, 2_000_000
    text = synth.random_text(n, sigma, 81)
    for x in range(1_000_000, 1_400_000, 4000):
        text[x:x + 500] = text[:500]
    rng = np.random.default_rng(82)
    starts = random_starts(n, 5000, rng, short=100)
    q, off = seed_batch(text, sigma, k, 83, Q=20_000, m_hi=150)
    with kb.KmerIndex(text, sigma, [k], mode=kb.MODE_CORRECT) as ix:
        ix.attach_records(starts)
        s = ix.seeds(q, off, k=k, max_occ=200)
        rec, _ = ix.locate(s.positions)
        Q = off.size - 1
        qid = np.repeat(np.arange(Q), np.diff(s.offsets.astype(np.int64)))
        trip = np.unique(np.stack([qid, s.seed_offsets.astype(np.int64), rec.astype(np.int64)]), axis=1)
        pairs, votes = np.unique(trip[[0, 2]], axis=1, return_counts=True)
        order = np.lexsort((pairs[1], -votes, pairs[0]))
        r = ix.record_votes(q, off, k=k, max_occ=200)
        assert np.array_equal(r.records, pairs[1][order]) and np.array_equal(r.votes, votes[order])
        assert np.array_equal(np.diff(r.offsets.astype(np.int64)), np.bincount(pairs[0], minlength=Q))


def test_adopted_key_range_parts(kb):
    import torch
    from kmer_index_b200 import sharded, synth
    sigma, n, k, parts = 4, 200_000, 12, 4
    text = synth.random_text(n, sigma, 71)
    text[20_000:40_000] = 0
    starts = random_starts(n, 300, np.random.default_rng(72), short=20)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream().cuda_stream
    idx = [kb.KmerIndex(text, sigma, [k], key_part=r, key_parts=parts, stream=stream or None, mode=kb.MODE_CORRECT)
           for r in range(parts)]
    try:
        q, off = seed_batch(text, sigma, k, 73)
        with pytest.raises(kb.KmerB200Error) as err:
            idx[0].record_votes(q, off, k=k)             # not adopted yet
        assert err.value.code == -5
        ps = [ix.element_part(0) for ix in idx]
        bufs, first = [], [0]
        dir_full = torch.empty(sigma ** k + 1, dtype=torch.int32, device=dev)
        for r, (ix, p) in enumerate(zip(idx, ps)):
            buf = torch.empty(max(p.n_kmers, 1), dtype=torch.int32, device=dev)
            if p.n_kmers:
                buf[:p.n_kmers].copy_(sharded._dev_view(p.d_positions, p.n_kmers, dev))
            bufs.append(buf)
            n_dir = p.key_hi - p.key_lo + (1 if r == parts - 1 else 0)
            ix.export_directory(0, first[-1], n_dir, dir_full.data_ptr() + 4 * p.key_lo)
            first.append(first[-1] + p.n_kmers)
        torch.cuda.synchronize()
        idx[0].adopt_element_parts(0, bufs, first, dir_full)
        idx[0].attach_records(starts)
        for max_occ in (0, 5):
            want = votes_truth(text, sigma, k, q, off, starts, max_occ)
            check_forms(idx[0], q, off, k, max_occ, 1, want, f"parts max_occ={max_occ}", device=False)
    finally:
        for ix in idx:
            ix.close()


def test_refusals(kb):
    import torch
    from kmer_index_b200 import synth
    n = 100_000
    text = synth.random_text(n, 4, 81)
    starts = random_starts(n, 50, np.random.default_rng(3), short=5)
    q, off = seed_batch(text, 4, 12, 82, Q=30)
    with kb.KmerIndex(text, 4, [10, 12], mode=kb.MODE_CORRECT) as ix:
        with pytest.raises(kb.KmerB200Error) as err:
            ix.record_votes(q, off, k=12)                # no records
        assert err.value.code == -1
        ix.attach_records(starts)
        for k in (11, 13, 0):
            with pytest.raises(kb.KmerB200Error) as err:
                ix.record_votes(q, off, k=k)
            assert err.value.code == -1
        ix.search_batch(q[:5], np.array([0, 5], np.uint64))   # an auxiliary k' = 5 element
        with pytest.raises(kb.KmerB200Error) as err:
            ix.record_votes(q, off, k=5)
        assert err.value.code == -1
        with pytest.raises(kb.KmerB200Error) as err:
            ix.record_votes(q, off, k=12, min_votes=0)
        assert err.value.code == -1
        with pytest.raises(ValueError):
            ix.record_votes(q, off)                      # several ks: k is needed
        bad = q.copy()
        bad[int(off[3]) + 2] = 4
        with pytest.raises(kb.KmerB200Error) as err:
            ix.record_votes(bad, off, k=12)
        assert err.value.code == -4
        short = np.array([0, 9, 1], np.uint8)            # shorter than k, still checked
        with pytest.raises(kb.KmerB200Error) as err:
            ix.record_votes(short, np.array([0, 3], np.uint64), k=12)
        assert err.value.code == -4
        import ctypes
        r = ctypes.c_void_p()
        assert ix._L.kmer_b200_record_votes(ix.handle, None, None, 0, 12, 0, 1, ctypes.byref(r)) == -1
        assert ix._L.kmer_b200_record_votes_device(ix.handle, None, None, 0, 0, 12, 0, 1, None) == -1
        want = votes_truth(text, 4, 12, q, off, starts)
        check_forms(ix, q, off, 12, 0, 1, want, "usable after refusals")
        empty = ix.record_votes(np.zeros(0, np.uint8), np.zeros(1, np.uint64), k=12)
        assert empty.offsets.tolist() == [0] and empty.records.size == 0 and empty.kmer_hits.size == 0
    sh = kb.KmerIndex(text[:60_063], 4, [12], shard_begin=0, n_total=n, halo=63, mode=kb.MODE_CORRECT)
    try:
        with pytest.raises(kb.KmerB200Error) as err:
            sh.record_votes(q, off, k=12)
        assert err.value.code in (-1, -5)
    finally:
        sh.close()
    if torch.cuda.device_count() >= 2:
        with kb.KmerIndex(text, 4, [12], devices=[0, 1]) as multi:
            with pytest.raises(kb.KmerB200Error) as err:
                multi.record_votes(q, off)
            assert err.value.code == -5


GUARD_CASE = r"""
import numpy as np
import kmer_index_b200 as kb
from kmer_index_b200 import synth
import sys
sys.path.insert(0, "tests")
from votes_truth import votes_truth
from collection_truth import random_starts
from test_gpu_seeds import seed_batch
rec = synth.random_text(70, 4, 90)
text = np.concatenate([np.tile(rec, 600), synth.random_text(200_000, 4, 91)]).astype(np.uint8)
starts = np.concatenate([np.arange(0, 600 * 70, 70), random_starts(200_000, 100, np.random.default_rng(92), short=10)[:] + 600 * 70]).astype(np.uint64)
q, off = seed_batch(text, 4, 14, 93, Q=500)
q = np.concatenate([q, rec[:60], text[50_000:62_000]]).astype(np.uint8)
off = np.append(off, [off[-1] + np.uint64(60), off[-1] + np.uint64(12_060)]).astype(np.uint64)
with kb.KmerIndex(text, 4, [14], mode=kb.MODE_CORRECT) as ix:
    ix.attach_records(starts)
    for max_occ, min_votes in ((0, 1), (7, 1), (0, 2)):
        r = ix.record_votes(q, off, k=14, max_occ=max_occ, min_votes=min_votes)
        want = votes_truth(text, 4, 14, q, off, starts, max_occ, min_votes)
        assert np.array_equal(r.offsets, want[0]) and np.array_equal(r.records, want[1]) and np.array_equal(r.votes, want[2])
        assert np.array_equal(r.kmer_hits, want[3])
    assert ix.stats()["votes_overflow"]["launches"] > 0
print("guard violations", kb.guard_violations())
"""


def test_vote_kernels_under_guarded_allocations(tmp_path):
    env = dict(os.environ, KMER_B200_GUARD="1")
    out = subprocess.run([sys.executable, "-c", GUARD_CASE], capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "guard violations 0" in out.stdout, out.stdout[-2000:]
