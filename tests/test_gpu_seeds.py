"""k-mer seeding on the device (KmerIndex.seeds and its device and count-only forms) against the numpy ground truth of
tests/seeds_truth.py, bit for bit: offsets, positions, status, seed offsets and k-mer counts."""
import os
import subprocess
import sys

import numpy as np
import pytest

from collection_truth import random_starts
from conftest import ROOT
from seeds_truth import assert_seeds_equal, query_kmers, seeds_truth
from test_seeds_cpu import SHAPES

pytestmark = pytest.mark.gpu
MAX_OCCS = (0, 1, 5, 10 ** 6)


@pytest.fixture(scope="module")
def kb():
    import kmer_index_b200
    return kmer_index_b200


def concat(*batches):
    qs = [q for q, _ in batches]
    lens = np.concatenate([np.diff(o.astype(np.int64)) for _, o in batches])
    off = np.zeros(lens.size + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    return np.concatenate(qs).astype(np.uint8), off


def seed_batch(text, sigma, k, seed, Q=240, m_hi=300):
    """Text windows (at 0, ending at n, anywhere), random reads, queries of 0 .. k - 1 symbols, reads up to m_hi symbols."""
    rng = np.random.default_rng(seed)
    n = text.size
    qs = []
    for i in range(Q):
        kind = i % 6
        m = int(rng.integers(k, m_hi + 1))
        if kind == 0:
            qs.append(text[:m])
        elif kind == 1:
            qs.append(text[n - m:])
        elif kind in (2, 3):
            s = int(rng.integers(0, n - m + 1))
            qs.append(text[s:s + m])
        elif kind == 4:
            qs.append(rng.integers(0, sigma, m).astype(np.uint8))
        else:
            qs.append(text[int(rng.integers(0, n - k)):][:i % k])   # 0 .. k - 1 symbols
    off = np.zeros(Q + 1, dtype=np.uint64)
    np.cumsum([x.size for x in qs], out=off[1:])
    return np.concatenate(qs).astype(np.uint8), off


def on_device(q, off):
    import torch
    dev = torch.device("cuda", 0)
    d_q = torch.from_numpy(q if q.size else np.zeros(1, np.uint8)).to(dev)
    d_off = torch.from_numpy(off.view(np.int64)).to(dev)
    torch.cuda.synchronize()
    return d_q, d_off


def host_arrays(r, Q, full=True):
    import torch
    dev = torch.device("cuda", 0)
    torch.cuda.synchronize()
    o = torch.as_tensor(r.offsets(), device=dev).cpu().numpy().astype(np.uint64)
    st = torch.as_tensor(r.status(), device=dev).cpu().numpy() if Q else np.zeros(0, np.uint8)
    kc = r.kmer_counts()
    kc = torch.as_tensor(kc, device=dev).cpu().numpy().view(np.uint32) if kc is not None and kc.__cuda_array_interface__["shape"][0] \
        else np.zeros(0, np.uint32)
    if not full:
        assert r.positions_ptr == 0 and r.seed_offsets() is None
        return o, st, kc
    p = torch.as_tensor(r.positions(), device=dev).cpu().numpy().view(np.uint32) if r.n_positions else np.zeros(0, np.uint32)
    j = torch.as_tensor(r.seed_offsets(), device=dev).cpu().numpy().view(np.uint32) if r.n_positions else np.zeros(0, np.uint32)
    return o, p, st, j, kc


def check_all_forms(ix, q, off, k, max_occ, want, label, device=True):
    """host, device and count-only forms against `want`"""
    r = ix.seeds(q, off, k=k, max_occ=max_occ)
    assert_seeds_equal((r.offsets, r.positions, r.status, r.seed_offsets, r.kmer_counts), want, label=f"{label} host")
    if not device:
        return
    Q = off.size - 1
    d_q, d_off = on_device(q, off)
    max_len = int(np.diff(off.astype(np.int64)).max(initial=1))
    full = ix.seeds_batch_device(d_q.data_ptr(), d_off.data_ptr(), Q, max_len, k=k, max_occ=max_occ)
    assert_seeds_equal(host_arrays(full, Q), want, label=f"{label} device")
    full.free()
    cnt = ix.count_seeds_batch_device(d_q.data_ptr(), d_off.data_ptr(), Q, max_len, k=k, max_occ=max_occ)
    o, st, kc = host_arrays(cnt, Q, full=False)
    cnt.free()
    assert_seeds_equal((o, st, kc), (want[0], want[2], want[4]), label=f"{label} count-only")


@pytest.mark.parametrize("shape", list(SHAPES))
def test_seeds_match_truth(kb, shape):
    """Every shape (dense and sparse directories, 32- and 64-bit keys, the two-window dna5 k = 20), every k of the
    multi-k index, every cap; and the seeds equal CORRECT-mode exact search of the batch's k-mers cut out as queries."""
    from kmer_index_b200 import synth
    sigma, ks = SHAPES[shape]
    text = synth.random_text(60_000, sigma, 31 + sigma)
    text[1000:1400] = 1 % sigma                       # a repeat: buckets of hundreds
    with kb.KmerIndex(text, sigma, ks) as ix, kb.KmerIndex(text, sigma, ks, directory_bits=10) as sparse:
        assert sparse.element_info(0).directory_shift > 0 or sigma ** min(ks) <= 1 << 10
        for k in ks:
            q, off = seed_batch(text, sigma, k, 100 + k)
            for max_occ in MAX_OCCS:
                want = seeds_truth(text, sigma, k, q, off, max_occ)
                check_all_forms(ix, q, off, k, max_occ, want, f"{shape} k={k} max_occ={max_occ}", device=k == ks[-1])
                if max_occ in (0, 5):
                    check_all_forms(sparse, q, off, k, max_occ, want, f"{shape} sparse k={k} max_occ={max_occ}", device=False)
            # the workaround: every k-mer as a query of its own through exact search
            _, qid, j = query_kmers(q, off, k, sigma)
            starts = off[:-1].astype(np.int64)[qid] + j
            kq = (q[starts[:, None] + np.arange(k)].reshape(-1) if starts.size else np.zeros(0, np.uint8))
            koff = np.arange(starts.size + 1, dtype=np.uint64) * np.uint64(k)
            exact = ix.search_batch(kq, koff, mode=kb.MODE_CORRECT)
            seeds = ix.seeds(q, off, k=k)
            assert np.array_equal(exact.positions, seeds.positions), f"{shape} k={k}: seeds != exact search of the k-mers"
            assert np.array_equal(np.diff(exact.offsets.astype(np.int64)), seeds.kmer_counts.astype(np.int64))


def test_collection_seeds(kb):
    import torch
    from kmer_index_b200 import synth
    sigma, k, n = 4, 12, 200_000
    text = synth.random_text(n, sigma, 51)
    rng = np.random.default_rng(52)
    starts = random_starts(n, 300, rng, short=30)
    q, off = seed_batch(text, sigma, k, 53, Q=400)
    # reads across every tenth junction: their k-mers that span it count only inside one record
    s = starts.astype(np.int64)
    junctions = [int(x) for x in s[1:-1:10] if 40 < x < n - 40]
    jq = np.concatenate([text[x - 30:x + 30] for x in junctions]).astype(np.uint8)
    joff = np.arange(len(junctions) + 1, dtype=np.uint64) * np.uint64(60)
    q, off = concat((q, off), (jq, joff))
    with kb.KmerIndex(text, sigma, [k], mode=kb.MODE_CORRECT) as ix:
        ix.attach_records(starts)
        for max_occ in MAX_OCCS:
            want = seeds_truth(text, sigma, k, q, off, max_occ, starts=starts)
            check_all_forms(ix, q, off, k, max_occ, want, f"collection max_occ={max_occ}")
        r = ix.seeds(q, off, k=k)
        p = r.positions.astype(np.int64)
        assert not np.any((s[None, :] > p[:, None]) & (s[None, :] < p[:, None] + k))
        # a junction k-mer: the in-record count, below the whole-text count
        plain = seeds_truth(text, sigma, k, q, off)
        assert np.all(r.kmer_counts <= plain[4]) and np.any(r.kmer_counts < plain[4])
        # planted reads inside records: locate_device puts the hit of each k-mer at its own place in the read's record
        planted = [(r_, int((s[r_ + 1] - s[r_]) // 3)) for r_ in range(s.size - 1) if s[r_ + 1] - s[r_] >= 100][:50]
        pq = np.concatenate([text[s[r_] + o:s[r_] + o + 60] for r_, o in planted]).astype(np.uint8)
        poff = np.arange(len(planted) + 1, dtype=np.uint64) * np.uint64(60)
        d_q, d_off = on_device(pq, poff)
        full = ix.seeds_batch_device(d_q.data_ptr(), d_off.data_ptr(), len(planted), 60, k=k)
        o_, p_, _, j_, _ = host_arrays(full, len(planted))
        rec, roff = ix.locate(torch.as_tensor(full.positions(), device="cuda"))
        rec, roff = rec.cpu().numpy(), roff.cpu().numpy()
        full.free()
        for i, (r_, o) in enumerate(planted):
            a, b = int(o_[i]), int(o_[i + 1])
            for j in range(60 - k + 1):
                at = np.nonzero((j_[a:b] == j) & (p_[a:b] == s[r_] + o + j))[0]
                assert at.size == 1, (i, j)
                assert rec[a + at[0]] == r_ and roff[a + at[0]] == o + j


def test_long_buckets_and_long_reads(kb):
    from kmer_index_b200 import synth
    sigma, k, n = 4, 16, 600_000
    text = synth.random_text(n, sigma, 61)
    text[100_000:250_000] = 2                          # a bucket of ~1.5e5 positions
    motif = synth.random_text(16, sigma, 62)
    for x in range(300_000, 300_000 + 16 * 3000, 16):  # buckets of ~3000
        text[x:x + 16] = motif
    rng = np.random.default_rng(63)
    starts = random_starts(n, 500, rng, short=20)
    qs = [text[150_000:150_040], text[300_000:300_100], text[299_990:300_060], text[5_000:25_000],
          synth.random_text(10 ** 6, sigma, 64)]
    qs[-1][500_000:500_200] = 2
    q = np.concatenate(qs).astype(np.uint8)
    off = np.zeros(len(qs) + 1, dtype=np.uint64)
    np.cumsum([x.size for x in qs], out=off[1:])
    with kb.KmerIndex(text, sigma, [k]) as ix:
        for max_occ in (0, 2048, 100):
            want = seeds_truth(text, sigma, k, q, off, max_occ)
            if max_occ == 0:
                assert want[4].max() > 10 ** 5 and np.any((want[4] > 2048) & (want[4] < 10 ** 4))
            check_all_forms(ix, q, off, k, max_occ, want, f"long max_occ={max_occ}")
        ix.attach_records(starts)
        for max_occ in (0, 100):
            want = seeds_truth(text, sigma, k, q, off, max_occ, starts=starts)
            check_all_forms(ix, q, off, k, max_occ, want, f"long collection max_occ={max_occ}")


def test_peer_position_parts(kb):
    """Positions left in key-range parts (read through pos_ptr): the same seeds as the whole index."""
    import torch
    from kmer_index_b200 import sharded, synth
    sigma, n = 4, 200_000
    text = synth.random_text(n, sigma, 71)
    text[20_000:40_000] = 0
    dev = torch.device("cuda", 0)
    for ks, parts in (([12], 4), ([5, 7, 9, 11, 13], 3)):
        stream = torch.cuda.current_stream().cuda_stream
        idx = [kb.KmerIndex(text, sigma, ks, key_part=r, key_parts=parts, stream=stream or None) for r in range(parts)]
        try:
            q, off = seed_batch(text, sigma, ks[-1], 72)
            with pytest.raises(kb.KmerB200Error) as err:
                idx[0].seeds(q, off, k=ks[0])            # a key-range part that has not been adopted
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
            for k in ks:
                for max_occ in (0, 5):
                    want = seeds_truth(text, sigma, k, q, off, max_occ)
                    check_all_forms(idx[0], q, off, k, max_occ, want, f"parts {ks} k={k} max_occ={max_occ}", device=False)
        finally:
            for ix in idx:
                ix.close()


def test_refusals(kb):
    import torch
    from kmer_index_b200 import synth
    n = 100_000
    text = synth.random_text(n, 4, 81)
    q, off = seed_batch(text, 4, 12, 82, Q=30)
    with kb.KmerIndex(text, 4, [10, 12]) as ix:
        for k in (11, 13, 0):
            with pytest.raises(kb.KmerB200Error) as err:
                ix.seeds(q, off, k=k)
            assert err.value.code == -1
        ix.search_batch(q[:5], np.array([0, 5], np.uint64), mode=kb.MODE_CORRECT)   # an auxiliary k' = 5 element
        with pytest.raises(kb.KmerB200Error) as err:
            ix.seeds(q, off, k=5)
        assert err.value.code == -1
        with pytest.raises(ValueError):
            ix.seeds(q, off)                          # several ks: k is needed
        bad = q.copy()
        bad[int(off[3]) + 2] = 4
        with pytest.raises(kb.KmerB200Error) as err:
            ix.seeds(bad, off, k=12)
        assert err.value.code == -4
        short = np.array([0, 9, 1], np.uint8)         # shorter than k, still checked
        with pytest.raises(kb.KmerB200Error) as err:
            ix.seeds(short, np.array([0, 3], np.uint64), k=12)
        assert err.value.code == -4
        assert_seeds_equal(tuple(getattr(ix.seeds(q, off, k=12), a) for a in
                                 ("offsets", "positions", "status", "seed_offsets", "kmer_counts")),
                           seeds_truth(text, 4, 12, q, off), label="usable after refusals")
        other = ix.search_approx(q, off, 1)
        assert other.seed_offsets is None and other.kmer_counts is None
    handles = [kb.KmerIndex(text, 4, [10, 12], shared_positions=True, mode=kb.MODE_CORRECT),
               kb.KmerIndex(text[:60_063], 4, [12], shard_begin=0, n_total=n, halo=63, mode=kb.MODE_CORRECT)]
    try:
        for ix in handles:
            with pytest.raises(kb.KmerB200Error) as err:
                ix.seeds(q, off, k=12)
            assert err.value.code == -5
    finally:
        for ix in handles:
            ix.close()
    if torch.cuda.device_count() >= 2:
        with kb.KmerIndex(text, 4, [12], devices=[0, 1]) as multi:
            with pytest.raises(kb.KmerB200Error) as err:
                multi.seeds(q, off)
            assert err.value.code == -5
    else:
        pytest.skip("a multi-device handle needs two GPUs")


GUARD_CASE = r"""
import numpy as np
import kmer_index_b200 as kb
from kmer_index_b200 import synth
import sys
sys.path.insert(0, "tests")
from seeds_truth import seeds_truth
from collection_truth import random_starts
from test_gpu_seeds import seed_batch
text = synth.random_text(300_000, 4, 91)
text[50_000:60_000] = 3
starts = random_starts(text.size, 100, np.random.default_rng(92), short=10)
q, off = seed_batch(text, 4, 14, 93, Q=500)
q = np.concatenate([q, text[49_000:61_000]]).astype(np.uint8)
off = np.append(off, off[-1] + np.uint64(12_000))
for coll in (False, True):
    with kb.KmerIndex(text, 4, [14], mode=kb.MODE_CORRECT) as ix:
        if coll:
            ix.attach_records(starts)
        for max_occ in (0, 7):
            r = ix.seeds(q, off, k=14, max_occ=max_occ)
            want = seeds_truth(text, 4, 14, q, off, max_occ, starts=starts if coll else None)
            assert np.array_equal(r.positions, want[1]) and np.array_equal(r.kmer_counts, want[4])
print("guard violations", kb.guard_violations())
"""


def test_seed_kernels_under_guarded_allocations(tmp_path):
    env = dict(os.environ, KMER_B200_GUARD="1")
    out = subprocess.run([sys.executable, "-c", GUARD_CASE], capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "guard violations 0" in out.stdout, out.stdout[-2000:]
