"""The k-mer spectrum on the device (KmerIndex.spectrum, frequent_kmers, occurrence_cutoff) against the numpy ground truth
of tests/spectrum_truth.py, bit for bit: histogram, info, frequent list and cutoff, on dense and sparse directories,
64-bit keys, views of a shared-positions index, a 70 000-occurrence bucket, directory sizes around the sweep's chunk
boundaries and collections with empty, short and adjacent records."""
import os
import subprocess
import sys

import numpy as np
import pytest

from collection_truth import random_starts
from conftest import ROOT
from spectrum_truth import counts_truth, cutoff, frequent, histogram

pytestmark = pytest.mark.gpu
FRACTIONS = (0.0, 0.0002, 0.01, 0.3, 0.99)


@pytest.fixture(scope="module")
def kb():
    import kmer_index_b200
    return kmer_index_b200


def check_spectrum(ix, text, sigma, k, starts=None, bins=(2, 5, 10001), label="", top=(1, 2, 3, 100)):
    """Every entry point of element k against the brute force."""
    h, c = counts_truth(text, sigma, k, starts)
    key_space = sigma ** k
    for b in bins:
        s = ix.spectrum(k=k, bins=b)
        assert np.array_equal(s.hist, histogram(c, b, key_space)), f"{label} k={k} bins={b}"
        assert (s.total, s.distinct, s.max_count) == (int(c.sum()), c.size, int(c.max()) if c.size else 0), f"{label} k={k}"
        assert s.key_space == min(key_space, 2 ** 64 - 1)
    for min_count in top:
        for limit in (None, 0, 1, 10):
            gh, gc = ix.frequent_kmers(k=k, min_count=min_count, limit=limit)
            wh, wc, n = frequent(h, c, min_count, limit)
            assert np.array_equal(gh, wh) and np.array_equal(gc, wc), f"{label} k={k} min_count={min_count} limit={limit}"
    for f in FRACTIONS:
        assert ix.occurrence_cutoff(f, k=k) == cutoff(c, f), f"{label} k={k} f={f}"
    return h, c


def test_dense_dna4_small_k(kb):
    from kmer_index_b200 import synth
    text = synth.random_text(50_000, 4, 1)
    with kb.KmerIndex(text, 4, [3, 6, 8]) as ix:
        for e, k in enumerate((3, 6, 8)):
            assert ix.element_info(e).directory_shift == 0
            check_spectrum(ix, text, 4, k, bins=(2, 3, 5, 100, 10001, 100_000), label="dense")


def test_sparse_dna4_k16(kb):
    from kmer_index_b200 import synth
    text = synth.random_text(1_000_000, 4, 2)
    text[300_000:300_500] = text[600_000:600_500]     # some repeats
    with kb.KmerIndex(text, 4, [16]) as ix:
        assert ix.element_info(0).directory_shift > 0
        check_spectrum(ix, text, 4, 16, label="sparse")


@pytest.mark.parametrize("sigma,k", [(5, 17), (27, 7)])
def test_sparse_64bit_keys(kb, sigma, k):
    from kmer_index_b200 import synth
    text = synth.random_text(300_000, sigma, 3 + sigma)
    text[1000:4000] = 1                               # one long run: a bucket of ~3000
    with kb.KmerIndex(text, sigma, [k]) as ix:
        info = ix.element_info(0)
        assert info.directory_shift > 0 and info.key_bits > 32
        check_spectrum(ix, text, sigma, k, label=f"sigma={sigma}")


def test_shared_positions_views(kb):
    from kmer_index_b200 import synth
    text = synth.random_text(200_000, 4, 4)
    text[50_000:50_300] = 2
    for n in (200_000, 9, 12):                        # the tail starts at the end of the text; a text as short as k_max
        t = text[:n]
        with kb.KmerIndex(t, 4, [5, 7, 9], shared_positions=True, mode=kb.MODE_CORRECT) as ix:
            for k in (5, 7, 9):
                check_spectrum(ix, t, 4, k, label=f"views n={n}")


def test_low_entropy_overflow(kb):
    """A 70 000-occurrence bucket: in the overflow bin, at the top of the frequent list, above the cutoff histogram."""
    from kmer_index_b200 import synth
    text = synth.random_text(400_000, 4, 5)
    text[100_000:170_020] = 0
    text[200_000:201_000] = np.tile([1, 2], 500)
    with kb.KmerIndex(text, 4, [8, 10]) as ix:
        for k in (8, 10):
            h, c = check_spectrum(ix, text, 4, k, label="low entropy", top=(1, 2, 500, 65_535, 65_536, 70_000, 70_022))
            gh, gc = ix.frequent_kmers(k=k, min_count=1, limit=1)
            assert gh[0] == 0 and gc[0] >= 70_000
            assert ix.spectrum(k=k, bins=100).hist[99] >= 1
            assert ix.occurrence_cutoff(0.0, k=k) == int(c.max())


@pytest.mark.parametrize("sigma,k", [(15, 1), (4, 2), (17, 1), (33, 1), (2, 11), (3, 7), (2, 12), (4, 11), (5, 10)])
def test_dense_sizes_around_chunks(kb, sigma, k):
    """sigma^k around the dense sweep's 16-entry thread chunk, the 2048-item tiles of the generic sweeps, and past one
    grid-stride round of the dense sweep (148 SMs x 8 CTAs x 256 threads x 16 entries = 4.85 M)."""
    from kmer_index_b200 import synth
    text = synth.random_text(300_000, sigma, 6 + sigma + k)
    with kb.KmerIndex(text, sigma, [k], directory_bits=32) as ix:
        assert ix.element_info(0).directory_shift == 0
        check_spectrum(ix, text, sigma, k, bins=(2, 4, 10001), label=f"size {sigma}^{k}", top=(1, 40))


def test_collections(kb):
    from kmer_index_b200 import synth
    rng = np.random.default_rng(7)
    text = synth.random_text(120_000, 4, 7)
    text[30_000:40_000] = 3
    cases = [random_starts(text.size, 400, rng, short=150), random_starts(text.size, 3000, rng, short=2000),
             np.array([0, 0, 0, 5, 5, 10, 22, 22, 23, 35, 47, 60_000, 60_012, text.size, text.size], dtype=np.uint64)]
    for starts in cases:
        for ks in ([5], [12], [16]):
            with kb.KmerIndex(text, 4, ks, mode=kb.MODE_CORRECT) as ix:
                ix.attach_records(starts)
                check_spectrum(ix, text, 4, ks[0], starts=starts, label=f"collection R={starts.size - 1}")


def test_collection_of_short_records(kb):
    """Every record shorter than k or exactly k long: only the k-long ones count; none at all gives an empty spectrum."""
    from kmer_index_b200 import synth
    text = synth.random_text(12 * 1000, 4, 8)
    starts = np.arange(0, text.size + 1, 12, dtype=np.uint64)
    with kb.KmerIndex(text, 4, [12, 13], mode=kb.MODE_CORRECT) as ix:
        ix.attach_records(starts)
        check_spectrum(ix, text, 4, 12, starts=starts, label="records of exactly k")
        s = ix.spectrum(k=13, bins=4)
        assert (s.total, s.distinct, s.max_count) == (0, 0, 0) and s.hist.tolist() == [4 ** 13, 0, 0, 0]
        assert ix.occurrence_cutoff(0.5, k=13) == 0
        gh, gc = ix.frequent_kmers(k=13, min_count=1)
        assert gh.size == 0 and gc.size == 0


def test_adopted_key_range_parts(kb):
    """Key-range parts refuse the spectrum until the assembled element is adopted; then it is the whole index's."""
    import torch
    from kmer_index_b200 import sharded, synth
    sigma, n, k, parts = 4, 200_000, 12, 3
    text = synth.random_text(n, sigma, 9)
    text[20_000:40_000] = 0
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream().cuda_stream
    idx = [kb.KmerIndex(text, sigma, [k], key_part=r, key_parts=parts, stream=stream or None) for r in range(parts)]
    try:
        with pytest.raises(kb.KmerB200Error) as err:
            idx[0].spectrum()
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
        check_spectrum(idx[0], text, sigma, k, label="adopted parts")
    finally:
        for ix in idx:
            ix.close()


def test_agrees_with_seeding(kb):
    """frequent_kmers(min_count=1) gives seeding's uncapped kmer_counts, and seeds(max_occ=cutoff) drops exactly the
    k-mers above the cutoff, on a plain and a collection index."""
    from kmer_index_b200 import synth
    from seeds_truth import query_kmers
    from test_gpu_seeds import seed_batch
    rng = np.random.default_rng(10)
    text = synth.random_text(300_000, 4, 10)
    text[10_000:14_000] = 1
    text[20_000:22_000] = np.tile([0, 3], 1000)
    starts = random_starts(text.size, 500, rng, short=100)
    k = 11
    q, off = seed_batch(text, 4, k, 11, Q=400)
    for coll in (False, True):
        with kb.KmerIndex(text, 4, [k], mode=kb.MODE_CORRECT) as ix:
            if coll:
                ix.attach_records(starts)
            gh, gc = ix.frequent_kmers(min_count=1)
            table = dict(zip(gh.tolist(), gc.tolist()))
            qh = query_kmers(q, off, k, 4)[0]
            counts = ix.seeds(q, off).kmer_counts
            assert [table.get(int(x), 0) for x in qh] == counts.tolist()
            h, c = counts_truth(text, 4, k, starts if coll else None)
            truth = dict(zip(h.tolist(), c.tolist()))
            for f in (0.0, 0.001, 0.05):
                cut = ix.occurrence_cutoff(f)
                assert cut == cutoff(c, f)
                capped = ix.seeds(q, off, max_occ=cut).kmer_counts
                above = np.array([truth.get(int(x), 0) > cut for x in qh])
                assert np.array_equal(capped == cut + 1, above), f"coll={coll} f={f}"
                assert np.array_equal(capped[~above], counts[~above])


def test_save_load_round_trip(kb, tmp_path):
    from kmer_index_b200 import synth
    text = synth.random_text(200_000, 4, 12)
    text[5000:9000] = 2
    path = str(tmp_path / "ix.kb")
    with kb.KmerIndex(text, 4, [7, 14]) as ix:
        want = [(ix.spectrum(k=k).hist, ix.frequent_kmers(k=k, min_count=3), ix.occurrence_cutoff(0.001, k=k)) for k in (7, 14)]
        ix.save(path)
    with kb.KmerIndex.load(path) as ix:
        for k, (hist, (fh, fc), cut) in zip((7, 14), want):
            assert np.array_equal(ix.spectrum(k=k).hist, hist)
            gh, gc = ix.frequent_kmers(k=k, min_count=3)
            assert np.array_equal(gh, fh) and np.array_equal(gc, fc)
            assert ix.occurrence_cutoff(0.001, k=k) == cut


def test_refusals(kb):
    import torch
    from kmer_index_b200 import synth
    n = 100_000
    text = synth.random_text(n, 4, 13)
    with kb.KmerIndex(text, 4, [10, 12]) as ix:
        ix.search_batch(text[:5], np.array([0, 5], np.uint64), mode=kb.MODE_CORRECT)   # an auxiliary k' = 5 element
        for k in (11, 13, 0, 5):
            for call in (lambda: ix.spectrum(k=k), lambda: ix.frequent_kmers(k=k), lambda: ix.occurrence_cutoff(0.1, k=k)):
                with pytest.raises(kb.KmerB200Error) as err:
                    call()
                assert err.value.code == -1
        for call in (lambda: ix.spectrum(k=10, bins=1), lambda: ix.spectrum(k=10, bins=(1 << 24) + 1),
                     lambda: ix.frequent_kmers(k=10, min_count=0), lambda: ix.occurrence_cutoff(1.0, k=10),
                     lambda: ix.occurrence_cutoff(-0.1, k=10), lambda: ix.occurrence_cutoff(float("nan"), k=10)):
            with pytest.raises(kb.KmerB200Error) as err:
                call()
            assert err.value.code == -1
        with pytest.raises(ValueError):
            ix.spectrum()                             # several ks: k is needed
        check_spectrum(ix, text, 4, 12, bins=(10001,), label="usable after refusals", top=(2,))
    with kb.KmerIndex(text[:60_063], 4, [12], shard_begin=0, n_total=n, halo=63, mode=kb.MODE_CORRECT) as shard:
        for call in (shard.spectrum, shard.frequent_kmers, lambda: shard.occurrence_cutoff(0.1)):
            with pytest.raises(kb.KmerB200Error) as err:
                call()
            assert err.value.code == -5
    if torch.cuda.device_count() >= 2:
        with kb.KmerIndex(text, 4, [12], devices=[0, 1]) as multi:
            with pytest.raises(kb.KmerB200Error) as err:
                multi.spectrum()
            assert err.value.code == -5


GUARD_CASE = r"""
import numpy as np
import kmer_index_b200 as kb
from kmer_index_b200 import synth
import sys
sys.path.insert(0, "tests")
from collection_truth import random_starts
from test_gpu_spectrum import check_spectrum
text = synth.random_text(300_000, 4, 14)
text[50_000:120_000] = 3
starts = random_starts(text.size, 200, np.random.default_rng(15), short=40)
for ks, coll, shared in (([6, 16], False, False), ([6, 16], True, False), ([5, 7, 9], False, True)):
    with kb.KmerIndex(text, 4, ks, mode=kb.MODE_CORRECT, shared_positions=shared) as ix:
        if coll:
            ix.attach_records(starts)
        for k in ks:
            check_spectrum(ix, text, 4, k, starts=starts if coll else None, bins=(3, 10001), top=(1, 66_000))
print("guard violations", kb.guard_violations())
"""


def test_spectrum_under_guarded_allocations():
    env = dict(os.environ, KMER_B200_GUARD="1")
    out = subprocess.run([sys.executable, "-c", GUARD_CASE], capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "guard violations 0" in out.stdout, out.stdout[-2000:]
