"""GPU parity at the BASELINE.json sizes.

Configs 1, 2, 4 (and config 3 on a query subsample / by counts): bit-exact against the C restatement oracle on
the full-size text. Config 5 (3 Gbp, 1e8 queries) is beyond what a CPU index can hold, so it is checked
through size-independent properties: ascending positions, every reported position verified against the text,
planted queries found, count-only == materialised, determinism (checksum), and an emulated 2-shard run giving
the same hit set.
"""
import numpy as np
import pytest

from conftest import assert_results_equal

pytestmark = pytest.mark.gpu

TEXT_SEED, QUERY_SEED = 205, 1239


@pytest.fixture(scope="module")
def kb():
    import kmer_index_b200
    return kmer_index_b200


def _free_host_gb():
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable"):
                return int(ln.split()[1]) / 1e6
    except OSError:
        pass
    return 0.0


FULL = [
    # label, sigma, ks, n, Q, m_lo, m_hi
    ("config1", 4, [10], 1_000_000, 10_000, 10, 10),
    ("config2", 4, [12], 100_000_000, 1_000_000, 13, 100),
    ("config4_dna15", 15, [8], 50_000_000, 1_000_000, 8, 8),
    ("config4_aa27", 27, [5], 50_000_000, 1_000_000, 5, 5),
]


@pytest.mark.parametrize("label,sigma,ks,n,Q,m_lo,m_hi", FULL)
def test_full_size_bit_exact_vs_oracle(kb, oracle_mod, label, sigma, ks, n, Q, m_lo, m_hi):
    from kmer_index_b200 import synth
    if _free_host_gb() < 16:
        pytest.skip("needs ~16 GB of host memory for the CPU oracle at this size")
    text = synth.random_text(n, sigma, TEXT_SEED)
    # half BASELINE-style random queries, half planted windows (random queries almost never hit for long m)
    q1, off1 = synth.random_queries(Q // 2, m_lo, m_hi, sigma, QUERY_SEED)
    q2, off2 = synth.stress_queries(text, Q - Q // 2, m_lo, m_hi, sigma, QUERY_SEED + 1) if n <= 2_000_000 else \
        _planted(text, Q - Q // 2, m_lo, m_hi, QUERY_SEED + 1)
    q = np.concatenate([q1, q2])
    off = np.concatenate([off1, off2[1:] + off1[-1]])
    with kb.KmerIndex(text, sigma, ks) as ix:
        got = ix.search_batch(q, off).as_tuple()
    with oracle_mod.Oracle(text, sigma, ks) as o:
        want = o.search(q, off)
    assert want[1].size > 0
    assert_results_equal(got, want, label=label)


def _planted(text, Q, m_lo, m_hi, seed):
    """Q windows of the text (vectorised; stress_queries loops in Python and is too slow for 5e5 queries)."""
    from kmer_index_b200 import synth
    n = text.size
    lens = synth.random_lengths(Q, m_lo, m_hi, seed)
    off = synth.offsets_from_lengths(lens)
    starts = synth.uniform_below(seed ^ 0xBEEF, 0, Q, n - m_hi).astype(np.int64)
    starts[::97] = n - lens[::97].astype(np.int64)              # some windows end exactly at the end of the text
    idx = np.repeat(starts - off[:-1].astype(np.int64), lens.astype(np.int64)) + np.arange(int(off[-1]), dtype=np.int64)
    return text[idx], off


@pytest.mark.parametrize("sigma,k", [(4, 12), (15, 6)])
def test_pipelined_text_upload_equals_plain(kb, sigma, k):
    """Host texts of 64 Mi symbols or more (2- and 4-bit alphabets) reach the device through the host threads' streaming
    pack, pinned ones partly as 1-byte ranks over the copy engine at the same time: the index must be the one the plain
    upload builds, and a rank >= sigma must be reported from either kind of chunk."""
    import os

    import torch

    from kmer_index_b200 import synth
    n = 70_000_037
    text = synth.random_text(n, sigma, TEXT_SEED + 3)
    pinned = torch.from_numpy(text).pin_memory()
    os.environ["KMER_B200_NO_TEXT_PIPELINE"] = "1"
    try:
        with kb.KmerIndex(text, sigma, [k]) as ix:
            want = ix.element_arrays(0)
    finally:
        del os.environ["KMER_B200_NO_TEXT_PIPELINE"]
    builds = [("pageable", text, None), ("pinned, calibrated share", pinned.numpy(), None),
              ("pinned, 34 % raw", pinned.numpy(), "34"), ("pinned, all raw", pinned.numpy(), "100")]
    for label, src, pct in builds:
        if pct is not None:
            os.environ["KMER_B200_HOST_RAW_PCT"] = pct
        try:
            with kb.KmerIndex(src, sigma, [k]) as ix:
                got = ix.element_arrays(0)
                moved = ix.build_transfer()
        finally:
            os.environ.pop("KMER_B200_HOST_RAW_PCT", None)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), label
        bits = 2 if sigma <= 4 else 4
        if label == "pageable":
            assert n * bits // 8 <= moved <= n * bits // 8 + 64, (label, moved)   # every chunk crossed the link packed
        elif pct == "100":
            assert moved == n, (label, moved)
        else:
            assert n * bits // 8 <= moved <= n, (label, moved)
    os.environ["KMER_B200_HOST_RAW_PCT"] = "50"
    try:
        for at in (3, 40_000_000, n - 1):                      # first chunk (raw), a packed chunk, the last word
            bad = pinned.numpy().copy()
            bad[at] = sigma
            with pytest.raises(kb.KmerB200Error) as e:
                kb.KmerIndex(torch.from_numpy(bad).pin_memory().numpy(), sigma, [k])
            assert e.value.code == -4, at
    finally:
        del os.environ["KMER_B200_HOST_RAW_PCT"]


def test_chunked_host_batch_equals_plain(kb):
    """Host batches >= 256 MiB are searched in pipelined chunks (H2D / search / D2H overlapped); the result must be
    the plain path's, offsets included."""
    import os

    from kmer_index_b200 import synth
    text = synth.random_text(20_000_000, 4, TEXT_SEED)
    q1, off1 = synth.random_queries(3_000_000, 12, 100, 4, QUERY_SEED)
    q2, off2 = _planted(text, 3_000_000, 12, 100, QUERY_SEED + 5)
    q = np.concatenate([q1, q2])
    off = np.concatenate([off1, off2[1:] + off1[-1]])
    assert q.size + 17 * (off.size - 1) >= (256 << 20)
    import torch
    pin_q, pin_off = torch.from_numpy(q).pin_memory(), torch.from_numpy(off).pin_memory()
    with kb.KmerIndex(text, 4, [12]) as ix:
        # pageable numpy input: packed as a stream on the host threads, cut into per-query words on the device
        packed = ix.search_batch(q, off).as_tuple()
        path = ix.last_search_host_path()
        assert path["pipeline"].startswith("streaming") and path["raw_chunk_pct"] == 0, path
        assert ix.last_search_transfer()[0] < q.size // 4 + 2 * (off.size - 1) + 4096
        # pinned input: part of the chunks cross the link as 1-byte ranks while the host threads pack the others
        mixed_auto = ix.search_batch(pin_q.numpy(), pin_off.numpy()).as_tuple()
        path_auto = ix.last_search_host_path()
        assert path_auto["pipeline"].startswith("streaming") and path_auto["host_pack_gbs"] > 0, path_auto
        mixed = {}
        try:
            for pct in (0, 30, 50, 100):
                os.environ["KMER_B200_HOST_RAW_PCT"] = str(pct)
                mixed[pct] = ix.search_batch(pin_q.numpy(), pin_off.numpy()).as_tuple()
                assert ix.last_search_host_path()["raw_chunk_pct"] == pct
            os.environ["KMER_B200_HOST_RAW_PCT"] = "50"
            bad = pin_q.numpy().copy()
            for at in (5, q.size // 2, q.size - 7):          # in a raw chunk or a stream chunk: reported either way
                bad[at] = 4
                with pytest.raises(kb.KmerB200Error) as e:
                    ix.search_batch(torch.from_numpy(bad).pin_memory().numpy(), pin_off.numpy())
                assert e.value.code == -4
                bad[at] = q[at]
            os.environ["KMER_B200_HOST_RAW_PCT"] = "100"
            piped = ix.search_batch(q, off).as_tuple()       # 1-byte ranks over PCIe, chunks pipelined
            # the offsets crossed the link as 16-bit lengths
            assert ix.last_search_transfer()[0] == q.size + 2 * (off.size - 1)
            # a query of 65 536 symbols or more: its chunk (the last one of 24) sends its offsets, the other chunks
            # lengths (CORRECT mode: the reference's table stops at 10 000 symbols)
            q_long = np.concatenate([q, text[1000:71_000]])
            off_long = np.concatenate([off, [off[-1] + 70_000]]).astype(np.uint64)
            piped_long = ix.search_batch(q_long, off_long, mode=kb.MODE_CORRECT).as_tuple()
            n_long = off_long.size - 1
            last = n_long - 23 * -(-n_long // 24)
            assert ix.last_search_transfer()[0] == q_long.size + 2 * (n_long - last) + 8 * (last + 1)
        finally:
            os.environ.pop("KMER_B200_HOST_RAW_PCT", None)
        # the same long query through the default choice. Pageable: the packed chunk that holds it refuses the batch
        # (its lengths travel as 16 bits), which is searched again with every chunk raw
        default_long = ix.search_batch(q_long, off_long, mode=kb.MODE_CORRECT).as_tuple()
        path_long = ix.last_search_host_path()
        assert path_long["pipeline"].startswith("streaming") and path_long["raw_chunk_pct"] == 100, path_long
        # pinned: the same unless the long query's chunk is one of the raw chunks
        pinned_long = ix.search_batch(torch.from_numpy(q_long).pin_memory().numpy(), off_long, mode=kb.MODE_CORRECT).as_tuple()
        assert ix.last_search_host_path()["pipeline"].startswith("streaming")
        os.environ["KMER_B200_NO_PIPELINE"] = "1"
        try:
            plain = ix.search_batch(q, off).as_tuple()
            plain_long = ix.search_batch(q_long, off_long, mode=kb.MODE_CORRECT).as_tuple()
        finally:
            del os.environ["KMER_B200_NO_PIPELINE"]
        bad = q.copy()
        bad[q.size // 2] = 4                                  # a rank >= sigma must be reported, not packed away
        with pytest.raises(kb.KmerB200Error) as e:
            ix.search_batch(bad, off)
        assert e.value.code == -4
    assert piped[1].size > 500_000
    assert_results_equal(piped, plain, label="pipelined vs plain")
    assert plain_long[0][-1] - plain_long[0][-2] == 1          # the long query occurs once, at position 1000
    assert_results_equal(piped_long, plain_long, label="pipelined with a 70 000-symbol query vs plain")
    assert_results_equal(default_long, plain_long, label="default pipeline choice with a 70 000-symbol query vs plain")
    assert_results_equal(pinned_long, plain_long, label="default pipeline choice, pinned, with a 70 000-symbol query vs plain")
    assert_results_equal(packed, plain, label="stream-packed pipeline (pageable input) vs plain")
    assert_results_equal(mixed_auto, plain, label=f"stream-packed + raw chunks ({path_auto}) vs plain")
    for pct, got in mixed.items():
        assert_results_equal(got, plain, label=f"stream-packed + {pct} % raw chunks vs plain")


def test_chunked_host_batch_8bit_equals_plain(kb):
    """An 8-bit alphabet (sigma 27) through the chunked pipeline: pageable input packed as a stream on the host threads
    (a byte reversal per word), pinned input sent as 1-byte ranks. Both must give the plain path's result, and a rank
    >= sigma must be reported from either."""
    import os

    import torch

    from kmer_index_b200 import synth
    sigma = 27
    text = synth.random_text(20_000_000, sigma, TEXT_SEED + 7)
    q1, off1 = synth.random_queries(3_000_000, 12, 100, sigma, QUERY_SEED + 7)
    q2, off2 = _planted(text, 3_000_000, 12, 100, QUERY_SEED + 8)
    q = np.concatenate([q1, q2])
    off = np.concatenate([off1, off2[1:] + off1[-1]])
    assert q.size + 17 * (off.size - 1) >= (256 << 20)
    pin_q = torch.from_numpy(q).pin_memory()
    with kb.KmerIndex(text, sigma, [5]) as ix:
        pageable = ix.search_batch(q, off).as_tuple()
        path = ix.last_search_host_path()
        assert path["pipeline"].startswith("streaming") and path["raw_chunk_pct"] == 0, path
        assert ix.last_search_transfer()[0] < q.size + 2 * (off.size - 1) + 4096
        pinned = ix.search_batch(pin_q.numpy(), off).as_tuple()
        path = ix.last_search_host_path()
        assert path["pipeline"].startswith("streaming") and path["raw_chunk_pct"] == 100, path
        assert ix.last_search_transfer()[0] == q.size + 2 * (off.size - 1)
        os.environ["KMER_B200_NO_PIPELINE"] = "1"
        try:
            plain = ix.search_batch(q, off).as_tuple()
        finally:
            del os.environ["KMER_B200_NO_PIPELINE"]
        for at in (3, q.size // 2, q.size - 1):
            bad = q.copy()
            bad[at] = sigma
            for label, src in (("pageable", bad), ("pinned", torch.from_numpy(bad).pin_memory().numpy())):
                with pytest.raises(kb.KmerB200Error) as e:
                    ix.search_batch(src, off)
                assert e.value.code == -4, (label, at)
    assert plain[1].size > 500_000
    assert_results_equal(pageable, plain, label="sigma 27, stream-packed chunks (pageable input) vs plain")
    assert_results_equal(pinned, plain, label="sigma 27, raw chunks (pinned input) vs plain")


def test_config3_full_text_counts_and_subsample(kb, oracle_mod):
    """multi_kmer_index<dna4,{5,7,9,11,13}> over 100 Mbp: all 1e6 queries by per-query hit COUNT against the oracle
    (1.4e10 positions do not fit a CPU result), and a subsample bit for bit."""
    from kmer_index_b200 import synth
    if _free_host_gb() < 24:
        pytest.skip("needs ~24 GB of host memory for the CPU oracle at this size")
    sigma, ks, n = 4, [5, 7, 9, 11, 13], 100_000_000
    text = synth.random_text(n, sigma, TEXT_SEED)
    q, off = synth.random_queries(1_000_000, 4, 40, sigma, QUERY_SEED)    # the BASELINE batch, all of it
    qs, offs = synth.random_queries(3_000, 6, 40, sigma, QUERY_SEED + 2)       # materialised on both sides
    qp, offp = _planted(text, 20_000, 6, 40, QUERY_SEED + 3)
    with kb.KmerIndex(text, sigma, ks) as ix, oracle_mod.Oracle(text, sigma, ks) as o:
        import torch
        dev = torch.device("cuda", 0)
        # all 10^6 queries: per-query count and status from the device count pass (the 1.4e10 positions of the full
        # batch are 56 GB -- they stay unmaterialised on both sides)
        d_q = torch.from_numpy(q).to(dev)
        d_off = torch.from_numpy(off.view(np.int64)).to(dev)
        torch.cuda.synchronize()
        res = ix.count_batch_device(d_q.data_ptr(), d_off.data_ptr(), off.size - 1, 40)
        c_off = torch.as_tensor(res.offsets(), device=dev).cpu().numpy().astype(np.uint64)
        c_status = torch.as_tensor(res.status(), device=dev).cpu().numpy()
        res.free()
        del d_q, d_off
        w_off, _, w_status = o.search(q, off, keep_positions=False)
        assert np.array_equal(c_status, w_status)
        assert np.array_equal(c_off, w_off)
        assert int(w_off[-1]) > 10_000_000_000
        # the first 2*10^5 of them materialised: same counts, ascending inside every query
        sub = 200_000
        got = ix.search_batch(q[:int(off[sub])], off[:sub + 1], copy=False)
        assert np.array_equal(got.status, w_status[:sub])
        assert np.array_equal(got.offsets, w_off[:sub + 1])
        pos = got.positions
        # ascending inside every query (sub-k results come from auxiliary elements or the sort kernel)
        d = np.diff(pos.astype(np.int64))
        boundaries = got.offsets[1:-1].astype(np.int64) - 1
        d[boundaries[(boundaries >= 0) & (boundaries < d.size)]] = 1
        assert (d > 0).all()
        del pos, d
        got.free()
        assert_results_equal(ix.search_batch(qs, offs).as_tuple(), o.search(qs, offs), label="config3 subsample")
        assert_results_equal(ix.search_batch(qp, offp).as_tuple(), o.search(qp, offp), label="config3 planted")


def test_config5_full_text_sample_bit_exact_vs_oracle(kb, oracle_mod):
    """kmer_index<dna4,16> over the full 3 Gbp text of config 5 against the CPU restatement on the SAME text, for a
    10^6-query sample: half BASELINE-random, half windows of the text (every length 16-64, some ending exactly at
    n), so the defective 53-63 plan and the rest-1..4 THROW rule are exercised with non-empty truth. The oracle holds
    only the buckets this batch can ask for (ko_create_restricted, pinned to the full restatement on the CPU), which
    is what makes 3 Gbp affordable on the host: one threaded scan of the text."""
    import torch

    from kmer_index_b200 import _capi, synth
    free, _ = torch.cuda.mem_get_info()
    if free < 100e9:
        pytest.skip("needs ~100 GB of device memory")
    if _free_host_gb() < 14:
        print("SKIPPED: config-5 full-size oracle comparison needs ~14 GB of host memory, have %.1f" % _free_host_gb())
        pytest.skip("needs ~14 GB of host memory")
    dev = torch.device("cuda", 0)
    L = _capi.lib()
    n, k, m_lo, m_hi = 3_000_000_000, 16, 16, 64
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sptr = stream.cuda_stream
    d_text = torch.empty(n, dtype=torch.uint8, device=dev)
    _capi.check(L.kmer_b200_synth_ranks_device(d_text.data_ptr(), n, 0, 4, TEXT_SEED, sptr))
    torch.cuda.synchronize()
    assert np.array_equal(d_text[:4096].cpu().numpy(), synth.random_text(4096, 4, TEXT_SEED))   # device generator == host generator
    # a stretch of period 16 (one random 16-mer repeated): windows inside it satisfy the defective plans non-trivially
    p_lo, p_len = 1_500_000_000, 1 << 16
    d_text[p_lo:p_lo + p_len] = d_text[p_lo:p_lo + 16].repeat(p_len // 16)
    text = d_text.cpu().numpy()
    Q = 1_000_000
    q1, off1 = synth.random_queries(Q // 2, m_lo, m_hi, 4, QUERY_SEED)
    q2, off2 = _planted(text, Q - Q // 2, m_lo, m_hi, QUERY_SEED + 1)
    n_periodic = 4096                                          # the last planted windows come from the periodic stretch
    lens2 = (off2[1:] - off2[:-1]).astype(np.int64)
    for j in range(n_periodic):
        i = lens2.size - 1 - j
        s0 = p_lo + 16 + (j * 7) % 4096
        q2[int(off2[i]):int(off2[i + 1])] = text[s0:s0 + int(lens2[i])]
    q = np.concatenate([q1, q2])
    off = np.concatenate([off1, off2[1:] + off1[-1]])
    lens = (off[1:] - off[:-1]).astype(np.int64)
    assert set(lens[Q // 2:].tolist()) == set(range(m_lo, m_hi + 1))
    ix = kb.KmerIndex(None, 4, [k], stream=sptr, text_device_ptr=d_text.data_ptr(), n=n)
    try:
        del d_text
        got = ix.search_batch(q, off).as_tuple()
        got_correct = ix.search_batch(q, off, mode=kb.MODE_CORRECT).as_tuple()
    finally:
        ix.close()
    with oracle_mod.Oracle(text, 4, [k], restrict_to=(q, off)) as o:
        want = o.search(q, off)
        ub = o.last_ub
    assert oracle_mod.Oracle.restricted_misses() == 0
    assert_results_equal(got, want, skip=ub, label="config5 full text")
    planted_lens, planted_status = lens[Q // 2:], want[2][Q // 2:]
    planted_counts = (want[0][1:] - want[0][:-1])[Q // 2:]
    rest = planted_lens % k
    # the sample does exercise what it is meant to: THROW with all parts present, non-empty defective plans
    assert int(((planted_status == 1) & (rest >= 1) & (rest <= 4)).sum()) > 1000
    # lengths 53-63 run the reference's defective plan (kmer_index.hpp:314): on a random text a planted window is NOT
    # found by it (false negative) -- reproduced bit for bit above; the periodic stretch below makes the plan non-empty
    defect = (planted_lens >= 53) & (planted_lens <= 63)
    assert int((planted_counts[defect] > 0).sum()) >= n_periodic // 8
    assert int((planted_counts[defect] == 0).sum()) > 1000
    assert int((want[0][1:] - want[0][:-1])[:Q // 2].sum()) > 1000                        # random queries with hits
    # CORRECT mode: every planted window is found at its origin; sorted lists
    c_off, c_pos, _ = got_correct
    assert int(((c_off[1:] - c_off[:-1])[Q // 2:] == 0).sum()) == 0


def test_config5_full_size_properties(kb):
    """kmer_index<dna4,16> over 3 Gbp, 1e8 queries of length 16-64, all on the device."""
    import torch

    from kmer_index_b200 import _capi, sharded
    free, _ = torch.cuda.mem_get_info()
    if free < 100e9:
        pytest.skip("needs ~100 GB of device memory")
    dev = torch.device("cuda", 0)
    L = _capi.lib()
    n, Q, m_lo, m_hi, k = 3_000_000_000, 100_000_000, 16, 64, 16
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sptr = stream.cuda_stream
    text = torch.empty(n, dtype=torch.uint8, device=dev)
    _capi.check(L.kmer_b200_synth_ranks_device(text.data_ptr(), n, 0, 4, TEXT_SEED, sptr))
    g = torch.Generator(device=dev)
    g.manual_seed(QUERY_SEED)
    lens = torch.randint(m_lo, m_hi + 1, (Q,), generator=g, device=dev, dtype=torch.int64)
    off = torch.zeros(Q + 1, dtype=torch.int64, device=dev)
    torch.cumsum(lens, 0, out=off[1:])
    n_sym = int(off[-1].item())
    q = torch.empty(n_sym, dtype=torch.uint8, device=dev)
    _capi.check(L.kmer_b200_synth_ranks_device(q.data_ptr(), n_sym, 0, 4, QUERY_SEED ^ 0xC0FFEE, sptr))
    # plant every 50th query: a window of the text (so long queries have true occurrences)
    planted = torch.arange(0, Q, 50, device=dev)
    starts = torch.randint(0, n - m_hi, (planted.numel(),), generator=g, device=dev, dtype=torch.int64)
    p_len = lens[planted]
    seg = torch.repeat_interleave(torch.arange(planted.numel(), device=dev), p_len)
    within = torch.arange(int(p_len.sum().item()), device=dev) - torch.repeat_interleave(torch.cumsum(p_len, 0) - p_len, p_len)
    q[off[planted][seg] + within] = text[starts[seg] + within]
    torch.cuda.synchronize()

    ix = kb.KmerIndex(None, 4, [k], stream=sptr, text_device_ptr=text.data_ptr(), n=n)
    try:
        res = ix.search_batch_device(q.data_ptr(), off.data_ptr(), Q, m_hi)
        r_off = torch.as_tensor(res.offsets(), device=dev)
        r_pos = torch.as_tensor(res.positions(), device=dev).view(torch.int32).to(torch.int64) & 0xFFFFFFFF
        r_st = torch.as_tensor(res.status(), device=dev)
        torch.cuda.synchronize()
        hits = int(r_off[-1].item())
        assert hits == r_pos.numel() and hits > planted.numel() // 4
        counts = r_off[1:] - r_off[:-1]
        # (1) status: THROW exactly for rest in 1..4 among queries that are OK-or-throw; no hits on non-OK
        rest = lens % k
        assert int(((r_st != 0) & (counts != 0)).sum().item()) == 0
        assert int(((r_st == 1) & ~((rest >= 1) & (rest <= 4))).sum().item()) == 0
        # (2) ascending inside every query
        d = r_pos[1:] - r_pos[:-1]
        inner = torch.ones(hits - 1, dtype=torch.bool, device=dev)
        ends = r_off[1:-1] - 1
        ends = ends[(ends >= 0) & (ends < hits - 1)]
        inner[ends] = False
        assert bool((d[inner] > 0).all().item())
        # (3) every reported position is a true occurrence of a prefix of the query it belongs to:
        #     verify the first 16 symbols and the last 16 symbols of the claimed match against the text
        qid = torch.repeat_interleave(torch.arange(Q, device=dev), counts)
        for shift_from_end in (False, True):
            for j in range(0, 16, 5):
                o = (lens[qid] - 1 - j) if shift_from_end else torch.full_like(qid, j)
                # lengths 53..63 run the reference's defective plan (only the parts are constrained)
                ok_len = (lens[qid] <= 52) | (lens[qid] == 64)
                a = text[r_pos + o]
                b = q[off[qid] + o]
                assert bool((a[ok_len] == b[ok_len]).all().item())
        # (4) planted queries whose plan is correct in the reference and does not throw are found at their origin
        pl_ok = (r_st[planted] == 0) & ((p_len <= 52) | (p_len == 64))
        lo = r_off[planted]
        hi = r_off[planted + 1]
        found = torch.zeros(planted.numel(), dtype=torch.bool, device=dev)
        width = int((hi - lo).max().item())
        for j in range(width):
            idx = torch.clamp(lo + j, max=hits - 1)
            found |= (lo + j < hi) & (r_pos[idx] == starts)
        assert bool(found[pl_ok].all().item())
        # (5) count-only pass agrees; (6) deterministic across runs
        checksum = int((r_pos * (qid + 1)).sum().item())
        res2 = ix.count_batch_device(q.data_ptr(), off.data_ptr(), Q, m_hi)
        assert torch.equal(torch.as_tensor(res2.offsets(), device=dev), r_off)
        res2.free()
        res3 = ix.search_batch_device(q.data_ptr(), off.data_ptr(), Q, m_hi)
        p3 = torch.as_tensor(res3.positions(), device=dev).view(torch.int32).to(torch.int64) & 0xFFFFFFFF
        torch.cuda.synchronize()
        assert int((p3 * (qid + 1)).sum().item()) == checksum
        res3.free()
        st_single, off_single = r_st.clone(), r_off.clone()
        res.free()
    finally:
        ix.close()
    del r_pos, qid, d, inner

    # (7) two position-range shards on the same GPU (built one after the other) give the same offsets and status
    per_shard = []
    shards = [sharded.shard_range(n, 2, r, halo=m_hi - 1) for r in range(2)]
    masks, pend, idxs = [], [], []
    try:
        for s in shards:
            sx = kb.KmerIndex(None, 4, [k], stream=sptr, text_device_ptr=text.data_ptr() + s.begin, n=s.length,
                              shard_begin=s.begin, n_total=n, halo=s.halo)
            idxs.append(sx)
            m = torch.zeros(Q, dtype=torch.int32, device=dev)
            pend.append(sx.search_sharded_begin(q.data_ptr(), off.data_ptr(), Q, m_hi, m.data_ptr()))
            masks.append(m)
        torch.cuda.synchronize()
        present = (masks[0] + masks[1]).to(torch.int32)
        total = torch.zeros(Q, dtype=torch.int64, device=dev)
        for sx, p in zip(idxs, pend):
            r = sx.search_sharded_finish(p, present.data_ptr(), Q)
            o = torch.as_tensor(r.offsets(), device=dev)
            total += o[1:] - o[:-1]
            assert torch.equal(torch.as_tensor(r.status(), device=dev), st_single)
            r.free()
        assert torch.equal(total, off_single[1:] - off_single[:-1])
    finally:
        for sx in idxs:
            sx.close()
