"""GPU parity: the CUDA path (through the C ABI) against the golden fixtures generated from the compiled
reference, against the C restatement oracle on larger seeded inputs, and against ground truth (CORRECT mode)."""
import contextlib

import numpy as np
import pytest

from conftest import assert_results_equal, golden_cases, load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def kb():
    import kmer_index_b200
    return kmer_index_b200


@pytest.mark.parametrize("name", golden_cases())
def test_cuda_matches_golden(kb, name):
    g = load_golden(name)
    with kb.KmerIndex(g["text"], int(g["sigma"]), g["ks"].tolist()) as ix:
        got = ix.search_batch(g["q"], g["q_off"]).as_tuple()
        assert_results_equal(got, (g["r_off"], g["r_pos"], g["r_status"]), skip=g["ub"].astype(bool), label=name)
        flat, o_ = g["scheme_flat"], 0
        for m, ln, multi in zip(g["scheme_m"], g["scheme_len"], g["scheme_multi"]):
            ks, use_multi = ix.scheme(int(m))
            assert ks == flat[o_:o_ + ln].tolist() and use_multi == bool(multi), (name, int(m))
            o_ += int(ln)


@pytest.mark.parametrize("name", golden_cases())
def test_cuda_matches_oracle_on_golden_inputs_including_ub(kb, oracle_mod, name):
    """On UB-flagged queries the product's defined behaviour is the oracle's ('not equal')."""
    g = load_golden(name)
    with kb.KmerIndex(g["text"], int(g["sigma"]), g["ks"].tolist()) as ix, \
            oracle_mod.Oracle(g["text"], int(g["sigma"]), g["ks"].tolist()) as o:
        assert_results_equal(ix.search_batch(g["q"], g["q_off"]).as_tuple(), o.search(g["q"], g["q_off"]), label=name)


@pytest.mark.parametrize("sigma,ks,n", [(4, [10], 1_000_000), (4, [12], 3_000_000), (4, [5, 7, 9, 11, 13], 500_000),
                                        (15, [8], 1_000_000), (27, [5], 1_000_000), (4, [16], 2_000_000),
                                        (4, [1], 5000), (5, [13], 300_000), (4, [3, 9, 16], 200_000),
                                        # hashes wider than 32 bits
                                        (4, [20], 300_000), (4, [31], 100_000), (15, [12], 200_000), (15, [16], 50_000),
                                        (27, [8], 100_000), (4, [12, 24], 100_000),
                                        # k-mers wider than one 64-bit packed window (two-window hash)
                                        (27, [9], 200_000), (27, [13], 100_000), (5, [17], 200_000), (5, [27], 50_000),
                                        (3, [40], 50_000), (2, [63], 20_000), (17, [15], 50_000), (27, [5, 9, 12], 50_000)])
def test_csr_matches_oracle(kb, oracle_mod, sigma, ks, n):
    """The index itself: positions stably sorted by hash == the reference's buckets in hash order."""
    from kmer_index_b200 import synth
    text = synth.random_text(n, sigma, 77 + n % 13)
    with kb.KmerIndex(text, sigma, ks) as ix, oracle_mod.Oracle(text, sigma, ks) as o:
        for e in range(len(ks)):
            h, p = ix.element_arrays(e)
            oh, op = o.element(e)
            assert np.array_equal(h.astype(np.uint64), oh), (ks, e)
            assert np.array_equal(p, op), (ks, e)


CASES = [
    # (label, sigma, ks, n, Q, m_lo, m_hi)
    ("c1", 4, [10], 1_000_000, 10_000, 10, 10),
    ("c2", 4, [12], 4_000_000, 20_000, 13, 100),
    ("c3", 4, [5, 7, 9, 11, 13], 2_000_000, 20_000, 4, 40),
    ("c4a", 15, [8], 2_000_000, 20_000, 8, 8),
    ("c4b", 27, [5], 2_000_000, 20_000, 5, 5),
    ("c5", 4, [16], 4_000_000, 20_000, 16, 64),
    ("short", 4, [12], 300_000, 4000, 1, 30),
    ("dna15_mix", 15, [8], 300_000, 6000, 1, 30),
    ("aa27_mix", 27, [5], 300_000, 6000, 1, 20),
    ("dna5", 5, [13], 300_000, 4000, 5, 40),
    # hashes wider than 32 bits (legal in the reference: k < 64 / log2(sigma), kmer_index.hpp:42)
    ("dna4_k20", 4, [20], 500_000, 6000, 10, 70),
    ("dna4_k31", 4, [31], 300_000, 4000, 20, 100),
    ("dna15_k10", 15, [10], 300_000, 6000, 5, 30),
    ("dna15_multi", 15, [10, 11, 12], 300_000, 6000, 5, 40),
    ("dna4_mixed", 4, [9, 21], 300_000, 6000, 5, 70),
    # k-mers wider than one 64-bit packed window (aa27 k >= 9, dna5 k >= 17)
    ("aa27_k12", 27, [12], 300_000, 6000, 6, 40),
    ("aa27_k9_10", 27, [9, 10], 300_000, 6000, 5, 45),
    ("dna5_k20", 5, [20], 300_000, 6000, 12, 70),
    ("dna5_k13_18_27", 5, [13, 18, 27], 200_000, 6000, 10, 90),
]


@pytest.mark.parametrize("label,sigma,ks,n,Q,m_lo,m_hi", CASES)
@pytest.mark.parametrize("qkind", ["random", "stress", "stress-noaux"])
def test_cuda_matches_oracle(kb, oracle_mod, label, sigma, ks, n, Q, m_lo, m_hi, qkind):
    from kmer_index_b200 import synth
    text = synth.random_text(n, sigma, 200 + len(label))
    if qkind == "random":
        q, off = synth.random_queries(Q, m_lo, m_hi, sigma, 1234 + len(label))
    else:
        q, off = synth.stress_queries(text, Q, m_lo, m_hi, sigma, 4321 + len(label))
    # "noaux": sub-k results come from the slab + segment-sort path instead of auxiliary k' = m elements
    with kb.KmerIndex(text, sigma, ks, aux_elements=qkind != "stress-noaux") as ix, oracle_mod.Oracle(text, sigma, ks) as o:
        want = o.search(q, off)
        for attempt in range(2):   # the second batch runs with the auxiliary elements already built
            got = ix.search_batch(q, off).as_tuple()
            assert_results_equal(got, want, label=f"{label}/{qkind}/{attempt}")
        if qkind != "random":
            assert want[1].size > 0


@pytest.mark.parametrize("sigma,ks,n,m_hi", [(4, [12], 200_000, 60), (4, [5, 7, 9, 11, 13], 200_000, 45),
                                             (15, [8], 100_000, 30), (4, [16], 100_000, 70),
                                             (27, [12], 100_000, 40), (5, [18], 100_000, 60)])
def test_correct_mode_matches_ground_truth(kb, oracle_mod, sigma, ks, n, m_hi):
    from kmer_index_b200 import synth
    text = synth.random_text(n, sigma, 31)
    text[1000:1400] = np.resize(np.array([0, 1, 1], dtype=np.uint8), 400)  # a repetitive stretch
    q, off = synth.stress_queries(text, 3000, 1, m_hi, sigma, 5150)
    with kb.KmerIndex(text, sigma, ks, mode=kb.MODE_CORRECT) as ix:
        got = ix.search_batch(q, off).as_tuple()
    want = oracle_mod.Oracle.truth(text, q, off)
    assert_results_equal(got, want, label=f"correct {ks}")


def test_edge_cases(kb):
    text = np.array([0, 1, 2, 3, 0, 1, 2, 3, 0, 1], dtype=np.uint8)
    with kb.KmerIndex(text, 4, [3]) as ix:
        # empty batch
        r = ix.search_batch(np.zeros(0, np.uint8), np.zeros(1, np.uint64))
        assert len(r) == 0 and r.offsets.tolist() == [0]
        # empty query inside a batch -> UNDEFINED status, no hits
        r = ix.search_batch(np.array([0, 1, 2], np.uint8), np.array([0, 0, 3], np.uint64))
        assert r.status.tolist() == [kb.QUERY_UNDEFINED, kb.QUERY_OK]
        assert r.positions.tolist() == [0, 4]
        # query longer than the text
        r = ix.search_batch(np.resize(text, 30), np.array([0, 30], np.uint64))
        assert r.status.tolist() == [0] and r.positions.size == 0
        # end of text: sub-k query matching only in the last k-1 positions (check_last_kmer)
        assert ix.search(np.array([0, 1], np.uint8)).tolist() == [0, 4, 8]
        assert ix.search(np.array([1], np.uint8)).tolist() == [1, 5, 9]
        # text of exactly k symbols
    with kb.KmerIndex(text[:3], 4, [3]) as ix:
        assert ix.search(np.array([0, 1, 2], np.uint8)).tolist() == [0]
        assert ix.search(np.array([1, 2], np.uint8)).tolist() == [1]
    # invalid rank is an error, not a silent wrong answer
    with pytest.raises(kb.KmerB200Error):
        kb.KmerIndex(np.array([0, 1, 2, 7, 1, 1], np.uint8), 4, [3])
    with pytest.raises(kb.KmerB200Error):
        kb.KmerIndex(text, 4, [40])   # k >= 64 / log2(sigma)
    with kb.KmerIndex(text, 4, [3]) as ix:
        with pytest.raises(kb.KmerB200Error):
            ix.search(np.array([0, 9, 1], np.uint8))
        # m > 10000 throws in the reference
        with pytest.raises(ValueError):
            ix.search(np.zeros(10001, np.uint8))
        # a sharded search that is begun and given up leaves the index usable
        import torch
        dq = torch.tensor([0, 1, 2, 1, 2, 3], dtype=torch.uint8, device="cuda")
        doff = torch.tensor([0, 3, 6], dtype=torch.int64, device="cuda")
        flags = torch.zeros(2, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()   # the index works on its own stream
        before = ix.device_bytes
        ix.search_sharded_abort(ix.search_sharded_begin(dq.data_ptr(), doff.data_ptr(), 2, 3, flags.data_ptr()))
        assert ix.device_bytes == before
        assert ix.search(np.array([0, 1, 2], np.uint8)).tolist() == [0, 4]


def _sharded_shape(sigma, ks, n, m_lo, m_hi, world, group, i):
    label = f"{sigma}-ks{i}-{n}-{m_lo}-{m_hi}-{world}" + (f"-G{group}" if group else "")
    return pytest.param(sigma, ks, n, m_lo, m_hi, world, group, id=label)


@pytest.mark.parametrize("fmt", [0, 1, "fused"])
@pytest.mark.parametrize("sigma,ks,n,m_lo,m_hi,world,group", [
    _sharded_shape(*shape, i) for i, shape in enumerate([
        (4, [16], 400_000, 16, 64, 2, 0), (4, [12], 300_000, 13, 64, 3, 0), (4, [5, 7, 9, 11, 13], 200_000, 4, 40, 2, 0),
        (15, [8], 200_000, 3, 20, 4, 0), (27, [12], 200_000, 8, 40, 2, 0)])] + [
    # the presence and deferred passes with G lanes per query forced (KMER_B200_GROUP)
    _sharded_shape(sigma, ks, n, m_lo, m_hi, world, group, i)
    for i, (sigma, ks, n, m_lo, m_hi, world) in ((2, (4, [5, 7, 9, 11, 13], 200_000, 4, 40, 2)), (3, (15, [8], 200_000, 3, 20, 4)))
    for group in (2, 4, 8)])
def test_sharded_search_emulated_on_one_gpu(kb, oracle_mod, monkeypatch, sigma, ks, n, m_lo, m_hi, world, group, fmt):
    """The sharded path (position-range shards with halo, presence OR, global-presence search, rank-order merge)
    run as `world` indices on one GPU must equal the unsharded reference-exact result."""
    import torch

    from kmer_index_b200 import sharded, synth
    from test_gpu_variants import kernel_summary, kernels_launched, lanes, template_args
    dev = torch.device("cuda", 0)
    stack = contextlib.ExitStack()
    if group:
        monkeypatch.setenv("KMER_B200_GROUP", str(group))
        names = stack.enter_context(kernels_launched())
    text = synth.random_text(n, sigma, 91)
    if group:
        text[30_000:31_500] = 1     # ~1500 consecutive hits for the constant queries, answered by the G-lane launch
    q, off = synth.stress_queries(text, 5000, m_lo, m_hi, sigma, 92)
    Q = off.size - 1
    d_q = torch.from_numpy(q).to(dev)
    d_off = torch.from_numpy(off.view(np.int64)).to(dev)
    stream = torch.cuda.current_stream().cuda_stream
    shards = [sharded.shard_range(n, world, r, halo=m_hi - 1) for r in range(world)]
    idx = [kb.KmerIndex(text[s.begin:s.begin + s.length], sigma, ks, shard_begin=s.begin, n_total=n, halo=s.halo,
                        stream=stream or None) for s in shards]
    try:
        masks, pending = [], []
        for ix in idx:
            m = torch.zeros(Q, dtype=torch.int64 if fmt == 0 else torch.int32, device=dev)
            if fmt == "fused":   # count pass with deferred presence rule
                pending.append(ix.search_sharded_begin(d_q.data_ptr(), d_off.data_ptr(), Q, m_hi, m.data_ptr()))
            else:
                ix.presence_batch_device(d_q.data_ptr(), d_off.data_ptr(), Q, m_hi, m.data_ptr(), fmt=fmt)
            torch.cuda.synchronize()
            masks.append(m)
        # what the NCCL exchange computes: OR of bit masks (fmt 0) / SUM of nibble flags (fmt 1, fused)
        present = sharded.fold_presence(torch.stack(masks)) if fmt == 0 else torch.stack(masks).sum(0).to(torch.int32)
        per_shard = []
        for i, ix in enumerate(idx):
            if fmt == "fused":
                r = ix.search_sharded_finish(pending[i], present.data_ptr(), Q)
            else:
                r = ix.search_batch_device_global(d_q.data_ptr(), d_off.data_ptr(), Q, m_hi, present.data_ptr(), fmt=fmt)
            torch.cuda.synchronize()
            o = torch.as_tensor(r.offsets(), device=dev).clone()
            p = (torch.as_tensor(r.positions(), device=dev).clone() if r.n_positions
                 else torch.empty(0, dtype=torch.int32, device=dev))
            st = torch.as_tensor(r.status(), device=dev).clone()
            r.free()
            per_shard.append((o, p, st))
        counts = torch.stack([o[1:] - o[:-1] for o, _, _ in per_shard])
        g_off, base = sharded.merge_offsets(counts)
        final = torch.empty(int(g_off[-1].item()), dtype=torch.int32, device=dev)
        for r, (o, p, _) in enumerate(per_shard):
            sharded.place_shard(final, o, p, base[r])
        got = (g_off.cpu().numpy().astype(np.uint64), final.cpu().numpy().view(np.uint32), per_shard[0][2].cpu().numpy())
        for _, _, st in per_shard[1:]:
            assert torch.equal(st, per_shard[0][2])
    finally:
        for ix in idx:
            ix.close()
        stack.close()
    with oracle_mod.Oracle(text, sigma, ks) as o:
        want = o.search(q, off)
    assert_results_equal(got, want, label=f"sharded x{world} {ks} G={group}")
    assert want[1].size > 0
    if group:
        # the presence pass (fmt 0, 1) or the deferred count pass (fused) ran with G lanes, and so did every other pass
        first_pass = "4" if fmt == "fused" else "2"
        assert lanes(names, "search_kernel") == {group}, kernel_summary(names)
        assert any(a[0] == first_pass for a in template_args(names, "search_kernel")), kernel_summary(names)


@pytest.mark.parametrize("sigma,ks,n,m_lo,m_hi,world", [(4, [16], 400_000, 16, 64, 2), (4, [5, 7, 9, 11, 13], 200_000, 4, 40, 3),
                                                       (27, [12], 200_000, 8, 40, 2), (4, [12], 300_000, 13, 64, 4),
                                                       (4, [12], 150_001, 13, 48, 2), (4, [5, 7, 9, 11, 13], 150_001, 4, 40, 3)])
def test_sharded_merged_finish_emulated_on_one_gpu(kb, oracle_mod, sigma, ks, n, m_lo, m_hi, world):
    """Merging inside the finish of shard 0 (kmer_b200_search_sharded_add_counts): the other shards' sparse counts
    are added before shard 0's offsets scan, its own hits land in place, the other lists are copied behind them.
    A batch that still needs the segment sort refuses (code -5) and is merged from the finished CSRs instead; the
    second batch (auxiliary elements built by then) takes the merged path. Both must equal the unsharded result."""
    import torch

    from kmer_index_b200 import sharded, synth
    dev = torch.device("cuda", 0)
    text = synth.random_text(n, sigma, 93)
    q, off = synth.stress_queries(text, 5000, m_lo, m_hi, sigma, 94)
    if n == 150_001:
        # a 70 000-symbol constant run: queries inside it have candidate lists far beyond 2048 entries and are
        # answered by the warp-per-query ("heavy") launch -- they must reach the hit list the merge works from
        text[20_000:90_000] = 0
        lens = (off[1:] - off[:-1]).astype(np.int64)
        for i in range(0, 900, 3):
            q[int(off[i]):int(off[i]) + int(lens[i])] = 0
    Q = off.size - 1
    d_q = torch.from_numpy(q).to(dev)
    d_off = torch.from_numpy(off.view(np.int64)).to(dev)
    stream = torch.cuda.current_stream().cuda_stream
    shards = [sharded.shard_range(n, world, r, halo=m_hi - 1) for r in range(world)]
    idx = [kb.KmerIndex(text[s.begin:s.begin + s.length], sigma, ks, shard_begin=s.begin, n_total=n, halo=s.halo,
                        stream=stream or None) for s in shards]
    with oracle_mod.Oracle(text, sigma, ks) as o:
        want = o.search(q, off)
    assert want[1].size > 0
    took_merged_path = False
    try:
        for attempt in range(2):
            masks = [torch.zeros(Q, dtype=torch.int32, device=dev) for _ in idx]
            pending = [ix.search_sharded_begin(d_q.data_ptr(), d_off.data_ptr(), Q, m_hi, m.data_ptr())
                       for ix, m in zip(idx, masks)]
            torch.cuda.synchronize()
            present = torch.stack(masks).sum(0).to(torch.int32)
            others, keep = [], []
            for r in range(1, world):
                # the sparse counts are available before the shard's own scan and write pass
                pc, pl = idx[r].search_sharded_peek(pending[r], present.data_ptr(), Q)
                pc, pl = torch.as_tensor(pc, device=dev), torch.as_tensor(pl, device=dev)
                early_q = torch.sort(pl[1:1 + int(pl[0].item())].to(torch.int64) & 0xFFFFFFFF).values
                early_c = pc[early_q].clone()
                early_q, early_c = early_q[early_c > 0], early_c[early_c > 0]
                res = idx[r].search_sharded_finish(pending[r], present.data_ptr(), Q)
                torch.cuda.synchronize()
                o_r = torch.as_tensor(res.offsets(), device=dev)
                p_r = (torch.as_tensor(res.positions(), device=dev).clone() if res.n_positions
                       else torch.empty(0, dtype=torch.int32, device=dev))
                q_r, c_r = sharded.sparse_lists(o_r, sharded._hit_ids(res, dev))
                assert torch.equal(q_r, early_q) and torch.equal(c_r, early_c)
                others.append((q_r.clone(), c_r.clone(), p_r))
                res.free()
            within = []
            try:
                for q_r, c_r, _ in others:
                    w = torch.empty(q_r.numel(), dtype=torch.int64, device=dev)
                    idx[0].search_sharded_add_counts(pending[0], present.data_ptr(), q_r.data_ptr(), c_r.data_ptr(),
                                                     q_r.numel(), w.data_ptr())
                    within.append(w)
                merged = True
            except kb.KmerB200Error as e:
                assert e.code == -5 and not within
                merged = False
            res0 = idx[0].search_sharded_finish(pending[0], present.data_ptr(), Q)
            torch.cuda.synchronize()
            offsets = torch.as_tensor(res0.offsets(), device=dev)
            positions = (torch.as_tensor(res0.positions(), device=dev) if res0.n_positions
                         else torch.empty(0, dtype=torch.int32, device=dev))
            if merged:
                took_merged_path = True
                for (q_r, c_r, p_r), w in zip(others, within):
                    sharded.place_lists(positions, offsets[q_r] + w, c_r, p_r)
                g_off, final = offsets, positions
            else:
                g_off, final = sharded.merge_lists(offsets, positions, sharded.sparse_lists(offsets, sharded._hit_ids(res0, dev)),
                                                   others)
            got = (g_off.cpu().numpy().astype(np.uint64), final.cpu().numpy().view(np.uint32),
                   torch.as_tensor(res0.status(), device=dev).cpu().numpy())
            res0.free()
            assert_results_equal(got, want, label=f"merged finish x{world} {ks} attempt {attempt} merged={merged}")
    finally:
        for ix in idx:
            ix.close()
    assert took_merged_path


@pytest.mark.parametrize("sigma,ks,n,parts", [(4, [12], 300_000, 4), (4, [16], 400_000, 8), (4, [5, 7, 9, 11, 13], 200_000, 3),
                                               (15, [8], 200_000, 2), (27, [5], 150_000, 5)])
def test_key_range_parts_assemble_to_the_whole_index(kb, oracle_mod, sigma, ks, n, parts):
    """Multi-GPU build of a replicated index, emulated on one GPU: `parts` indices, each holding the k-mers of one
    key-range part, are concatenated (positions part after part, directory entries offset by the earlier parts'
    k-mer counts) and adopted -- the result must equal the index built in one piece, CSR and answers. Before the
    adoption a part answers with exactly its own share of every hit list."""
    import torch

    from kmer_index_b200 import sharded, synth
    dev = torch.device("cuda", 0)
    text = synth.random_text(n, sigma, 71)
    text[1000:1400] = 0                                      # a long bucket that lands in one part
    q, off = synth.stress_queries(text, 4000, 1, 48, sigma, 72)
    stream = torch.cuda.current_stream().cuda_stream
    idx = [kb.KmerIndex(text, sigma, ks, key_part=r, key_parts=parts, stream=stream or None) for r in range(parts)]
    try:
        with oracle_mod.Oracle(text, sigma, ks) as o:
            want = o.search(q, off)
            want_csr = [o.element(e) for e in range(len(ks))]
        exact = (off[1:] - off[:-1]) == ks[0] if len(ks) == 1 else None
        if exact is not None:
            # exact-k queries: the bucket of the query lives in exactly one part; the parts' hit counts add up
            per_part = [ix.search_batch(q, off) for ix in idx]
            total = sum((r.offsets[1:] - r.offsets[:-1]).astype(np.int64) for r in per_part)
            assert np.array_equal(total[exact], (want[0][1:] - want[0][:-1]).astype(np.int64)[exact])
        for e, k in enumerate(ks):
            ps = [ix.element_part(e) for ix in idx]
            assert sum(p.n_kmers for p in ps) == n - k + 1
            assert ps[0].key_lo == 0 and ps[-1].key_hi == sigma ** k
            pos_full = torch.empty(n - k + 1, dtype=torch.int32, device=dev)
            dir_full = torch.empty(sigma ** k + 1, dtype=torch.int32, device=dev)
            base = 0
            for r, (ix, p) in enumerate(zip(idx, ps)):
                assert p.key_hi - p.key_lo + 1 == p.directory_entries
                if r:
                    assert p.key_lo == ps[r - 1].key_hi
                pos_full[base:base + p.n_kmers].copy_(sharded._dev_view(p.d_positions, p.n_kmers, dev))
                n_dir = p.key_hi - p.key_lo + (1 if r == parts - 1 else 0)
                ix.export_directory(e, base, n_dir, dir_full.data_ptr() + 4 * p.key_lo)
                base += p.n_kmers
            torch.cuda.synchronize()
            idx[0].adopt_element(e, pos_full, dir_full)
            h, p_ = idx[0].element_arrays(e)
            assert np.array_equal(p_, want_csr[e][1]) and np.array_equal(h, want_csr[e][0])
        for attempt in range(2):     # the second batch runs with the auxiliary elements the first one built
            assert_results_equal(idx[0].search_batch(q, off).as_tuple(), want, label=f"assembled {ks} x{parts}/{attempt}")
    finally:
        for ix in idx:
            ix.close()


@pytest.mark.parametrize("sigma,ks,n,parts", [(4, [12], 300_000, 4), (4, [16], 400_000, 8), (4, [5, 7, 9, 11, 13], 200_000, 3)])
def test_positions_left_in_parts_answer_like_the_whole_index(kb, oracle_mod, sigma, ks, n, parts):
    """Peer-positions multi-GPU index, emulated on one GPU: the directory is assembled whole, the position array stays
    in the key-range parts (here: separate buffers of the same GPU) and kmer_b200_adopt_element_parts points at them."""
    import torch

    from kmer_index_b200 import sharded, synth
    dev = torch.device("cuda", 0)
    text = synth.random_text(n, sigma, 73)
    text[1000:4400] = 0                                      # a bucket beyond the heavy threshold, in one part
    q, off = synth.stress_queries(text, 4000, 1, 48, sigma, 74)
    stream = torch.cuda.current_stream().cuda_stream
    idx = [kb.KmerIndex(text, sigma, ks, key_part=r, key_parts=parts, stream=stream or None) for r in range(parts)]
    try:
        with oracle_mod.Oracle(text, sigma, ks) as o:
            want = o.search(q, off)
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
            with pytest.raises(kb.KmerB200Error):
                idx[0].element_arrays(e)                     # the positions are not one array any more
        for attempt in range(2):
            assert_results_equal(idx[0].search_batch(q, off).as_tuple(), want, label=f"positions in parts {ks} x{parts}/{attempt}")
        if len(ks) == 1:
            assert_results_equal(idx[0].search_batch(q, off, mode=kb.MODE_CORRECT).as_tuple(), oracle_mod.Oracle.truth(text, q, off),
                                 label="positions in parts, CORRECT mode")
    finally:
        for ix in idx:
            ix.close()


@pytest.mark.parametrize("sigma,k,n,parts", [(4, 12, 300_000, 4), (4, 16, 400_000, 8), (4, 10, 3_000_000, 2)])
def test_directory_parts_travel_as_bucket_sizes(kb, sigma, k, n, parts):
    """The replicated multi-GPU build ships every part's directory as one byte per bucket and rebuilds the whole
    directory with a prefix sum: must equal the directory assembled from the 4-byte entries; a bucket of >= 255 k-mers
    is reported instead of being truncated."""
    import torch

    from kmer_index_b200 import synth
    dev = torch.device("cuda", 0)
    text = synth.random_text(n, sigma, 81)
    stream = torch.cuda.current_stream().cuda_stream
    idx = [kb.KmerIndex(text, sigma, [k], key_part=r, key_parts=parts, stream=stream or None) for r in range(parts)]
    try:
        key_space = sigma ** k
        ps = [ix.element_part(0) for ix in idx]
        dir_a = torch.empty(key_space + 1, dtype=torch.int32, device=dev)
        sizes = torch.empty(key_space, dtype=torch.uint8, device=dev)
        base = 0
        for r, (ix, p) in enumerate(zip(idx, ps)):
            ix.export_directory(0, base, p.key_hi - p.key_lo + (1 if r == parts - 1 else 0), dir_a.data_ptr() + 4 * p.key_lo)
            assert ix.export_bucket_sizes(0, sizes.data_ptr() + p.key_lo) == 0
            base += p.n_kmers
        torch.cuda.synchronize()
        dir_b = torch.full((key_space + 1,), -1, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()                                  # the index works on its own stream
        idx[0].directory_from_sizes(sizes.data_ptr(), key_space, dir_b.data_ptr())
        torch.cuda.synchronize()
        assert torch.equal(dir_a, dir_b)
        assert int(dir_b[-1].item()) == n - k + 1
    finally:
        for ix in idx:
            ix.close()
    low = text.copy()
    low[1000:1400] = 0                                            # one bucket of ~390 k-mers
    with kb.KmerIndex(low, sigma, [k], key_part=0, key_parts=parts) as ix:
        scratch = torch.empty(key_space, dtype=torch.uint8, device=dev)
        assert ix.export_bucket_sizes(0, scratch.data_ptr()) >= 1


@pytest.mark.parametrize("sigma,k,n,m_hi,parts,mode", [(4, 16, 500_000, 64, 4, 0), (4, 12, 300_000, 100, 3, 0), (4, 12, 300_000, 60, 8, 1),
                                                        (15, 8, 200_000, 40, 2, 0), (27, 5, 150_000, 24, 5, 0)])
def test_routed_search_on_key_range_parts_emulated(kb, oracle_mod, sigma, k, n, m_hi, parts, mode):
    """The partitioned multi-GPU search, all ranks emulated on one GPU: `parts` indices each hold one key-range part,
    every "rank" routes its slice of the batch to the owners of the queries' first k-mers (send blocks), owners search
    what they received and send results back, origins restore batch order. The three all-to-all exchanges are plain
    tensor copies here. Result must equal the oracle (REFERENCE_EXACT incl. the whole-text presence rules through the
    shared bitmap; CORRECT against the plain scan)."""
    import torch

    from kmer_index_b200 import synth
    dev = torch.device("cuda", 0)
    text = synth.random_text(n, sigma, 61)
    text[5000:9000] = np.resize(text[100:100 + k], 4000)      # a periodic stretch: the defective plans become non-empty
    text[20_000:24_000] = 0                                    # and a long bucket
    q, off = synth.stress_queries(text, 6000, k, m_hi, sigma, 62)
    Q = off.size - 1
    stream = torch.cuda.current_stream().cuda_stream
    idx = [kb.KmerIndex(text, sigma, [k], key_part=r, key_parts=parts, stream=stream or None, mode=mode) for r in range(parts)]
    try:
        if mode == 0:
            with oracle_mod.Oracle(text, sigma, [k]) as o:
                want = o.search(q, off)
        else:
            want = oracle_mod.Oracle.truth(text, q, off)
        # presence bitmap: every part exports its slice, the slices are disjoint -> sum == or
        words = idx[0].presence_words(0)
        bits = torch.zeros(words, dtype=torch.int64, device=dev)
        for ix in idx:
            part = torch.zeros(words, dtype=torch.int64, device=dev)
            torch.cuda.synchronize()
            ix.presence_export(0, part.data_ptr())      # enqueued on the index's own stream
            torch.cuda.synchronize()
            bits += part
        torch.cuda.synchronize()
        for ix in idx:
            ix.presence_attach(0, bits)
        for attempt in range(2):
            slack = 0.0 if attempt == 0 else 0.01              # the second round starts with blocks that overflow
            lo = [r * Q // parts for r in range(parts + 1)]
            d_q = torch.from_numpy(q).to(dev)
            d_off = [torch.from_numpy((off[lo[r]:lo[r + 1] + 1] - off[lo[r]]).view(np.int64)).to(dev) for r in range(parts)]
            q_ptr = [d_q.data_ptr() + int(off[lo[r]]) for r in range(parts)]
            Ql = [lo[r + 1] - lo[r] for r in range(parts)]
            plan_q = max(Ql)
            while True:
                plan = idx[0].route_plan(plan_q, m_hi, parts, slack)
                send = [torch.empty(parts * plan.block_bytes, dtype=torch.uint8, device=dev) for _ in range(parts)]
                status = [torch.empty(max(Ql[r], 1), dtype=torch.uint8, device=dev) for r in range(parts)]
                sent = [idx[r].route_queries(q_ptr[r], d_off[r].data_ptr(), Ql[r], plan, send[r].data_ptr(), status[r].data_ptr())
                        for r in range(parts)]
                need = max(max(s) for s in sent)
                if need <= plan.capacity:
                    break
                assert attempt == 1
                slack = 1.05 * need * parts / plan_q + 0.05
            B, RB = plan.block_bytes, plan.return_block_bytes
            recv = [torch.cat([send[r][o * B:(o + 1) * B] for r in range(parts)]) for o in range(parts)]       # all-to-all
            ret_send, owner_res, pos_splits = [], [], []
            for o in range(parts):
                rs = torch.empty(parts * RB, dtype=torch.uint8, device=dev)
                res, splits = idx[o].search_routed(recv[o].data_ptr(), plan, rs.data_ptr())
                ret_send.append(rs)
                owner_res.append(res)
                pos_splits.append(splits)
            torch.cuda.synchronize()
            got_off, got_pos, got_st = [np.zeros(1, np.uint64)], [], []
            for r in range(parts):
                ret_recv = torch.cat([ret_send[o][r * RB:(r + 1) * RB] for o in range(parts)])                # all-to-all
                recv_splits = [pos_splits[o][r] for o in range(parts)]
                chunks = []
                for o in range(parts):
                    p_o = (torch.as_tensor(owner_res[o].positions(), device=dev) if owner_res[o].n_positions
                           else torch.empty(0, dtype=torch.int32, device=dev))
                    a = sum(pos_splits[o][:r])
                    chunks.append(p_o[a:a + pos_splits[o][r]])
                pos_recv = torch.cat(chunks) if chunks else torch.empty(0, dtype=torch.int32, device=dev)     # all-to-all-v
                out = idx[r].unroute(send[r].data_ptr(), ret_recv.data_ptr(), plan, sent[r], pos_recv.data_ptr(), recv_splits, Ql[r],
                                     status[r].data_ptr())
                torch.cuda.synchronize()
                o_ = torch.as_tensor(out.offsets(), device=dev).cpu().numpy().astype(np.uint64)
                got_off.append(o_[1:] + got_off[-1][-1])
                got_pos.append(torch.as_tensor(out.positions(), device=dev).cpu().numpy().view(np.uint32) if out.n_positions
                               else np.zeros(0, np.uint32))
                got_st.append(torch.as_tensor(out.status(), device=dev).cpu().numpy())
                out.free()
            for res in owner_res:
                res.free()
            got = (np.concatenate(got_off), np.concatenate(got_pos), np.concatenate(got_st))
            assert_results_equal(got, want, label=f"routed x{parts} k={k} mode={mode} attempt {attempt}")
        assert want[1].size > 1000
    finally:
        for ix in idx:
            ix.close()


@pytest.mark.parametrize("sigma,ks", [(4, [12]), (4, [5, 7, 9, 11, 13]), (15, [8]), (4, [20])])
def test_heavy_buckets_take_the_warp_path(kb, oracle_mod, sigma, ks):
    """A text with one enormous bucket (a long constant run): the index-wide average bucket is ~1, so queries get
    one or two lanes each -- except those whose candidate list is long, which are handed to the warp-per-query
    launch. Results must not depend on which launch answered."""
    from kmer_index_b200 import synth
    text = synth.random_text(150_000, sigma, 5)
    text[20_000:90_000] = 0
    text[100_000:100_300] = np.resize(np.array([1, 0, 0], dtype=np.uint8), 300)
    q, off = synth.stress_queries(text, 3000, 1, 48, sigma, 6, low_sigma=2)
    # make sure the batch contains constant queries of many lengths (they hit the 70 000-element buckets)
    lens = (off[1:] - off[:-1]).astype(np.int64)
    for i in range(0, 600, 3):
        q[int(off[i]):int(off[i]) + int(lens[i])] = 0
    with kb.KmerIndex(text, sigma, ks) as ix, oracle_mod.Oracle(text, sigma, ks) as o:
        want = o.search(q, off)
        for attempt in range(2):
            got = ix.search_batch(q, off).as_tuple()
            assert_results_equal(got, want, label=f"heavy {ks}/{attempt}")
        assert int((want[0][1:] - want[0][:-1]).max()) > 2048
    with kb.KmerIndex(text, sigma, ks, mode=kb.MODE_CORRECT) as ix:
        assert_results_equal(ix.search_batch(q, off).as_tuple(), oracle_mod.Oracle.truth(text, q, off), label="heavy correct")


@pytest.mark.parametrize("sigma,ks", [(4, [12]), (4, [5, 7, 9, 11, 13]), (15, [10]), (27, [5]), (27, [12])])
def test_save_load_round_trip(kb, oracle_mod, tmp_path, sigma, ks):
    """Construct once, load later: the loaded index answers exactly like the built one (and like the oracle)."""
    from kmer_index_b200 import synth
    text = synth.random_text(120_000, sigma, 3)
    q, off = synth.stress_queries(text, 3000, 1, 45, sigma, 4)
    path = str(tmp_path / "index.kmerb200")
    with kb.KmerIndex(text, sigma, ks) as ix:
        built = ix.search_batch(q, off).as_tuple()
        arrays = [ix.element_arrays(e) for e in range(len(ks))]
        ix.save(path)
    with kb.KmerIndex.load(path) as ld:
        assert ld.ks == list(ks) and ld.n == text.size
        assert_results_equal(ld.search_batch(q, off).as_tuple(), built, label="loaded vs built")
        for e in range(len(ks)):
            h, p = ld.element_arrays(e)
            assert np.array_equal(h, arrays[e][0]) and np.array_equal(p, arrays[e][1])
    with oracle_mod.Oracle(text, sigma, ks) as o:
        assert_results_equal(built, o.search(q, off), label="built vs oracle")
    with pytest.raises(kb.KmerB200Error):
        bad = tmp_path / "bad.bin"
        bad.write_bytes(b"not an index" * 100)
        kb.KmerIndex.load(str(bad))


@pytest.mark.parametrize("alphabet,ks", [("dna4", [12]), ("dna15", [8]), ("aa27", [5])])
def test_character_input_matches_rank_input(kb, alphabet, ks):
    """Texts/queries given as characters (device-side translation through a 256-entry table) == given as ranks."""
    from kmer_index_b200 import synth
    sigma = kb.ALPHABETS[alphabet]
    chars = np.frombuffer(kb.ALPHABET_CHARS[alphabet].encode(), dtype=np.uint8)
    text = synth.random_text(100_003, sigma, 8)
    q, off = synth.stress_queries(text, 500, 1, 30, sigma, 9)
    queries = [chars[q[int(off[i]):int(off[i + 1])]].tobytes() for i in range(off.size - 1)]
    queries[3] = queries[3].lower()                       # case-insensitive
    lut = kb.char_lut(alphabet)
    with kb.KmerIndex(text, sigma, ks) as a, kb.KmerIndex(chars[text].tobytes(), sigma, ks, lut=lut) as b:
        want = a.search_batch(q, off).as_tuple()
        assert_results_equal(b.search_batch_text(queries).as_tuple(), want, label="chars")
        assert_results_equal(b.search_batch(q, off).as_tuple(), want, label="ranks on char-built index")
        with pytest.raises(kb.KmerB200Error):
            b.search_batch_text([b"ACG?T"])
    with pytest.raises(kb.KmerB200Error):
        kb.KmerIndex(b"ACGTNACGT" * 10, 4, [3], lut=kb.char_lut("dna4"))   # N is not in dna4


@pytest.mark.parametrize("sigma,ks", [(4, [12]), (4, [9, 13]), (27, [5]), (4, [3])])
def test_long_queries_up_to_the_table_limit(kb, oracle_mod, sigma, ks):
    """Queries of hundreds to 9999 symbols (kmer_index.hpp:401: the scheme table covers lengths < 10000): many
    parts per query, packed query staged over several rounds, a full warp per query."""
    from kmer_index_b200 import synth
    text = synth.random_text(60_000, sigma, 12)
    text[30_000:42_000] = np.resize(text[100:160], 12_000)        # a long periodic stretch: multi-part matches exist
    lens = [200, 777, 1024, 2047, 4999, 9998, 9999, 10000, 10001]
    qs = []
    for i, m in enumerate(lens * 3):
        start = [0, 30_000 + 17, 60_000 - m if m <= 60_000 else 0][i % 3]
        piece = text[start:start + m]
        if piece.size < m:
            piece = np.resize(piece, m)
        qs.append(piece.copy())
    qs[5][-1] ^= 1                                                  # a near miss
    q = np.concatenate(qs)
    off = np.zeros(len(qs) + 1, dtype=np.uint64)
    np.cumsum([x.size for x in qs], out=off[1:])
    with kb.KmerIndex(text, sigma, ks) as ix, oracle_mod.Oracle(text, sigma, ks) as o:
        got = ix.search_batch(q, off).as_tuple()
        want = o.search(q, off)
        ub = o.last_ub
    assert_results_equal(got, want, label=f"long {ks}")
    assert set(want[2].tolist()) >= {0, 1, 2}                      # OK, THROW (m > 10000) and UNDEFINED (m == 10000)
    with kb.KmerIndex(text, sigma, ks, mode=kb.MODE_CORRECT) as ix:
        keep = np.array([x.size < 10000 for x in qs])
        got = ix.search_batch(q, off).as_tuple()
        truth = oracle_mod.Oracle.truth(text, q, off)
        for i in np.flatnonzero(keep):
            assert np.array_equal(got[1][int(got[0][i]):int(got[0][i + 1])], truth[1][int(truth[0][i]):int(truth[0][i + 1])]), i
    del ub


@pytest.mark.parametrize("directory_bits", [12, 18, 30])
def test_sparse_directory_and_accounting_variants(kb, oracle_mod, directory_bits):
    """directory_bits caps the directory (hash >> shift indexing + binary search in the sorted hashes); profile=2
    runs the count pass that also sums the gathered sectors. Neither may change a result."""
    from kmer_index_b200 import synth
    text = synth.random_text(200_000, 4, 21)
    q, off = synth.stress_queries(text, 4000, 1, 60, 4, 22)
    with oracle_mod.Oracle(text, 4, [12]) as o:
        want = o.search(q, off)
    with kb.KmerIndex(text, 4, [12], directory_bits=directory_bits, profile=2) as ix:
        info = ix.element_info(0)
        assert info.directory_shift == max(0, 24 - directory_bits)
        assert_results_equal(ix.search_batch(q, off).as_tuple(), want, label=f"dir_bits={directory_bits}")
        assert ix.last_search_gathers > 0
        st = ix.stats()
        assert st["search_count"]["launches"] >= 1 and st["search_count"]["device_ms"] > 0


def _fasta(records, width, crlf=False, comments=False):
    nl = b"\r\n" if crlf else b"\n"
    out = []
    for name, seq in records:
        out.append(b">" + name + nl)
        if comments:
            out.append(b";a comment line" + nl)
        for i in range(0, len(seq), width):
            out.append(seq[i:i + width] + nl)
    return b"".join(out)


@pytest.mark.parametrize("variant", ["fasta", "fasta-crlf-comments", "fasta-no-final-newline", "fasta-headerless-start", "fastq"])
def test_fasta_fastq_parsed_on_the_device(kb, variant):
    """Multi-record FASTA / FASTQ bytes -> concatenated ranks + record table (device parser) == a plain Python parser;
    an index over the records finds every planted window in its record, and matches that span a record boundary are
    recognisable."""
    from kmer_index_b200 import synth
    chars = np.frombuffer(b"ACGT", dtype=np.uint8)
    rng = np.random.default_rng(5)
    lens = [3000, 1, 64, 70_001, 2047, 2048, 2049, 10, 500_000]
    seqs = [chars[synth.random_text(m, 4, 100 + i)].tobytes() for i, m in enumerate(lens)]
    seqs[3] = seqs[3].lower()                                       # soft-masked: case-insensitive table
    recs = [(f"rec{i} some description".encode(), s) for i, s in enumerate(seqs)]
    if variant == "fastq":
        data = b"".join(b"@" + n + b"\n" + s + b"\n+\n" + bytes(rng.integers(33, 74, len(s), dtype=np.uint8)) + b"\n" for n, s in recs)
    else:
        data = _fasta(recs, 61, crlf="crlf" in variant, comments="comments" in variant)
        if variant == "fasta-no-final-newline":
            data = data.rstrip(b"\n")
        if variant == "fasta-headerless-start":
            data = seqs[0][:100] + b"\n" + data
            recs = [(b"", seqs[0][:100])] + recs
    want = np.concatenate([np.frombuffer(s.upper(), dtype=np.uint8) for _, s in recs])
    want = np.searchsorted(chars, want).astype(np.uint8)
    want_starts = np.concatenate([[0], np.cumsum([len(s) for _, s in recs])]).astype(np.uint64)
    with kb.parse_sequences(data, "dna4") as r:
        assert len(r) == len(recs) and r.n_symbols == want.size
        assert np.array_equal(r.starts, want_starts)
        for i, (name, _) in enumerate(recs):
            assert r.name(i).encode() == name
        with r.index([12]) as ix:
            h, p = ix.element_arrays(0)
            qs, truth = [], []
            for i in [j for j, (_, sq) in enumerate(recs) if len(sq) >= 43][:4] + [len(recs) - 1]:
                s0 = int(want_starts[i]) + 7
                qs.append(want[s0:s0 + 36])           # 3 x k: a length on which the reference's plan is the correct one
                truth.append((i, 7))
            q = np.concatenate(qs)
            off = np.arange(0, 36 * len(qs) + 1, 36, dtype=np.uint64)
            res = ix.search_batch(q, off)
            for j, (rec_i, o_i) in enumerate(truth):
                pos = res.to_vector(j)
                rec, o = r.locate(pos, 36)
                assert (rec_i, o_i) in set(zip(rec.tolist(), o.tolist()))
            # a window that starts 5 symbols before a record boundary only exists because records are concatenated
            s0 = int(want_starts[1]) - 5
            res = ix.search_batch(want[s0:s0 + 24], np.array([0, 24], dtype=np.uint64))
            rec, _ = r.locate(res.to_vector(0), 24)
            assert rec.size >= 1 and (rec == 0xFFFFFFFF).any()
    with kb.KmerIndex(want, 4, [12]) as ref:
        h2, p2 = ref.element_arrays(0)
    assert np.array_equal(p, p2) and np.array_equal(h, h2)
    with pytest.raises(kb.KmerB200Error):
        kb.parse_sequences(b">x\nACGTNACGT\n", "dna4")            # N is not in dna4
