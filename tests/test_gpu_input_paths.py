"""The two paths that turn the caller's bytes into what the search kernels read, checked against plain references.

A. The device FASTA / FASTQ parser (kmer_b200_parse_sequences: three passes over 2048-byte tiles, line state carried
   across tiles by one 1024-thread CTA) against the line-by-line Python parser of tests/fastx_truth.py: the ranks read
   back from the device, the record starts, header offsets, names and symbol count. Line feeds, '\\r', markers and
   record starts are placed on tile and 8-byte thread edges on purpose; inputs of more than 2048 and 4096 tiles make
   every thread of the carry kernel walk several tiles; every alphabet; refusals.
B. The chunked host-batch pipeline (search_batch_host_chunked: 24 chunks, packed ones cut into per-query words on the
   device by align_stream_kernel, raw ones sent as 1-byte ranks) against the single-copy path of the same index
   (KMER_B200_NO_PIPELINE=1) bit for bit, and on a sample against the C restatement oracle (reference mode) and the
   plain scan (MODE_CORRECT). Each run asserts the pipeline, the raw share, the exact host-to-device bytes and how many
   times align_stream_kernel ran, so an override that does nothing fails the case."""
import contextlib
import ctypes as C
import os
from collections import Counter

import numpy as np
import pytest

import fastx_truth
from collection_truth import truth_per_record
from conftest import assert_results_equal

pytestmark = pytest.mark.gpu

TILE = 2048
RESIDUES = (0, 1, 7, 8, TILE - 1)   # tile start, 2048 t + 1, the last byte of a thread's 8, the first of the next, 2048 t - 1


@pytest.fixture(scope="module")
def kb():
    import kmer_index_b200
    return kmer_index_b200


@contextlib.contextmanager
def overrides(**env):
    """set (value) or clear (None) environment variables for the block"""
    old = {k: os.environ.get(k) for k in env}
    for k, v in env.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = str(v)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


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


# ================================================================ A. FASTA / FASTQ parsing on the device

def device_ranks(kb, r):
    import torch
    if r.n_symbols == 0:
        return np.zeros(0, np.uint8)
    ptr = int(r._L.kmer_b200_records_ranks_device(r._h))
    return torch.as_tensor(kb._DevArray(ptr, r.n_symbols, "|u1", r), device="cuda").cpu().numpy()


def assert_parsed(kb, data, alphabet, fmt=0, label=""):
    """the device parser's records == the Python parser's"""
    want = fastx_truth.parse(data, alphabet, fmt)
    with kb.parse_sequences(data, alphabet, fmt) as r:
        assert r.n_symbols == want.ranks.size, (label, r.n_symbols, want.ranks.size)
        got = device_ranks(kb, r)
        diff = np.flatnonzero(got != want.ranks)
        assert diff.size == 0, f"{label}: ranks differ first at symbol {diff[:1]}"
        assert np.array_equal(r.starts, want.starts), (label, r.starts[:8], want.starts[:8])
        assert np.array_equal(r.header_offsets, want.header_offsets), label
        assert [r.name(i) for i in range(len(r))] == want.names, label
    return want


def refused(kb, data, alphabet, fmt=0):
    """the error code of a parse that must fail; the Python parser refuses the same input"""
    with pytest.raises(ValueError):
        fastx_truth.parse(data, alphabet, fmt)
    with pytest.raises(kb.KmerB200Error) as e:
        kb.parse_sequences(data, alphabet, fmt)
    return e.value.code


def _seq(rng, alphabet, m, lower=False):
    from kmer_index_b200 import ALPHABET_CHARS
    chars = np.frombuffer(ALPHABET_CHARS[alphabet].encode(), dtype=np.uint8)
    s = chars[rng.integers(0, chars.size, m)].tobytes()
    if lower and m:                                       # a soft-masked stretch
        a = int(rng.integers(0, m))
        b = int(rng.integers(a, m + 1))
        s = s[:a] + s[a:b].lower() + s[b:]
    return s


def _name(rng, length):
    return rng.integers(33, 127, length, dtype=np.uint8).tobytes()   # printable, no blank, no '\r'


def _qual(rng, m):
    q = rng.integers(33, 127, m, dtype=np.uint8).tobytes()
    if m and rng.random() < 0.3:
        q = (b"@" if rng.random() < 0.5 else b"+") + q[1:]   # a quality line that looks like a header or a '+' line
    return q


def random_layout(rng, alphabet, fmt, size, widths=(60, 61), crlf=False, unwrapped=0):
    """records until `size` bytes: names of 0-40 bytes (5 % of 5000), sequences of 0-3000 symbols (10 % empty), soft-masked
    stretches; FASTA: line widths from `widths`, blanks and tabs inside lines, blank lines, comment lines, sometimes
    sequence before the first header; FASTQ: quality lines that start with '@' or '+'. unwrapped > 0: the first record
    is one line of that many symbols."""
    eol = b"\r\n" if crlf else b"\n"
    out = bytearray()
    if fmt == 1 and rng.random() < 0.3:
        out += _seq(rng, alphabet, int(rng.integers(1, 200))) + eol
    first = True
    while len(out) < size:
        name = _name(rng, 5000 if rng.random() < 0.05 else int(rng.integers(0, 40)))
        r = rng.random()
        m = unwrapped if first and unwrapped else 0 if r < 0.1 else int(rng.integers(1, 30)) if r < 0.3 else int(rng.integers(30, 3000))
        seq = _seq(rng, alphabet, m, lower=rng.random() < 0.2)
        if fmt == 1:
            w = m if first and unwrapped else int(rng.choice(widths))
            out += b">" + name + eol
            for i in range(0, m, w):
                line = seq[i:i + w]
                if rng.random() < 0.05:
                    j = int(rng.integers(0, len(line) + 1))
                    line = line[:j] + (b" " if rng.random() < 0.5 else b"\t") + line[j:]
                out += line + eol
                if rng.random() < 0.03:
                    out += eol
                if rng.random() < 0.03:
                    out += b";" + _name(rng, 20) + eol
        else:
            out += b"@" + name + eol + seq + eol + b"+" + eol + _qual(rng, m) + eol
        first = False
    return bytes(out)


def edge_layout(fmt, crlf, seed, alphabet="dna4"):
    """dna4 records whose header is padded so that one event lands on each residue of RESIDUES (mod 2048) in turn: the
    header's line feed, the '\\r' of its CRLF, the first sequence line's line feed, and the next record's marker (after
    a non-empty and after an empty record: two headers meet there). Returns the bytes and [(offset, expected byte)]."""
    rng = np.random.default_rng(seed)
    eol = b"\r\n" if crlf else b"\n"
    marker = b">" if fmt == 1 else b"@"
    events = [("header_lf", False), ("seq_lf", False), ("next_record", False), ("next_record", True)]
    if crlf:
        events.append(("header_cr", False))
    out, landed = bytearray(), []

    def record(name, seq, qual):
        if fmt == 1:
            return b">" + name + eol + b"".join(seq[i:i + 61] + eol for i in range(0, len(seq), 61))
        return b"@" + name + eol + seq + eol + b"+" + eol + qual + eol

    for event, empty in events:
        for res in RESIDUES:
            m = 0 if empty else int(rng.integers(1, 200))
            seq, qual = _seq(rng, alphabet, m), _qual(rng, m)
            rec0 = record(b"", seq, qual)
            lf = rec0.index(b"\n")
            at = {"header_lf": lf, "header_cr": lf - 1, "seq_lf": rec0.index(b"\n", lf + 1) if m else -1,
                  "next_record": len(rec0)}[event]
            target = (len(out) + at) // TILE * TILE + res
            if target < len(out) + at:
                target += TILE
            out += record(_name(rng, target - len(out) - at), seq, qual)
            landed.append((target, {"header_lf": b"\n", "seq_lf": b"\n", "header_cr": b"\r", "next_record": marker}[event]))
    out += record(b"last", _seq(rng, alphabet, 50), _qual(rng, 50))
    data = bytes(out)
    for at, byte in landed:
        assert data[at:at + 1] == byte, (at, byte)
    return data, landed


@pytest.mark.parametrize("crlf", [False, True], ids=["lf", "crlf"])
@pytest.mark.parametrize("fmt", [1, 2], ids=["fasta", "fastq"])
def test_line_feeds_markers_and_record_starts_on_tile_edges(kb, fmt, crlf):
    for seed in (1, 2):
        data, landed = edge_layout(fmt, crlf, seed)
        assert len({at % TILE for at, _ in landed}) == len(RESIDUES)
        assert_parsed(kb, data, "dna4", fmt, label=f"seed {seed}")
        # the same layout shifted by one byte (a blank first line for FASTA; FASTQ: a longer first name)
        shifted = b"\n" + data if fmt == 1 else b"@x" + data[1:]
        assert_parsed(kb, shifted, "dna4", fmt, label=f"seed {seed} shifted")


@pytest.mark.parametrize("size", [2, 2047, 2048, 2049, 4096])
@pytest.mark.parametrize("fmt", [1, 2], ids=["fasta", "fastq"])
def test_input_sizes_around_one_and_two_tiles(kb, fmt, size):
    rng = np.random.default_rng(size * 3 + fmt)
    for i in range(6):
        body = random_layout(rng, "dna4", fmt, size + 100, widths=(7, 60, 61), crlf=i % 2 == 1)
        data = body[:size]
        assert_parsed(kb, data, "dna4", fmt, label=f"{size} bytes, layout {i}")
        assert_parsed(kb, data[:-1] + b"\n", "dna4", fmt, label=f"{size} bytes ending in a line feed, layout {i}")


def test_one_byte_inputs(kb):
    for data in (b">", b"@", b"A", b"a", b"\n", b"\r", b";"):
        assert_parsed(kb, data, "dna4", 0, label=repr(data))
    assert refused(kb, b"N", "dna4") == -4


@pytest.mark.parametrize("size", [5_000_000, 9_000_000])
@pytest.mark.parametrize("fmt", [1, 2], ids=["fasta", "fastq"])
def test_more_tiles_than_carry_threads(kb, fmt, size):
    """> 2048 and > 4096 tiles: every thread of the 1024-thread carry kernel walks 3 or 5 tiles; a record of one line of
    10^6 symbols leaves ~490 tiles in a row without a line feed"""
    tiles = -(-size // TILE)
    assert tiles > 2048 and tiles % 1024 != 0
    rng = np.random.default_rng(size + fmt)
    data = random_layout(rng, "dna5", fmt, size + 10_000, widths=(60, 61, 2049), unwrapped=1_000_000)[:size]
    want = assert_parsed(kb, data, "dna5", fmt)
    assert want.ranks.size > 1_000_000 and want.starts.size > 100


@pytest.mark.parametrize("widths", [(1,), (7,), (60,), (61,), (2047,), (2048,), (2049,), (1, 2048, 61, 2049)],
                         ids=lambda w: "-".join(map(str, w)))
def test_fasta_layouts(kb, widths):
    """line widths, 5000-byte headers, empty records, comment lines, blank lines, blanks and tabs inside sequence lines,
    soft-masked sequence"""
    rng = np.random.default_rng(sum(widths))
    size = 60_000 if widths == (1,) else 300_000
    for crlf in (False, True):
        assert_parsed(kb, random_layout(rng, "dna4", 1, size, widths=widths, crlf=crlf), "dna4", 1, label=f"crlf={crlf}")


def test_one_unwrapped_line_of_a_million_symbols(kb):
    rng = np.random.default_rng(17)
    for fmt in (1, 2):
        data = random_layout(rng, "dna15", fmt, 1_100_000, unwrapped=1_000_000)
        assert_parsed(kb, data, "dna15", fmt)


def test_fastq_content(kb):
    """quality lines that start with '@' or '+', empty sequence and quality lines, trailing blank lines"""
    rng = np.random.default_rng(23)
    recs = [(b"q%d" % i, _seq(rng, "dna4", m)) for i, m in enumerate([5, 0, 3, 0, 0, 40, 1])]
    quals = [(b"@" if i % 2 == 0 else b"+") + b"I" * (len(s) - 1) if s else b"" for i, (_, s) in enumerate(recs)]
    data = b"".join(b"@" + n + b"\n" + s + b"\n+\n" + q + b"\n" for (n, s), q in zip(recs, quals))
    want = assert_parsed(kb, data, "dna4", 2)
    assert len(want.names) == len(recs)
    for tail in (b"\n", b"\n\n", b"\n\n\n\n\n", b"\r\n"):
        got = assert_parsed(kb, data + tail, "dna4", 2, label=repr(tail))
        assert len(got.names) == len(recs), f"a trailing {tail!r} must not add a record"
    # the example of a FASTQ file that ends with a blank line: two records, not three
    with kb.parse_sequences(b"@a\nACGT\n+\nIIII\n@b\nGG\n+\nII\n\n", "dna4", 2) as r:
        assert len(r) == 2 and r.starts.tolist() == [0, 4, 6] and r.header_offsets.tolist() == [0, 15]
    for i in range(20):                                    # random files, some ending in blank lines, some in CRLF
        crlf = i % 3 == 2
        data = random_layout(rng, "dna4", 2, int(rng.integers(100, 20_000)), crlf=crlf)
        if i % 2:
            data += (b"\r\n" if crlf else b"\n") * int(rng.integers(1, 6))
        assert_parsed(kb, data, "dna4", 0, label=f"layout {i}")


@pytest.mark.parametrize("alphabet", ["dna4", "dna5", "dna15", "aa27"])
def test_every_alphabet(kb, alphabet):
    rng = np.random.default_rng(len(alphabet) * 101)
    for i in range(20):
        fmt = 1 + i % 2
        data = random_layout(rng, alphabet, fmt, int(rng.integers(1, 40_000)), widths=(7, 60, 61, 2048), crlf=i % 4 >= 2)
        assert_parsed(kb, data, alphabet, 0 if i % 5 == 0 else fmt, label=f"layout {i}")


def test_refusals_and_loud_failures(kb):
    # a character outside the alphabet in every position class: first byte, on tile edges, last byte
    assert refused(kb, b"NACGT\n>a\nACGT\n", "dna4") == -4
    line = bytearray(b">a\n" + b"A" * 9000 + b"\n")
    for at in (TILE - 1, TILE, 2 * TILE - 1, 2 * TILE, 3 * TILE + 7, 3 * TILE + 8):
        bad = bytearray(line)
        bad[at] = ord("N")
        assert refused(kb, bytes(bad), "dna4", 1) == -4, at
    assert refused(kb, b">a\nACGT\n>b\nACGN", "dna4") == -4
    assert refused(kb, b"@a\nACGT\n+\nIIII\n@b\nACGX\n+\nIIII", "dna5") == -4
    assert refused(kb, b">a\nAC>GT\n", "dna4") == -4                                 # a marker inside a sequence line
    # any byte in a header, a comment, a '+' line or a quality line is accepted
    junk = bytes(b for b in range(256) if b != ord("\n"))
    assert_parsed(kb, b">" + junk + b"\nACGT\n;" + junk + b"\nGG\n>" + junk + b"\n", "dna4", 1)
    assert_parsed(kb, b"@" + junk + b"\nACGT\n+" + junk + b"\n" + junk + b"\n@b\nG\n+\nI\n", "dna4", 2)
    # formats: 3 and empty input refused; 0 picks FASTQ exactly when the first byte is '@'
    with pytest.raises(kb.KmerB200Error) as e:
        kb.parse_sequences(b">a\nACGT\n", "dna4", 3)
    assert e.value.code == -1
    with pytest.raises(kb.KmerB200Error) as e:
        kb.parse_sequences(b"", "dna4", 0)
    assert e.value.code == -1
    fastq = b"@a\nACGT\n+\nIIII\n"
    with kb.parse_sequences(fastq, "dna4", 0) as r:
        assert r.n_symbols == 4 and r.name(0) == "a"
    assert_parsed(kb, fastq, "dna4", 0)
    assert refused(kb, b"\n" + fastq, "dna4", 0) == -4      # not '@' first: FASTA, and '@a' is a sequence line
    assert refused(kb, fastq, "dna4", 1) == -4
    for data in (b">a\nACGT\n", b";c\n>a\nACGT\n", b"ACGT\n>a\nGG\n"):
        assert_parsed(kb, data, "dna4", 0)
    # a blank line between FASTQ records fails loudly: the next '@' line falls on a sequence line
    assert refused(kb, b"@a\nACGT\n+\nIIII\n\n@b\nGG\n+\nII\n", "dna4", 2) == -4
    assert refused(kb, b"@a\r\nACGT\r\n+\r\nIIII\r\n\r\n@b\r\nGG\r\n+\r\nII\r\n", "dna4", 0) == -4


def test_collection_index_over_parsed_records(kb):
    """records with empty ones and records that start on tile edges, indexed as a collection: search == the per-record
    scan over the Python parser's ranks and starts"""
    data, _ = edge_layout(1, False, 7)
    want = fastx_truth.parse(data, "dna4", 1)
    starts = want.starts
    assert (np.diff(starts.astype(np.int64)) == 0).sum() >= len(RESIDUES)   # empty records
    text = want.ranks
    rng = np.random.default_rng(8)
    qs = []
    for i in range(400):
        m = int(rng.integers(0, 41))
        kind = i % 3
        if kind == 0:                                    # random
            qs.append(rng.integers(0, 4, m).astype(np.uint8))
            continue
        if kind == 1:                                    # a window anywhere
            p = int(rng.integers(0, text.size - m + 1))
        else:                                            # a window around a record start
            s = int(starts[int(rng.integers(1, starts.size - 1))])
            p = min(max(0, s - m // 2), text.size - m)
        qs.append(text[p:p + m].copy())
    off = np.zeros(len(qs) + 1, np.uint64)
    np.cumsum([x.size for x in qs], out=off[1:])
    q = np.concatenate(qs)
    truth = truth_per_record(text, starts, q, off, 0)
    with kb.parse_sequences(data, "dna4", 1) as r:
        assert np.array_equal(r.starts, starts)
        with r.index([5, 9], collection=True) as ix:
            got = ix.search_batch(q, off, mode=kb.MODE_CORRECT).as_tuple()
    assert truth[1].size > 400
    assert_results_equal(got, truth, label="collection over parsed records")


# ================================================================ B. chunked host batches

CHUNKS = 24          # search_batch_host_chunked: kChunks
PIPELINE = "streaming host pack + raw chunks"
RUN_LO, RUN = 1_000_000, 6000   # a constant run of the texts: candidate lists of ~6000 > 2048


def chunk_bounds(Q):
    per = -(-Q // CHUNKS)
    return [min(c * per, Q) for c in range(CHUNKS + 1)]


def raw_chunks(pct):
    """raw_chunk_choice: which chunks travel as 1-byte ranks at a raw share of pct %"""
    acc, raw = (99 if pct else 0), []
    for _ in range(CHUNKS):
        acc += min(pct, 100)
        raw.append(acc >= 100)
        if acc >= 100:
            acc -= 100
    return raw


def h2d_bytes(off, bits, pct):
    """host-to-device bytes of a chunked batch: per chunk its ranks (raw) or its packed stream and one padding word, then
    16-bit lengths -- or the chunk's offsets when a query of a raw chunk has 65 536 symbols or more"""
    off = np.asarray(off, dtype=np.int64)
    lens = np.diff(off)
    c0, raw, spw, total = chunk_bounds(lens.size), raw_chunks(pct), 64 // bits, 0
    for c in range(CHUNKS):
        qa, qb = c0[c], c0[c + 1]
        if qa == qb:
            continue
        n_sym = int(off[qb] - off[qa])
        total += n_sym if raw[c] else (-(-n_sym // spw) + 1) * 8
        total += 2 * (qb - qa) if lens[qa:qb].max() < 65536 else 8 * (qb - qa + 1)
    return total


def packed_chunks(Q, pct):
    c0, raw = chunk_bounds(Q), raw_chunks(pct)
    return sum(1 for c in range(CHUNKS) if c0[c + 1] > c0[c] and not raw[c])


def pipelined(ix, q, off, bits, mode=None, pct=None, expect_pct=None):
    """a search through the chunked pipeline (KMER_B200_HOST_RAW_PCT=pct unless None): the path, the raw share, the exact
    host-to-device bytes and one align_stream_kernel launch per packed chunk are asserted. Returns (result, raw share)."""
    from kmer_index_b200 import MODE_DEFAULT
    with overrides(KMER_B200_HOST_RAW_PCT=pct, KMER_B200_NO_PIPELINE=None), kernels_launched() as names:
        got = ix.search_batch(q, off, mode=MODE_DEFAULT if mode is None else mode).as_tuple()
    path = ix.last_search_host_path()
    assert path["pipeline"] == PIPELINE, path
    raw_pct = path["raw_chunk_pct"]
    if expect_pct is not None:
        assert raw_pct == expect_pct, path
    assert ix.last_search_transfer()[0] == h2d_bytes(off, bits, raw_pct), (raw_pct, ix.last_search_transfer())
    aligned = sum(v for k, v in names.items() if k.startswith("align_stream_kernel"))
    assert aligned == packed_chunks(len(off) - 1, raw_pct), (aligned, raw_pct)
    return got, raw_pct


def single_copy(ix, q, off, mode=None):
    from kmer_index_b200 import MODE_DEFAULT
    with overrides(KMER_B200_NO_PIPELINE=1):
        got = ix.search_batch(q, off, mode=MODE_DEFAULT if mode is None else mode).as_tuple()
    assert ix.last_search_host_path()["pipeline"] == "single copy"
    return got


def take(off, data, idx):
    """CSR rows idx of (off, data)"""
    off = np.asarray(off, dtype=np.int64)
    lens = off[idx + 1] - off[idx]
    new = np.zeros(idx.size + 1, np.int64)
    np.cumsum(lens, out=new[1:])
    return new.astype(np.uint64), data[np.repeat(off[idx] - new[:-1], lens) + np.arange(new[-1])]


def check_sample(oracle_mod, text, sigma, k, q, off, sample, got, correct, label):
    """rows `sample` of a result against the oracle (reference mode) or the plain scan (MODE_CORRECT)"""
    qs_off, qs = take(off, q, sample)
    g_off, g_pos = take(got[0], got[1], sample)
    g = (g_off, g_pos, got[2][sample])
    if correct:
        w_off, w_pos, _ = oracle_mod.Oracle.truth(text, qs, qs_off)
        assert np.array_equal(g_off, w_off) and np.array_equal(g_pos, w_pos), label
        assert (g[2][np.diff(qs_off) > 0] == 0).all(), label
    else:
        with oracle_mod.Oracle(text, sigma, [k]) as o:
            want = o.search(qs, qs_off)
            ub = o.last_ub
        assert_results_equal(g, want, skip=ub, label=label)
    assert g_pos.size > 0, label


def make_text(sigma, seed, n=2_000_003):
    from kmer_index_b200 import synth
    text = synth.random_text(n, sigma, seed)
    text[RUN_LO:RUN_LO + RUN] = 0
    return text


def make_batch(text, sigma, Q, m_lo, m_hi, seed):
    """Q queries of m_lo..m_hi symbols: windows of the text whose starts take every residue mod 16, windows at position 0
    and ending at n, random queries, constant runs (candidate lists > 2048), one query of every length 0..m_hi, empty
    queries scattered and one whole chunk of them, a query of m_hi symbols second in chunk 0 and last in chunk 1.
    Returns (ranks, offsets, sample): the sample is 2000 random queries and every one of those edge queries."""
    from kmer_index_b200 import synth
    rng = np.random.default_rng(seed)
    n = text.size
    lens = rng.integers(m_lo, m_hi + 1, Q).astype(np.int64)
    kind = rng.integers(0, 3, Q)                                    # 1: random, else a window of the text
    start = rng.integers(0, (n - m_hi) // 16, Q) * 16 + np.arange(Q) % 16
    c0 = chunk_bounds(Q)
    pick = rng.permutation(Q)
    pick = pick[(pick < c0[5]) | (pick >= c0[6])]                  # chunk 5 is left to empty queries
    at_ends, runs, every = pick[:64], pick[64:264], pick[264:265 + m_hi]
    kind[at_ends] = 0
    start[at_ends[:32]] = 0
    start[at_ends[32:]] = n - lens[at_ends[32:]]
    kind[runs] = 0
    start[runs] = RUN_LO + rng.integers(0, RUN - m_hi, runs.size)
    kind[every] = 1
    lens[every] = np.arange(m_hi + 1)
    empties = pick[265 + m_hi:265 + m_hi + Q // 200]
    lens[empties] = 0
    lens[c0[5]:c0[6]] = 0                                           # a chunk of nothing but empty queries
    longest = np.array([1, c0[2] - 1])
    lens[longest] = m_hi
    kind[longest] = 1
    pool = np.concatenate([text, synth.random_text(1 << 22, sigma, seed + 1)])
    src = np.where(kind == 1, n + rng.integers(0, (1 << 22) - m_hi, Q), start)
    off = np.zeros(Q + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    q = np.empty(int(off[-1]), np.uint8)
    for b in range(0, Q, 1 << 15):                                   # gathered in blocks: bounded index arrays
        e = min(Q, b + (1 << 15))
        o = off[b:e + 1]
        q[o[0]:o[-1]] = pool[np.repeat(src[b:e] - (o[:-1] - o[0]), lens[b:e]) + np.arange(o[-1] - o[0])]
    edges = np.concatenate([at_ends, runs, every, empties[:64], longest, [c0[c] for c in range(1, CHUNKS)],
                            [c0[c] - 1 for c in range(1, CHUNKS)], [c0[5], c0[6] - 1]])
    sample = np.union1d(rng.choice(Q, 2000, replace=False), edges).astype(np.int64)
    assert q.size + 17 * Q >= 256 << 20                             # large enough to be chunked
    return q, off.astype(np.uint64), sample


def lengthen(q, off, i, sym=0):
    """the batch with one more symbol at the end of query i"""
    off2 = off.copy()
    off2[i + 1:] += 1
    return np.insert(q, int(off[i + 1]), np.uint8(sym)), off2


_BATCHES = {}


def four_bit_batch(alphabet):
    """(text, sigma, k, ranks, offsets, sample) of the 4-bit alphabets: ~2e6 queries of 0-256 symbols, built once"""
    if alphabet not in _BATCHES:
        from kmer_index_b200 import ALPHABETS
        sigma, k = ALPHABETS[alphabet], {"dna5": 13, "dna15": 8}[alphabet]
        text = make_text(sigma, 31 + sigma)
        _BATCHES[alphabet] = (text, sigma, k) + make_batch(text, sigma, 2_000_000, k, 256, 41 + sigma)
    return _BATCHES[alphabet]


@pytest.mark.parametrize("alphabet", ["dna5", "dna15"])
def test_four_bit_alphabets_through_the_pipeline(kb, oracle_mod, alphabet):
    """4-bit alphabets (pack32x4 on the host, align_stream_kernel at 4 bits): pageable input, every chunk packed; pinned
    input at raw shares 0, 50, 100 % and the calibrated share; the packed-chunk limit of 256 symbols and one symbol
    beyond it; a rank >= sigma in the last symbol of a packed chunk and in a raw chunk"""
    import torch
    text, sigma, k, q, off, sample = four_bit_batch(alphabet)
    Q = off.size - 1
    assert int(np.diff(off).max()) == 256                            # exactly 16 words: accepted in a packed chunk
    pin_t = torch.from_numpy(q).pin_memory()
    pin = pin_t.numpy()
    with kb.KmerIndex(text, sigma, [k]) as ix:
        plain = single_copy(ix, q, off)
        plain_c = single_copy(ix, q, off, kb.MODE_CORRECT)
        packed, _ = pipelined(ix, q, off, 4, expect_pct=0)
        assert_results_equal(packed, plain, label="pageable, every chunk packed")
        packed_c, _ = pipelined(ix, q, off, 4, mode=kb.MODE_CORRECT, expect_pct=0)
        assert_results_equal(packed_c, plain_c, label="pageable, every chunk packed, MODE_CORRECT")
        for pct in (0, 50, 100):
            got, _ = pipelined(ix, pin, off, 4, pct=pct, expect_pct=pct)
            assert_results_equal(got, plain, label=f"pinned, {pct} % raw")
        got, auto = pipelined(ix, pin, off, 4)
        assert ix.last_search_host_path()["host_pack_gbs"] > 0
        assert_results_equal(got, plain, label=f"pinned, calibrated share ({auto} % raw)")
        # 257 symbols in query 1 (chunk 0): the packed chunk refuses, the batch is searched again with every chunk raw
        q1, off1 = lengthen(q, off, 1)
        longer, _ = pipelined(ix, q1, off1, 4, expect_pct=100)
        assert_results_equal(longer, single_copy(ix, q1, off1), label="a 257-symbol query")
        # a rank >= sigma in the last symbol of a packed chunk (not a whole word: the scalar tail) or in a raw chunk
        c0 = chunk_bounds(Q)
        c = next(c for c in range(1, CHUNKS) if int(off[c0[c + 1]] - off[c0[c]]) % 16 and c != 5)
        at = int(off[c0[c + 1]]) - 1
        for label, arr, pct in (("packed", q, None), ("raw", pin, 100)):
            keep = arr[at]
            arr[at] = sigma
            try:
                with overrides(KMER_B200_HOST_RAW_PCT=pct), pytest.raises(kb.KmerB200Error) as e:
                    ix.search_batch(arr, off)
            finally:
                arr[at] = keep
            assert e.value.code == -4, label
    check_sample(oracle_mod, text, sigma, k, q, off, sample, packed, False, "pipelined vs oracle")
    check_sample(oracle_mod, text, sigma, k, q, off, sample, packed_c, True, "pipelined MODE_CORRECT vs plain scan")
    check_sample(oracle_mod, text, sigma, k, q1, off1, np.union1d(sample[:200], [1]), longer, False, "257 symbols vs oracle")


@pytest.mark.parametrize("alphabet,k,bits,Q,m_lo", [("dna4", 12, 2, 700_000, 350), ("aa27", 5, 8, 2_400_000, 100)],
                         ids=["2bit", "8bit"])
def test_packed_chunk_limits_and_empty_queries(kb, oracle_mod, alphabet, k, bits, Q, m_lo):
    """a query of exactly 16 words stays in a packed chunk; one symbol more reruns the pageable batch with every chunk
    raw. The batch has empty queries scattered and a chunk of nothing else (a stream of one padding word, stride 1)."""
    sigma = kb.ALPHABETS[alphabet]
    m_max = 16 * (64 // bits)
    text = make_text(sigma, 50 + bits)
    q, off, sample = make_batch(text, sigma, Q, m_lo, m_max, 60 + bits)
    c0 = chunk_bounds(Q)
    assert off[c0[5]] == off[c0[6]] and int(np.diff(off).max()) == m_max
    with kb.KmerIndex(text, sigma, [k]) as ix:
        got, _ = pipelined(ix, q, off, bits, expect_pct=0)
        assert_results_equal(got, single_copy(ix, q, off), label="packed")
        q1, off1 = lengthen(q, off, 1)
        longer, _ = pipelined(ix, q1, off1, bits, expect_pct=100)
        assert_results_equal(longer, single_copy(ix, q1, off1), label=f"a {m_max + 1}-symbol query")
        if bits == 2:
            # 16-bit lengths in an all-raw run: a query of 65 535 symbols is sent as a length, one of 65 536 makes its
            # chunk (the last) send offsets
            for m in (65_535, 65_536):
                ql = np.concatenate([q, text[7:7 + m]])
                offl = np.append(off, off[-1] + np.uint64(m))
                got_long, _ = pipelined(ix, ql, offl, bits, mode=kb.MODE_CORRECT, pct=100, expect_pct=100)
                n_long = offl.size - 1
                assert (ix.last_search_transfer()[0] == ql.size + 2 * n_long) == (m == 65_535)
                assert_results_equal(got_long, single_copy(ix, ql, offl, kb.MODE_CORRECT), label=f"a {m}-symbol query")
                check_sample(oracle_mod, text, sigma, k, ql, offl, np.append(sample[:100], n_long - 1), got_long, True,
                             f"a {m}-symbol query vs plain scan")
    check_sample(oracle_mod, text, sigma, k, q, off, sample, got, False, "packed vs oracle")
    check_sample(oracle_mod, text, sigma, k, q1, off1, np.union1d(sample[:200], [1]), longer, False, "longer vs oracle")


def test_offsets_that_do_not_start_at_zero(kb):
    """4096 bytes of ranks >= sigma in front of the batch, every offset shifted by 4096: never read, never validated"""
    import torch
    text, sigma, k, q, off, _ = four_bit_batch("dna5")
    pre = (np.arange(4096) % (256 - sigma) + sigma).astype(np.uint8)
    q2, off2 = np.concatenate([pre, q]), off + np.uint64(4096)
    pin_t = torch.from_numpy(q2).pin_memory()
    with kb.KmerIndex(text, sigma, [k]) as ix:
        want, _ = pipelined(ix, q, off, 4, expect_pct=0)
        got, _ = pipelined(ix, q2, off2, 4, expect_pct=0)
        assert_results_equal(got, want, label="pageable")
        got, _ = pipelined(ix, pin_t.numpy(), off2, 4, pct=50, expect_pct=50)
        assert_results_equal(got, want, label="pinned, 50 % raw")
        assert_results_equal(single_copy(ix, q2, off2), want, label="single copy")


def test_pointer_batch_large_enough_to_be_chunked(kb):
    """kmer_b200_search_batch_ptrs gathers into a pageable buffer: every chunk packed, the flat batch's result"""
    from kmer_index_b200 import _capi
    text, sigma, k, q, off, _ = four_bit_batch("dna5")
    Q = off.size - 1
    ptrs = np.uint64(q.ctypes.data) + off[:-1]
    lens = np.diff(off).astype(np.uint64)
    with kb.KmerIndex(text, sigma, [k]) as ix:
        want, _ = pipelined(ix, q, off, 4, expect_pct=0)
        r = C.c_void_p()
        with kernels_launched() as names:
            _capi.check(ix._L.kmer_b200_search_batch_ptrs(ix.handle, ptrs.ctypes.data, lens.ctypes.data, Q, kb.MODE_DEFAULT,
                                                          C.byref(r)))
        got = ix._host_result(r, Q, True).as_tuple()
        path = ix.last_search_host_path()
        assert path["pipeline"] == PIPELINE and path["raw_chunk_pct"] == 0, path
        assert ix.last_search_transfer()[0] == h2d_bytes(off, 4, 0)
        assert sum(v for n, v in names.items() if n.startswith("align_stream_kernel")) == packed_chunks(Q, 0)
    assert_results_equal(got, want, label="pointer batch")


def test_dna5_character_input(kb):
    """characters with N (either case) through create_from_text and search_batch_text == ranks"""
    from kmer_index_b200 import synth
    chars = np.frombuffer(kb.ALPHABET_CHARS["dna5"].encode(), dtype=np.uint8)
    text = synth.random_text(100_003, 5, 71)
    text[5000:5400] = 3                                   # a run of N
    q, off = synth.stress_queries(text, 600, 1, 30, 5, 72)
    queries = [chars[q[int(off[i]):int(off[i + 1])]].tobytes() for i in range(off.size - 1)]
    queries = [x.lower() if i % 7 == 3 else x for i, x in enumerate(queries)]
    text_chars = chars[text].tobytes()
    text_chars = text_chars[:5200] + text_chars[5200:5300].lower() + text_chars[5300:]
    assert sum(x.count(b"N") + x.count(b"n") for x in queries) > 100
    lut = kb.char_lut("dna5")
    with kb.KmerIndex(text, 5, [5, 9]) as a, kb.KmerIndex(text_chars, 5, [5, 9], lut=lut) as b:
        want = a.search_batch(q, off).as_tuple()
        assert_results_equal(b.search_batch_text(queries).as_tuple(), want, label="characters")
        assert_results_equal(b.search_batch(q, off).as_tuple(), want, label="ranks on the character-built index")
        assert_results_equal(a.search_batch_text(queries, lut=lut).as_tuple(), want, label="characters on the rank-built index")
        with pytest.raises(kb.KmerB200Error) as e:
            b.search_batch_text([b"ACGXT"])
        assert e.value.code == -4
