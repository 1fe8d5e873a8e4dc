"""Plain Python restatement of the FASTA / FASTQ parser (kmer_b200_parse_sequences), line by line, written to be read
rather than to be fast. The rules it states:

  FASTA: a line that starts with '>' starts a record (its header: the line without the '>', a trailing '\\r' dropped);
         a line that starts with ';' is a comment; every other line is sequence. '\\r', space and tab are dropped from
         sequence lines. Sequence before the first header -- or a file without one -- is an unnamed first record.
  FASTQ: records of four lines: '@' header, sequence, '+' line, qualities. Only the sequence line is read. A line in
         header position that is empty (trailing blank lines) starts no record; a blank line between records therefore
         moves the next '@' line into sequence position, where '@' is refused.
  Sequence characters go through char_lut(alphabet); one outside the alphabet raises ValueError.

parse(data, alphabet, fmt) -> Parsed(ranks, starts, header_offsets, names). fmt 0 picks FASTQ exactly when the first
byte is '@'. header_offsets[i] is the byte offset of record i's header line (NO_HEADER for the unnamed first record).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

NO_HEADER = 0xFFFFFFFFFFFFFFFF
DROPPED = b"\r \t"


@dataclass
class Parsed:
    ranks: np.ndarray            # uint8, all records back to back
    starts: np.ndarray           # uint64 [R + 1]: where each record's sequence starts in ranks, then len(ranks)
    header_offsets: np.ndarray   # uint64 [R]
    names: list                  # str [R]


def lut_of(alphabet: str) -> np.ndarray:
    from kmer_index_b200 import char_lut
    return char_lut(alphabet)


def _name(line: bytes) -> str:
    if line.endswith(b"\r"):
        line = line[:-1]
    return line[1:].decode(errors="replace")


def parse(data: bytes, alphabet: str, fmt: int = 0) -> Parsed:
    from kmer_index_b200 import ALPHABETS
    if fmt not in (0, 1, 2):
        raise ValueError(f"unknown format {fmt}")
    if not data:
        raise ValueError("empty input")
    if fmt == 0:
        fmt = 2 if data[:1] == b"@" else 1
    lut, sigma = lut_of(alphabet), ALPHABETS[alphabet]
    seq = bytearray()
    starts, headers, names = [], [], []
    at = 0
    for line_no, line in enumerate(data.split(b"\n")):
        if fmt == 1:
            is_header, is_seq = line.startswith(b">"), not (line.startswith(b">") or line.startswith(b";"))
        else:
            is_header = line_no % 4 == 0 and line[:1] not in (b"", b"\r")
            is_seq = line_no % 4 == 1
        if is_header:
            starts.append(len(seq))
            headers.append(at)
            names.append(_name(line))
        if is_seq:
            ranks = lut[np.frombuffer(line.translate(None, DROPPED), dtype=np.uint8)]
            if (ranks >= sigma).any():
                raise ValueError(f"the sequence line at byte {at} holds a character outside {alphabet}")
            seq += ranks.tobytes()
        at += len(line) + 1
    if not starts or starts[0] > 0:
        starts.insert(0, 0)
        headers.insert(0, NO_HEADER)
        names.insert(0, "")
    return Parsed(np.frombuffer(bytes(seq), dtype=np.uint8).copy(), np.array(starts + [len(seq)], dtype=np.uint64),
                  np.array(headers, dtype=np.uint64), names)
