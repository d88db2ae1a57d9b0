"""FASTQ ingestion into the packed batch layout the C ABI takes (concatenated bytes + uint64 offsets).

Mirrors zoe's ``FastQReader`` (src/data/records/fastq/reader.rs:87-185): single-line records only, ``@`` header,
non-empty sequence, ``+`` separator, quality string of the sequence's length made of graphic ASCII; the same
conditions are errors here (``ValueError`` with zoe's messages).
"""
from __future__ import annotations

import io
from itertools import zip_longest
from typing import BinaryIO, Iterable, Iterator, List, Tuple, Union

import numpy as np


def _chop(line: bytes) -> bytes:
    if line.endswith(b"\n"):
        line = line[:-1]
    if line.endswith(b"\r"):
        line = line[:-1]
    return line


def read_fastq(src: Union[str, bytes, BinaryIO, Iterable[bytes]]) -> Iterator[Tuple[str, bytes, bytes]]:
    """Yields ``(header, sequence, quality)`` per record."""
    if isinstance(src, str):
        fh: Iterable[bytes] = open(src, "rb")
    elif isinstance(src, (bytes, bytearray)):
        fh = io.BytesIO(bytes(src))
    else:
        fh = src
    it = iter(fh)
    for first in it:
        if not first.startswith(b"@"):
            raise ValueError("Missing '@' symbol at header line beginning! Ensure that the FASTQ file is not multi-line.")
        header = _chop(first[1:])
        if not header:
            raise ValueError("Missing FASTQ header!")
        name = header.decode("utf-8")
        seq = _chop(next(it, b""))
        if not seq:
            raise ValueError(f"Missing FASTQ sequence! See header: {name}")
        plus = next(it, b"")
        if not plus.startswith(b"+"):
            raise ValueError(f"Missing '+' line! Ensure that the FASTQ file is not multi-line. See header: {name}")
        qual = _chop(next(it, b""))
        if len(qual) != len(seq):
            if not qual:
                raise ValueError(f"Missing FASTQ quality scores! See header: {name}")
            raise ValueError(f"Sequence and quality score length mismatch ({len(seq)} ≠ {len(qual)})! See: {name}")
        if any(c < 33 or c > 126 for c in qual):
            raise ValueError(f"Quality scores must be graphic ASCII! See: {name}")
        yield name, seq, qual


def pack_fastq(src) -> Tuple[List[str], np.ndarray, np.ndarray, List[bytes]]:
    """``(headers, buf, offs, quals)``: the streamed-batch layout of ``zoe_cuda_sw_*_batch``."""
    names, seqs, quals = [], [], []
    for name, seq, qual in read_fastq(src):
        names.append(name)
        seqs.append(seq)
        quals.append(qual)
    buf, offs = _packed(seqs)
    return names, buf, offs, quals


def _mate_name(header: str) -> str:
    """The read name of a mate's header: its first whitespace token without a trailing ``/1`` or ``/2``."""
    name = header.split(None, 1)[0] if header.strip() else ""
    return name[:-2] if name.endswith(("/1", "/2")) else name


def read_fastq_pairs(r1, r2) -> Iterator[Tuple[str, bytes, bytes, bytes, bytes]]:
    """Yields ``(name, seq1, qual1, seq2, qual2)`` per read pair of two paired-end FASTQ files (record i of ``r1`` and
    of ``r2`` are the mates of pair i).  ``ValueError`` when the files differ in record count or a pair's names differ
    (names compared as :func:`_mate_name` gives them)."""
    for k, (a, b) in enumerate(zip_longest(read_fastq(r1), read_fastq(r2))):
        if a is None or b is None:
            raise ValueError(f"R1 and R2 differ in record count: {'R1' if a is None else 'R2'} ends after {k} records")
        n1, n2 = _mate_name(a[0]), _mate_name(b[0])
        if n1 != n2:
            raise ValueError(f"mate names differ at record {k + 1}: {n1!r} in R1, {n2!r} in R2")
        yield n1, a[1], a[2], b[1], b[2]


def _packed(seqs: List[bytes]):
    offs = np.zeros(len(seqs) + 1, dtype=np.uint64)
    if seqs:
        offs[1:] = np.cumsum([len(s) for s in seqs], dtype=np.uint64)
    buf = np.frombuffer(b"".join(seqs), dtype=np.uint8) if seqs else np.zeros(1, dtype=np.uint8)
    return np.ascontiguousarray(buf), offs


def pack_fastq_pairs(r1, r2):
    """``(names, buf1, offs1, quals1, buf2, offs2, quals2)``: the two mate batches of
    ``CudaProfiles.align_paired_best_hit_arrays``."""
    names, s1, q1, s2, q2 = [], [], [], [], []
    for name, a, qa, b, qb in read_fastq_pairs(r1, r2):
        names.append(name)
        s1.append(a)
        q1.append(qa)
        s2.append(b)
        q2.append(qb)
    (buf1, offs1), (buf2, offs2) = _packed(s1), _packed(s2)
    return names, buf1, offs1, q1, buf2, offs2, q2
