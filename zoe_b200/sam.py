"""SAM emission for alignments produced by the CUDA path -- the caller side of zoe's SW path.

Mirrors (paths relative to the zoe repository):
  * ``SamData::from_alignment``  src/data/records/sam/mod.rs:216-245  (POS = ref_range.start + 1, CIGAR =
    ``AlignmentStates::to_cigar_unchecked``, RNEXT ``*``, PNEXT 0, TLEN 0, ``AS:i:<score>``)
  * ``SamData::unmapped``        src/data/records/sam/mod.rs:201-214  (FLAG 4, POS 0, MAPQ 255, CIGAR/SEQ/QUAL ``*``)
  * ``Display for SamData``      src/data/records/sam/std_traits.rs:3-43 (tab-separated, missing SEQ/QUAL as ``*``)

Results of the best-hit search (``CudaProfiles.align_best_hit_arrays``) become one primary record per read:
``sam_lines_best_hit``.

Results of the paired-end best-hit search (``CudaProfiles.align_paired_best_hit_arrays``) become two records per read
pair, mate 1 first, with the paired FLAG bits, RNEXT, PNEXT and TLEN: ``sam_lines_paired``.

Results of the both-strand search pass their strands as ``strand``: a reverse-strand pair is written as SAM writes a read
that maps to the reverse strand -- FLAG bit 16 set, SEQ reverse-complemented, QUAL reversed (its POS and CIGAR already
refer to the reverse complement).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Iterable, List, Optional, Sequence

import numpy as np

from . import _lib
from .alignment import Alignment, MaybeAligned, Strand, reverse_complement

_OPS = {0: "M", 1: "I", 2: "D", 4: "S"}


@dataclass
class SamData:
    qname: str
    flag: int
    rname: str
    pos: int
    mapq: int
    cigar: str
    seq: bytes
    qual: bytes
    rnext: str = "*"
    pnext: int = 0
    tlen: int = 0
    opt_fields: List[str] = field(default_factory=list)

    @classmethod
    def from_alignment(cls, alignment: Alignment, qname: str, flag: int, rname: str, mapq: int, seq: bytes,
                       qual: bytes) -> "SamData":
        return cls(qname, flag, rname, alignment.ref_range[0] + 1, mapq, alignment.states, seq, qual,
                   opt_fields=[f"AS:i:{int(alignment.score)}"])

    @classmethod
    def unmapped(cls, qname: str, rname: str) -> "SamData":
        return cls(qname, 4, rname, 0, 255, "", b"*", b"*")

    def __str__(self) -> str:
        seq = self.seq.decode("ascii", "replace") if self.seq else "*"
        qual = self.qual.decode("ascii", "replace") if self.qual else "*"
        s = "\t".join([self.qname, str(self.flag), self.rname, str(self.pos), str(self.mapq), self.cigar or "*",
                       self.rnext, str(self.pnext), str(self.tlen), seq, qual])
        for f in self.opt_fields:
            s += "\t" + f
        return s


def _oriented(reverse: bool, flag: int, seq: bytes, qual: bytes):
    """FLAG, SEQ and QUAL of a record on the forward strand, or on the reverse strand (FLAG 16)."""
    if not reverse:
        return flag, seq, qual
    return flag | 16, reverse_complement(seq), qual if qual == b"*" else qual[::-1]


def sam_records(result: Sequence[Sequence[MaybeAligned]], qnames: Sequence[str], rnames: Sequence[str],
                seqs: Sequence[bytes], quals: Optional[Sequence[bytes]] = None, mapq: int = 255, flag: int = 0,
                strand: Optional[Sequence[Sequence[Strand]]] = None):
    """``CudaProfiles.sw_align_batch(SeqSrc.Query(reads))`` -> one :class:`SamData` per (read, reference) pair;
    pairs that are not ``Some`` become ``SamData::unmapped`` records.  ``strand[i][j]`` (the both-strand search):
    ``Strand.Reverse`` pairs become reverse-strand records."""
    out = []
    for i, row in enumerate(result):
        for j, m in enumerate(row):
            if m.is_some():
                f, seq, qual = _oriented(strand is not None and strand[i][j] is Strand.Reverse, flag, bytes(seqs[i]),
                                         bytes(quals[i]) if quals is not None else b"*")
                out.append(SamData.from_alignment(m.unwrap(), qnames[i], f, rnames[j], mapq, seq, qual))
            else:
                out.append(SamData.unmapped(qnames[i], rnames[j]))
    return out


def sam_lines_from_arrays(a: dict, n_profiled: int, qnames: Sequence[str], rnames: Sequence[str], buf: np.ndarray,
                          offs: np.ndarray, quals: Optional[Sequence[bytes]] = None, mapq: int = 255,
                          flag: int = 0, strand: Optional[np.ndarray] = None) -> Iterable[str]:
    """The same records straight from ``CudaProfiles.align_arrays`` (no per-pair Python objects): yields SAM lines in
    pair order (read-major).  ``strand`` (flat, pair index; e.g. ``align_both_strands_arrays(...)["strand"]``): pairs
    with strand 1 become reverse-strand records."""
    n = len(offs) - 1
    cig, coff = a["cigar"], a["cigar_off"]
    for i in range(n):
        seq = bytes(buf[int(offs[i]):int(offs[i + 1])])
        qual = bytes(quals[i]) if quals is not None else b"*"
        for j in range(n_profiled):
            k = i * n_profiled + j
            if int(a["status"][k]) != _lib.SOME:
                yield str(SamData.unmapped(qnames[i], rnames[j]))
                continue
            words = cig[int(coff[k]):int(coff[k + 1])]
            cigar = "".join(f"{int(w) >> 4}{_OPS[int(w) & 15]}" for w in words)
            f, s, q = _oriented(strand is not None and int(strand[k]) == 1, flag, seq, qual)
            rec = SamData(qnames[i], f, rnames[j], int(a["ref_start"][k]) + 1, mapq, cigar, s, q,
                          opt_fields=[f"AS:i:{int(a['score'][k])}"])
            yield str(rec)


def sam_lines_best_hit(a: dict, qnames: Sequence[str], rnames: Sequence[str], buf: np.ndarray, offs: np.ndarray,
                       quals: Optional[Sequence[bytes]] = None, mapq: int = 255, flag: int = 0) -> Iterable[str]:
    """One SAM line per read from ``CudaProfiles.align_best_hit_arrays``: a Some winner maps to ``rnames[hit]`` at
    ``ref_start + 1`` with its CIGAR and ``AS:i:score``, plus ``XS:i:runner_up`` when the runner-up is above 0; a strand-1
    winner is a reverse-strand record (FLAG 16, reverse-complemented SEQ, reversed QUAL).  Any other read is
    ``SamData::unmapped`` with RNAME ``*``."""
    n = len(offs) - 1
    cig, coff = a["cigar"], a["cigar_off"]
    for i in range(n):
        if int(a["status"][i]) != _lib.SOME:
            yield str(SamData.unmapped(qnames[i], "*"))
            continue
        seq = bytes(buf[int(offs[i]):int(offs[i + 1])])
        qual = bytes(quals[i]) if quals is not None else b"*"
        words = cig[int(coff[i]):int(coff[i + 1])]
        cigar = "".join(f"{int(w) >> 4}{_OPS[int(w) & 15]}" for w in words)
        f, s, q = _oriented(int(a["strand"][i]) == 1, flag, seq, qual)
        tags = [f"AS:i:{int(a['score'][i])}"]
        if int(a["runner_up"][i]) > 0:
            tags.append(f"XS:i:{int(a['runner_up'][i])}")
        yield str(SamData(qnames[i], f, rnames[int(a["hit"][i])], int(a["ref_start"][i]) + 1, mapq, cigar, s, q,
                          opt_fields=tags))


def sam_lines_paired(a: dict, qnames: Sequence[str], rnames: Sequence[str], buf1: np.ndarray, offs1: np.ndarray,
                     buf2: np.ndarray, offs2: np.ndarray, quals1: Optional[Sequence[bytes]] = None,
                     quals2: Optional[Sequence[bytes]] = None, mapq: int = 255) -> Iterable[str]:
    """Two SAM lines per read pair from ``CudaProfiles.align_paired_best_hit_arrays``, mate 1 then mate 2.

    FLAG: 0x1 always, 0x2 for a proper pair, 0x4 / 0x8 when the record's own / its mate's result is not Some, 0x10 /
    0x20 for its own / its mate's reverse strand when mapped, 0x40 for mate 1, 0x80 for mate 2.  A mapped mate is written
    as :func:`sam_lines_best_hit` writes a read (RNAME ``rnames[hit]``, POS, CIGAR, oriented SEQ and QUAL, ``AS`` and
    ``XS``), with RNEXT ``=`` and PNEXT at its mate's POS, and TLEN ``tlen`` for mate 1, ``-tlen`` for mate 2.  An
    unmapped mate of a mapped one takes its mate's RNAME and POS (the SAM recommended practice), so both records'
    PNEXT point there; it keeps its SEQ and QUAL as given.  A pair with no mapped mate gets RNAME ``*`` and POS 0
    (FLAG 77 and 141)."""
    cig, coff = a["cigar"], a["cigar_off"]
    bufs, offs, quals = (buf1, buf2), (offs1, offs2), (quals1, quals2)
    for i in range(len(offs1) - 1):
        k = (2 * i, 2 * i + 1)
        mapped = [int(a["status"][x]) == _lib.SOME for x in k]
        rev = [int(a["strand"][x]) == 1 for x in k]
        pos = [int(a["ref_start"][x]) + 1 if mapped[m] else 0 for m, x in enumerate(k)]
        if mapped[0] != mapped[1]:  # the unmapped mate is placed at its mate
            pos = [max(pos)] * 2
        rname = rnames[int(a["hit"][i])] if any(mapped) else "*"
        for m in range(2):
            o = 1 - m
            flag = 0x1 | (0x40 if m == 0 else 0x80)
            flag |= 0x2 if int(a["proper"][i]) else 0
            flag |= 0 if mapped[m] else 0x4
            flag |= 0 if mapped[o] else 0x8
            flag |= 0x10 if mapped[m] and rev[m] else 0
            flag |= 0x20 if mapped[o] and rev[o] else 0
            seq = bytes(bufs[m][int(offs[m][i]):int(offs[m][i + 1])])
            qual = bytes(quals[m][i]) if quals[m] is not None else b"*"
            rnext, pnext = ("=", pos[o]) if any(mapped) else ("*", 0)
            if not mapped[m]:
                yield str(SamData(qnames[i], flag, rname, pos[m], mapq, "", seq or b"*", qual or b"*", rnext, pnext, 0))
                continue
            x = k[m]
            words = cig[int(coff[x]):int(coff[x + 1])]
            cigar = "".join(f"{int(w) >> 4}{_OPS[int(w) & 15]}" for w in words)
            _, s, q = _oriented(rev[m], 0, seq, qual)
            tags = [f"AS:i:{int(a['score'][x])}"]
            if int(a["runner_up"][x]) > 0:
                tags.append(f"XS:i:{int(a['runner_up'][x])}")
            tlen = int(a["tlen"][i]) if m == 0 else -int(a["tlen"][i])
            yield str(SamData(qnames[i], flag, rname, pos[m], mapq, cigar, s, q, rnext, pnext, tlen, opt_fields=tags))
