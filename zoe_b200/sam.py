"""SAM emission for alignments produced by the CUDA path -- the caller side of zoe's SW path.

Mirrors (paths relative to the zoe repository):
  * ``SamData::from_alignment``  src/data/records/sam/mod.rs:216-245  (POS = ref_range.start + 1, CIGAR =
    ``AlignmentStates::to_cigar_unchecked``, RNEXT ``*``, PNEXT 0, TLEN 0, ``AS:i:<score>``)
  * ``SamData::unmapped``        src/data/records/sam/mod.rs:201-214  (FLAG 4, POS 0, MAPQ 255, CIGAR/SEQ/QUAL ``*``)
  * ``Display for SamData``      src/data/records/sam/std_traits.rs:3-43 (tab-separated, missing SEQ/QUAL as ``*``)

Results of the best-hit search (``CudaProfiles.align_best_hit_arrays``) become one primary record per read:
``sam_lines_best_hit``.

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
