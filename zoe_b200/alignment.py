"""Host-side mirror of zoe's interface for the SW path, over the C-ABI CUDA library.

zoe names mirrored here (paths relative to the zoe repository):
  * ``ProfileError``   -- src/alignment/errors.rs:6-15 (raised by validate_profile_args,
                          src/alignment/profile.rs:32-44)
  * ``MaybeAligned``   -- src/alignment/types/output.rs:18-25 (Some / Overflowed / Unmapped)
  * ``Alignment``      -- src/alignment/types/output.rs:264-279
  * ``SeqSrc``         -- src/alignment/mod.rs:157-162
  * ``CudaProfiles``   -- the batched counterpart of ``SharedProfiles``
                          (src/alignment/profile_set.rs:552-560) with ``new_with_w128/256/512``
                          (profile_set.rs:434-483) and ``sw_score_from_i8`` / ``sw_align_from_i8``
                          semantics (profile_set.rs:71-78, 136-145), applied to a whole batch.

All arithmetic happens in the CUDA library; this module only marshals buffers.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from enum import Enum
from typing import Generic, Iterable, Optional, Sequence, TypeVar

import numpy as np

from . import _lib
from .matrices import WeightMatrix

T = TypeVar("T")


class ProfileError(ValueError):
    """zoe's ``ProfileError`` (errors.rs:6-15)."""

    EmptySequence = "EmptySequence"
    GapOpenOutOfRange = "GapOpenOutOfRange"
    GapExtendOutOfRange = "GapExtendOutOfRange"
    BadGapWeights = "BadGapWeights"

    def __init__(self, kind: str, message: str = ""):
        super().__init__(f"{kind}: {message}" if message else kind)
        self.kind = kind


class ZoeCudaError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"zoe_cuda error {code}: {message}")
        self.code = code


_PROFILE_ERRORS = {
    _lib.E_EMPTY_SEQUENCE: ProfileError.EmptySequence,
    _lib.E_GAP_OPEN_RANGE: ProfileError.GapOpenOutOfRange,
    _lib.E_GAP_EXTEND_RANGE: ProfileError.GapExtendOutOfRange,
    _lib.E_BAD_GAP_WEIGHTS: ProfileError.BadGapWeights,
}


class Status(Enum):
    Some = 0
    Overflowed = 1
    Unmapped = 2


@dataclass(frozen=True)
class MaybeAligned(Generic[T]):
    """Tri-state alignment outcome (output.rs:18-25)."""

    status: Status
    value: Optional[T] = None

    @classmethod
    def some(cls, v: T) -> "MaybeAligned[T]":
        return cls(Status.Some, v)

    def is_some(self) -> bool:
        return self.status is Status.Some

    def unwrap(self) -> T:
        if self.status is not Status.Some:
            raise ValueError(f"called unwrap() on MaybeAligned::{self.status.name}")
        return self.value  # type: ignore[return-value]


MaybeAligned.Overflowed = MaybeAligned(Status.Overflowed)  # type: ignore[attr-defined]
MaybeAligned.Unmapped = MaybeAligned(Status.Unmapped)  # type: ignore[attr-defined]


@dataclass(frozen=True)
class SeqSrc(Generic[T]):
    """Which role the *non-profile* sequences play (alignment/mod.rs:157-162)."""

    kind: str
    seq: T

    @classmethod
    def Query(cls, seq: T) -> "SeqSrc[T]":
        return cls("Query", seq)

    @classmethod
    def Reference(cls, seq: T) -> "SeqSrc[T]":
        return cls("Reference", seq)


@dataclass(frozen=True)
class Alignment:
    """zoe's ``Alignment<u32>`` (output.rs:264-279); ``states`` rendered as a CIGAR string."""

    score: int
    ref_range: tuple
    query_range: tuple
    states: str
    ref_len: int
    query_len: int


@dataclass(frozen=True)
class ScoreAndRanges:
    """zoe's ``ScoreAndRanges<u32>`` (src/alignment/types/output.rs): score + 0-based half-open ranges."""

    score: int
    ref_range: tuple
    query_range: tuple


_CIGAR_OPS = {0: "M", 1: "I", 2: "D", 4: "S"}


class Strand(Enum):
    """Which strand of a streamed sequence a both-strand result belongs to."""

    Forward = 0
    Reverse = 1


def _complement_table() -> bytes:
    # the Python copy of the device table (csrc/strands.cuh, complement_base)
    t = bytearray(range(256))
    for a, b in (b"AT", b"TA", b"UA", b"CG", b"GC", b"RY", b"YR", b"KM", b"MK", b"BV", b"VB", b"DH", b"HD"):
        t[a] = b
        t[a | 0x20] = b | 0x20
    return bytes(t)


_COMPLEMENT = _complement_table()


def reverse_complement(seq: bytes) -> bytes:
    """The reverse complement the both-strand search aligns: bytes reversed, each mapped through the complement table
    (A<->T, C<->G, U->A, R<->Y, K<->M, B<->V, D<->H; S, W, N and every other byte unchanged; lowercase keeps its case)."""
    return bytes(seq).translate(_COMPLEMENT)[::-1]


def _pack(seqs: Sequence[bytes]):
    offs = np.zeros(len(seqs) + 1, dtype=np.uint64)
    if len(seqs):
        offs[1:] = np.cumsum([len(s) for s in seqs], dtype=np.uint64)
    buf = np.frombuffer(b"".join(seqs), dtype=np.uint8) if len(seqs) else np.zeros(0, dtype=np.uint8)
    if buf.size == 0:
        buf = np.zeros(1, dtype=np.uint8)
    return np.ascontiguousarray(buf), offs


def _p(a: np.ndarray, ty):
    return a.ctypes.data_as(C.POINTER(ty))


@dataclass(frozen=True)
class BestHit:
    """One streamed sequence's result of the best-hit search: the chosen profiled sequence ``index`` and ``strand``, the
    alignment of that pair (of the reverse complement for ``Strand.Reverse``), and ``runner_up``, the best Some score
    against any other profiled sequence (0 if none; SAM ``XS``)."""

    index: int
    strand: Strand
    result: MaybeAligned
    runner_up: int


@dataclass(frozen=True)
class PairedHit:
    """One read pair's result of the paired-end best-hit search: the profiled sequence ``index`` both mates were placed
    on, ``proper`` (the mates point inward within the insert bounds), ``tlen`` (mate 1's SAM TLEN; mate 2's is
    ``-tlen``) and a :class:`BestHit` per mate, whose ``strand`` is the mate's strand in the chosen orientation."""

    index: int
    proper: bool
    tlen: int
    mate1: BestHit
    mate2: BestHit


class CudaProfiles:
    """A set of profiled sequences resident on one or more B200s.

    ``CudaProfiles.new_with_w256(targets, matrix, gap_open, gap_extend)`` corresponds to building one
    ``SharedProfiles::new_with_w256`` per target; ``sw_score_batch(seqs)[i][j]`` then equals
    ``profiles[j].sw_score_from_i8(seqs[i])`` and ``sw_align_batch(SeqSrc.Query(seqs))[i][j]`` equals
    ``profiles[j].sw_align_from_i8(SeqSrc::Query(seqs[i]))``.
    """

    def __init__(self, targets: Iterable[bytes], matrix: WeightMatrix, gap_open: int, gap_extend: int,
                 lanes=(32, 16, 8), devices: Optional[Sequence[int]] = None, n_devices: int = 1,
                 profiled_is_query: bool = False):
        self._h = C.c_void_p()
        self._lib = _lib.load()
        targets = [bytes(t) for t in targets]
        # zoe validates the profile arguments before anything touches a device
        if not (-127 <= gap_open <= 0):
            raise ProfileError(ProfileError.GapOpenOutOfRange, str(gap_open))
        if not (-127 <= gap_extend <= 0):
            raise ProfileError(ProfileError.GapExtendOutOfRange, str(gap_extend))
        if gap_extend < gap_open:
            raise ProfileError(ProfileError.BadGapWeights, f"open {gap_open} extend {gap_extend}")
        if any(len(t) == 0 for t in targets) or not targets:
            raise ProfileError(ProfileError.EmptySequence)
        if devices is not None:
            ids = (C.c_int * len(devices))(*devices)
            rc = self._lib.zoe_cuda_create(C.byref(self._h), ids, len(devices))
        else:
            rc = self._lib.zoe_cuda_create(C.byref(self._h), None, n_devices)
        if rc:
            raise ZoeCudaError(rc, "zoe_cuda_create failed (no usable CUDA device?)")
        self.matrix = matrix
        self.targets = targets
        self.gap_open, self.gap_extend = gap_open, gap_extend
        self.profiled_is_query = bool(profiled_is_query)
        w = np.ascontiguousarray(matrix.weights, dtype=np.int8)
        lut = np.ascontiguousarray(matrix.mapping.index_map, dtype=np.uint8)
        self._check(self._lib.zoe_cuda_set_scoring(self._h, _p(w, C.c_int8), matrix.S, _p(lut, C.c_uint8), gap_open,
                                                    gap_extend, int(profiled_is_query)))
        self._check(self._lib.zoe_cuda_set_lanes(self._h, *lanes))
        buf, offs = _pack(targets)
        self._check(self._lib.zoe_cuda_set_profiled(self._h, _p(buf, C.c_uint8), _p(offs, C.c_uint64), len(targets)))
        self.lanes = tuple(lanes)

    # lane presets: profile_set.rs:434-483
    @classmethod
    def new_with_w128(cls, targets, matrix, gap_open, gap_extend, **kw):
        return cls(targets, matrix, gap_open, gap_extend, lanes=(16, 8, 4), **kw)

    @classmethod
    def new_with_w256(cls, targets, matrix, gap_open, gap_extend, **kw):
        return cls(targets, matrix, gap_open, gap_extend, lanes=(32, 16, 8), **kw)

    @classmethod
    def new_with_w512(cls, targets, matrix, gap_open, gap_extend, **kw):
        return cls(targets, matrix, gap_open, gap_extend, lanes=(64, 32, 16), **kw)

    ALIGN_AUTO, ALIGN_FULL, ALIGN_WINDOW = 0, 1, 2

    def set_align_options(self, mode: int = 0, checkpoint_log2: int = 6, slack: int = 16):
        """Tuning of the align pipeline (never changes results): see ``zoe_cuda_set_align_options``."""
        self._check(self._lib.zoe_cuda_set_align_options(self._h, mode, checkpoint_log2, slack))

    def set_memory_budget(self, scratch_bytes: int = 0):
        """Bound the device scratch of one align / ranges / 3-pass call (0 = automatic); larger batches run in chunks."""
        self._check(self._lib.zoe_cuda_set_memory_budget(self._h, int(scratch_bytes)))

    def set_width_policy(self, first_bits: int = 8, last_bits: int = 32, unsigned: bool = False):
        """Which zoe integer types may report a result: ``(8, 32)`` = ``sw_*_from_i8`` (default), ``(16, 32)`` =
        ``..._from_i16``, ``(32, 32)`` = ``..._from_i32`` (profile_set.rs:71-179); ``first == last`` = a standalone
        ``StripedProfile<T, N, S>``; ``unsigned`` = zoe's u8/u16/u32 profiles over the biased matrix."""
        self._check(self._lib.zoe_cuda_set_width_policy(self._h, first_bits, last_bits, int(unsigned)))

    def _check(self, rc: int):
        if rc == 0:
            return
        msg = self._lib.zoe_cuda_last_error(self._h).decode(errors="replace")
        if rc in _PROFILE_ERRORS:
            raise ProfileError(_PROFILE_ERRORS[rc], msg)
        raise ZoeCudaError(rc, msg)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.zoe_cuda_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def n_profiled(self) -> int:
        return len(self.targets)

    # ---- raw array API (what bench.py times) ----
    def sw_score_arrays(self, buf: np.ndarray, offs: np.ndarray):
        """Scores for a packed batch: returns (score u32, status u8, tier u8), each ``[n, n_profiled]``."""
        n = len(offs) - 1
        pairs = n * self.n_profiled
        score = np.zeros(max(pairs, 1), dtype=np.uint32)
        status = np.zeros(max(pairs, 1), dtype=np.uint8)
        tier = np.zeros(max(pairs, 1), dtype=np.uint8)
        self._check(self._lib.zoe_cuda_sw_score_batch(self._h, _p(buf, C.c_uint8), _p(offs, C.c_uint64), n,
                                                      _p(score, C.c_uint32), _p(status, C.c_uint8), _p(tier, C.c_uint8)))
        shape = (n, self.n_profiled)
        return score[:pairs].reshape(shape), status[:pairs].reshape(shape), tier[:pairs].reshape(shape)

    def sw_score_both_strands_arrays(self, buf: np.ndarray, offs: np.ndarray):
        """:meth:`sw_score_arrays` of the both-strand search: (score, status, tier, strand), each ``[n, n_profiled]``;
        strand 0 = the sequence as given won, 1 = its reverse complement."""
        n = len(offs) - 1
        pairs = n * self.n_profiled
        score = np.zeros(max(pairs, 1), dtype=np.uint32)
        status = np.zeros(max(pairs, 1), dtype=np.uint8)
        tier = np.zeros(max(pairs, 1), dtype=np.uint8)
        strand = np.zeros(max(pairs, 1), dtype=np.uint8)
        self._check(self._lib.zoe_cuda_sw_score_both_strands_batch(
            self._h, _p(buf, C.c_uint8), _p(offs, C.c_uint64), n, _p(score, C.c_uint32), _p(status, C.c_uint8),
            _p(tier, C.c_uint8), _p(strand, C.c_uint8)))
        shape = (n, self.n_profiled)
        return (score[:pairs].reshape(shape), status[:pairs].reshape(shape), tier[:pairs].reshape(shape),
                strand[:pairs].reshape(shape))

    def sw_score_into(self, buf: np.ndarray, offs: np.ndarray, score: np.ndarray, status: np.ndarray, tier: np.ndarray):
        """Like :meth:`sw_score_arrays` but writes into caller-owned (ideally pinned) output arrays."""
        self._check(self._lib.zoe_cuda_sw_score_batch(self._h, _p(buf, C.c_uint8), _p(offs, C.c_uint64), len(offs) - 1,
                                                      _p(score, C.c_uint32), _p(status, C.c_uint8), _p(tier, C.c_uint8)))

    def stream_handle(self, dev_index: int = 0) -> int:
        return int(self._lib.zoe_cuda_stream(self._h, dev_index) or 0)

    def stage(self, buf: np.ndarray, offs: np.ndarray):
        self._check(self._lib.zoe_cuda_stage_streamed(self._h, _p(buf, C.c_uint8), _p(offs, C.c_uint64), len(offs) - 1))
        self._staged_n = len(offs) - 1

    def run_score_staged(self):
        self._check(self._lib.zoe_cuda_run_score_staged(self._h))

    def run_align_staged(self):
        self._check(self._lib.zoe_cuda_run_align_staged(self._h))

    def fetch_scores(self):
        pairs = self._staged_n * self.n_profiled
        score = np.zeros(max(pairs, 1), dtype=np.uint32)
        status = np.zeros(max(pairs, 1), dtype=np.uint8)
        tier = np.zeros(max(pairs, 1), dtype=np.uint8)
        self._check(self._lib.zoe_cuda_fetch_scores(self._h, _p(score, C.c_uint32), _p(status, C.c_uint8),
                                                    _p(tier, C.c_uint8)))
        shape = (self._staged_n, self.n_profiled)
        return score[:pairs].reshape(shape), status[:pairs].reshape(shape), tier[:pairs].reshape(shape)

    def last_timing(self):
        t, k, n = C.c_float(0), C.c_float(0), C.c_uint32(0)
        self._lib.zoe_cuda_last_timing(self._h, C.byref(t), C.byref(k), C.byref(n))
        return {"total_ms": t.value, "dp_kernel_ms": k.value, "kernel_launches": n.value}

    def last_stats(self):
        s = _lib.Stats()
        self._lib.zoe_cuda_last_stats(self._h, C.byref(s))
        return s.as_dict()

    def dpx_peak(self, kind: int = 0):
        g, ms = C.c_double(0), C.c_float(0)
        self._check(self._lib.zoe_cuda_dpx_peak(self._h, kind, C.byref(g), C.byref(ms)))
        return g.value, ms.value

    def align_arrays(self, buf: np.ndarray, offs: np.ndarray, cigar_cap: Optional[int] = None, three_pass: bool = False):
        """Alignments for a packed batch; returns a dict of flat arrays (pair index = i*n_profiled+j).
        ``three_pass``: ``sw_align_from_i8_3pass`` (ranges + banded box alignment) instead of ``sw_align_from_i8``."""
        return self._align_arrays(buf, offs, cigar_cap, three_pass, both_strands=False)

    def align_both_strands_arrays(self, buf: np.ndarray, offs: np.ndarray, cigar_cap: Optional[int] = None,
                                  three_pass: bool = False):
        """:meth:`align_arrays` of the both-strand search: every pair's better strand, plus a ``"strand"`` array
        (0 forward, 1 reverse complement; a reverse result's ranges and CIGAR refer to the reverse complement)."""
        return self._align_arrays(buf, offs, cigar_cap, three_pass, both_strands=True)

    def _align_arrays(self, buf, offs, cigar_cap, three_pass: bool, both_strands: bool):
        n = len(offs) - 1
        pairs = max(n * self.n_profiled, 1)
        out = {
            "score": np.zeros(pairs, dtype=np.uint32), "status": np.zeros(pairs, dtype=np.uint8),
            "tier": np.zeros(pairs, dtype=np.uint8), "ref_start": np.zeros(pairs, dtype=np.uint32),
            "ref_end": np.zeros(pairs, dtype=np.uint32), "query_start": np.zeros(pairs, dtype=np.uint32),
            "query_end": np.zeros(pairs, dtype=np.uint32), "cigar_off": np.zeros(pairs + 1, dtype=np.uint64),
            "hazard": np.zeros(pairs, dtype=np.uint8),
        }
        if both_strands:
            out["strand"] = np.zeros(pairs, dtype=np.uint8)
        cap = int(cigar_cap) if cigar_cap else max(16 * pairs, 1024)
        for _ in range(2):
            out["cigar"] = np.zeros(cap, dtype=np.uint32)
            rc = self._align_call(buf, offs, out, three_pass)
            if rc == _lib.E_CIGAR_CAP:
                cap = int(out["cigar_off"][0]) + 16
                continue
            self._check(rc)
            break
        else:
            self._check(rc)
        return out

    def _align_call(self, buf: np.ndarray, offs: np.ndarray, out: dict, three_pass: bool) -> int:
        """One align / 3-pass call into ``out``; the both-strand entry point when ``out`` has a ``"strand"`` array."""
        args = [self._h, _p(buf, C.c_uint8), _p(offs, C.c_uint64), len(offs) - 1, _p(out["score"], C.c_uint32),
                _p(out["status"], C.c_uint8), _p(out["tier"], C.c_uint8), _p(out["ref_start"], C.c_uint32),
                _p(out["ref_end"], C.c_uint32), _p(out["query_start"], C.c_uint32), _p(out["query_end"], C.c_uint32),
                _p(out["cigar"], C.c_uint32), _p(out["cigar_off"], C.c_uint64), len(out["cigar"])]
        if "strand" in out:
            strand = _p(out["strand"], C.c_uint8)
            if three_pass:
                return self._lib.zoe_cuda_sw_align_3pass_both_strands_batch(*args, strand)
            return self._lib.zoe_cuda_sw_align_both_strands_batch(*args, _p(out["hazard"], C.c_uint8), strand)
        if three_pass:
            return self._lib.zoe_cuda_sw_align_3pass_batch(*args)
        return self._lib.zoe_cuda_sw_align_batch(*args, _p(out["hazard"], C.c_uint8))

    def align_into(self, buf: np.ndarray, offs: np.ndarray, out: dict, three_pass: bool = False):
        """Like :meth:`align_arrays` but into caller-owned (ideally pinned) arrays; ``out['cigar']`` is the capacity.
        With a ``"strand"`` array in ``out``, the both-strand search (:meth:`align_both_strands_arrays`)."""
        self._check(self._align_call(buf, offs, out, three_pass))

    def run_3pass_staged(self):
        self._check(self._lib.zoe_cuda_run_3pass_staged(self._h))

    def ranges_arrays(self, buf: np.ndarray, offs: np.ndarray):
        """``sw_score_ranges`` for a packed batch: dict of flat arrays (pair index = i*n_profiled+j)."""
        return self._ranges_arrays(buf, offs, both_strands=False)

    def ranges_both_strands_arrays(self, buf: np.ndarray, offs: np.ndarray):
        """:meth:`ranges_arrays` of the both-strand search, plus a ``"strand"`` array (0 forward, 1 reverse complement)."""
        return self._ranges_arrays(buf, offs, both_strands=True)

    def _ranges_arrays(self, buf: np.ndarray, offs: np.ndarray, both_strands: bool):
        n = len(offs) - 1
        pairs = max(n * self.n_profiled, 1)
        out = {k: np.zeros(pairs, dtype=np.uint32) for k in ("score", "ref_start", "ref_end", "query_start", "query_end")}
        out.update({k: np.zeros(pairs, dtype=np.uint8) for k in ("status", "tier")})
        if both_strands:
            out["strand"] = np.zeros(pairs, dtype=np.uint8)
        self.ranges_into(buf, offs, out)
        return out

    def ranges_into(self, buf: np.ndarray, offs: np.ndarray, out: dict):
        """Like :meth:`ranges_arrays` but into caller-owned (ideally pinned) arrays.  With a ``"strand"`` array in
        ``out``, the both-strand search (:meth:`ranges_both_strands_arrays`)."""
        args = [self._h, _p(buf, C.c_uint8), _p(offs, C.c_uint64), len(offs) - 1, _p(out["score"], C.c_uint32),
                _p(out["status"], C.c_uint8), _p(out["tier"], C.c_uint8), _p(out["ref_start"], C.c_uint32),
                _p(out["ref_end"], C.c_uint32), _p(out["query_start"], C.c_uint32), _p(out["query_end"], C.c_uint32)]
        if "strand" in out:
            self._check(self._lib.zoe_cuda_sw_score_ranges_both_strands_batch(*args, _p(out["strand"], C.c_uint8)))
        else:
            self._check(self._lib.zoe_cuda_sw_score_ranges_batch(*args))

    def run_ranges_staged(self):
        self._check(self._lib.zoe_cuda_run_ranges_staged(self._h))

    def sw_score_ranges_batch(self, src: "SeqSrc"):
        """``out[i][j] == profiles[j].sw_score_ranges_from_i8(SeqSrc::X(seqs[i]))`` as
        ``MaybeAligned[ScoreAndRanges]`` (profile_set.rs:313-322)."""
        self._check_src(src)
        seqs = [bytes(s) for s in src.seq]
        buf, offs = _pack(seqs)
        return self._ranges_rows(len(seqs), self.ranges_arrays(buf, offs))

    def _check_src(self, src: "SeqSrc"):
        want_pq = src.kind == "Reference"  # streamed sequences are references <=> profiled are queries
        if want_pq != self.profiled_is_query:
            raise ValueError(
                f"this CudaProfiles was built with profiled_is_query={self.profiled_is_query}; "
                f"SeqSrc.{src.kind} needs the opposite orientation")

    def _ranges_rows(self, n: int, a: dict):
        out = []
        for i in range(n):
            row = []
            for j in range(self.n_profiled):
                k = i * self.n_profiled + j
                st = int(a["status"][k])
                if st != _lib.SOME:
                    row.append(self._maybe(st, None))
                else:
                    row.append(MaybeAligned.some(ScoreAndRanges(
                        int(a["score"][k]), (int(a["ref_start"][k]), int(a["ref_end"][k])),
                        (int(a["query_start"][k]), int(a["query_end"][k])))))
            out.append(row)
        return out

    def align_flag_bytes(self, n_seqs: int, seq_len: int) -> int:
        """Bytes of direction flags one align pass writes (8 lanes x 32 B per column per sequence pair for <= 152 rows)."""
        cols = sum(len(t) for t in self.targets)
        lanes_words = {True: 8 * 8}  # G=8, NW=8 (K=19) -- the short-read layout
        return int((n_seqs + 1) // 2 * cols * lanes_words[True] * 4) if seq_len <= 152 else 0

    # ---- zoe-shaped API ----
    def sw_score_batch(self, seqs: Sequence[bytes]):
        """``[[MaybeAligned[int]]]``: ``out[i][j] == profiles[j].sw_score_from_i8(seqs[i])``."""
        buf, offs = _pack([bytes(s) for s in seqs])
        score, status, _ = self.sw_score_arrays(buf, offs)
        return [[self._maybe(int(status[i, j]), int(score[i, j])) for j in range(self.n_profiled)]
                for i in range(len(seqs))]

    @staticmethod
    def _maybe(status: int, value):
        if status == _lib.SOME:
            return MaybeAligned.some(value)
        return MaybeAligned.Overflowed if status == _lib.OVERFLOWED else MaybeAligned.Unmapped  # type: ignore

    def sw_align_3pass_batch(self, src: SeqSrc):
        """``out[i][j] == profiles[j].sw_align_from_i8_3pass(SeqSrc::X(seqs[i]))`` (profile_set.rs:213-231)."""
        return self.sw_align_batch(src, three_pass=True)

    def sw_align_batch(self, src: SeqSrc, three_pass: bool = False):
        """``out[i][j] == profiles[j].sw_align_from_i8(SeqSrc::X(seqs[i]))`` for the SeqSrc given."""
        self._check_src(src)
        seqs = [bytes(s) for s in src.seq]
        buf, offs = _pack(seqs)
        return self._alignment_rows(seqs, self.align_arrays(buf, offs, three_pass=three_pass))

    def _alignment_rows(self, seqs: Sequence[bytes], a: dict):
        out = []
        for i in range(len(seqs)):
            row = []
            for j in range(self.n_profiled):
                k = i * self.n_profiled + j
                st = int(a["status"][k])
                if st != _lib.SOME:
                    row.append(self._maybe(st, None))
                    continue
                lo, hi = int(a["cigar_off"][k]), int(a["cigar_off"][k + 1])
                cig = "".join(f"{int(w) >> 4}{_CIGAR_OPS[int(w) & 15]}" for w in a["cigar"][lo:hi])
                streamed_len, prof_len = len(seqs[i]), len(self.targets[j])
                if self.profiled_is_query:
                    ref_len, query_len = streamed_len, prof_len
                else:
                    ref_len, query_len = prof_len, streamed_len
                row.append(MaybeAligned.some(Alignment(
                    int(a["score"][k]), (int(a["ref_start"][k]), int(a["ref_end"][k])),
                    (int(a["query_start"][k]), int(a["query_end"][k])), cig, ref_len, query_len)))
            out.append(row)
        return out

    # ---- both-strand search: every streamed sequence and its reverse complement, the better strand per pair ----
    def _with_strand(self, rows, strand: np.ndarray):
        return [[(m, Strand(int(strand[i * self.n_profiled + j]))) for j, m in enumerate(row)] for i, row in enumerate(rows)]

    def sw_score_both_strands_batch(self, seqs: Sequence[bytes]):
        """``[[(MaybeAligned[int], Strand)]]``: the better of ``sw_score_batch([s])`` and
        ``sw_score_batch([reverse_complement(s)])`` per pair; ties go to ``Strand.Forward``."""
        buf, offs = _pack([bytes(s) for s in seqs])
        score, status, _, strand = self.sw_score_both_strands_arrays(buf, offs)
        return [[(self._maybe(int(status[i, j]), int(score[i, j])), Strand(int(strand[i, j])))
                 for j in range(self.n_profiled)] for i in range(len(seqs))]

    def sw_score_ranges_both_strands_batch(self, src: "SeqSrc"):
        """``[[(MaybeAligned[ScoreAndRanges], Strand)]]``; a reverse result's ranges refer to the reverse complement."""
        self._check_src(src)
        seqs = [bytes(s) for s in src.seq]
        buf, offs = _pack(seqs)
        a = self.ranges_both_strands_arrays(buf, offs)
        return self._with_strand(self._ranges_rows(len(seqs), a), a["strand"])

    def sw_align_both_strands_batch(self, src: SeqSrc, three_pass: bool = False):
        """``[[(MaybeAligned[Alignment], Strand)]]``: the better strand of every pair, aligned as the single-strand
        call aligns it; a reverse result's ranges and CIGAR refer to the reverse complement (SAM FLAG 16)."""
        self._check_src(src)
        seqs = [bytes(s) for s in src.seq]
        buf, offs = _pack(seqs)
        a = self.align_both_strands_arrays(buf, offs, three_pass=three_pass)
        return self._with_strand(self._alignment_rows(seqs, a), a["strand"])

    def sw_align_3pass_both_strands_batch(self, src: SeqSrc):
        """The 3-pass alignment (:meth:`sw_align_3pass_batch`) of the both-strand search."""
        return self.sw_align_both_strands_batch(src, three_pass=True)

    # ---- best-hit search: each streamed sequence's best profiled sequence and strand, chosen on the device ----
    def sw_score_best_hit_arrays(self, buf: np.ndarray, offs: np.ndarray, both_strands: bool = False):
        """Per streamed sequence (flat arrays of ``n``): ``hit`` (u32), ``strand`` (u8), the winner's ``score`` /
        ``status`` / ``tier`` and ``runner_up`` (u32), as ``zoe_cuda_sw_score_best_hit_batch`` defines them."""
        n = len(offs) - 1
        out = self._best_hit_outputs(n)
        self._check(self._lib.zoe_cuda_sw_score_best_hit_batch(
            self._h, _p(buf, C.c_uint8), _p(offs, C.c_uint64), n, int(both_strands), _p(out["hit"], C.c_uint32),
            _p(out["strand"], C.c_uint8), _p(out["score"], C.c_uint32), _p(out["status"], C.c_uint8),
            _p(out["tier"], C.c_uint8), _p(out["runner_up"], C.c_uint32)))
        return {k: v[:n] for k, v in out.items()}

    def align_best_hit_arrays(self, buf: np.ndarray, offs: np.ndarray, both_strands: bool = False,
                              three_pass: bool = False, cigar_cap: Optional[int] = None):
        """:meth:`sw_score_best_hit_arrays` plus the alignment of each selected pair: ``ref_start`` ... ``query_end``,
        ``hazard``, ``cigar`` and ``cigar_off`` (``n + 1``), indexed by streamed sequence."""
        n = len(offs) - 1
        m = max(n, 1)
        out = self._best_hit_outputs(n)
        out.update({k: np.zeros(m, dtype=np.uint32) for k in ("ref_start", "ref_end", "query_start", "query_end")})
        out["hazard"] = np.zeros(m, dtype=np.uint8)
        out["cigar_off"] = np.zeros(m + 1, dtype=np.uint64)
        cap = int(cigar_cap) if cigar_cap else max(16 * m, 1024)
        for _ in range(2):
            out["cigar"] = np.zeros(cap, dtype=np.uint32)
            rc = self._lib.zoe_cuda_sw_align_best_hit_batch(
                self._h, _p(buf, C.c_uint8), _p(offs, C.c_uint64), n, int(both_strands), int(three_pass),
                _p(out["hit"], C.c_uint32), _p(out["strand"], C.c_uint8), _p(out["score"], C.c_uint32),
                _p(out["status"], C.c_uint8), _p(out["tier"], C.c_uint8), _p(out["runner_up"], C.c_uint32),
                _p(out["ref_start"], C.c_uint32), _p(out["ref_end"], C.c_uint32), _p(out["query_start"], C.c_uint32),
                _p(out["query_end"], C.c_uint32), _p(out["cigar"], C.c_uint32), _p(out["cigar_off"], C.c_uint64),
                len(out["cigar"]), _p(out["hazard"], C.c_uint8))
            if rc == _lib.E_CIGAR_CAP:
                cap = int(out["cigar_off"][0]) + 16
                continue
            self._check(rc)
            break
        else:
            self._check(rc)
        for k in out:
            if k not in ("cigar", "cigar_off"):
                out[k] = out[k][:n]
        out["cigar_off"] = out["cigar_off"][:n + 1]
        return out

    @staticmethod
    def _best_hit_outputs(n: int) -> dict:
        m = max(n, 1)
        return {"hit": np.zeros(m, dtype=np.uint32), "strand": np.zeros(m, dtype=np.uint8),
                "score": np.zeros(m, dtype=np.uint32), "status": np.zeros(m, dtype=np.uint8),
                "tier": np.zeros(m, dtype=np.uint8), "runner_up": np.zeros(m, dtype=np.uint32)}

    def sw_align_best_hit_batch(self, src: SeqSrc, both_strands: bool = False, three_pass: bool = False):
        """One :class:`BestHit` per streamed sequence: its best profiled sequence (and strand, with ``both_strands``),
        aligned as :meth:`sw_align_batch` aligns that pair."""
        self._check_src(src)
        seqs = [bytes(s) for s in src.seq]
        buf, offs = _pack(seqs)
        return self._best_hit_rows(seqs, self.align_best_hit_arrays(buf, offs, both_strands, three_pass))

    def _best_hit_rows(self, seqs: Sequence[bytes], a: dict):
        out = []
        for i, s in enumerate(seqs):
            j, strand = int(a["hit"][i]), Strand(int(a["strand"][i]))
            st = int(a["status"][i])
            if st != _lib.SOME:
                m = self._maybe(st, None)
            else:
                lo, hi = int(a["cigar_off"][i]), int(a["cigar_off"][i + 1])
                cig = "".join(f"{int(w) >> 4}{_CIGAR_OPS[int(w) & 15]}" for w in a["cigar"][lo:hi])
                streamed_len, prof_len = len(s), len(self.targets[j])
                ref_len, query_len = (streamed_len, prof_len) if self.profiled_is_query else (prof_len, streamed_len)
                m = MaybeAligned.some(Alignment(
                    int(a["score"][i]), (int(a["ref_start"][i]), int(a["ref_end"][i])),
                    (int(a["query_start"][i]), int(a["query_end"][i])), cig, ref_len, query_len))
            out.append(BestHit(j, strand, m, int(a["runner_up"][i])))
        return out

    # ---- paired-end best-hit search: each read pair's profiled sequence and orientation, chosen from both mates ----
    def sw_score_paired_best_hit_arrays(self, buf1: np.ndarray, offs1: np.ndarray, buf2: np.ndarray, offs2: np.ndarray):
        """``hit`` per pair (``n`` entries) and, per mate at index ``2 i + m``, ``strand``, ``score``, ``status``,
        ``tier`` and ``runner_up``, as ``zoe_cuda_sw_score_paired_best_hit_batch`` defines them.  Mate 1 of pair ``i`` is
        sequence ``i`` of (buf1, offs1), mate 2 sequence ``i`` of (buf2, offs2)."""
        n = self._pair_count(offs1, offs2)
        out = self._best_hit_outputs(2 * n)
        out["hit"] = np.zeros(max(n, 1), dtype=np.uint32)
        self._check(self._lib.zoe_cuda_sw_score_paired_best_hit_batch(
            self._h, _p(buf1, C.c_uint8), _p(offs1, C.c_uint64), _p(buf2, C.c_uint8), _p(offs2, C.c_uint64), n,
            _p(out["hit"], C.c_uint32), _p(out["strand"], C.c_uint8), _p(out["score"], C.c_uint32),
            _p(out["status"], C.c_uint8), _p(out["tier"], C.c_uint8), _p(out["runner_up"], C.c_uint32)))
        return {k: v[:n] if k == "hit" else v[:2 * n] for k, v in out.items()}

    def align_paired_best_hit_arrays(self, buf1: np.ndarray, offs1: np.ndarray, buf2: np.ndarray, offs2: np.ndarray,
                                     three_pass: bool = False, *, min_insert: int, max_insert: int,
                                     cigar_cap: Optional[int] = None):
        """:meth:`sw_score_paired_best_hit_arrays` plus ``proper`` (u8) and ``tlen`` (i32) per pair and, per mate,
        its alignment: ``ref_start`` ... ``query_end``, ``hazard``, ``cigar`` and ``cigar_off`` (``2 n + 1``)."""
        n = self._pair_count(offs1, offs2)
        m = max(2 * n, 1)
        out = self._best_hit_outputs(2 * n)
        out["hit"] = np.zeros(max(n, 1), dtype=np.uint32)
        out["proper"] = np.zeros(max(n, 1), dtype=np.uint8)
        out["tlen"] = np.zeros(max(n, 1), dtype=np.int32)
        out.update({k: np.zeros(m, dtype=np.uint32) for k in ("ref_start", "ref_end", "query_start", "query_end")})
        out["hazard"] = np.zeros(m, dtype=np.uint8)
        out["cigar_off"] = np.zeros(m + 1, dtype=np.uint64)
        cap = int(cigar_cap) if cigar_cap else max(16 * m, 1024)
        for _ in range(2):
            out["cigar"] = np.zeros(cap, dtype=np.uint32)
            rc = self._lib.zoe_cuda_sw_align_paired_best_hit_batch(
                self._h, _p(buf1, C.c_uint8), _p(offs1, C.c_uint64), _p(buf2, C.c_uint8), _p(offs2, C.c_uint64), n,
                int(three_pass), int(min_insert), int(max_insert), _p(out["hit"], C.c_uint32),
                _p(out["proper"], C.c_uint8), _p(out["tlen"], C.c_int32), _p(out["strand"], C.c_uint8),
                _p(out["score"], C.c_uint32), _p(out["status"], C.c_uint8), _p(out["tier"], C.c_uint8),
                _p(out["runner_up"], C.c_uint32), _p(out["ref_start"], C.c_uint32), _p(out["ref_end"], C.c_uint32),
                _p(out["query_start"], C.c_uint32), _p(out["query_end"], C.c_uint32), _p(out["cigar"], C.c_uint32),
                _p(out["cigar_off"], C.c_uint64), len(out["cigar"]), _p(out["hazard"], C.c_uint8))
            if rc == _lib.E_CIGAR_CAP:
                cap = int(out["cigar_off"][0]) + 16
                continue
            self._check(rc)
            break
        else:
            self._check(rc)
        for k in out:
            if k in ("hit", "proper", "tlen"):
                out[k] = out[k][:n]
            elif k != "cigar":
                out[k] = out[k][:2 * n + 1] if k == "cigar_off" else out[k][:2 * n]
        return out

    @staticmethod
    def _pair_count(offs1: np.ndarray, offs2: np.ndarray) -> int:
        if len(offs1) != len(offs2):
            raise ValueError(f"mate batches differ in size: {len(offs1) - 1} and {len(offs2) - 1} sequences")
        return len(offs1) - 1

    def sw_align_paired_best_hit_batch(self, mates1: Sequence[bytes], mates2: Sequence[bytes], three_pass: bool = False,
                                       *, min_insert: int, max_insert: int):
        """One :class:`PairedHit` per read pair ``(mates1[i], mates2[i])`` (an FR library): the profiled sequence and
        orientation that the two mates support best together, each mate aligned as :meth:`sw_align_batch` aligns it
        (its reverse complement when its strand is ``Strand.Reverse``)."""
        m1, m2 = [bytes(s) for s in mates1], [bytes(s) for s in mates2]
        if len(m1) != len(m2):
            raise ValueError(f"mate lists differ in length: {len(m1)} and {len(m2)}")
        (buf1, offs1), (buf2, offs2) = _pack(m1), _pack(m2)
        a = self.align_paired_best_hit_arrays(buf1, offs1, buf2, offs2, three_pass, min_insert=min_insert,
                                              max_insert=max_insert)
        mates = [s for pair in zip(m1, m2) for s in pair]
        rows = self._best_hit_rows(mates, dict(a, hit=np.repeat(a["hit"], 2)))
        return [PairedHit(int(a["hit"][i]), bool(a["proper"][i]), int(a["tlen"][i]), rows[2 * i], rows[2 * i + 1])
                for i in range(len(m1))]
