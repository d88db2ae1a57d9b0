"""Pass 3 of the 3-pass alignment (sw_3pass.cuh) at its routing and kernel edges, against the CPU oracle.

A pair that needs a DP goes to one of five code paths, chosen from its box (rn streamed rows x qn profiled columns, from
passes 1-2) and its current band width bw (0 = sw_scalar_align on the whole box):
  * "shared-ring": tp_dp_kernel, banded, (H, E) ring in shared memory (bw <= 15);
  * "global-ring": tp_dp_kernel, banded, ring in the pair's scratch (bw >= 16 under ZOE_CUDA_TP_THREAD);
  * "warp-band":   tp_band_warp_kernel, banded (bw >= 16);
  * "warp-box":    tp_band_warp_kernel, scalar box of more than 65 536 cells with qn + 2 <= 24 576;
  * "thread-box":  tp_dp_kernel, scalar box (small, or a row too long for the warp kernel's shared memory).
The corpus below is built from reads with known indels, so that the box and the first band width follow from the
construction; the oracle's box and accepted width then say which widths pass 3 tries and which kernel runs each attempt.
Every group is checked pair by pair (status, score, tier, both ranges, CIGAR) in both orientations, once with the
default routing and once with every pair on the single-thread kernel, and last_stats() must equal the totals the oracle
implies, band attempts included.

The band never leaves the matrix before the last row: the first width is |rn - qn| + 1, so rn < qn + bw and
rows_done = min(rn, qn + bw) is rn.  The nearest edge is an insertion, rn = qn + bw - 1, whose last row holds two cells.
"""
import os
import re

import numpy as np
import pytest

from oracle import oracle as O
from test_3pass_gpu import (ROOT, TP_BOX_CELLS, TP_RING, TP_WCAP_CAP, check_3pass, osc, tp_attempts, tp_is_large,
                            tp_ring_size, tp_row_cells)
from zoe_b200 import WeightMatrix, synth

W25 = WeightMatrix.new_dna_matrix(2, -5, b"N")
W42 = WeightMatrix.new_dna_matrix(4, -2, b"N")
W54 = WeightMatrix.new_dna_matrix(5, -4, b"N")
BENCH, TIES, FREE = (W25, -10, -1), (W42, -3, -1), (W54, 0, 0)  # FREE: gaps cost nothing, N scores 0 against anything
SCORINGS = (BENCH, TIES, FREE)

FIRST_WIDTHS = (1, 2, 15, 16, 17, 31, 32, 33, 47, 48, 64)  # accepted at the first width
DOUBLED_WIDTHS = (8, 16, 32, 64)                          # accepted after doubling from width 1
CHUNK_EDGES = (31, 32, 33, 63, 64, 65, 96, 97)            # warp-kernel scalar rows around its 32-column chunks
ROWS_PAST_2_20 = 1 << 20


def tp_route(bw, rn, qn, thread_only=False):
    """Kernel and storage of one attempt, as run_3pass_on_device and the two kernels decide it.  Every round's warp
    capacity covers the widest large row up to TP_WCAP_CAP, so the choice depends on the pair alone."""
    if not thread_only and tp_is_large(bw, rn, qn) and tp_row_cells(bw, qn) + 2 <= TP_WCAP_CAP:
        return "warp-band" if bw else "warp-box"
    if bw == 0:
        return "thread-box"
    return "shared-ring" if tp_ring_size(bw) <= TP_RING else "global-ring"


def pair_classes(rn, qn, path):
    """The edges one DP pair reaches, from its box and the oracle's path."""
    att = tp_attempts(rn, qn, path)
    out = {("route", tp_route(bw, rn, qn)) for bw in att}
    out |= {("thread-route", tp_route(bw, rn, qn, thread_only=True)) for bw in att}
    if path & 0xff == 1:
        out.add(("first" if len(att) == 1 else "doubled", att[-1]))
        if len(att) == 1 and att[0] >= 16:
            out.add(("first-wide", "rn>qn" if rn > qn else "rn<qn" if rn < qn else "rn=qn"))
    else:
        if len(att) > 1:
            out.add(("scalar-after-doubling", tp_route(0, rn, qn)))
        if rn * qn in (TP_BOX_CELLS, TP_BOX_CELLS + 256):
            out.add(("box-cells", rn * qn, tp_route(0, rn, qn)))
        if qn in CHUNK_EDGES and tp_route(0, rn, qn) == "warp-box" and len(att) == 1:
            out.add(("warp-box-qn", qn))
        if qn + 2 in (TP_WCAP_CAP, TP_WCAP_CAP + 1):
            out.add(("wcap", qn, tp_route(0, rn, qn)))
        if rn > ROWS_PAST_2_20:
            out.add(("rows-past-2^20", tp_route(0, rn, qn)))
    return out


# ---- the corpus: groups of (targets, reads) aligned in one call each, with the edges each group must reach ----
def _cat(*parts):
    return np.concatenate([np.asarray(p, dtype=np.uint8) for p in parts])


def _n(k):
    return np.full(k, ord("N"), dtype=np.uint8)


def banded_group(rng):
    """Reads cut from one target with a deletion / insertion of d bases (first width d + 1), or with an insertion and a
    deletion of k bases that cancel (rn == qn, first width 1, accepted at the first power of two >= k)."""
    t = synth.random_dna(rng, 40000)
    reads, a = [], 0
    F = 150
    for bw0 in FIRST_WIDTHS[1:]:
        d = bw0 - 1
        reads.append(_cat(t[a:a + F], t[a + F + d:a + 2 * F + d]))  # deletion: rn = qn - d
        a += 2 * F + d + 50
        reads.append(_cat(t[a:a + F], synth.random_dna(rng, d), t[a + F:a + 2 * F]))  # insertion: rn = qn + d
        a += 2 * F + 50
    L = 40
    for k in (1, 5, 8, 12, 16, 20, 32, 40, 64):
        reads.append(_cat(t[a:a + F], synth.random_dna(rng, k), t[a + F:a + F + L], t[a + F + L + k:a + 2 * F + L + k]))
        a += 2 * F + L + k + 50
    # a k = 66 deviation: widths 1 .. 64 fail and 128 > (qn - 1) / 2, so the scalar box: 256 x 256 (thread kernel) and,
    # with one more inserted base, 257 x 256 (warp kernel)
    for extra in (0, 1):
        F2, L2, k = 65, 60, 66
        reads.append(_cat(t[a:a + F2], synth.random_dna(rng, k + extra), t[a + F2:a + F2 + L2],
                          t[a + F2 + L2 + k:a + 2 * F2 + L2 + k]))
        a += 2 * F2 + L2 + k + 50
    assert a <= len(t)
    expects = {("first", w) for w in FIRST_WIDTHS} | {("doubled", w) for w in DOUBLED_WIDTHS}
    expects |= {("first-wide", "rn>qn"), ("first-wide", "rn<qn"), ("scalar-after-doubling", "thread-box"),
                ("scalar-after-doubling", "warp-box"), ("box-cells", 65536, "thread-box"), ("box-cells", 65792, "warp-box"),
                ("route", "shared-ring"), ("route", "warp-band"), ("route", "thread-box"), ("route", "warp-box"),
                ("thread-route", "global-ring")}
    return [t], reads, expects


def chunk_edge_group(rng):
    """Profiled A + B of qn bases, streamed A + N * L + B with rn * qn > 65 536: under free gaps every base must match,
    so the box is the whole pair, a scalar box from the start (|rn - qn| + 1 > (qn - 1) / 2) on the warp kernel."""
    targets, reads = [], []
    for qn in CHUNK_EDGES:
        p = synth.random_dna(rng, qn)
        h = qn // 2
        targets.append(p)
        reads.append(_cat(p[:h], _n(TP_BOX_CELLS // qn + 1), p[h:]))
    expects = {("warp-box-qn", qn) for qn in CHUNK_EDGES} | {("thread-route", "thread-box")}
    return targets, reads, expects


def wcap_group(rng):
    """Profiled A + N * D + B of 24 574 and 24 575 columns, streamed A + B (3 000 rows): the first box row plus its two
    guard slots fills the warp kernel's 24 576-int rows, the second does not fit and goes to the thread kernel, whose
    scalar row lives in global memory.  Both in one call, so one round launches both kernels on large boxes."""
    a, b = synth.random_dna(rng, 1500), synth.random_dna(rng, 1500)
    targets = [_cat(a, _n(qn - 3000), b) for qn in (TP_WCAP_CAP - 2, TP_WCAP_CAP - 1)]
    expects = {("wcap", TP_WCAP_CAP - 2, "warp-box"), ("wcap", TP_WCAP_CAP - 1, "thread-box")}
    return targets, [_cat(a, b)], expects


def rows_2_20_group(rng):
    """Profiled A + B (64 bases), streamed A + N * 1 048 600 + B: under free gaps the first best cell is at box row
    1 048 663, past the 20 bits a packed best-cell key of the warp kernel kept."""
    a, b = synth.random_dna(rng, 32), synth.random_dna(rng, 32)
    expects = {("rows-past-2^20", "warp-box")}
    return [_cat(a, b)], [_cat(a, _n(1_048_600), b)], expects


GROUPS = {"banded": (banded_group, 31), "chunk_edges": (chunk_edge_group, 32), "wcap": (wcap_group, 33),
          "rows_2_20": (rows_2_20_group, 34)}


def build_group(name):
    fn, seed = GROUPS[name]
    return fn(np.random.default_rng(seed))


def oracle_dp_pairs(targets, reads, wm, go, ge):
    """(rn, qn, path) of every pair that needs a DP, from the oracle alone (the box and path do not depend on the
    orientation: zoe computes them un-inverted and inverts the alignment at the end)."""
    sc = osc(wm, go, ge)
    out = []
    for s in reads:
        for t in targets:
            t, s = bytes(t), bytes(s)
            rc, _aln, _tier, path = O.sw_align_3pass_from(t, s, sc)
            if rc == O.SOME and path & 0xff:
                _, _, rr, qr, _ = O.sw_score_ranges_from(t, s, sc)
                out.append((rr[1] - rr[0], qr[1] - qr[0], path))
    return out


# ---- CPU: the routing constants and the corpus ----
def test_routing_constants_match_the_source():
    """A change to pass 3's routing fails here, on any machine."""
    flat = lambda p: re.sub(r"\s+", " ", open(os.path.join(ROOT, "zoe_b200", "csrc", p)).read())
    cuh, cu = flat("sw_3pass.cuh"), flat("zoe_cuda.cu")
    assert f"constexpr uint32_t kTpRing = {TP_RING}," in cuh
    assert "uint32_t r = kTpRing; while (r < 2 * bw + 2) r *= 2;" in cuh
    assert f"return bw != 0 ? tp_ring_size(bw) > kTpRing : (unsigned long long)rn * qn > {TP_BOX_CELLS}ull;" in cuh
    assert "return bw != 0 ? 2 * bw + 2 : qn;" in cuh
    # the thread kernel leaves a pair to the warp kernel, and the warp kernel takes it, on the same test
    assert "if (tp_is_large(bw, rn, qn) && tp_row_cells(bw, qn) + 2 <= t.warp_wcap) return;" in cuh
    assert "if (!tp_is_large(bw, rn, qn) || tp_row_cells(bw, qn) + 2 > wcap) continue;" in cuh
    # first width, widest band, doubling (classification, both DP kernels)
    assert "uint32_t bw = (rn > qn ? rn - qn : qn - rn) + 1; if (bw > (qn - 1) / 2) bw = 0;" in cuh
    assert cuh.count("const uint32_t max_bw = (qn - 1) / 2; const uint32_t nbw = 2 * bw <= max_bw ? 2 * bw : 0u;") == 2
    assert TP_WCAP_CAP == 24 * 1024
    assert ("if (wide > 0 && !getenv(\"ZOE_CUDA_TP_THREAD\")) { wcap = (uint32_t)std::min<unsigned long long>"
            "((wide + 2 + 31) & ~31ull, 24 * 1024);") in cu
    # one warp still fits at the cap, so a pair within it is never left without a kernel
    assert "warps = (uint32_t)std::min<size_t>(16, (200 * 1024) / ((size_t)wcap * 8));" in cu
    assert (200 * 1024) // (TP_WCAP_CAP * 8) >= 1


def test_routing_model():
    assert [tp_ring_size(b) for b in (1, 15, 16, 31, 32)] == [32, 32, 64, 64, 128]
    assert tp_route(15, 400, 300) == "shared-ring" and tp_route(16, 400, 300) == "warp-band"
    assert tp_route(16, 400, 300, thread_only=True) == "global-ring"
    assert tp_route(0, 256, 256) == "thread-box" and tp_route(0, 257, 256) == "warp-box"
    assert tp_route(0, 3000, 24574) == "warp-box" and tp_route(0, 3000, 24575) == "thread-box"
    assert tp_attempts(300, 300, 1 | (8 << 8)) == [1, 2, 4, 8]
    assert tp_attempts(256, 256, 2) == [1, 2, 4, 8, 16, 32, 64, 0]
    assert tp_attempts(2146, 31, 2) == [0]
    with pytest.raises(AssertionError):
        tp_attempts(300, 300, 1 | (12 << 8))  # not a width the doubling tries


@pytest.mark.parametrize("name", list(GROUPS))
def test_corpus_reaches_its_edges(name):
    targets, reads, expects = build_group(name)
    reached = set()
    for wm, go, ge in SCORINGS:
        for rn, qn, path in oracle_dp_pairs(targets, reads, wm, go, ge):
            reached |= pair_classes(rn, qn, path)
    assert expects <= reached, sorted(expects - reached, key=str)


def test_corpus_covers_every_edge():
    declared = set()
    for name in GROUPS:
        declared |= build_group(name)[2]
    routes = ("shared-ring", "warp-band", "warp-box", "thread-box")
    want = ({("first", w) for w in FIRST_WIDTHS} | {("doubled", w) for w in DOUBLED_WIDTHS}
            | {("warp-box-qn", q) for q in CHUNK_EDGES} | {("route", r) for r in routes}
            | {("thread-route", "global-ring"), ("thread-route", "thread-box"), ("first-wide", "rn>qn"),
               ("first-wide", "rn<qn"), ("scalar-after-doubling", "thread-box"), ("scalar-after-doubling", "warp-box"),
               ("box-cells", 65536, "thread-box"), ("box-cells", 65792, "warp-box"), ("wcap", 24574, "warp-box"),
               ("wcap", 24575, "thread-box"), ("rows-past-2^20", "warp-box")})
    assert want <= declared, sorted(want - declared, key=str)


# ---- GPU: every group, both orientations, default routing and the single-thread kernel ----
@pytest.mark.gpu
@pytest.mark.parametrize("thread_only", [False, True], ids=["default", "thread"])
@pytest.mark.parametrize("name", list(GROUPS))
def test_group_against_oracle(name, thread_only):
    targets, reads, expects = build_group(name)
    saved = os.environ.pop("ZOE_CUDA_TP_THREAD", None)
    if thread_only:
        os.environ["ZOE_CUDA_TP_THREAD"] = "1"
    reached = set()
    try:
        for wm, go, ge in SCORINGS:
            for pq in (False, True):
                _stats, dp = check_3pass(targets, reads, wm, go, ge, profiled_is_query=pq)
                for _i, _j, rn, qn, path in dp:
                    reached |= pair_classes(rn, qn, path)
    finally:
        os.environ.pop("ZOE_CUDA_TP_THREAD", None)
        if saved is not None:
            os.environ["ZOE_CUDA_TP_THREAD"] = saved
    assert expects <= reached, sorted(expects - reached, key=str)
