"""GPU parity: zoe_cuda_sw_align_3pass_batch (through the C ABI) vs the CPU oracle's literal restatement of
sw_align_3pass (src/alignment/sw/three_pass.rs:21-104, banded.rs:40-133) with the ProfileSets escalation
(profile_set.rs:213-290).  Bit-exact: status, score, tier, both ranges and the CIGAR string."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from zoe_b200 import BLOSUM_62, CudaProfiles, DNA_PROFILE_MAP, SeqSrc, WeightMatrix, synth
from zoe_b200.alignment import Status

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W25 = WeightMatrix.new_dna_matrix(2, -5, b"N")
W42 = WeightMatrix.new_dna_matrix(4, -2, b"N")


def osc(wm, go, ge):
    return O.Scoring(wm.weights, wm.mapping.index_map, go, ge)


# ---- pass 3 routing, restated from sw_3pass.cuh and run_3pass_on_device (test_3pass_band_edges_gpu.py pins the constants) ----
TP_RING = 32                 # kTpRing: (H, E) entries a banded attempt keeps in shared memory
TP_BOX_CELLS = 65536         # scalar boxes above this many cells are "large"
TP_WCAP_CAP = 24 * 1024      # row cells + 2 the warp kernel can hold at most (two int rows per warp in shared memory)


def tp_ring_size(bw):
    r = TP_RING
    while r < 2 * bw + 2:
        r *= 2
    return r


def tp_is_large(bw, rn, qn):
    return tp_ring_size(bw) > TP_RING if bw else rn * qn > TP_BOX_CELLS


def tp_row_cells(bw, qn):
    return 2 * bw + 2 if bw else qn


def tp_kernel(bw, rn, qn, thread_only=False):
    """Which kernel runs an attempt at width `bw` (0: the scalar box): "warp" (tp_band_warp_kernel), "shared" (tp_dp_kernel,
    banded, ring in shared memory), "global" (tp_dp_kernel, banded, ring in the pair's scratch) or "thread" (tp_dp_kernel,
    scalar).  Every round's warp capacity covers the widest large row up to the cap, so the rule is per pair."""
    if not thread_only and tp_is_large(bw, rn, qn) and tp_row_cells(bw, qn) + 2 <= TP_WCAP_CAP:
        return "warp"
    if bw == 0:
        return "thread"
    return "shared" if tp_ring_size(bw) <= TP_RING else "global"


def tp_attempts(rn, qn, path):
    """Widths pass 3 tries on a DP pair, in order (0 = the scalar box), from the oracle's box and path (1 | accepted
    width << 8 banded, 2 scalar fallback): |rn - qn| + 1, doubled while it stays <= (qn - 1) / 2 (three_pass.rs:66-84)."""
    assert path & 0xff in (1, 2), path
    max_bw = (qn - 1) // 2
    bw = abs(rn - qn) + 1
    out = []
    while 0 < bw <= max_bw:
        out.append(bw)
        if path & 0xff == 1 and bw == path >> 8:
            return out
        bw *= 2
    assert path == 2, (rn, qn, path, out)  # an accepted width the doubling never tries
    return out + [0]


def check_3pass(targets, seqs, wm, go=-10, ge=-1, profiled_is_query=False, lanes=(32, 16, 8), policy=None):
    """Every pair against the oracle; last_stats() against the oracle's paths, band attempts included.  Returns the stats
    and, per DP pair, (i, j, rn, qn, path) with the box of passes 1-2 (rows streamed, columns profiled)."""
    targets = [bytes(t) for t in targets]
    seqs = [bytes(s) for s in seqs]
    prof = CudaProfiles(targets, wm, go, ge, lanes=lanes, profiled_is_query=profiled_is_query)
    if policy:
        prof.set_width_policy(*policy)
    src = SeqSrc.Reference(seqs) if profiled_is_query else SeqSrc.Query(seqs)
    got = prof.sw_align_3pass_batch(src)
    stats = prof.last_stats()
    sc = osc(wm, go, ge)
    paths = {0: 0, 1: 0, 2: 0}
    attempts = 0
    dp = []
    for i, s in enumerate(seqs):
        for j, t in enumerate(targets):
            standalone = policy and policy[0] == policy[1]  # a standalone StripedProfile<T, N, S>
            if standalone:
                rc, aln, path = O.striped_align_3pass(t, s, sc, policy[0], lanes[0], signed=not policy[2],
                                                      streamed_is_query=not profiled_is_query)
            else:
                rc, aln, _tier, path = O.sw_align_3pass_from(t, s, sc, lanes=lanes, first_bits=policy[0] if policy else 8,
                                                             streamed_is_query=not profiled_is_query)
            g = got[i][j]
            assert g.status.value == rc, (i, j, g, rc, aln)
            if rc == O.SOME:
                a = g.unwrap()
                assert (a.score, a.ref_range, a.query_range, a.states, a.ref_len, a.query_len) == \
                       (aln.score, aln.ref_range, aln.query_range, aln.cigar, aln.ref_len, aln.query_len), (i, j, a, aln, path)
                paths[path & 0xff] += 1
                if path & 0xff:
                    # the box pass 3 ran on: the ranges of passes 1-2, un-inverted
                    if standalone:
                        _, _, rr, qr = O.striped_score_ranges(t, s, sc, policy[0], lanes[0], signed=not policy[2])
                    else:
                        _, _, rr, qr, _ = O.sw_score_ranges_from(t, s, sc, lanes=lanes,
                                                                 first_bits=policy[0] if policy else 8)
                    rn, qn = rr[1] - rr[0], qr[1] - qr[0]
                    attempts += sum(1 for bw in tp_attempts(rn, qn, path) if bw)
                    dp.append((i, j, rn, qn, path))
    assert (stats["tp_nogaps"], stats["tp_banded"], stats["tp_scalar"], stats["tp_band_attempts"]) == \
           (paths[0], paths[1], paths[2], attempts), (stats, paths, attempts)
    prof.close()
    return stats, dp


def test_doc_example():
    # profile_set.rs:192-208: sw_align_from_i8_3pass(SeqSrc::Reference(reference)).score == 26
    prof = CudaProfiles.new_with_w256([b"CGTTCGCCATAAAGGGGG"], W42, -3, -1, profiled_is_query=True)
    r = prof.sw_align_3pass_batch(SeqSrc.Reference([b"ATGCATCGATCGATCGATCGATCGATCGATGC"]))
    a = r[0][0].unwrap()
    assert (a.score, a.query_range, a.ref_range) == (26, (0, 15), (14, 31))
    prof.close()
    check_3pass([b"CGTTCGCCATAAAGGGGG", b"CTCAGATTG"], [b"ATGCATCGATCGATCGATCGATCGATCGATGC", b"GGCCACAGGATTGAG"], W42, -3, -1,
                profiled_is_query=True)
    check_3pass([b"CGTTCGCCATAAAGGGGG", b"CTCAGATTG"], [b"ATGCATCGATCGATCGATCGATCGATCGATGC", b"GGCCACAGGATTGAG"], W42, -3, -1)


def test_config3_sample():
    targets, reads = synth.config3(ROOT, n_reads=400, seed=92)
    stats, _ = check_3pass(targets, list(reads), W25)
    assert stats["tp_nogaps"] > 100 and stats["tp_banded"] > 5


def test_random_pairs_many_scorings_both_orientations():
    rng = np.random.default_rng(73)
    tot = {"tp_nogaps": 0, "tp_banded": 0, "tp_scalar": 0}
    for (ma, mi, go, ge) in [(2, -5, -10, -1), (4, -2, -3, -1), (1, -1, -4, -2), (3, -1, -4, -1), (1, -1, -1, -1),
                             (5, -4, 0, 0), (2, -1, -2, -1)]:
        wm = WeightMatrix.new_dna_matrix(ma, mi, b"N")
        targets = [synth.random_dna(rng, int(L)) for L in (37, 300, 64, 513)]
        seqs = []
        for _ in range(61):
            L = int(rng.integers(1, 150))
            s = synth.random_dna(rng, L)
            if L > 24:
                t = targets[int(rng.integers(0, 4))]
                k = min(L - 4, len(t) - 2, 120)
                st = int(rng.integers(0, len(t) - k + 1))
                frag = synth._mutate(rng, t[st:st + k], 0.06, 0.05, 0.05, np.frombuffer(b"ACGT", dtype=np.uint8))
                k2 = min(len(frag), L - 2)
                s[2:2 + k2] = frag[:k2]
            seqs.append(s)
        seqs.append(np.zeros(0, dtype=np.uint8))
        for st, _ in (check_3pass(targets, seqs, wm, go, ge),
                      check_3pass(targets[:2], seqs[:30], wm, go, ge, profiled_is_query=True, lanes=(16, 8, 4))):
            for k in tot:
                tot[k] += st[k]
    assert all(v > 0 for v in tot.values()), tot


def test_long_gaps_force_band_doubling_and_scalar_fallback():
    # reads with a long deletion / insertion: |dr - dq| + 1 starts wide; very short boxes: max_bandwidth 0 -> scalar
    rng = np.random.default_rng(9)
    t = synth.random_dna(rng, 400)
    seqs = [np.concatenate([t[20:80], t[120:180]]), np.concatenate([t[200:260], synth.random_dna(rng, 25), t[260:330]]),
            np.concatenate([t[10:60], t[64:110], t[118:170]]), t[5:8].copy(), t[300:302].copy(),
            np.concatenate([t[40:70], synth.random_dna(rng, 3), t[70:100], t[103:140]])]
    stats, _ = check_3pass([t], seqs, W42, -3, -1)
    assert stats["tp_band_attempts"] >= stats["tp_banded"]
    check_3pass([t], seqs, W42, -3, -1, profiled_is_query=True)
    check_3pass([t], seqs, W25)


def test_repeats_and_ties():
    wm = WeightMatrix.new_dna_matrix(1, -1, b"N")
    targets = [b"ACACACACACACACACACAC", b"AAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAA", b"ACGTACGTACGTACGTACGTACGT"]
    seqs = [b"ACACAC", b"CACACACA", b"AAAAAAAAAA", b"A", b"ACGTACGT", b"GTACGTAC", b"TTTTTT", b"ACGTTTACGT", b"CACAAACACA",
            b"ACGTACTACGTACGGTACGT", b"ACACATTACACAC"]
    check_3pass(targets, seqs, wm, -2, -1)
    check_3pass(targets, seqs, wm, -2, -1, profiled_is_query=True)


def test_protein_and_width_policies():
    targets, q = synth.config5(n_queries=40)
    check_3pass(targets, list(q), BLOSUM_62)
    rng = np.random.default_rng(5)
    t = [synth.random_dna(rng, 200)]
    seqs = [t[0][10:150].copy(), synth.random_dna(rng, 90), t[0][:64].copy(), np.concatenate([t[0][10:60], t[0][66:150]])]
    check_3pass(t, seqs, W25, policy=(16, 32, False), profiled_is_query=True)
    check_3pass(t, seqs, W25, policy=(32, 32, False), lanes=(8, 8, 8))
    # unsigned standalone profiles over the biased matrix: u8 overflows where i8 would not (limit 255 - bias - 1)
    check_3pass(t, seqs, W25, policy=(8, 8, True), lanes=(16, 16, 16), profiled_is_query=True)
    check_3pass(t, seqs, W25, policy=(16, 16, True), lanes=(16, 16, 16))
    w = WeightMatrix.new(DNA_PROFILE_MAP, 127, -5, b"N")
    stats, _ = check_3pass([b"A" * 600], [b"A" * 600, b"A" * 300, b"A" * 100 + b"C" + b"A" * 100], w)
    assert stats["tier32"] == 1


def test_edge_cases_and_cigar_capacity():
    prof = CudaProfiles.new_with_w256([b"ACGTACGTAC", b"A"], W25, -10, -1)
    r = prof.sw_align_3pass_batch(SeqSrc.Query([b"", b"C", b"TTTT", b"ACGTACGTAC", b"A", b"GGACGTACGTACGG"]))
    assert r[0][0].status is Status.Unmapped and r[0][1].status is Status.Unmapped
    assert r[1][1].status is Status.Unmapped
    a = r[3][0].unwrap()
    assert (a.score, a.ref_range, a.query_range, a.states) == (20, (0, 10), (0, 10), "10M")
    a = r[5][0].unwrap()
    assert (a.score, a.ref_range, a.query_range, a.states) == (20, (0, 10), (2, 12), "2S10M2S")
    # too small a CIGAR buffer: the call reports the capacity it needs, then succeeds
    buf, offs = synth.fixed_len_batch(np.frombuffer(b"ACGTACGTAC" * 4, dtype=np.uint8).reshape(4, 10))
    out = prof.align_arrays(buf, offs, cigar_cap=1, three_pass=True)
    assert int(out["cigar_off"][-1]) == 4 * (1 + 2)  # per read: "10M" vs the first target, "1M9S" vs "A"
    prof.close()
