"""Every score, align, ranges and 3-pass kernel instantiation against the oracle, at its row-bucket and width edges.

The host picks one (G, K) instantiation of each kernel family per batch: the tightest row capacity G * K of
kScoreKernels that holds the batch's longest streamed sequence.  The protein path picks a K of the shared-rows kernels
from the longest profiled sequence, and its streaming variant when every streamed sequence has 64 residues or more.
A batch of random reads up to 150 nt only ever runs the (8, 19) kernels, so this file builds one batch per bucket whose
longest read is exactly the bucket's capacity, plus batches that sit exactly at the thresholds where the dispatcher
switches between the packed 16-bit and the 32-bit kernels.  Every comparison is exact: status, score, tier, both
ranges and the CIGAR.

References: the vectorised CPU port (oracle.cpu_baseline, pinned to the C oracle by test_cpu_baseline.py) for every
score and align pair, and the plain-C oracle for ranges, 3-pass and a sample of the align pairs."""
import os
import re

import numpy as np
import pytest

from oracle import cpu_baseline as CB
from oracle import oracle as O
from zoe_b200 import BLOSUM_62, CudaProfiles, DNA_PROFILE_MAP, SeqSrc, WeightMatrix, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ZOE_CUDA_CU = os.path.join(ROOT, "zoe_b200", "csrc", "zoe_cuda.cu")

# ---- the dispatcher's tables (checked against zoe_cuda.cu by test_tables_match_the_dispatcher) ----
# (G, K) of every entry of kScoreKernels: score, align, ranges and 3-pass kernels of G * K rows
SCORE_KERNELS = [(8, 4), (8, 8), (8, 13), (8, 16), (8, 19), (8, 24), (8, 32),
                 (16, 19), (16, 24), (16, 32), (32, 10), (32, 20), (32, 24), (32, 32)]
ROW_BUCKETS = sorted(g * k for g, k in SCORE_KERNELS)
# K of sw_score_rows_kernel<32, K> and sw_score_rows_stream_kernel<32, K> (kRowsKernels, kRowsStreamKernels)
ROWS_KERNEL_K = [8, 12, 16, 18, 20, 24, 28, 32]
MAX_ROWS_SINGLE_PASS = 1024  # longer streamed sequences take the long-row kernels
ROWS_STREAM_MIN_LEN = 64     # the streaming rows kernel needs every streamed sequence this long
PACKED_BOUND = 60000         # score: min(longest streamed, longest profiled) x max weight from here on runs 32-bit directly


def packed_overflow_threshold(w):
    """Score: a packed lane at or above this is flagged and its sequence re-run at 32 bits."""
    return 32767 - w - 1


def ranges_packed_bound(w, go):
    """Ranges: packed 16-bit kernels only while min(longest streamed, longest profiled) x w is below this (go < 0)."""
    return 32767 - w - 1 + go


# Instantiations no input can launch: listed so that a coverage table can name them, kept in the build.
UNREACHABLE = {
    # bound = rows x max weight <= 256 x 127 = 32512 < 32767 - 127 - 1: no packed lane of these buckets can be flagged
    **{f"sw_score_kernel<{g},{k},false,1,GapRt": "packed lanes of <= 256 rows never overflow (256 x 127 < 32639)"
       for g, k in SCORE_KERNELS if g * k <= 256},
    # ranges run 32-bit only when rows x w >= 32767 - w - 1 - go; with w, -go <= 127 that needs more than 192 rows
    **{f"sw_ends_kernel<{g},{k},false>": "ranges of <= 192 rows stay packed (192 x 127 < 32767 - 128 - 127)"
       for g, k in SCORE_KERNELS if g * k <= 192},
}


def _block(src, name):
    m = re.search(re.escape(name) + r"\[\]\s*=\s*\{(.*?)\n\};", src, re.S)
    assert m, name
    return m.group(1)


def test_tables_match_the_dispatcher():
    """Adding or removing an instantiation without adding it to this sweep fails here, on any machine."""
    src = open(ZOE_CUDA_CU).read()
    assert [(int(g), int(k)) for g, k in re.findall(r"ZK\((\d+),\s*(\d+)\)", _block(src, "kScoreKernels"))] == SCORE_KERNELS
    assert len(set(ROW_BUCKETS)) == len(ROW_BUCKETS)  # one kernel per capacity: the longest read picks it alone
    for table, kern in (("kRowsKernels", "sw_score_rows_kernel"), ("kRowsStreamKernels", "sw_score_rows_stream_kernel")):
        rows = re.findall(r"\{(\d+),\s*" + kern + r"<32,\s*(\d+)>\}", _block(src, table))
        assert [int(a) for a, _ in rows] == ROWS_KERNEL_K and [int(b) for _, b in rows] == ROWS_KERNEL_K, table
    flat = re.sub(r"\s+", " ", src)
    assert "constexpr int kMaxRowsSinglePass = 32 * 32;" in flat and 32 * 32 == MAX_ROWS_SINGLE_PASS
    assert f"ctx->staged_min_len >= {ROWS_STREAM_MIN_LEN}" in flat
    assert f"ctx->staged_max_len >= {ROWS_STREAM_MIN_LEN}" in flat  # the rows path needs one sequence that long
    assert flat.count(f"bool packed_ok = bound < {PACKED_BOUND};") == 2  # single-pass and long-row score paths
    assert "if (bound >= (uint64_t)(kPackedLimit - ctx->max_weight - 1))" in flat
    assert "constexpr int kPackedLimit = kHalfMax ? 0x7C00 : 32767;" in re.sub(r"\s+", " ", open(
        os.path.join(ROOT, "zoe_b200", "csrc", "sw_score.cuh")).read())
    assert "const bool packed = bound < (uint64_t)(32767 - std::max(ctx->max_weight, 0) - 1 - ctx->go);" in flat
    assert packed_overflow_threshold(127) == 32639 and ranges_packed_bound(127, -127) == 32512
    # the GapImm sweep of test_gap_imm_gpu.py walks the same buckets
    from test_gap_imm_gpu import ROW_BUCKETS as gap_imm_buckets
    assert gap_imm_buckets == ROW_BUCKETS


# ---- inputs ----
W25 = WeightMatrix.new_dna_matrix(2, -5, b"N")
W42 = WeightMatrix.new_dna_matrix(4, -2, b"N")
# (matrix, go, ge): the benchmark scoring, whose packed score kernels have the penalties compiled in (GapImm), and a
# tie-heavy scoring with run-time penalties whose walks meet E == H == F ties (literal kernels)
SCORINGS = [(W25, -10, -1), (W42, -3, -1)]
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def osc(wm, go, ge):
    return O.Scoring(wm.weights, wm.mapping.index_map, go, ge)


def tandem(rng, L):
    unit = synth.random_dna(rng, int(rng.integers(1, 5)))
    return np.resize(unit, L).astype(np.uint8)


def related(rng, t, L):
    """A mutated stretch of t (substitutions and short indels) of exactly L bases, padded with random bases."""
    st = int(rng.integers(0, max(len(t) - L, 0) + 1))
    frag = synth._mutate(rng, t[st:st + L + 8], 0.05, 0.02, 0.02, ACGT)[:L]
    pad = L - len(frag)
    left = int(rng.integers(0, pad + 1))
    return np.concatenate([synth.random_dna(rng, left), frag, synth.random_dna(rng, pad - left)]).astype(np.uint8)


def bucket_inputs(cap, prev, n, seed):
    """Three profiled sequences (longer than cap with a tandem-repeat stretch, mid-sized, a few dozen columns) and n
    (odd) streamed sequences whose longest is exactly cap.  Lengths 0 and 1 sit next to a cap-long read in the same
    packed task (sequences 2t and 2t + 1 share one); prev + 1 and cap - 1 are the bucket's inner edges."""
    rng = np.random.default_rng(seed)
    long_t = synth.random_dna(rng, cap + 150)
    long_t[cap // 2:cap // 2 + 60] = tandem(rng, 60)
    targets = [long_t, synth.random_dna(rng, max(cap // 2, 40) + 3), synth.random_dna(rng, 37)]
    lens = [cap, 0, cap, 1, prev + 1, cap - 1, cap] + [int(x) for x in rng.integers(prev + 1, cap + 1, n - 7)]
    reads = []
    for i, L in enumerate(lens):
        kind = i % 6
        if L < 2 or kind == 4:
            reads.append(synth.random_dna(rng, L))
        elif kind == 5:
            reads.append(tandem(rng, L))
        else:  # mostly mutated stretches of the long target, some of the mid-sized one
            reads.append(related(rng, targets[1] if kind == 3 else long_t, L))
    assert max(len(r) for r in reads) == cap and len(reads) % 2 == 1
    return targets, reads


def port_score(targets, buf, offs, wm, go, ge):
    pbuf, poff = synth.pack(targets)
    return CB.score_batch(pbuf, poff, buf, offs, wm.weights, wm.mapping.index_map, go, ge, width_bits=256)


def port_align(targets, buf, offs, wm, go, ge, profiled_is_query):
    pbuf, poff = synth.pack(targets)
    return CB.align_batch(pbuf, poff, buf, offs, wm.weights, wm.mapping.index_map, go, ge, width_bits=256,
                          streamed_is_query=not profiled_is_query)


def assert_align_equal(got, want, n_pairs, what):
    assert np.array_equal(got["status"][:n_pairs], want["status"]), what
    assert np.array_equal(got["tier"][:n_pairs], want["tier"]), what
    assert CB.compare_alignments(got, want, n_pairs) == 0, what


def cigar_str(a, k):
    ops = "MIDNS"
    return "".join(f"{int(w) >> 4}{ops[int(w) & 15]}" for w in a["cigar"][int(a["cigar_off"][k]):int(a["cigar_off"][k + 1])])


def ranges_oracle(targets, reads, sc, profiled_is_query):
    return [[O.sw_score_ranges_from(bytes(t), bytes(s), sc, streamed_is_query=not profiled_is_query)
             for t in targets] for s in reads]


def assert_ranges_equal(got, want, what):
    nt = len(want[0])
    for i, row in enumerate(want):
        for j, (rc, score, rr, qr, tier) in enumerate(row):
            k = i * nt + j
            g = (int(got["status"][k]), int(got["tier"][k]))
            assert g == (rc, tier), (what, i, j, g, rc, tier)
            if rc == O.SOME:
                g = (int(got["score"][k]), (int(got["ref_start"][k]), int(got["ref_end"][k])),
                     (int(got["query_start"][k]), int(got["query_end"][k])))
                assert g == (score, rr, qr), (what, i, j, g, score, rr, qr)


def with_env(name, fn):
    saved = os.environ.pop(name, None)
    os.environ[name] = "1"
    try:
        return fn()
    finally:
        os.environ.pop(name)
        if saved is not None:
            os.environ[name] = saved


# ---- 2. one batch per row bucket ----
@pytest.mark.gpu
@pytest.mark.parametrize("G,K", SCORE_KERNELS)
def test_row_bucket_against_oracle(G, K):
    from test_3pass_gpu import check_3pass
    cap = G * K
    prev = max([b for b in ROW_BUCKETS if b < cap], default=0)
    targets, reads = bucket_inputs(cap, prev, 31 if cap >= 512 else 51, seed=cap)
    buf, offs = synth.pack(reads)
    n_pairs = len(reads) * len(targets)
    pinned = hazard = fallback = 0
    for wm, go, ge in SCORINGS:
        sc = osc(wm, go, ge)
        want_score = port_score(targets, buf, offs, wm, go, ge)
        for pq in (False, True):
            what = (cap, go, pq)
            prof = CudaProfiles.new_with_w256(targets, wm, go, ge, profiled_is_query=pq)
            got = prof.sw_score_arrays(buf, offs)
            for g, w, name in zip(got, want_score, ("score", "status", "tier")):
                assert np.array_equal(g, w), (what, name)
            want = port_align(targets, buf, offs, wm, go, ge, pq)
            for mode in (CudaProfiles.ALIGN_FULL, CudaProfiles.ALIGN_WINDOW):
                # window: the smallest checkpoint spacing (raised to G) and a 1-column slack, so walks leave their window
                prof.set_align_options(mode, 2, 1)
                a = prof.align_arrays(buf, offs)
                assert_align_equal(a, want, n_pairs, (what, mode))
                st = prof.last_stats()
                if mode == CudaProfiles.ALIGN_WINDOW:
                    pinned += st["window_pinned"]
                    fallback += st["window_fallback"]
                if go == -3:
                    hazard += st["hazard"]
            for i in range(0, len(reads), 5):  # the plain-C oracle on a sample
                j = (i // 5) % len(targets)
                rc, aln, tier = O.sw_align_from(bytes(targets[j]), bytes(reads[i]), sc, streamed_is_query=not pq)
                k = i * len(targets) + j
                assert (int(a["status"][k]), int(a["tier"][k])) == (rc, tier), (what, i, j)
                if rc == O.SOME:
                    got_a = (int(a["score"][k]), (int(a["ref_start"][k]), int(a["ref_end"][k])),
                             (int(a["query_start"][k]), int(a["query_end"][k])), cigar_str(a, k))
                    assert got_a == (aln.score, aln.ref_range, aln.query_range, aln.cigar), (what, i, j)
            # ranges: the scan + pin + reverse-scan path, and the forward ends kernel (read on every call)
            want_r = ranges_oracle(targets, reads, sc, pq)
            assert_ranges_equal(prof.ranges_arrays(buf, offs), want_r, (what, "ranges"))
            assert_ranges_equal(with_env("ZOE_CUDA_RANGES_SLOW", lambda: prof.ranges_arrays(buf, offs)), want_r,
                                (what, "ranges slow"))
            prof.close()
            check_3pass(targets, reads, wm, go, ge, profiled_is_query=pq)
    assert pinned > 0  # recurring maxima: the pin sweep ran
    if G == 32:
        assert fallback > 0  # walks longer than the slack went to the literal kernels
    if cap >= 512:
        assert hazard > 0  # the literal kernels ran at this row count


@pytest.mark.gpu
@pytest.mark.parametrize("cap", [256, 512, 1024])  # one bucket per G
def test_window_pass_a_from_global_memory(cap):
    """A profiled panel beyond the 96 KB staging area: pass A reads the codes from global memory."""
    rng = np.random.default_rng(300 + cap)
    panel = [synth.random_dna(rng, int(L)) for L in rng.integers(2300, 2700, 40)]
    assert sum(len(t) for t in panel) > 96 * 1024
    prev = max(b for b in ROW_BUCKETS if b < cap)
    reads = [related(rng, panel[i % 40], int(L)) for i, L in enumerate([cap, prev + 1, cap - 1, 1, cap])]
    reads.append(tandem(rng, cap // 2))
    reads.append(synth.random_dna(rng, cap))
    buf, offs = synth.pack(reads)
    for wm, go, ge in SCORINGS:
        prof = CudaProfiles.new_with_w256(panel, wm, go, ge)
        prof.set_align_options(CudaProfiles.ALIGN_WINDOW, 6, 16)
        a = prof.align_arrays(buf, offs)
        prof.close()
        assert_align_equal(a, port_align(panel, buf, offs, wm, go, ge, False), len(reads) * len(panel), (cap, go))


# ---- 3. width edges at exact thresholds ----
W127 = WeightMatrix.new(DNA_PROFILE_MAP, 127, -5, b"N")
W100 = WeightMatrix.new(DNA_PROFILE_MAP, 100, -100, b"N")


def self_match_targets(rng, lens):
    return [np.concatenate([synth.random_dna(rng, 20), np.full(L, ord("A"), np.uint8), synth.random_dna(rng, 20)])
            for L in lens]


@pytest.mark.gpu
def test_score_packed_overflow_threshold():
    """256 x 127 = 32512 stays packed (no pair can be flagged); 257 x 127 = 32639 reaches the threshold and is re-run."""
    rng = np.random.default_rng(61)
    targets = self_match_targets(rng, [300]) + [synth.random_dna(rng, 90)]
    for lens, rerun in (([256, 255, 100, 0, 256], False), ([257, 256, 1, 120, 258], True), ([258, 256, 255], True)):
        reads = [np.full(L, ord("A"), np.uint8) for L in lens] + [synth.random_dna(rng, 200)]
        buf, offs = synth.pack(reads)
        for go, ge in ((-10, -1), (-11, -1)):  # GapImm and run-time packed kernels
            prof = CudaProfiles.new_with_w256(targets, W127, go, ge)
            got = prof.sw_score_arrays(buf, offs)
            st = prof.last_stats()
            prof.close()
            for g, w in zip(got, port_score(targets, buf, offs, W127, go, ge)):
                assert np.array_equal(g, w), (lens, go)
            assert (st["rerun_wide"] > 0) == rerun, (lens, st)
            assert (got[0][:, 0] >= packed_overflow_threshold(127)).any() == rerun


@pytest.mark.gpu
@pytest.mark.parametrize("wm,prof_lens", [(W100, (599, 600, 601)), (W127, (472, 473))])
@pytest.mark.parametrize("cap", [768, 1024])
def test_score_bound_goes_wide_directly(wm, prof_lens, cap):
    """min(longest streamed, longest profiled) x w below 60000: packed + re-run of the flagged; from 60000 on: 32-bit."""
    w = int(wm.weights.max())
    rng = np.random.default_rng(cap + w)
    for P in prof_lens:
        targets = [np.full(P, ord("A"), np.uint8), synth.random_dna(rng, 50)]
        reads = [np.full(L, ord("A"), np.uint8) for L in (cap, P, P - 1, 300)] + [synth.random_dna(rng, cap - 5)]
        buf, offs = synth.pack(reads)
        prof = CudaProfiles.new_with_w256(targets, wm, -10, -1)
        got = prof.sw_score_arrays(buf, offs)
        st = prof.last_stats()
        prof.close()
        for g, want in zip(got, port_score(targets, buf, offs, wm, -10, -1)):
            assert np.array_equal(g, want), (P, cap)
        assert int(got[0][1, 0]) == P * w
        assert (st["rerun_wide"] > 0) == (P * w < PACKED_BOUND), (P, st)  # direct 32-bit runs re-run nothing


@pytest.mark.gpu
@pytest.mark.parametrize("go", [-127, -126])
def test_ranges_packed_bound(go):
    """256 rows x 127: 32512 < 32767 - 128 + go holds for go = -126 (packed ends kernel), not for -127 (32-bit)."""
    rng = np.random.default_rng(67)
    assert (256 * 127 < ranges_packed_bound(127, go)) == (go == -126)
    targets = self_match_targets(rng, [256, 120]) + [synth.random_dna(rng, 41)]
    reads = [np.full(L, ord("A"), np.uint8) for L in (256, 0, 255, 1, 193)]
    reads += [related(rng, targets[0], 200), tandem(rng, 256)]
    buf, offs = synth.pack(reads)
    sc = osc(W127, go, -1)
    want = ranges_oracle(targets, reads, sc, False)
    prof = CudaProfiles.new_with_w256(targets, W127, go, -1)
    assert_ranges_equal(prof.ranges_arrays(buf, offs), want, go)
    assert_ranges_equal(with_env("ZOE_CUDA_RANGES_SLOW", lambda: prof.ranges_arrays(buf, offs)), want, (go, "slow"))
    prof.close()
    assert want[0][0][1] == 256 * 127


# a matrix whose self-match scores hit any integer: A-A 127, C-C 1 (mismatch -5, bias 5)
def _tier_matrix():
    w = np.where(np.eye(len(DNA_PROFILE_MAP), dtype=bool), 1, -5).astype(np.int8)
    a = DNA_PROFILE_MAP.to_index(ord("A"))
    w[a, a] = 127
    return WeightMatrix(DNA_PROFILE_MAP, w)


W_TIER = _tier_matrix()


def scoring_exactly(s):
    """A sequence whose best local alignment against any sequence containing it scores exactly s under W_TIER."""
    return b"A" * (s // 127) + b"C" * (s % 127)


TIER_EDGES = {None: [253, 254, 255, 65533, 65534, 65535],  # signed chain i8 -> i16 -> i32: limits 254 and 65534
              (8, 8, True): [248, 249, 250],                    # unsigned u8 over the biased matrix: 255 - 5 - 1
              (16, 16, True): [65528, 65529, 65530]}            # unsigned u16: 65535 - 5 - 1


def tier_oracle(entry, t, s, sc, policy, lanes):
    """(status, score, ref_range, query_range, cigar) of one pair; ranges and CIGAR None where the entry has none."""
    if policy:
        b = policy[0]
        if entry == "score":
            rc, v = O.striped_score(t, s, sc, b, lanes, signed=False)
            return rc, v, None, None, None
        if entry == "ranges":
            rc, v, rr, qr = O.striped_score_ranges(t, s, sc, b, lanes, signed=False, streamed_is_query=True)
            return rc, v, rr, qr, None
        fn = O.striped_align if entry == "align" else O.striped_align_3pass
        rc, a = fn(t, s, sc, b, lanes, signed=False, streamed_is_query=True)[:2]
    else:
        if entry == "score":
            rc, v, _ = O.sw_score_from(t, s, sc)
            return rc, v, None, None, None
        if entry == "ranges":
            rc, v, rr, qr, _ = O.sw_score_ranges_from(t, s, sc, streamed_is_query=True)
            return rc, v, rr, qr, None
        fn = O.sw_align_from if entry == "align" else O.sw_align_3pass_from
        rc, a = fn(t, s, sc, streamed_is_query=True)[:2]
    return (rc, a.score, a.ref_range, a.query_range, a.cigar) if rc == O.SOME else (rc, 0, None, None, None)


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["score", "align", "ranges", "3pass"])
@pytest.mark.parametrize("policy", list(TIER_EDGES), ids=["signed", "u8", "u16"])
def test_tier_limits(policy, entry):
    """Scores one below, at and one above each tier limit, through each entry point, against the oracle."""
    assert W_TIER.get_bias() == 5 and int(W_TIER.weights.max()) == 127
    scores = TIER_EDGES[policy]
    sc = osc(W_TIER, -10, -1)
    seqs = [scoring_exactly(v) for v in scores]
    targets = [b"G" * 5 + s + b"T" * 5 for s in seqs]  # every read scores its own value against its own target
    lanes = 16 if policy and policy[0] == 16 else 32      # standalone profiles of 256-bit vectors
    prof = CudaProfiles(targets, W_TIER, -10, -1, lanes=(lanes,) * 3 if policy else (32, 16, 8))
    if policy:
        prof.set_width_policy(*policy)
    buf, offs = synth.pack([np.frombuffer(s, dtype=np.uint8) for s in seqs])
    if entry == "score":
        score, status, tier = (x.ravel() for x in prof.sw_score_arrays(buf, offs))
        got = {"score": score, "status": status, "tier": tier}
    elif entry == "ranges":
        got = prof.ranges_arrays(buf, offs)
    else:
        got = prof.align_arrays(buf, offs, three_pass=entry == "3pass")
    prof.close()
    nt = len(targets)
    for i, s in enumerate(seqs):
        for j, t in enumerate(targets):
            k = i * nt + j
            rc, v, rr, qr, cig = tier_oracle(entry, t, s, sc, policy, lanes)
            g, w = [int(got["status"][k])], [rc]
            if rc != O.SOME:
                assert g == w, (entry, policy, i, j)
                continue
            g.append(int(got["score"][k]))
            w.append(v)
            if rr is not None:
                g += [(int(got["ref_start"][k]), int(got["ref_end"][k])), (int(got["query_start"][k]), int(got["query_end"][k]))]
                w += [rr, qr]
            if cig is not None:
                g.append(cigar_str(got, k))
                w.append(cig)
            assert g == w, (entry, policy, i, j)
            if i == j:
                assert v == scores[i]
    # the diagonal: below and at a limit fits the narrow type; above it escalates (signed) or overflows (unsigned)
    diag = [int(got["status"][i * nt + i]) for i in range(len(seqs))]
    if policy:
        assert diag == [O.SOME, O.SOME, O.OVERFLOWED], diag
    else:
        assert [int(got["tier"][i * nt + i]) for i in range(len(seqs))] == [8, 8, 16, 16, 16, 32]


@pytest.mark.gpu
def test_align_packed_overflow_beyond_u16_is_overflowed():
    """Reduced case: under u16 (standalone, unsigned), a 524-base self match scoring 65530 overflows the packed fill,
    whose 32-bit re-run then finds it beyond u16 (limit 65529).  The pair stayed on the literal kernels' list with
    score 0, which tier_for maps to the first tier, and the align call failed with an internal score mismatch."""
    s = scoring_exactly(65530)
    prof = CudaProfiles([b"G" * 5 + s + b"T" * 5], W_TIER, -10, -1, lanes=(16, 16, 16))
    prof.set_width_policy(16, 16, True)
    buf, offs = synth.pack([np.frombuffer(s, dtype=np.uint8)])
    a = prof.align_arrays(buf, offs)
    st = prof.last_stats()
    prof.close()
    assert (int(a["status"][0]), int(a["score"][0]), int(a["cigar_off"][1])) == (O.OVERFLOWED, 0, 0)
    assert st["rerun_wide"] == 1 and st["overflowed"] == 1


# ---- 4. protein shared-rows kernels ----
AA = np.frombuffer(b"ACDEFGHIKLMNPQRSTVWY", dtype=np.uint8)


def protein_batch(rng, targets, lens):
    out = []
    for i, L in enumerate(lens):
        q = AA[rng.integers(0, 20, L)]
        t = targets[i % len(targets)]
        w = min(L, len(t)) - 2
        if w > 10 and i % 3:
            st = int(rng.integers(0, len(t) - w + 1))
            keep = rng.random(w) > 0.3
            q[1:1 + w] = np.where(keep, t[st:st + w], q[1:1 + w])
        out.append(q)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("K", ROWS_KERNEL_K)
def test_protein_rows_kernels(K):
    """Profiled lengths 32 K and 32 K_prev + 1 pick sw_score_rows*_kernel<32, K>; shortest streamed 64 -> the
    streaming variant, 63 -> the non-streaming one."""
    k_prev = max([k for k in ROWS_KERNEL_K if k < K], default=0)
    rng = np.random.default_rng(500 + K)
    targets = [AA[rng.integers(0, 20, 32 * K)], AA[rng.integers(0, 20, 32 * k_prev + 1)], AA[rng.integers(0, 20, 45)]]
    for shortest in (ROWS_STREAM_MIN_LEN, ROWS_STREAM_MIN_LEN - 1):
        lens = [shortest, 1000, shortest + 1, 32 * K] + [int(x) for x in rng.integers(shortest, 1001, 17)]
        reads = protein_batch(rng, targets, lens)
        assert len(reads) % 2 == 1
        buf, offs = synth.pack(reads)
        prof = CudaProfiles.new_with_w256(targets, BLOSUM_62, -10, -1)
        got = prof.sw_score_arrays(buf, offs)
        prof.close()
        for g, w in zip(got, port_score(targets, buf, offs, BLOSUM_62, -10, -1)):
            assert np.array_equal(g, w), (K, shortest)
    # packed lanes that overflow (match weight 120) with a bound below 60000: flagged pairs re-run at 32 bits
    wide = WeightMatrix(BLOSUM_62.mapping, np.where(np.eye(25, dtype=bool), 120, -4).astype(np.int8))
    P = min(32 * K, 480)
    t = AA[rng.integers(0, 20, P)]
    for shortest in (ROWS_STREAM_MIN_LEN, ROWS_STREAM_MIN_LEN - 1):
        reads = [t.copy(), t[:shortest].copy(), AA[rng.integers(0, 20, 200)], t[P // 4:].copy(), t[: P - 1].copy()]
        buf, offs = synth.pack(reads)
        prof = CudaProfiles.new_with_w256([t], wide, -10, -1)
        got = prof.sw_score_arrays(buf, offs)
        st = prof.last_stats()
        prof.close()
        for g, w in zip(got, port_score([t], buf, offs, wide, -10, -1)):
            assert np.array_equal(g, w), (K, shortest, "wide")
        assert int(got[0][0, 0]) == 120 * P
        assert (st["rerun_wide"] > 0) == (120 * P >= packed_overflow_threshold(120)), st


# ---- 5. which instantiations run, read from the profiler's kernel trace ----
def _norm(name):
    name = re.sub(r"\s+", "", name).replace("(anonymousnamespace)::", "")
    return re.sub(r"\b\w+::", "", name)


def expected_kernels():
    exp = []
    for g, k in SCORE_KERNELS:
        for ns in (1, 2):
            exp += [f"sw_score_kernel<{g},{k},true,{ns},GapRt", f"sw_score_kernel<{g},{k},true,{ns},GapImm<10,1>"]
        exp += [f"sw_align_fill_kernel<{g},{k},true>", f"sw_align_scan_kernel<{g},{k},true,false>",
                f"sw_align_scan_kernel<{g},{k},false,false>", f"sw_align_scan_kernel<{g},{k},true,true>",
                f"sw_align_winfill_kernel<{g},{k},true>", f"sw_align_winfill_kernel<{g},{k},false>",
                f"sw_ends_kernel<{g},{k},true>"]
    for k in ROWS_KERNEL_K:
        exp += [f"sw_score_rows_kernel<32,{k}>", f"sw_score_rows_stream_kernel<32,{k}>"]
    return exp


def run_compact_sweep():
    """Sections 2 and 4 in small: every bucket through score (one and three profiled sequences, both scorings), align
    (full, window, window over a > 96 KB panel) and ranges (default, ZOE_CUDA_RANGES_SLOW); every rows K both ways."""
    rng = np.random.default_rng(7)
    panel = [synth.random_dna(rng, int(L)) for L in rng.integers(2300, 2700, 40)]
    for g, k in SCORE_KERNELS:
        cap = g * k
        prev = max([b for b in ROW_BUCKETS if b < cap], default=0)
        targets, reads = bucket_inputs(cap, prev, 9, seed=cap + 1)
        buf, offs = synth.pack(reads)
        for wm, go, ge in SCORINGS:
            for tset in (targets[:1], targets):
                prof = CudaProfiles.new_with_w256(tset, wm, go, ge)
                prof.sw_score_arrays(buf, offs)
                prof.close()
        prof = CudaProfiles.new_with_w256(targets, W42, -3, -1)
        for mode in (CudaProfiles.ALIGN_FULL, CudaProfiles.ALIGN_WINDOW):
            prof.set_align_options(mode, 6, 16)
            prof.align_arrays(buf, offs)
        prof.ranges_arrays(buf, offs)
        with_env("ZOE_CUDA_RANGES_SLOW", lambda: prof.ranges_arrays(buf, offs))
        prof.close()
        prof = CudaProfiles.new_with_w256(panel, W25, -10, -1)
        prof.set_align_options(CudaProfiles.ALIGN_WINDOW, 6, 16)
        pbuf, poff = synth.pack([related(rng, panel[i], L) for i, L in enumerate([cap, prev + 1, cap])])
        prof.align_arrays(pbuf, poff)
        prof.close()
    for K in ROWS_KERNEL_K:
        targets = [AA[rng.integers(0, 20, 32 * K)]]
        for shortest in (ROWS_STREAM_MIN_LEN, ROWS_STREAM_MIN_LEN - 1):
            buf, offs = synth.pack(protein_batch(rng, targets, [shortest, 300, 200]))
            prof = CudaProfiles.new_with_w256(targets, BLOSUM_62, -10, -1)
            prof.sw_score_arrays(buf, offs)
            prof.close()


@pytest.mark.gpu
def test_every_listed_instantiation_is_launched():
    torch = pytest.importorskip("torch")
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        run_compact_sweep()
        torch.cuda.synchronize()
    names = {_norm(e.name) for e in p.events() if "kernel" in e.name}
    launched = lambda pat: any(pat in n for n in names)
    missing = [e for e in expected_kernels() if not launched(e)]
    assert not missing, (len(missing), missing[:20], sorted(n for n in names if n.startswith(("sw_", "void")))[:20])
    unexpected = [e for e in UNREACHABLE if launched(e)]
    assert not unexpected, unexpected
