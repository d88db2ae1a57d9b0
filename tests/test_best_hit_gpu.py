"""GPU: the best-hit search (zoe_cuda_sw_score_best_hit_batch / zoe_cuda_sw_align_best_hit_batch).  Per read, the winner
is the candidate (profiled j, strand s) of highest both-strand rank (Overflowed > Some by score > Unmapped; ties to the
smallest j, then the forward strand), and the align entry point returns exactly what the single-strand align call
returns for that pair."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from zoe_b200 import CudaProfiles, SeqSrc, Strand, WeightMatrix, _lib, reverse_complement, synth
from zoe_b200.alignment import _pack

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W25 = WeightMatrix.new_dna_matrix(2, -5, b"N")
W42 = WeightMatrix.new_dna_matrix(4, -2, b"N")
SCORINGS = [(W25, -10, -1), (W42, -3, -1)]  # compiled-in penalties (GapImm); run-time penalties with hazard pairs
OPS = {0: "M", 1: "I", 2: "D", 4: "S"}
ALIGN_KEYS = ["ref_start", "ref_end", "query_start", "query_end"]


def rank(status, score):
    status, score = np.asarray(status), np.asarray(score)
    return np.where(status == _lib.OVERFLOWED, np.int64(1) << 40,
                    np.where(status == _lib.SOME, score.astype(np.int64) + 1, 0))


def select_rule(status, score, tier):
    """The selection applied to candidate arrays ``[n, P, S]``: (hit, strand, score, status, tier, runner_up)."""
    n, P, S = status.shape
    key = rank(status, score).reshape(n, P * S)            # candidate c = j * S + s
    c = np.argmax(key, axis=1)                             # first maximum: smallest j, then forward
    hit, strand = c // S, c % S
    rows = np.arange(n)
    st, sc, ti = status[rows, hit, strand], score[rows, hit, strand], tier[rows, hit, strand]
    some = status == _lib.SOME
    other = np.ones((n, P), bool)
    other[rows, hit] = False
    masked = np.where(some & other[:, :, None], score.astype(np.int64), 0).reshape(n, -1)
    ru = np.where(st == _lib.SOME, masked.max(axis=1), 0)
    return hit, strand, sc, st, ti, ru


def profiles(targets, wm, go, ge, pq=False, **kw):
    return CudaProfiles.new_with_w256([bytes(t) for t in targets], wm, go, ge, profiled_is_query=pq, **kw)


def cigar_str(words):
    return "".join(f"{int(w) >> 4}{OPS[int(w) & 15]}" for w in words)


# ---- 1. oracle parity ------------------------------------------------------------------------------------------------
def oracle_score(target, read, sc):
    rc, s, t = O.sw_score_from(target, read, sc)
    return (rc, s if rc == 0 else 0, t)  # the score call reports a tier for every status


def oracle_align(three_pass, target, read, sc, pq):
    if three_pass:
        rc, a, t, _ = O.sw_align_3pass_from(target, read, sc, streamed_is_query=not pq)
    else:
        rc, a, t = O.sw_align_from(target, read, sc, streamed_is_query=not pq)
    return (rc, a.score, t, tuple(a.ref_range), tuple(a.query_range), a.cigar) if rc == 0 else (rc, 0, 0, None, None, None)


@pytest.mark.parametrize("three_pass", [False, True])
@pytest.mark.parametrize("both", [False, True])
@pytest.mark.parametrize("pq", [False, True])
@pytest.mark.parametrize("scoring", [0, 1])
def test_oracle_parity(seqs, three_pass, both, pq, scoring):
    wm, go, ge = SCORINGS[scoring]
    sc = O.Scoring(wm.weights, wm.mapping.index_map, go, ge)
    targets = [seqs[k] for k in ("H5_HA", "H1_HA", "KJ907631", "KJ907623")]
    rng = np.random.default_rng(21)
    reads = [bytes(r) for r in synth.illumina_reads(rng, [np.frombuffer(t, np.uint8) for t in targets], 60)]
    reads += [bytes(synth.random_dna(rng, int(L))) for L in rng.integers(20, 151, 12)]
    prof = profiles(targets, wm, go, ge, pq)
    buf, offs = _pack(reads)
    a = prof.align_best_hit_arrays(buf, offs, both_strands=both, three_pass=three_pass)
    s = prof.sw_score_best_hit_arrays(buf, offs, both_strands=both)
    S = 2 if both else 1
    cand = np.zeros((len(reads), len(targets), S, 3), dtype=np.int64)
    for i, r in enumerate(reads):
        for j, t in enumerate(targets):
            for st in range(S):
                cand[i, j, st] = oracle_score(t, r if st == 0 else reverse_complement(r), sc)
    hit, strand, score, status, tier, ru = select_rule(cand[..., 0], cand[..., 1], cand[..., 2])
    for out in (a, s):
        for key, want in (("hit", hit), ("strand", strand), ("score", score), ("status", status), ("tier", tier),
                          ("runner_up", ru)):
            assert np.array_equal(out[key], want), key
    for i, r in enumerate(reads):
        if status[i] != _lib.SOME:
            assert a["cigar_off"][i] == a["cigar_off"][i + 1] and all(a[k][i] == 0 for k in ALIGN_KEYS)
            continue
        seq = r if strand[i] == 0 else reverse_complement(r)
        want = oracle_align(three_pass, targets[hit[i]], seq, sc, pq)
        got = (_lib.SOME, int(a["score"][i]), int(a["tier"][i]), (int(a["ref_start"][i]), int(a["ref_end"][i])),
               (int(a["query_start"][i]), int(a["query_end"][i])),
               cigar_str(a["cigar"][int(a["cigar_off"][i]):int(a["cigar_off"][i + 1])]))
        assert got == want, (i, hit[i], strand[i])
    assert len(set(hit[status == _lib.SOME].tolist())) > 1
    if both:
        assert 0 < strand.sum() < len(reads)
    prof.close()


# ---- 2. self-consistency at scale --------------------------------------------------------------------------------------
def candidates(prof, buf, offs, both):
    """[n, P, S] score-call results of every candidate."""
    n, P = len(offs) - 1, prof.n_profiled
    if not both:
        sc, st, ti = prof.sw_score_arrays(buf, offs)
        return st[:, :, None], sc[:, :, None], ti[:, :, None]
    seqs = [bytes(buf[int(offs[i]):int(offs[i + 1])]) for i in range(n)]
    f = prof.sw_score_arrays(buf, offs)
    r = prof.sw_score_arrays(*_pack([reverse_complement(s) for s in seqs]))
    return tuple(np.stack([f[k], r[k]], axis=2) for k in (1, 0, 2))


def single_align(prof, buf, offs, both, three_pass):
    """[n, P] align results of both strands (strand-1 results from a call on the reverse complements)."""
    f = prof.align_arrays(buf, offs, three_pass=three_pass)
    if not both:
        return [f]
    seqs = [bytes(buf[int(offs[i]):int(offs[i + 1])]) for i in range(len(offs) - 1)]
    return [f, prof.align_arrays(*_pack([reverse_complement(s) for s in seqs]), three_pass=three_pass)]


def assert_matches_rule(prof, buf, offs, both, three_pass, a=None):
    n, P = len(offs) - 1, prof.n_profiled
    st, sc, ti = candidates(prof, buf, offs, both)
    hit, strand, score, status, tier, ru = select_rule(st, sc, ti)
    if a is None:
        a = prof.align_best_hit_arrays(buf, offs, both_strands=both, three_pass=three_pass)
    s = prof.sw_score_best_hit_arrays(buf, offs, both_strands=both)
    for out in (a, s):
        for key, want in (("hit", hit), ("strand", strand), ("score", score), ("status", status), ("tier", tier),
                          ("runner_up", ru)):
            assert np.array_equal(out[key], want), key
    # every alignment output equals column `hit` of the single-strand align call on the winning strand
    ref = single_align(prof, buf, offs, both, three_pass)
    k = np.arange(n) * P + hit
    some = status == _lib.SOME
    for key in ["score", "status", "tier"] + ALIGN_KEYS + ([] if three_pass else ["hazard"]):
        want = np.zeros(n, dtype=a[key].dtype)
        for sd, r in enumerate(ref):
            sel = strand == sd
            want[sel] = r[key][k[sel]]
        if key in ALIGN_KEYS + ["hazard"]:
            want[~some] = 0
        else:
            want[~some] = a[key][~some]  # not aligned: the score pass's values, checked above
        assert np.array_equal(a[key], want), key
    if three_pass:
        assert not a["hazard"].any()
    lens = np.zeros(n, dtype=np.int64)
    words = []
    for i in range(n):
        if not some[i]:
            continue
        r = ref[strand[i]]
        lo, hi = int(r["cigar_off"][k[i]]), int(r["cigar_off"][k[i] + 1])
        lens[i] = hi - lo
        words.append(r["cigar"][lo:hi])
    want_off = np.zeros(n + 1, dtype=np.uint64)
    want_off[1:] = np.cumsum(lens)
    assert np.array_equal(a["cigar_off"], want_off)
    total = int(want_off[-1])
    assert np.array_equal(a["cigar"][:total], np.concatenate(words) if words else np.zeros(0, np.uint32))
    return a


@pytest.mark.parametrize("three_pass", [False, True])
@pytest.mark.parametrize("both", [False, True])
def test_config2_matches_rule(both, three_pass):
    targets, reads = synth.config2(n_reads=50_000)
    prof = profiles(targets, W25, -10, -1)
    buf, offs = synth.fixed_len_batch(reads)
    a = assert_matches_rule(prof, buf, offs, both, three_pass)
    n, P, S = len(reads), len(targets), 2 if both else 1
    for score_only in (True, False):
        if score_only:
            prof.sw_score_best_hit_arrays(buf, offs, both_strands=both)
        else:
            prof.align_best_hit_arrays(buf, offs, both_strands=both, three_pass=three_pass)
        st = prof.last_stats()
        assert st["tier8"] + st["tier16"] + st["tier32"] + st["overflowed"] + st["unmapped"] == S * n * P
        assert st["tier8"] > 0 and st["tier16"] > 0
    aligned = int((a["status"] == _lib.SOME).sum())
    cells = S * 150 * n * sum(len(t) for t in targets)
    cells += sum(150 * len(targets[int(j)]) for j in a["hit"][a["status"] == _lib.SOME])
    assert st["pairs"] == S * n * P + aligned and st["cells"] == cells
    assert st["tier8"] + st["tier16"] + st["tier32"] + st["overflowed"] + st["unmapped"] == S * n * P
    prof.close()


# ---- 3. ties and statuses --------------------------------------------------------------------------------------------
def test_ties_and_statuses(seqs):
    ha = seqs["KJ907631"]
    x = ha[100:150]
    palindrome = x + reverse_complement(x)
    frag = ha[300:450]
    prof = profiles([seqs["H1_HA"], ha, ha], W25, -10, -1)  # duplicate profiled sequences 1 and 2
    reads = [frag, reverse_complement(frag), palindrome, b"N" * 60, b""]
    buf, offs = _pack(reads)
    for three_pass in (False, True):
        a = prof.align_best_hit_arrays(buf, offs, both_strands=True, three_pass=three_pass)
        assert list(a["hit"]) == [1, 1, 1, 0, 0]                      # the lowest j of the duplicates; Unmapped -> 0
        assert list(a["strand"]) == [0, 1, 0, 0, 0]                   # the palindrome: forward
        assert list(a["status"]) == [_lib.SOME] * 3 + [_lib.UNMAPPED] * 2
        assert a["score"][0] == a["score"][1] == 300
        # runner-up: the duplicate j = 2 scores the same; the winner's other strand does not count
        assert a["runner_up"][0] == 300 and a["runner_up"][3] == 0 and a["runner_up"][4] == 0
    # runner-up ignores the winner's other strand: this read scores 300 on both strands of j = 0
    solo = profiles([ha, seqs["H1_HA"]], W25, -10, -1)
    twin = frag + reverse_complement(frag)
    a = solo.sw_score_best_hit_arrays(*_pack([twin]), both_strands=True)
    f, r = solo.sw_score_arrays(*_pack([twin])), solo.sw_score_arrays(*_pack([reverse_complement(twin)]))
    assert f[0][0, 0] == r[0][0, 0] >= 300
    j1 = [int(x[0][0, 1]) for x in (f, r) if x[1][0, 1] == _lib.SOME]
    assert (int(a["hit"][0]), int(a["strand"][0])) == (0, 0) and a["runner_up"][0] == max(j1, default=0) < 300
    solo.close()
    # an Overflowed candidate on j = 1 beats a Some candidate on j = 0 (i8 only: a 150-nt self match scores 300 > 254)
    prof2 = profiles([frag[:60], frag], W25, -10, -1)
    prof2.set_width_policy(8, 8)
    for three_pass in (False, True):
        a = prof2.align_best_hit_arrays(*_pack([frag]), three_pass=three_pass)
        assert (int(a["hit"][0]), int(a["status"][0]), int(a["runner_up"][0])) == (1, _lib.OVERFLOWED, 0)
        assert a["cigar_off"][1] == 0
    prof.close()
    prof2.close()


def test_empty_buckets_and_zoe_rows(seqs):
    rng = np.random.default_rng(3)
    used = [seqs["KJ907631"], seqs["H1_HA"]]
    targets = [b"N" * 1700, used[0], b"N" * 1700, used[1]]  # N scores 0: these can win no read
    reads = [bytes(r) for r in synth.illumina_reads(rng, [np.frombuffer(t, np.uint8) for t in used], 300, random_frac=0.0)]
    prof = profiles(targets, W25, -10, -1)
    buf, offs = _pack(reads)
    a = assert_matches_rule(prof, buf, offs, True, False)
    assert set(a["hit"][a["status"] == _lib.SOME].tolist()) == {1, 3}  # profiled sequences 0 and 2 win no read
    rows = prof.sw_align_best_hit_batch(SeqSrc.Query(reads), both_strands=True)
    full = prof.sw_align_batch(SeqSrc.Query(reads[:20]))
    for i, b in enumerate(rows[:20]):
        assert b.index == int(a["hit"][i]) and b.strand is Strand(int(a["strand"][i]))
        assert b.runner_up == int(a["runner_up"][i])
        if b.strand is Strand.Forward and b.result.is_some():
            assert b.result == full[i][b.index]
    prof.close()


# ---- 4. other paths --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("three_pass", [False, True])
def test_mixed_long_short(seqs, three_pass):
    rng = np.random.default_rng(5)
    targets = [seqs["KJ907631"], seqs["H1_HA"]]
    short = [bytes(r) for r in synth.illumina_reads(rng, [np.frombuffer(t, np.uint8) for t in targets], 40)]
    ha = targets[0]
    long_ = [ha[100:1600], reverse_complement(ha[50:1550]), bytes(synth.random_dna(rng, 1500)), targets[1][10:1200]]
    reads = short[:20] + long_ + short[20:]
    prof = profiles(targets, W25, -10, -1)
    a = assert_matches_rule(prof, *_pack(reads), True, three_pass)
    assert a["status"][20] == _lib.SOME and a["strand"][21] == 1 and a["hit"][23] == 1
    prof.close()


def test_config4_slice_3pass():
    targets, reads = synth.config4(n_reads=120)
    genome = bytes(targets[0])
    panel = [genome[:15000], genome[15000:]]
    prof = profiles(panel, W25, -10, -1)
    a = assert_matches_rule(prof, *_pack([bytes(r) for r in reads]), True, True)
    assert len(set(a["hit"].tolist())) == 2
    prof.close()


@pytest.mark.parametrize("three_pass", [False, True])
def test_memory_budget_chunks(three_pass):
    targets, reads = synth.config2(n_reads=4000, seed_reads=9)
    prof = profiles(targets, W42, -3, -1)
    buf, offs = synth.fixed_len_batch(reads)
    want = prof.align_best_hit_arrays(buf, offs, both_strands=True, three_pass=three_pass)
    prof.set_memory_budget(1 << 20)
    got = assert_matches_rule(prof, buf, offs, True, three_pass)
    for key in want:
        assert np.array_equal(got[key], want[key]), key
    prof.close()


def test_large_panel_column_groups():
    rng = np.random.default_rng(17)
    panel = [synth.random_dna(rng, 1600) for _ in range(70)]  # 112 KB: more than the score kernel stages at once
    reads = synth.illumina_reads(np.random.default_rng(18), panel, 3000)
    prof = profiles(panel, W25, -10, -1)
    for three_pass in (False, True):
        a = assert_matches_rule(prof, *synth.fixed_len_batch(reads), True, three_pass)
        assert len(set(a["hit"][a["status"] == _lib.SOME].tolist())) > 50
    prof.close()


# ---- 5. CIGAR capacity and the context afterwards ----------------------------------------------------------------------
def raw_align_best_hit(prof, buf, offs, both, three_pass, cap):
    """One zoe_cuda_sw_align_best_hit_batch call (no retry): (return code, cigar_off)."""
    import ctypes as C
    n = len(offs) - 1
    p = lambda a, t: a.ctypes.data_as(C.POINTER(t))  # noqa: E731
    u32 = [np.zeros(max(n, 1), dtype=np.uint32) for _ in range(7)]
    u8 = [np.zeros(max(n, 1), dtype=np.uint8) for _ in range(4)]
    coff = np.zeros(n + 1, dtype=np.uint64)
    cig = np.zeros(max(cap, 1), dtype=np.uint32)
    rc = prof._lib.zoe_cuda_sw_align_best_hit_batch(
        prof._h, p(buf, C.c_uint8), p(offs, C.c_uint64), n, int(both), int(three_pass), p(u32[0], C.c_uint32),
        p(u8[0], C.c_uint8), p(u32[1], C.c_uint32), p(u8[1], C.c_uint8), p(u8[2], C.c_uint8), p(u32[2], C.c_uint32),
        p(u32[3], C.c_uint32), p(u32[4], C.c_uint32), p(u32[5], C.c_uint32), p(u32[6], C.c_uint32), p(cig, C.c_uint32),
        p(coff, C.c_uint64), cap, p(u8[3], C.c_uint8))
    return rc, coff


@pytest.mark.parametrize("three_pass", [False, True])
def test_cigar_cap_and_context_restored(three_pass):
    targets, reads = synth.config2(n_reads=3000, seed_reads=12)
    prof = profiles(targets, W42, -3, -1)
    buf, offs = synth.fixed_len_batch(reads)
    before_s = prof.sw_score_arrays(buf, offs)
    before_a = prof.align_arrays(buf, offs, three_pass=three_pass)
    ref = prof.align_best_hit_arrays(buf, offs, both_strands=True, three_pass=three_pass)
    need = int(ref["cigar_off"][-1])
    assert need > 0
    rc, coff = raw_align_best_hit(prof, buf, offs, True, three_pass, need - 1)
    assert rc == _lib.E_CIGAR_CAP and int(coff[0]) == need
    rc, coff = raw_align_best_hit(prof, buf, offs, True, three_pass, need)
    assert rc == 0 and np.array_equal(coff, ref["cigar_off"])
    after_s = prof.sw_score_arrays(buf, offs)
    after_a = prof.align_arrays(buf, offs, three_pass=three_pass)
    for x, y in zip(before_s, after_s):
        assert np.array_equal(x, y)
    for key in before_a:
        assert np.array_equal(before_a[key], after_a[key]), key
    prof.close()


# ---- 6. devices and kernels ------------------------------------------------------------------------------------------
def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.skipif("_n_gpus() < 2")
@pytest.mark.parametrize("three_pass", [False, True])
def test_two_gpus_match_one(three_pass):
    targets, reads = synth.config2(n_reads=20_001, seed_reads=14)
    buf, offs = synth.fixed_len_batch(reads)
    one = profiles(targets, W25, -10, -1)
    two = profiles(targets, W25, -10, -1, n_devices=2)
    a = one.align_best_hit_arrays(buf, offs, both_strands=True, three_pass=three_pass)
    b = two.align_best_hit_arrays(buf, offs, both_strands=True, three_pass=three_pass)
    for key in a:
        assert np.array_equal(a[key], b[key]), key
    one.close()
    two.close()


_TRACE = r"""
import sys
import torch
from torch.profiler import ProfilerActivity, profile
sys.path.insert(0, sys.argv[1])
from zoe_b200 import CudaProfiles, WeightMatrix, synth
targets, reads = synth.config2(n_reads=500, seed_reads=15)
buf, offs = synth.fixed_len_batch(reads)
prof = CudaProfiles.new_with_w256([bytes(t) for t in targets], WeightMatrix.new_dna_matrix(2, -5, b"N"), -10, -1)
with profile(activities=[ProfilerActivity.CUDA]) as p:
    prof.align_best_hit_arrays(buf, offs, both_strands=True)
    torch.cuda.synchronize()
prof.close()
print(" ".join(e.name for e in p.events()))
"""


def test_kernels_in_profiler_trace():
    # In a process of its own: after a torch.profiler session that traced this library's kernels, a later session in
    # the same process recorded no kernels (tests/test_both_strands_gpu.py's trace test, run after this file).
    import subprocess
    import sys

    names = subprocess.run([sys.executable, "-c", _TRACE, ROOT], capture_output=True, text=True, check=True).stdout
    for k in ("best_hit_select_kernel", "best_hit_gather_kernel", "best_hit_scatter_kernel"):
        assert k in names, k
