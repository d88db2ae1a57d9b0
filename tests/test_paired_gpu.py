"""GPU: the paired-end best-hit search (zoe_cuda_sw_score_paired_best_hit_batch / zoe_cuda_sw_align_paired_best_hit_batch).
Per pair, the winner is the candidate (profiled j, orientation o) -- mate 1 on strand o, mate 2 on strand 1 - o -- of
highest key (Overflowed mates, then the sum of the Some scores; ties to the smallest j, then o = 0); each Some mate is
aligned exactly as the single-strand align call aligns it, and tlen / proper follow from the mates' panel ranges."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import oracle as O
from zoe_b200 import CudaProfiles, PairedHit, WeightMatrix, _lib, reverse_complement, synth
from zoe_b200.alignment import _pack

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W25 = WeightMatrix.new_dna_matrix(2, -5, b"N")
W42 = WeightMatrix.new_dna_matrix(4, -2, b"N")
SCORINGS = [(W25, -10, -1), (W42, -3, -1)]
OPS = {0: "M", 1: "I", 2: "D", 4: "S"}
ALIGN_KEYS = ["ref_start", "ref_end", "query_start", "query_end"]
MATE_KEYS = ["strand", "score", "status", "tier", "runner_up"]


def profiles(targets, wm, go, ge, pq=False, **kw):
    return CudaProfiles.new_with_w256([bytes(t) for t in targets], wm, go, ge, profiled_is_query=pq, **kw)


def cigar_str(words):
    return "".join(f"{int(w) >> 4}{OPS[int(w) & 15]}" for w in words)


# ---- the pair rule in numpy ----------------------------------------------------------------------------------------------
def pair_rule(status, score, tier):
    """Candidate arrays ``[n, 2 (mate), P, 2 (strand)]`` -> ``hit`` [n] and the per-mate outputs [2n] (index 2i + m)."""
    n, _, P, _ = status.shape
    st1, sc1 = status[:, 0], score[:, 0].astype(np.int64)               # [n, P, o]: mate 1 on strand o
    st2, sc2 = status[:, 1, :, ::-1], score[:, 1, :, ::-1].astype(np.int64)  # mate 2 on strand 1 - o
    ovf = (st1 == _lib.OVERFLOWED).astype(np.int64) + (st2 == _lib.OVERFLOWED)
    total = np.where(st1 == _lib.SOME, sc1, 0) + np.where(st2 == _lib.SOME, sc2, 0)
    key = (ovf << 40) + total                                            # candidate c = 2 j + o
    c = np.argmax(key.reshape(n, 2 * P), axis=1)                          # first maximum: smallest j, then o = 0
    hit, o = c // 2, c % 2
    rows = np.arange(n)
    out = {k: np.zeros((n, 2), dtype=np.int64) for k in MATE_KEYS}
    other = np.ones((n, P), bool)
    other[rows, hit] = False
    for m in range(2):
        s = o if m == 0 else 1 - o
        out["strand"][:, m] = s
        st = status[rows, m, hit, s]
        out["status"][:, m] = st
        out["score"][:, m] = score[rows, m, hit, s]
        out["tier"][:, m] = tier[rows, m, hit, s]
        masked = np.where((status[:, m] == _lib.SOME) & other[:, :, None], score[:, m].astype(np.int64), 0)
        out["runner_up"][:, m] = np.where(st == _lib.SOME, masked.reshape(n, -1).max(axis=1), 0)
    return hit, {k: v.reshape(-1) for k, v in out.items()}


def pair_outputs(status, strand, start, end, min_insert, max_insert):
    """tlen and proper from per-mate arrays [2n] (panel ranges)."""
    st, sd = status.reshape(-1, 2), strand.reshape(-1, 2)
    s, e = start.reshape(-1, 2).astype(np.int64), end.reshape(-1, 2).astype(np.int64)
    both = (st == _lib.SOME).all(axis=1)
    extent = e.max(axis=1) - s.min(axis=1)
    o = sd[:, 0]
    tlen = np.where((s[:, 0] < s[:, 1]) | ((s[:, 0] == s[:, 1]) & (o == 0)), extent, -extent)
    fwd, rev = np.where(o == 0, s[:, 0], s[:, 1]), np.where(o == 0, s[:, 1], s[:, 0])
    proper = both & (fwd <= rev) & (extent >= min_insert) & (extent <= max_insert)
    return np.where(both, tlen, 0), proper.astype(np.uint8)


def panel_range(a, pq):
    return (a["query_start"], a["query_end"]) if pq else (a["ref_start"], a["ref_end"])


def interleave(m1, m2):
    return [s for pair in zip(m1, m2) for s in pair]


# ---- 1. oracle parity ------------------------------------------------------------------------------------------------
def oracle_score(target, read, sc):
    rc, s, t = O.sw_score_from(target, read, sc)
    return (rc, s if rc == 0 else 0, t)


def oracle_align(three_pass, target, read, sc, pq):
    if three_pass:
        rc, a, t, _ = O.sw_align_3pass_from(target, read, sc, streamed_is_query=not pq)
    else:
        rc, a, t = O.sw_align_from(target, read, sc, streamed_is_query=not pq)
    return (rc, a.score, t, tuple(a.ref_range), tuple(a.query_range), a.cigar) if rc == 0 else (rc, 0, 0, None, None, None)


def oracle_pairs(targets, seed):
    rng = np.random.default_rng(seed)
    arrs = [np.frombuffer(t, np.uint8) for t in targets]
    m1, m2, _ = synth.paired_reads(rng, arrs, 60, read_len=120, insert_mean=320, insert_sd=60)
    m1, m2 = [bytes(x) for x in m1], [bytes(x) for x in m2]
    for L1, L2 in rng.integers(20, 151, (6, 2)):  # random mates, alone or beside a true mate
        m1.append(bytes(synth.random_dna(rng, int(L1))))
        m2.append(bytes(synth.random_dna(rng, int(L2))) if L2 % 2 else m2[int(L1) % 60])
    m1 += [b"", targets[0][200:320], b"A"]  # a 0-length and a 1-base mate
    m2 += [reverse_complement(targets[1][400:520]), b"", b"C"]
    return m1, m2


@pytest.mark.parametrize("three_pass", [False, True])
@pytest.mark.parametrize("pq", [False, True])
@pytest.mark.parametrize("scoring", [0, 1])
def test_oracle_parity(seqs, three_pass, pq, scoring):
    wm, go, ge = SCORINGS[scoring]
    sc = O.Scoring(wm.weights, wm.mapping.index_map, go, ge)
    targets = [seqs[k] for k in ("H5_HA", "H1_HA", "KJ907631", "KJ907623")]
    m1, m2 = oracle_pairs(targets, 31)
    n, P = len(m1), len(targets)
    prof = profiles(targets, wm, go, ge, pq)
    (b1, o1), (b2, o2) = _pack(m1), _pack(m2)
    a = prof.align_paired_best_hit_arrays(b1, o1, b2, o2, three_pass, min_insert=200, max_insert=450)
    s = prof.sw_score_paired_best_hit_arrays(b1, o1, b2, o2)
    cand = np.zeros((n, 2, P, 2, 3), dtype=np.int64)
    for i in range(n):
        for m, r in enumerate((m1[i], m2[i])):
            for j, t in enumerate(targets):
                for sd in range(2):
                    cand[i, m, j, sd] = oracle_score(t, r if sd == 0 else reverse_complement(r), sc)
    hit, want = pair_rule(cand[..., 0], cand[..., 1], cand[..., 2])
    for out in (a, s):
        assert np.array_equal(out["hit"], hit)
        for key in MATE_KEYS:
            assert np.array_equal(out[key], want[key]), key
    mates = interleave(m1, m2)
    for k, r in enumerate(mates):
        if want["status"][k] != _lib.SOME:
            assert a["cigar_off"][k] == a["cigar_off"][k + 1] and all(a[x][k] == 0 for x in ALIGN_KEYS)
            continue
        seq = r if want["strand"][k] == 0 else reverse_complement(r)
        exp = oracle_align(three_pass, targets[hit[k // 2]], seq, sc, pq)
        got = (_lib.SOME, int(a["score"][k]), int(a["tier"][k]), (int(a["ref_start"][k]), int(a["ref_end"][k])),
               (int(a["query_start"][k]), int(a["query_end"][k])),
               cigar_str(a["cigar"][int(a["cigar_off"][k]):int(a["cigar_off"][k + 1])]))
        assert got == exp, (k, hit[k // 2])
    tlen, proper = pair_outputs(a["status"], a["strand"], *panel_range(a, pq), 200, 450)
    assert np.array_equal(a["tlen"], tlen) and np.array_equal(a["proper"], proper)
    assert 0 < int(proper.sum()) < n and (tlen > 0).any() and (tlen < 0).any()
    assert len(set(hit.tolist())) > 1 and 0 < int(want["strand"][0::2].sum()) < n
    assert list(want["status"][-6:-2]) == [_lib.UNMAPPED, _lib.SOME, _lib.SOME, _lib.UNMAPPED]
    prof.close()


# ---- 2. the rule applied to single-strand calls, at scale ----------------------------------------------------------------
def candidates(prof, m1, m2):
    """[n, 2, P, 2] single-strand score-call results: mate 1, rc(mate 1), mate 2, rc(mate 2)."""
    calls = [[prof.sw_score_arrays(*_pack(x)) for x in (m, [reverse_complement(s) for s in m])] for m in (m1, m2)]
    return tuple(np.stack([np.stack([calls[m][sd][k] for sd in range(2)], axis=2) for m in range(2)], axis=1)
                 for k in (1, 0, 2))


def assert_matches_rule(prof, m1, m2, three_pass, min_insert=0, max_insert=1000, a=None):
    n = len(m1)
    (b1, o1), (b2, o2) = _pack(m1), _pack(m2)
    hit, want = pair_rule(*candidates(prof, m1, m2))
    if a is None:
        a = prof.align_paired_best_hit_arrays(b1, o1, b2, o2, three_pass, min_insert=min_insert, max_insert=max_insert)
    s = prof.sw_score_paired_best_hit_arrays(b1, o1, b2, o2)
    for out in (a, s):
        assert np.array_equal(out["hit"], hit)
        for key in MATE_KEYS:
            assert np.array_equal(out[key], want[key]), key
    # the aligned mates equal the single-strand align call on the selected sequences, column hit
    mates = interleave(m1, m2)
    sel = [r if sd == 0 else reverse_complement(r) for r, sd in zip(mates, want["strand"])]
    ref = prof.align_arrays(*_pack(sel), three_pass=three_pass)
    P = prof.n_profiled
    k = np.arange(2 * n) * P + np.repeat(hit, 2)
    some = want["status"] == _lib.SOME
    for key in ["score", "status", "tier"] + ALIGN_KEYS + ([] if three_pass else ["hazard"]):
        exp = ref[key][k].copy()
        if key in ALIGN_KEYS + ["hazard"]:
            exp[~some] = 0
        else:
            exp[~some] = a[key][~some]
        assert np.array_equal(a[key], exp), key
    if three_pass:
        assert not a["hazard"].any()
    lo, hi = ref["cigar_off"][k].astype(np.int64), ref["cigar_off"][k + 1].astype(np.int64)
    lens = np.where(some, hi - lo, 0)
    want_off = np.zeros(2 * n + 1, dtype=np.uint64)
    want_off[1:] = np.cumsum(lens)
    assert np.array_equal(a["cigar_off"], want_off)
    words = [ref["cigar"][lo[x]:hi[x]] for x in np.nonzero(some)[0]]
    total = int(want_off[-1])
    assert np.array_equal(a["cigar"][:total], np.concatenate(words) if words else np.zeros(0, np.uint32))
    tlen, proper = pair_outputs(a["status"], a["strand"], *panel_range(a, prof.profiled_is_query), min_insert,
                                max_insert)
    assert np.array_equal(a["tlen"], tlen) and np.array_equal(a["proper"], proper)
    return a


def config2_pairs(n, seed=41):
    targets = synth.config2(n_reads=0)[0]
    m1, m2, truth = synth.paired_reads(np.random.default_rng(seed), targets, n)
    return targets, [bytes(x) for x in m1], [bytes(x) for x in m2], truth


@pytest.mark.parametrize("three_pass", [False, True])
def test_config2_matches_rule(three_pass):
    targets, m1, m2, truth = config2_pairs(200_000)
    prof = profiles(targets, W25, -10, -1)
    a = assert_matches_rule(prof, m1, m2, three_pass, 200, 500)
    n, P = len(m1), len(targets)
    (b1, o1), (b2, o2) = _pack(m1), _pack(m2)
    prof.sw_score_paired_best_hit_arrays(b1, o1, b2, o2)
    st = prof.last_stats()  # the score pass over every candidate
    assert st["pairs"] == 4 * n * P and st["tier8"] + st["tier16"] + st["tier32"] + st["overflowed"] + st["unmapped"] == 4 * n * P
    prof.align_paired_best_hit_arrays(b1, o1, b2, o2, three_pass, min_insert=200, max_insert=500)
    st = prof.last_stats()
    some = a["status"] == _lib.SOME
    cells = 2 * 150 * 2 * n * sum(len(t) for t in targets)
    cells += sum(150 * len(targets[int(j)]) for j in np.repeat(a["hit"], 2)[some])
    assert st["pairs"] == 4 * n * P + int(some.sum()) and st["cells"] == cells
    # most pairs land on their true segment in the true orientation, and most of those are proper
    ok = (a["hit"] == truth["target"]) & (a["strand"][0::2] == truth["strand"]) & some.reshape(-1, 2).all(axis=1)
    assert ok.mean() > 0.75 and a["proper"].mean() > 0.65
    prof.close()


# ---- 3. edges ------------------------------------------------------------------------------------------------------------
def test_ties_between_j_and_o(seqs):
    ha = seqs["KJ907631"]
    x = ha[100:150]
    pal = x + reverse_complement(x)
    prof = profiles([seqs["H1_HA"], ha, ha], W25, -10, -1)  # duplicate profiled sequences 1 and 2
    m1 = [ha[300:450], pal, reverse_complement(ha[700:850])]  # pair 2 points outward
    m2 = [reverse_complement(ha[500:650]), pal, ha[900:1050]]
    for three_pass in (False, True):
        a = assert_matches_rule(prof, m1, m2, three_pass)
        assert list(a["hit"]) == [1, 1, 1]                 # the lowest j of the duplicates
        assert list(a["strand"]) == [0, 1, 0, 1, 1, 0]      # palindromic mates: o = 0
        assert list(a["runner_up"][:2]) == [300, 300]       # the duplicate scores the same
        assert list(a["tlen"]) == [350, 50, 350] and list(a["proper"]) == [1, 1, 0]
    prof.close()


def test_overflowed_beats_larger_some_sum(seqs):
    ha = seqs["KJ907631"]
    frag, other = ha[300:450], ha[1000:1100]
    # j = 0: mate 1 scores 120 and mate 2 200 (key (0, 320)); j = 1: mate 1 overflows i8 (300 > 254), mate 2 is
    # barely Some there (key (1, small))
    prof = profiles([frag[:60] + other, frag], W25, -10, -1)
    prof.set_width_policy(8, 8)
    m1, m2 = [frag], [reverse_complement(other)]
    for three_pass in (False, True):
        a = assert_matches_rule(prof, m1, m2, three_pass)
        assert int(a["hit"][0]) == 1 and int(a["status"][0]) == _lib.OVERFLOWED
        assert a["cigar_off"][1] == 0 and a["tlen"][0] == 0 and a["proper"][0] == 0
    st, sc, _ = candidates(prof, m1, m2)
    assert st[0, 0, 0, 0] == st[0, 1, 0, 1] == _lib.SOME and sc[0, 0, 0, 0] + sc[0, 1, 0, 1] >= 320
    prof.close()


def test_unmapped_mates(seqs):
    ha = seqs["KJ907631"]
    prof = profiles([seqs["H1_HA"], ha], W25, -10, -1)
    m1 = [ha[300:450], b"N" * 80, b"", b"N" * 40]
    m2 = [b"N" * 90, reverse_complement(ha[500:650]), b"", b""]
    for three_pass in (False, True):
        a = assert_matches_rule(prof, m1, m2, three_pass)
        assert list(a["status"]) == [_lib.SOME, _lib.UNMAPPED, _lib.UNMAPPED, _lib.SOME] + [_lib.UNMAPPED] * 4
        assert list(a["hit"]) == [1, 1, 0, 0] and list(a["strand"][4:]) == [0, 1, 0, 1]
        assert not a["tlen"].any() and not a["proper"].any()
    rows = prof.sw_align_paired_best_hit_batch(m1, m2, min_insert=0, max_insert=1000)
    assert isinstance(rows[0], PairedHit) and rows[0].index == 1 and rows[0].mate1.result.is_some()
    assert not rows[0].mate2.result.is_some() and not rows[2].mate1.result.is_some()
    prof.close()


@pytest.mark.parametrize("three_pass", [False, True])
def test_mixed_long_short(seqs, three_pass):
    targets = [seqs["KJ907631"], seqs["H1_HA"]]
    rng = np.random.default_rng(43)
    s1, s2, _ = synth.paired_reads(rng, [np.frombuffer(t, np.uint8) for t in targets], 30)
    m1, m2 = [bytes(x) for x in s1], [bytes(x) for x in s2]
    ha = targets[0]
    m1[5], m2[5] = ha[100:1300], reverse_complement(ha[400:1600])  # a long pair
    m1[9] = ha[200:1400]                                            # a long mate beside a short one
    prof = profiles(targets, W25, -10, -1)
    a = assert_matches_rule(prof, m1, m2, three_pass, 100, 2000)
    assert a["status"][10] == a["status"][11] == _lib.SOME and a["proper"][5] == 1 and a["tlen"][5] == 1500
    prof.close()


@pytest.mark.parametrize("three_pass", [False, True])
def test_memory_budget_chunks(three_pass):
    targets, m1, m2, _ = config2_pairs(3000, seed=44)
    prof = profiles(targets, W42, -3, -1)
    (b1, o1), (b2, o2) = _pack(m1), _pack(m2)
    want = prof.align_paired_best_hit_arrays(b1, o1, b2, o2, three_pass, min_insert=200, max_insert=500)
    prof.set_memory_budget(1 << 20)
    got = assert_matches_rule(prof, m1, m2, three_pass, 200, 500)
    for key in want:
        assert np.array_equal(got[key], want[key]), key
    prof.close()


def raw_align_paired(prof, m1, m2, three_pass, cap, min_insert=0, max_insert=1000):
    """One zoe_cuda_sw_align_paired_best_hit_batch call (no retry): (return code, cigar_off)."""
    n = len(m1)
    (b1, o1), (b2, o2) = _pack(m1), _pack(m2)
    p = lambda a, t: a.ctypes.data_as(C.POINTER(t))  # noqa: E731
    hit, tlen = np.zeros(max(n, 1), np.uint32), np.zeros(max(n, 1), np.int32)
    proper = np.zeros(max(n, 1), np.uint8)
    u32 = [np.zeros(max(2 * n, 1), dtype=np.uint32) for _ in range(6)]
    u8 = [np.zeros(max(2 * n, 1), dtype=np.uint8) for _ in range(4)]
    coff = np.zeros(2 * n + 1, dtype=np.uint64)
    cig = np.zeros(max(cap, 1), dtype=np.uint32)
    rc = prof._lib.zoe_cuda_sw_align_paired_best_hit_batch(
        prof._h, p(b1, C.c_uint8), p(o1, C.c_uint64), p(b2, C.c_uint8), p(o2, C.c_uint64), n, int(three_pass),
        min_insert, max_insert, p(hit, C.c_uint32), p(proper, C.c_uint8), p(tlen, C.c_int32), p(u8[0], C.c_uint8),
        p(u32[0], C.c_uint32), p(u8[1], C.c_uint8), p(u8[2], C.c_uint8), p(u32[1], C.c_uint32), p(u32[2], C.c_uint32),
        p(u32[3], C.c_uint32), p(u32[4], C.c_uint32), p(u32[5], C.c_uint32), p(cig, C.c_uint32), p(coff, C.c_uint64),
        cap, p(u8[3], C.c_uint8))
    return rc, coff


@pytest.mark.parametrize("three_pass", [False, True])
def test_cigar_cap_bad_insert_and_context_restored(three_pass):
    targets, m1, m2, _ = config2_pairs(2000, seed=45)
    prof = profiles(targets, W42, -3, -1)
    buf, offs = _pack(m1)
    before_s = prof.sw_score_arrays(buf, offs)
    before_a = prof.align_arrays(buf, offs, three_pass=three_pass)
    (b1, o1), (b2, o2) = _pack(m1), _pack(m2)
    ref = prof.align_paired_best_hit_arrays(b1, o1, b2, o2, three_pass, min_insert=0, max_insert=1000)
    need = int(ref["cigar_off"][-1])
    assert need > 0
    rc, coff = raw_align_paired(prof, m1, m2, three_pass, need - 1)
    assert rc == _lib.E_CIGAR_CAP and int(coff[0]) == need
    rc, coff = raw_align_paired(prof, m1, m2, three_pass, need, min_insert=501, max_insert=500)
    assert rc == _lib.E_BAD_ARG
    rc, coff = raw_align_paired(prof, m1, m2, three_pass, need)
    assert rc == 0 and np.array_equal(coff, ref["cigar_off"])
    after_s = prof.sw_score_arrays(buf, offs)
    after_a = prof.align_arrays(buf, offs, three_pass=three_pass)
    for x, y in zip(before_s, after_s):
        assert np.array_equal(x, y)
    for key in before_a:
        assert np.array_equal(before_a[key], after_a[key]), key
    with pytest.raises(ValueError):
        prof.sw_score_paired_best_hit_arrays(b1, o1, b2, o2[:-1])
    prof.close()


# ---- 4. devices and kernels ------------------------------------------------------------------------------------------
def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.skipif("_n_gpus() < 2")
@pytest.mark.parametrize("three_pass", [False, True])
def test_two_gpus_match_one(three_pass):
    targets, m1, m2, _ = config2_pairs(10_001, seed=46)
    (b1, o1), (b2, o2) = _pack(m1), _pack(m2)
    one = profiles(targets, W25, -10, -1)
    two = profiles(targets, W25, -10, -1, n_devices=2)
    a = one.align_paired_best_hit_arrays(b1, o1, b2, o2, three_pass, min_insert=200, max_insert=500)
    b = two.align_paired_best_hit_arrays(b1, o1, b2, o2, three_pass, min_insert=200, max_insert=500)
    for key in a:
        assert np.array_equal(a[key], b[key]), key
    one.close()
    two.close()


_TRACE = r"""
import sys
import torch
from torch.profiler import ProfilerActivity, profile
sys.path.insert(0, sys.argv[1])
import numpy as np
from zoe_b200 import CudaProfiles, WeightMatrix, synth
targets = synth.config2(n_reads=0)[0]
m1, m2, _ = synth.paired_reads(np.random.default_rng(47), targets, 500)
(b1, o1), (b2, o2) = synth.fixed_len_batch(m1), synth.fixed_len_batch(m2)
prof = CudaProfiles.new_with_w256([bytes(t) for t in targets], WeightMatrix.new_dna_matrix(2, -5, b"N"), -10, -1)
with profile(activities=[ProfilerActivity.CUDA]) as p:
    prof.align_paired_best_hit_arrays(b1, o1, b2, o2, min_insert=200, max_insert=500)
    torch.cuda.synchronize()
prof.close()
print(" ".join(e.name for e in p.events()))
"""


def test_kernels_in_profiler_trace():
    # in a process of its own, as tests/test_best_hit_gpu.py's trace test
    import subprocess
    import sys

    names = subprocess.run([sys.executable, "-c", _TRACE, ROOT], capture_output=True, text=True, check=True).stdout
    for k in ("strand_expand_kernel", "pair_select_kernel", "pair_finalize_kernel", "best_hit_gather_kernel"):
        assert k in names, k
