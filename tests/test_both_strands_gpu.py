"""GPU: the both-strand search (zoe_cuda_sw_*_both_strands_batch).  For every pair the result must be the better of the
single-strand result for the read and for its reverse complement (Overflowed > Some by score > Unmapped, ties to the
forward strand), with every output of the winning strand unchanged."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from zoe_b200 import CudaProfiles, Strand, WeightMatrix, ZoeCudaError, _lib, reverse_complement, synth
from zoe_b200.alignment import _pack
from zoe_b200.matrices import ByteIndexMap

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W25 = WeightMatrix.new_dna_matrix(2, -5, b"N")
W42 = WeightMatrix.new_dna_matrix(4, -2, b"N")
SCORINGS = [(W25, -10, -1), (W42, -3, -1)]  # compiled-in penalties (GapImm); run-time penalties with hazard pairs
OPS = {0: "M", 1: "I", 2: "D", 4: "S"}


def rank(status, score):
    return np.where(status == _lib.OVERFLOWED, np.int64(1) << 40, np.where(status == _lib.SOME, score.astype(np.int64) + 1, 0))


def pick(f, r):
    """The selection rule applied to two single-strand result tuples (status, score, ...)."""
    rf = rank(np.array(f[0]), np.array(f[1]))
    rr = rank(np.array(r[0]), np.array(r[1]))
    return (r, 1) if rr > rf else (f, 0)


def cigar_str(words):
    return "".join(f"{int(w) >> 4}{OPS[int(w) & 15]}" for w in words)


def profiles(targets, wm, go, ge, pq=False):
    return CudaProfiles.new_with_w256([bytes(t) for t in targets], wm, go, ge, profiled_is_query=pq)


# ---- 1. oracle parity ------------------------------------------------------------------------------------------------
def oracle_result(kind, target, read, sc, pq):
    """(status, score, tier, ref_range, query_range, cigar) of the single-strand call, from the C oracle."""
    if kind == "score":
        rc, s, t = O.sw_score_from(target, read, sc)
        return (rc, s if rc == 0 else 0, t if rc == 0 else 0, None, None, None)
    if kind == "ranges":
        rc, s, rr, qr, t = O.sw_score_ranges_from(target, read, sc, streamed_is_query=not pq)
        return (rc, s, t, rr, qr, None) if rc == 0 else (rc, 0, 0, None, None, None)
    if kind == "align":
        rc, a, t = O.sw_align_from(target, read, sc, streamed_is_query=not pq)
    else:
        rc, a, t, _ = O.sw_align_3pass_from(target, read, sc, streamed_is_query=not pq)
    return (rc, a.score, t, tuple(a.ref_range), tuple(a.query_range), a.cigar) if rc == 0 else (rc, 0, 0, None, None, None)


def run_both(prof, kind, seqs):
    """Flat dict of the both-strand outputs for a list of reads."""
    buf, offs = _pack([bytes(s) for s in seqs])
    if kind == "score":
        score, status, tier, strand = prof.sw_score_both_strands_arrays(buf, offs)
        return {"score": score.ravel(), "status": status.ravel(), "tier": tier.ravel(), "strand": strand.ravel()}
    if kind == "ranges":
        return prof.ranges_both_strands_arrays(buf, offs)
    return prof.align_both_strands_arrays(buf, offs, three_pass=kind == "3pass")


def run_single(prof, kind, seqs):
    buf, offs = _pack([bytes(s) for s in seqs])
    if kind == "score":
        score, status, tier = prof.sw_score_arrays(buf, offs)
        return {"score": score.ravel(), "status": status.ravel(), "tier": tier.ravel()}
    if kind == "ranges":
        return prof.ranges_arrays(buf, offs)
    return prof.align_arrays(buf, offs, three_pass=kind == "3pass")


def got_result(kind, a, k):
    st = int(a["status"][k])
    if st != _lib.SOME:
        return (st, 0, 0, None, None, None)
    if kind == "score":
        return (st, int(a["score"][k]), int(a["tier"][k]), None, None, None)
    rr, qr = (int(a["ref_start"][k]), int(a["ref_end"][k])), (int(a["query_start"][k]), int(a["query_end"][k]))
    cig = None if kind == "ranges" else cigar_str(a["cigar"][int(a["cigar_off"][k]):int(a["cigar_off"][k + 1])])
    return (st, int(a["score"][k]), int(a["tier"][k]), rr, qr, cig)


def parity_reads(seqs_fixture):
    rng = np.random.default_rng(11)
    ha = synth.golden_ha(ROOT)
    reads = [bytes(r) for r in synth.illumina_reads(rng, [ha], 240)]  # both strands
    reads += [bytes(synth.random_dna(rng, int(L))) for L in rng.integers(20, 151, 40)]
    return [ha], reads


@pytest.mark.parametrize("kind", ["score", "ranges", "align", "3pass"])
@pytest.mark.parametrize("pq", [False, True])
@pytest.mark.parametrize("scoring", [0, 1])
def test_oracle_parity(seqs, kind, pq, scoring):
    wm, go, ge = SCORINGS[scoring]
    sc = O.Scoring(wm.weights, wm.mapping.index_map, go, ge)
    for targets, reads in (parity_reads(seqs), ([seqs["H5_HA"]], [seqs["H1_HA"], reverse_complement(seqs["H1_HA"])])):
        prof = profiles(targets, wm, go, ge, pq)
        a = run_both(prof, kind, reads)
        n_rev = 0
        for i, r in enumerate(reads):
            for j, t in enumerate(targets):
                k = i * len(targets) + j
                want, strand = pick(oracle_result(kind, bytes(t), r, sc, pq),
                                    oracle_result(kind, bytes(t), reverse_complement(r), sc, pq))
                assert (got_result(kind, a, k), int(a["strand"][k])) == (want, strand), (kind, pq, i, j)
                n_rev += strand
        if len(reads) > 2:
            assert 0 < n_rev < len(reads)
        prof.close()


# ---- 2. self-consistency at scale --------------------------------------------------------------------------------------
def select_np(f, r, keys, cigar=False):
    """The selection rule applied element-wise to two single-strand array dicts (and their CIGAR streams)."""
    rev = rank(r["status"], r["score"]) > rank(f["status"], f["score"])
    out = {k: np.where(rev, r[k], f[k]) for k in keys}
    out["strand"] = rev.astype(np.uint8)
    if cigar:
        n = len(rev)
        lo = np.where(rev, r["cigar_off"][:n], f["cigar_off"][:n]).astype(np.int64)
        ln = np.where(rev, np.diff(r["cigar_off"]), np.diff(f["cigar_off"])).astype(np.int64)
        off = np.zeros(n + 1, dtype=np.uint64)
        off[1:] = np.cumsum(ln)
        src = np.repeat(lo - off[:-1].astype(np.int64), ln) + np.arange(int(off[-1]))
        fc, rc_ = f["cigar"], r["cigar"]
        from_rev = np.repeat(rev, ln)
        out["cigar_off"] = off
        out["cigar"] = np.where(from_rev, rc_[np.minimum(src, len(rc_) - 1)], fc[np.minimum(src, len(fc) - 1)])
    return out


def assert_consistent(prof, kind, seqs):
    both = run_both(prof, kind, seqs)
    f = run_single(prof, kind, seqs)
    r = run_single(prof, kind, [reverse_complement(s) for s in seqs])
    keys = ["score", "status", "tier"] + ([] if kind == "score" else ["ref_start", "ref_end", "query_start", "query_end"])
    keys += ["hazard"] if kind == "align" else []
    want = select_np(f, r, keys, cigar=kind in ("align", "3pass"))
    pairs = len(seqs) * prof.n_profiled
    for key in keys + ["strand"]:
        assert np.array_equal(both[key][:pairs], want[key][:pairs]), key
    if kind in ("align", "3pass"):
        assert np.array_equal(both["cigar_off"][:pairs + 1], want["cigar_off"])
        total = int(want["cigar_off"][-1])
        assert np.array_equal(both["cigar"][:total], want["cigar"][:total])
    return both


@pytest.mark.parametrize("kind", ["ranges", "align", "3pass"])
def test_config3_matches_two_single_strand_calls(kind):
    targets, reads = synth.config3(ROOT, n_reads=50_000)
    prof = profiles(targets, W25, -10, -1)
    both = assert_consistent(prof, kind, [bytes(r) for r in reads])
    # true-origin reads (score >= 200) are reverse-complemented with probability 1/2 by the generator
    mapped = (both["status"][:len(reads)] == _lib.SOME) & (both["score"][:len(reads)] >= 200)
    frac = both["strand"][:len(reads)][mapped].mean()
    assert mapped.mean() > 0.8 and 0.45 < frac < 0.55, (mapped.mean(), frac)
    prof.close()


def test_config2_score_matches_two_single_strand_calls():
    targets, reads = synth.config2(n_reads=20_000)
    prof = profiles(targets, W25, -10, -1)
    seqs = [bytes(r) for r in reads]
    assert_consistent(prof, "score", seqs)
    # the statistics count both strands
    buf, offs = _pack(seqs)
    prof.sw_score_both_strands_arrays(buf, offs)
    st = prof.last_stats()
    pairs = 2 * len(seqs) * prof.n_profiled
    assert st["pairs"] == pairs and st["cells"] == 2 * 150 * len(seqs) * sum(len(t) for t in targets)
    assert st["tier8"] + st["tier16"] + st["tier32"] + st["overflowed"] + st["unmapped"] == pairs
    prof.close()


# ---- 3. ties and statuses --------------------------------------------------------------------------------------------
def test_ties_and_statuses():
    ha = bytes(synth.golden_ha(ROOT))
    x = ha[100:150]
    palindrome = x + reverse_complement(x)
    assert reverse_complement(palindrome) == palindrome
    reads = [palindrome, b"N" * 60, b"", b"A", ha[300:450], reverse_complement(ha[300:450])]
    prof = profiles([ha], W25, -10, -1)
    for kind in ("score", "ranges", "align", "3pass"):
        a = run_both(prof, kind, reads)
        st, strand = a["status"][:len(reads)], a["strand"][:len(reads)]
        assert strand[0] == 0 and st[0] == _lib.SOME, kind                   # palindrome: equal scores
        assert strand[1] == 0 and st[1] == _lib.UNMAPPED, kind               # both strands Unmapped
        assert strand[2] == 0 and st[2] == _lib.UNMAPPED, kind               # 0-length read
        assert strand[3] == 0 and st[3] == _lib.SOME and a["score"][3] == 2, kind  # 1 base: A and T both occur
        assert list(strand[4:6]) == [0, 1] and a["score"][4] == a["score"][5] == 300, kind
    # Overflowed beats Some, in each direction: i8 only, a 150-nt self match scores 300 > 254
    prof.set_width_policy(8, 8)
    for kind in ("score", "ranges", "align", "3pass"):
        a = run_both(prof, kind, [ha[300:450], reverse_complement(ha[300:450])])
        assert list(a["status"][:2]) == [_lib.OVERFLOWED] * 2 and list(a["strand"][:2]) == [0, 1], kind
    prof.close()


# ---- 4. the complement table on the device ---------------------------------------------------------------------------
def test_device_complement_table():
    letters = b"ACGTURYKMBVDHSWN"
    m = ByteIndexMap(letters, b"N")
    wm = WeightMatrix.new(m, 1, -1)
    read = letters + letters.lower()
    comp = dict(zip(b"ACGTURYKMBVDHSWN", b"TGCAAYRMKVBHDSWN"))
    expected = bytes(comp[b & ~0x20] | (b & 0x20) for b in read)[::-1]
    assert reverse_complement(read) == expected
    prof = profiles([expected], wm, -10, -1)
    for kind in ("score", "ranges", "align", "3pass"):
        a = run_both(prof, kind, [read])
        assert (int(a["status"][0]), int(a["score"][0]), int(a["strand"][0])) == (_lib.SOME, len(read), 1), kind
    prof.close()


# ---- 5. paths other than short reads ---------------------------------------------------------------------------------
def test_mixed_long_short_align_vs_oracle():
    rng = np.random.default_rng(5)
    ha = synth.golden_ha(ROOT)
    short = [bytes(r) for r in synth.illumina_reads(rng, [ha], 12)]
    long_ = [bytes(ha[100:1600]), reverse_complement(bytes(ha[50:1550])), bytes(synth.random_dna(rng, 1500))]
    reads = short[:6] + long_ + short[6:]
    prof = profiles([ha], W25, -10, -1)
    a = run_both(prof, "align", reads)
    sc = O.Scoring(W25.weights, W25.mapping.index_map, -10, -1)
    for i, r in enumerate(reads):
        want, strand = pick(oracle_result("align", bytes(ha), r, sc, False),
                            oracle_result("align", bytes(ha), reverse_complement(r), sc, False))
        assert (got_result("align", a, i), int(a["strand"][i])) == (want, strand), i
    assert list(a["strand"][6:9]) == [0, 1, a["strand"][8]]
    prof.close()


@pytest.mark.parametrize("kind", ["ranges", "3pass"])
def test_config4_slice(kind):
    targets, reads = synth.config4(n_reads=150)
    prof = profiles(targets, W25, -10, -1)
    both = assert_consistent(prof, kind, [bytes(r) for r in reads])
    assert 0.3 < both["strand"][:len(reads)].mean() < 0.7
    prof.close()


@pytest.mark.parametrize("kind", ["ranges", "align", "3pass"])
def test_memory_budget_chunks(kind):
    targets, reads = synth.config3(ROOT, n_reads=3000, seed=9)
    seqs = [bytes(r) for r in reads]
    prof = profiles(targets, W42, -3, -1)
    want = run_both(prof, kind, seqs)
    prof.set_memory_budget(4 << 20)
    got = assert_consistent(prof, kind, seqs)
    for key, v in want.items():
        assert np.array_equal(got[key][:len(v)] if key != "cigar" else got[key][:int(want["cigar_off"][-1])],
                              v if key != "cigar" else v[:int(want["cigar_off"][-1])]), key
    prof.close()


@pytest.mark.parametrize("three_pass", [False, True])
def test_cigar_cap_reports_selected_need(three_pass):
    targets, reads = synth.config3(ROOT, n_reads=2000, seed=12)
    seqs = [bytes(r) for r in reads]
    prof = profiles(targets, W42, -3, -1)
    buf, offs = _pack(seqs)
    ref = prof.align_both_strands_arrays(buf, offs, three_pass=three_pass)
    need_sel = int(ref["cigar_off"][len(seqs)])
    need_both = int(prof.align_arrays(buf, offs, three_pass=three_pass)["cigar_off"][len(seqs)]) + int(
        prof.align_arrays(*_pack([reverse_complement(s) for s in seqs]), three_pass=three_pass)["cigar_off"][len(seqs)])
    assert need_sel < need_both
    out = {k: np.zeros_like(v) for k, v in ref.items()}
    out["cigar"] = np.zeros(need_sel - 1, dtype=np.uint32)
    with pytest.raises(ZoeCudaError) as e:
        prof.align_into(buf, offs, out, three_pass=three_pass)
    assert e.value.code == _lib.E_CIGAR_CAP and int(out["cigar_off"][0]) == need_sel
    out["cigar"] = np.zeros(need_sel, dtype=np.uint32)
    prof.align_into(buf, offs, out, three_pass=three_pass)
    for key in ref:
        assert np.array_equal(out[key][:need_sel] if key == "cigar" else out[key], ref[key][:need_sel] if key == "cigar" else ref[key]), key
    prof.close()


def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.skipif("_n_gpus() < 2")
@pytest.mark.parametrize("kind", ["score", "ranges", "align", "3pass"])
def test_two_gpus_match_one(kind):
    targets, reads = synth.config3(ROOT, n_reads=20_001, seed=13)
    seqs = [bytes(r) for r in reads]
    one = CudaProfiles.new_with_w256([bytes(t) for t in targets], W25, -10, -1)
    two = CudaProfiles.new_with_w256([bytes(t) for t in targets], W25, -10, -1, n_devices=2)
    a, b = run_both(one, kind, seqs), run_both(two, kind, seqs)
    for key in a:
        assert np.array_equal(a[key], b[key]), key
    one.close()
    two.close()


# ---- 6. the new kernels run ------------------------------------------------------------------------------------------
def test_kernels_in_profiler_trace():
    import torch
    from torch.profiler import ProfilerActivity, profile

    targets, reads = synth.config3(ROOT, n_reads=500, seed=14)
    seqs = [bytes(r) for r in reads]
    prof = profiles(targets, W25, -10, -1)
    for kind in ("score", "ranges", "align", "3pass"):
        with profile(activities=[ProfilerActivity.CUDA]) as p:
            run_both(prof, kind, seqs)
            torch.cuda.synchronize()
        names = " ".join(e.name for e in p.events())
        assert "strand_expand_kernel" in names and "strand_select_kernel" in names, kind
        if kind in ("align", "3pass"):
            assert "strand_cigar_gather_kernel" in names, kind
    prof.close()
