"""GPU: the packed score kernels with the gap penalties compiled in (GapImm, used for the scorings listed in
kGapImmPairs) against the oracle, and against the run-time-penalty kernels (ZOE_CUDA_NO_GAP_IMM) in the same process."""
import os

import numpy as np
import pytest

from oracle import cpu_baseline as CB
from oracle import oracle as O
from zoe_b200 import CudaProfiles, WeightMatrix, synth

pytestmark = pytest.mark.gpu
W25 = WeightMatrix.new_dna_matrix(2, -5, b"N")
# row capacity G * K of every packed score kernel (kScoreKernels): a batch runs the tightest fit for its longest read
ROW_BUCKETS = [32, 64, 104, 128, 152, 192, 256, 304, 320, 384, 512, 640, 768, 1024]


def make(targets, wm, go, ge, no_imm=False):
    saved = os.environ.pop("ZOE_CUDA_NO_GAP_IMM", None)
    if no_imm:
        os.environ["ZOE_CUDA_NO_GAP_IMM"] = "1"
    try:  # the switch is read when the context is created
        return CudaProfiles.new_with_w256([bytes(t) for t in targets], wm, go, ge)
    finally:
        os.environ.pop("ZOE_CUDA_NO_GAP_IMM", None)
        if saved is not None:
            os.environ["ZOE_CUDA_NO_GAP_IMM"] = saved


def related_reads(rng, targets, lens, mut=0.08):
    """Reads of the given lengths, each a mutated stretch of a random target (forward strand) or random bases."""
    out = []
    for L in lens:
        t = targets[int(rng.integers(0, len(targets)))]
        if L <= len(t) and rng.random() < 0.8:
            st = int(rng.integers(0, len(t) - L + 1))
            r = t[st:st + L].copy()
            sub = rng.random(L) < mut
            r[sub] = synth.random_dna(rng, int(sub.sum()))
        else:
            r = synth.random_dna(rng, L)
        out.append(r)
    return out


def cpu_scores(targets, buf, offs, wm, go, ge):
    pbuf, poff = synth.pack(targets)
    return CB.score_batch(pbuf, poff, buf, offs, wm.weights, wm.mapping.index_map, go, ge)


def assert_same(got, want):
    for g, w, what in zip(got, want, ("score", "status", "tier")):
        assert np.array_equal(np.asarray(g), np.asarray(w)), what


@pytest.mark.parametrize("go,ge", [(-10, -1), (-11, -2)])  # (10, 1) is listed (GapImm); (11, 2) is not (GapRt)
def test_config2_reads_vs_oracle(go, ge):
    targets, reads = synth.config2(n_reads=3000, seed_reads=17)
    buf, offs = synth.fixed_len_batch(reads)
    prof = make(targets, W25, go, ge)
    score, status, tier = prof.sw_score_arrays(buf, offs)
    prof.close()
    c_score, c_status, c_tier = cpu_scores(targets, buf, offs, W25, go, ge)
    assert np.array_equal(status, c_status)
    ok = c_status == O.SOME
    assert np.array_equal(score[ok], c_score[ok]) and np.array_equal(tier[ok], c_tier[ok])
    assert (tier == 16).any() and (tier == 8).any()
    sc = O.Scoring(W25.weights, W25.mapping.index_map, go, ge)
    for i in range(0, 3000, 150):  # the plain-C oracle on a sample
        for j, t in enumerate(targets):
            rc, s_, t_ = O.sw_score_from(bytes(t), bytes(reads[i]), sc)
            assert (int(status[i, j]), int(score[i, j]), int(tier[i, j])) == (rc, s_, t_), (i, j)


def test_same_results_with_and_without_compiled_penalties():
    rng = np.random.default_rng(23)
    c2_targets, c2_reads = synth.config2(n_reads=50_000, seed_reads=29)
    panel = [synth.random_dna(rng, int(L)) for L in rng.integers(1500, 2600, 60)]  # > 96 KB: swept group by group
    assert sum(len(t) for t in panel) > 96 * 1024
    cases = [(c2_targets, list(c2_reads))]
    lo = 1
    for cap in ROW_BUCKETS:  # one batch per kernel: its longest read is exactly the bucket's capacity
        lens = list(rng.integers(lo, cap + 1, 299)) + [cap]
        cases.append((c2_targets, related_reads(rng, c2_targets, lens)))
        lo = cap + 1
    cases.append((c2_targets[:1], related_reads(rng, c2_targets[:1], [150] * 501)))  # one profiled sequence: NS = 1
    cases.append((c2_targets[:3], related_reads(rng, c2_targets[:3], [150] * 500)))  # odd count: a lone last stream
    cases.append((panel, related_reads(rng, panel, list(rng.integers(100, 153, 2001)))))
    for targets, reads in cases:
        buf, offs = synth.pack(reads)
        got = {}
        for no_imm in (False, True):
            prof = make(targets, W25, -10, -1, no_imm=no_imm)
            got[no_imm] = prof.sw_score_arrays(buf, offs)
            prof.close()
        assert_same(got[False], got[True])
    # the large panel against the CPU port as well
    c_score, c_status, c_tier = cpu_scores(panel, buf, offs, W25, -10, -1)
    assert_same(got[False], (c_score, c_status, c_tier))


def test_packed_overflow_still_escalates():
    """Match weight 100: a stretch of 330+ matching bases reaches the packed overflow threshold (32767 - 100), so those
    pairs are re-run by the 32-bit kernel (which reads the penalties from ScoreParams) and must still be exact; reads of
    300 nt or less cannot overflow and keep their packed result.  The reads stay below 600 nt: from a bound of 600 x 100
    on, a batch skips the packed kernel and runs at 32 bits directly."""
    wm = WeightMatrix.new_dna_matrix(100, -100, b"N")
    targets, _ = synth.config2(n_reads=1)
    rng = np.random.default_rng(37)
    reads = related_reads(rng, targets, list(rng.integers(150, 600, 300)), mut=0.002)
    buf, offs = synth.pack(reads)
    prof = make(targets, wm, -10, -1)
    got = prof.sw_score_arrays(buf, offs)
    assert prof.last_stats()["rerun_wide"] > 0
    prof.close()
    c_score, c_status, c_tier = cpu_scores(targets, buf, offs, wm, -10, -1)
    assert_same(got, (c_score, c_status, c_tier))
    assert (got[0] >= 32767 - 100).any() and (got[0] < 32767 - 100).any()  # both kernels carry results
    prof = make(targets, wm, -10, -1, no_imm=True)
    assert_same(got, prof.sw_score_arrays(buf, offs))
    prof.close()
