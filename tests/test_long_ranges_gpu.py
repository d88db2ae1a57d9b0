"""GPU parity of the long-row ranges pipeline (sw_ends_long_kernel forward + reverse, streamed sequences > 1024
residues) against the oracle's literal restatement of sw_simd_score_ranges (striped.rs:355-388) -- zoe's functions take
any length, so do zoe_cuda_sw_score_ranges_batch and everything built on it."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from zoe_b200 import BLOSUM_62, CudaProfiles, DNA_PROFILE_MAP, SeqSrc, WeightMatrix, synth
from test_ranges_gpu import check_ranges, W25, W42

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def golden(name):
    with open(os.path.join(ROOT, "tests", "golden", name), "rb") as f:
        return f.read().strip()


def ont_reads(rng, genome, n, lo, hi):
    reads = []
    for _ in range(n):
        L = int(rng.integers(lo, hi + 1))
        s = int(rng.integers(0, len(genome) - L + 1))
        frag = genome[s:s + L]
        if rng.random() < 0.3:
            frag = synth._COMP[frag[::-1]]
        reads.append(synth._mutate(rng, frag, 0.06, 0.04, 0.04, synth._ACGT))
    return reads


def test_cy137594_self_alignment_ranges():
    # sw/test.rs:264-280: CY137594 (1 686 nt) against itself scores 3372; the ranges are the whole sequence
    s = golden("CY137594.txt")
    assert len(s) > 1024
    prof = CudaProfiles.new_with_w256([s], W25, -10, -1)
    a = prof.sw_score_ranges_batch(SeqSrc.Query([s]))[0][0].unwrap()
    prof.close()
    assert (a.score, a.ref_range, a.query_range) == (3372, (0, len(s)), (0, len(s)))
    check_ranges([s], [s, s[100:1500], s[::-1]], W25)


def test_long_reads_vs_genome_both_orientations():
    rng = np.random.default_rng(21)
    genome = synth.random_dna(rng, 7000)
    reads = ont_reads(rng, genome, 10, 1100, 3200) + [synth.random_dna(rng, 1500)]
    check_ranges([genome], reads, W25)
    check_ranges([genome], reads[:4], W25, profiled_is_query=True)


def test_mixed_short_and_long_batch_and_panel():
    rng = np.random.default_rng(22)
    g1, g2 = synth.random_dna(rng, 4000), synth.random_dna(rng, 1300)
    reads = ont_reads(rng, g1, 4, 1025, 2000) + ont_reads(rng, g1, 5, 40, 300) + ont_reads(rng, g2, 2, 800, 1300)
    reads += [np.zeros(0, dtype=np.uint8), synth.random_dna(rng, 1)]
    check_ranges([g1, g2], reads, W25)
    check_ranges([g1, g2], reads[:6], W42, go=-3, ge=-1)


def test_long_protein_and_unpacked_path():
    rng = np.random.default_rng(23)
    t = synth._AA20[rng.integers(0, 20, 1800)]
    q = [synth._mutate(rng, t[100:1400], 0.2, 0.02, 0.02, synth._AA20), synth._AA20[rng.integers(0, 20, 1200)]]
    check_ranges([t], q, BLOSUM_62)
    # match 127: the packed 16-bit lanes could overflow -> the 32-bit instantiation
    w = WeightMatrix.new(DNA_PROFILE_MAP, 127, -5, b"N")
    g = synth.random_dna(rng, 2500)
    check_ranges([g], [g[200:1500].copy(), g[:1100].copy()], w)


def test_long_path_forced_on_short_reads():
    # the chunked-row pipeline on config-3 reads (one chunk, many pairs): end-cell ties, unmapped reads, both halves
    targets, reads = synth.config3(ROOT, n_reads=300)
    os.environ["ZOE_CUDA_RANGES_LONG"] = "1"
    try:
        check_ranges(targets, list(reads), W25)
        rng = np.random.default_rng(24)
        seqs = [synth.random_dna(rng, int(k)) for k in rng.integers(1, 400, 120)]
        check_ranges([synth.random_dna(rng, 900), synth.random_dna(rng, 77)], seqs, W42, go=-3, ge=-1)
    finally:
        os.environ.pop("ZOE_CUDA_RANGES_LONG", None)


def test_3pass_cigars_for_long_reads():
    # SURVEY 8(f).1: the memory-light alignment is what gives long reads a CIGAR (three_pass.rs:21-104)
    from test_3pass_gpu import check_3pass
    rng = np.random.default_rng(25)
    genome = synth.random_dna(rng, 5000)
    reads = ont_reads(rng, genome, 7, 1100, 2600) + [synth.random_dna(rng, 1300), genome[500:1700].copy()]
    stats, _ = check_3pass([genome], reads, W25)
    assert stats["tp_banded"] > 0
    check_3pass([genome], reads[:3], W25, profiled_is_query=True)
    s = golden("CY137594.txt")
    check_3pass([s], [s], W25)  # zoe's self-alignment fixture: 1686M, no gaps


def test_3pass_warp_kernel_scalar_fallback_and_wide_bands():
    # boxes whose band attempts fail up to (qn - 1) / 2 end in sw_scalar_align on the whole box (three_pass.rs:81-84):
    # a read made of two distant pieces of the target forces bands wider than any doubling reaches
    from test_3pass_gpu import check_3pass
    rng = np.random.default_rng(26)
    g = synth.random_dna(rng, 3000)
    chimera = np.concatenate([g[100:700], g[1900:2500]])           # 1200 nt, a 1200-column deletion in the middle
    shifted = np.concatenate([g[200:900], synth.random_dna(rng, 300), g[900:1500]])  # a 300-nt insertion
    reads = [chimera, shifted] + ont_reads(rng, g, 3, 1100, 1600)
    stats, _ = check_3pass([g], reads, WeightMatrix.new_dna_matrix(2, -5, b"N"), go=-3, ge=-1)
    assert stats["tp_band_attempts"] > stats["tp_banded"]


def test_sw_align_batch_takes_long_and_mixed_batches():
    # ADVICE r1: one long read must not fail the whole zoe_cuda_sw_align_batch call; zoe's sw_simd_align has no limit
    from test_align_gpu import check_align
    rng = np.random.default_rng(27)
    g = synth.random_dna(rng, 2200)
    long_reads = ont_reads(rng, g, 3, 1030, 1500)
    short_reads = ont_reads(rng, g, 6, 30, 400)
    check_align([g], long_reads, W25)                                   # all long
    check_align([g, g[300:900].copy()], [short_reads[0], long_reads[0], short_reads[1], short_reads[2], long_reads[1]], W25)
    check_align([g], [long_reads[2], short_reads[3]], W42, go=-3, ge=-1, profiled_is_query=True)
    s = golden("CY137594.txt")
    check_align([s], [s], W25)                                          # sw/test.rs:264-280, aligned on the GPU
