// strands.cuh -- both-strand search (zoe_cuda_sw_*_both_strands_batch): the strand expansion in front of the DP
// pipelines and the strand selection behind them (DESIGN.md 4.8).  The DP kernels never see a strand: they run on a
// doubled batch in which sequence 2i is streamed sequence i and sequence 2i+1 its reverse complement.
#pragma once
#include <cstdint>

namespace zoe_cuda {

// The complement table of the both-strand search (the Python copy is zoe_b200.alignment._COMPLEMENT): A<->T, C<->G,
// U->A, the IUPAC pairs R<->Y, K<->M, B<->V, D<->H; S, W, N and every other byte map to themselves; lowercase letters
// map the same way and keep their case.
__host__ __device__ constexpr uint8_t complement_base(uint8_t c) {
    const uint8_t lower = (c >= 'a' && c <= 'z') ? 0x20 : 0;
    switch (c & ~lower) {
        case 'A': return 'T' | lower;
        case 'T': return 'A' | lower;
        case 'U': return 'A' | lower;
        case 'C': return 'G' | lower;
        case 'G': return 'C' | lower;
        case 'R': return 'Y' | lower;
        case 'Y': return 'R' | lower;
        case 'K': return 'M' | lower;
        case 'M': return 'K' | lower;
        case 'B': return 'V' | lower;
        case 'V': return 'B' | lower;
        case 'D': return 'H' | lower;
        case 'H': return 'D' | lower;
        default: return c;
    }
}

// Source mappings of strand_expand_kernel.  at(i) gives expanded read i's bytes, its length and its position in the
// concatenation of all n reads; total(n) is that concatenation's length.
// One staged shard: read i is sequence i.
struct ExpandSingle {
    const uint8_t *seq;
    const uint64_t *off;  // n + 1 entries
    __device__ __forceinline__ const uint8_t *at(uint64_t i, uint64_t *pos, uint64_t *len) const {
        *pos = off[i];
        *len = off[i + 1] - *pos;
        return seq + *pos;
    }
    __device__ __forceinline__ uint64_t total(uint64_t n) const { return off[n]; }
};

// A staged shard of read pairs (paired.cuh): the mate-1 sequences, then the mate-2 sequences at seq + off1[n_pairs].
// Read 2i + m is mate m of pair i, so the reads are the mates interleaved by pair.
struct ExpandPairs {
    const uint8_t *seq;
    const uint64_t *off1, *off2;  // n_pairs + 1 entries each, each relative to its own mates' first byte
    uint64_t n_pairs;
    __device__ __forceinline__ const uint8_t *at(uint64_t i, uint64_t *pos, uint64_t *len) const {
        const uint64_t p = i >> 1, a1 = off1[p], l1 = off1[p + 1] - a1, a2 = off2[p];
        *pos = a1 + a2 + ((i & 1) ? l1 : 0);
        *len = (i & 1) ? off2[p + 1] - a2 : l1;
        return (i & 1) ? seq + off1[n_pairs] + a2 : seq + a1;
    }
    __device__ __forceinline__ uint64_t total(uint64_t) const { return off1[n_pairs] + off2[n_pairs]; }
};

// Doubles n reads of a staged shard: out sequence 2i is read i, 2i+1 its reverse complement, at offsets 2 pos_i and
// 2 pos_i + len_i (off2 gets 2n + 1 entries).  One warp per read; memory-bound.
template <class Src>
__global__ void __launch_bounds__(256) strand_expand_kernel(const Src src, uint64_t n, uint8_t *__restrict__ seq2,
                                                            uint64_t *__restrict__ off2) {
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    const uint32_t lane = threadIdx.x & 31;
    for (uint64_t i = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += warps) {
        uint64_t a, len;
        const uint8_t *s = src.at(i, &a, &len);
        uint8_t *fwd = seq2 + 2 * a, *rev = fwd + len;
        for (uint64_t k = lane; k < len; k += 32) {
            fwd[k] = s[k];
            rev[k] = complement_base(s[len - 1 - k]);
        }
        if (lane == 0) {
            off2[2 * i] = 2 * a;
            off2[2 * i + 1] = 2 * a + len;
            if (i + 1 == n) off2[2 * n] = 2 * src.total(n);
        }
    }
}

// Per-pair outputs of a doubled run gathered for the selected strand.  in32[0] is the score and in8[0] the status:
// they decide the strand.  cig_off (may be null): the doubled run's CIGAR offsets; the selected CIGAR lengths go to
// cig_count.
struct StrandSelectParams {
    const uint32_t *in32[5];
    uint32_t *out32[5];
    const uint8_t *in8[3];
    uint8_t *out8[3];
    int n32, n8;
    const uint64_t *cig_off;
    uint32_t *cig_count;
    uint8_t *strand;
    uint64_t n_out;  // pairs of the real shard
    uint32_t n_prof;
};

// Rank of a result: Overflowed > Some(score), ordered by score, > Unmapped.
__device__ __forceinline__ uint64_t strand_rank(uint8_t status, uint32_t score) {
    return status == 1 ? ~0ull : status == 0 ? (uint64_t)score + 1 : 0ull;
}

// Output pair (i, j) takes the reverse strand (doubled pair (2i+1, j)) only when it ranks strictly above the forward
// one (2i, j): every tie goes to the forward strand.
__global__ void strand_select_kernel(const StrandSelectParams p) {
    const uint64_t o = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= p.n_out) return;
    const uint64_t i = o / p.n_prof, j = o - i * p.n_prof;
    const uint64_t f = 2 * i * p.n_prof + j, r = f + p.n_prof;
    const bool rev = strand_rank(p.in8[0][r], p.in32[0][r]) > strand_rank(p.in8[0][f], p.in32[0][f]);
    const uint64_t s = rev ? r : f;
#pragma unroll
    for (int k = 0; k < 5; ++k)
        if (k < p.n32) p.out32[k][o] = p.in32[k][s];
#pragma unroll
    for (int k = 0; k < 3; ++k)
        if (k < p.n8) p.out8[k][o] = p.in8[k][s];
    if (p.cig_off) p.cig_count[o] = (uint32_t)(p.cig_off[s + 1] - p.cig_off[s]);
    if (p.strand) p.strand[o] = rev ? 1 : 0;
}

// Copies the selected strand's CIGAR words of every output pair to their compacted offsets.  One warp per pair.
__global__ void __launch_bounds__(256) strand_cigar_gather_kernel(const uint32_t *__restrict__ cig_in,
                                                                  const uint64_t *__restrict__ off_in,
                                                                  const uint8_t *__restrict__ strand, uint64_t n_out,
                                                                  uint32_t n_prof, const uint64_t *__restrict__ off_out,
                                                                  uint32_t *__restrict__ cig_out) {
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    const uint32_t lane = threadIdx.x & 31;
    for (uint64_t o = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); o < n_out; o += warps) {
        const uint64_t i = o / n_prof, j = o - i * n_prof;
        const uint64_t s = (2 * i + strand[o]) * n_prof + j;
        const uint64_t a = off_in[s], len = off_in[s + 1] - a, b = off_out[o];
        for (uint64_t k = lane; k < len; k += 32) cig_out[b + k] = cig_in[a + k];
    }
}

}  // namespace zoe_cuda
