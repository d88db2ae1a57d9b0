// paired.cuh -- paired-end best-hit search (zoe_cuda_sw_*_paired_best_hit_batch, DESIGN.md 4.10): the pair-aware
// selection and the pair outputs around the best-hit machinery of best_hit.cuh.  The two mate batches are expanded
// (strands.cuh, ExpandPairs) into one quadrupled batch: sequence 4i + 2m + s is mate m of pair i on strand s, which is the
// doubled layout of the both-strand search for the 2n mates interleaved by pair.  The score pass, the buckets, the
// alignments and the CIGAR gather run on it unchanged; only the selection and the pair outputs are new.
#pragma once
#include <cstdint>

namespace zoe_cuda {

// Outputs of the selection: pair_hit per pair, the rest per mate at 2i + m (the per-read buffers of the best-hit search).
struct PairSelectParams {
    const uint32_t *score;  // score pass, 4 n_pairs x n_prof: row 4i + 2m + s is mate m of pair i on strand s
    const uint8_t *status, *tier;
    uint64_t n_pairs;
    uint32_t n_prof;
    uint32_t *pair_hit, *hit, *score_out, *runner_up;
    uint8_t *strand, *status_out, *tier_out;
};

// Candidate (j, o) puts mate 1 on strand o and mate 2 on strand 1 - o.  Its key, highest wins: the number of
// Overflowed mates, then the sum of the Some scores (33 bits), then the inverted candidate index c = 2 j + o so that
// ties go to the smallest j, then to o = 0.  66 bits: hi = (overflowed << 33) | sum, lo = ~c.
struct PairKey {
    uint64_t hi;
    uint32_t lo;
};

__device__ __forceinline__ bool pair_key_above(const PairKey &a, const PairKey &b) {
    return a.hi > b.hi || (a.hi == b.hi && a.lo > b.lo);
}

// One group of W lanes per pair (W = 1 while the 2 n_prof candidates fit a warp's width, 32 beyond); each lane takes
// every W-th candidate.  Pass 1 finds the winner; pass 2 each mate's runner-up, its largest Some score among candidates
// of another profiled sequence, on either strand.
template <int W>
__global__ void __launch_bounds__(256) pair_select_kernel(const PairSelectParams p) {
    const uint64_t groups = (uint64_t)gridDim.x * (blockDim.x / W);
    const uint32_t lane = threadIdx.x % W;
    const uint32_t P = p.n_prof, nc = 2 * P;
    for (uint64_t i = (uint64_t)blockIdx.x * (blockDim.x / W) + threadIdx.x / W; i < p.n_pairs; i += groups) {
        const uint64_t base = 4 * i * P;
        PairKey best{0, 0};
        for (uint32_t c = lane; c < nc; c += W) {
            const uint32_t j = c >> 1, o = c & 1;
            const uint64_t q1 = base + (uint64_t)o * P + j, q2 = base + (uint64_t)(3 - o) * P + j;
            const uint8_t s1 = p.status[q1], s2 = p.status[q2];
            const uint64_t ovf = (s1 == 1) + (s2 == 1);
            const uint64_t sum = (uint64_t)(s1 == 0 ? p.score[q1] : 0u) + (s2 == 0 ? p.score[q2] : 0u);
            const PairKey k{(ovf << 33) | sum, ~c};
            if (pair_key_above(k, best)) best = k;
        }
#pragma unroll
        for (int d = W / 2; d >= 1; d >>= 1) {
            const PairKey o{__shfl_xor_sync(0xffffffffu, best.hi, d, W), __shfl_xor_sync(0xffffffffu, best.lo, d, W)};
            if (pair_key_above(o, best)) best = o;
        }
        const uint32_t c = ~best.lo, hit = c >> 1, o = c & 1;
        uint32_t ru[2] = {0, 0};
        for (uint32_t k = lane; k < nc; k += W) {
            const uint32_t j = k >> 1, t = k & 1;
            if (j == hit) continue;
#pragma unroll
            for (int m = 0; m < 2; ++m) {
                const uint64_t r = base + (uint64_t)(2 * m + t) * P + j;
                if (p.status[r] == 0) ru[m] = max(ru[m], p.score[r]);
            }
        }
#pragma unroll
        for (int d = W / 2; d >= 1; d >>= 1) {
            ru[0] = max(ru[0], __shfl_xor_sync(0xffffffffu, ru[0], d, W));
            ru[1] = max(ru[1], __shfl_xor_sync(0xffffffffu, ru[1], d, W));
        }
        if (lane == 0) {
            p.pair_hit[i] = hit;
#pragma unroll
            for (int m = 0; m < 2; ++m) {
                const uint32_t s = m == 0 ? o : 1 - o;
                const uint64_t q = base + (uint64_t)(2 * m + s) * P + hit, r = 2 * i + m;
                const uint8_t st = p.status[q];
                p.hit[r] = hit;
                p.strand[r] = (uint8_t)s;
                p.score_out[r] = p.score[q];
                p.status_out[r] = st;
                p.tier_out[r] = p.tier[q];
                p.runner_up[r] = st == 0 ? ru[m] : 0;
            }
        }
    }
}

// Pair outputs from the per-mate outputs in mate order.  A mate's panel range is [ref_start, ref_end) when the
// profiled sequences are references, [query_start, query_end) when they are queries.
struct PairFinalizeParams {
    const uint8_t *status, *strand;
    const uint32_t *start, *end;  // the panel-range buffers
    uint64_t n_pairs;
    uint32_t min_insert, max_insert;
    uint8_t *proper;
    int32_t *tlen;
};

// tlen (mate 1's TLEN) is +extent when mate 1 starts first, or at the same start with mate 1 forward, else -extent;
// proper: the forward mate starts at or before the reverse one (the mates point inward) and the extent is within the
// insert bounds.  Both are 0 unless both mates are Some.  One thread per pair.
__global__ void __launch_bounds__(256) pair_finalize_kernel(const PairFinalizeParams p) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < p.n_pairs; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t a = 2 * i, b = a + 1;
        if (p.status[a] != 0 || p.status[b] != 0) {
            p.proper[i] = 0;
            p.tlen[i] = 0;
            continue;
        }
        const uint32_t s1 = p.start[a], s2 = p.start[b];
        const uint32_t extent = max(p.end[a], p.end[b]) - min(s1, s2);
        const bool o = p.strand[a] != 0;
        p.tlen[i] = (s1 < s2 || (s1 == s2 && !o)) ? (int32_t)extent : -(int32_t)extent;
        const uint32_t fwd = o ? s2 : s1, rev = o ? s1 : s2;
        p.proper[i] = fwd <= rev && extent >= p.min_insert && extent <= p.max_insert;
    }
}

}  // namespace zoe_cuda
