// best_hit.cuh -- best-hit search (zoe_cuda_sw_*_best_hit_batch, DESIGN.md 4.9): the selection, bucketing, gather and
// scatter around the unchanged score and align pipelines.  The score pass covers every candidate (read i or its reverse
// complement, against every profiled sequence j); best_hit_select_kernel picks each read's winner; the align entry point
// then buckets the Some winners by (hit, length class), gathers each bucket into a compact batch, aligns it against the
// one profiled sequence `hit` and scatters the results back to read order.
#pragma once
#include <cstdint>

#include "strands.cuh"

namespace zoe_cuda {

// Per-read outputs of the selection.
struct BestHitSelectParams {
    const uint32_t *score;  // score pass, (S * n) x n_prof: row S i + s is read i on strand s
    const uint8_t *status, *tier;
    uint64_t n;             // reads of the shard
    uint32_t n_prof;
    uint32_t n_strands;     // 1, or 2 (both strands: the doubled batch of strands.cuh)
    uint32_t *hit, *score_out, *runner_up;
    uint8_t *strand, *status_out, *tier_out;
};

// Candidate key: the both-strand rank (strands.cuh) above the candidate index c = j * n_strands + s, inverted so that the
// largest key is the highest rank with the smallest j, then the forward strand.  The rank takes 33 bits.
__device__ __forceinline__ uint64_t best_hit_key(uint8_t status, uint32_t score, uint32_t c) {
    const uint64_t rank = status == 1 ? 0x1ffffffffull : strand_rank(status, score);
    return (rank << 31) | (uint64_t)(0x7fffffffu - c);
}

// One group of W lanes per read (W = 1 for small panels, 32 for large ones); each lane takes every W-th candidate.
// Pass 1 finds the winner; pass 2 the runner-up, the largest Some score among candidates of another profiled sequence.
template <int W>
__global__ void __launch_bounds__(256) best_hit_select_kernel(const BestHitSelectParams p) {
    const uint64_t groups = (uint64_t)gridDim.x * (blockDim.x / W);
    const uint32_t lane = threadIdx.x % W;
    const uint32_t nc = p.n_prof * p.n_strands;
    for (uint64_t i = (uint64_t)blockIdx.x * (blockDim.x / W) + threadIdx.x / W; i < p.n; i += groups) {
        const uint64_t base = i * p.n_strands * p.n_prof;
        uint64_t best = 0;
        for (uint32_t c = lane; c < nc; c += W) {
            const uint32_t j = c / p.n_strands, s = c - j * p.n_strands;
            const uint64_t q = base + (uint64_t)s * p.n_prof + j;
            best = max(best, best_hit_key(p.status[q], p.score[q], c));
        }
#pragma unroll
        for (int d = W / 2; d >= 1; d >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, d, W));
        const uint32_t c = 0x7fffffffu - (uint32_t)(best & 0x7fffffffu);
        const uint32_t hit = c / p.n_strands, s = c - hit * p.n_strands;
        const uint64_t q = base + (uint64_t)s * p.n_prof + hit;
        const uint8_t st = p.status[q];
        uint32_t ru = 0;
        if (st == 0)
            for (uint32_t k = lane; k < nc; k += W) {
                const uint32_t j = k / p.n_strands, t = k - j * p.n_strands;
                const uint64_t r = base + (uint64_t)t * p.n_prof + j;
                if (j != hit && p.status[r] == 0) ru = max(ru, p.score[r]);
            }
#pragma unroll
        for (int d = W / 2; d >= 1; d >>= 1) ru = max(ru, __shfl_xor_sync(0xffffffffu, ru, d, W));
        if (lane == 0) {
            p.hit[i] = hit;
            p.strand[i] = (uint8_t)s;
            p.score_out[i] = p.score[q];
            p.status_out[i] = st;
            p.tier_out[i] = p.tier[q];
            p.runner_up[i] = ru;
        }
    }
}

// Bucket table of one device, n_keys keys, 64-bit words: [count | longest | shortest | residues | start | cursor] x n_keys.
// The first five blocks are what the host reads back.
enum BestHitTab { kBhCount = 0, kBhMax = 1, kBhMin = 2, kBhSum = 3, kBhStart = 4, kBhCursor = 5, kBhTabRows = 6 };

// Key of each Some winner (hit, or 2 hit + long when the long / short split applies; ~0 = not aligned) and the bucket
// counts, lengths and residues.  With smem, a block first accumulates in shared memory (n_keys * 32 bytes).
__global__ void __launch_bounds__(256) best_hit_bucket_count_kernel(const uint32_t *__restrict__ hit,
                                                                    const uint8_t *__restrict__ status,
                                                                    const uint64_t *__restrict__ off, uint32_t n_strands,
                                                                    uint64_t n, bool split_long, uint32_t n_keys,
                                                                    bool smem, uint32_t *__restrict__ key,
                                                                    unsigned long long *__restrict__ tab) {
    extern __shared__ unsigned long long s_tab[];
    unsigned long long *t = smem ? s_tab : tab;
    if (smem) {
        for (uint32_t k = threadIdx.x; k < n_keys; k += blockDim.x) {
            s_tab[kBhCount * n_keys + k] = 0;
            s_tab[kBhMax * n_keys + k] = 0;
            s_tab[kBhMin * n_keys + k] = ~0ull;
            s_tab[kBhSum * n_keys + k] = 0;
        }
        __syncthreads();
    }
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        if (status[i] != 0) {
            key[i] = ~0u;
            continue;
        }
        const uint64_t len = off[n_strands * i + 1] - off[n_strands * i];
        const uint32_t k = split_long ? 2 * hit[i] + (len > 1024 ? 1 : 0) : hit[i];
        key[i] = k;
        atomicAdd(&t[kBhCount * n_keys + k], 1ull);
        atomicMax(&t[kBhMax * n_keys + k], (unsigned long long)len);
        atomicMin(&t[kBhMin * n_keys + k], (unsigned long long)len);
        atomicAdd(&t[kBhSum * n_keys + k], (unsigned long long)len);
    }
    if (smem) {
        __syncthreads();
        for (uint32_t k = threadIdx.x; k < n_keys; k += blockDim.x) {
            if (s_tab[kBhCount * n_keys + k] == 0) continue;
            atomicAdd(&tab[kBhCount * n_keys + k], s_tab[kBhCount * n_keys + k]);
            atomicMax(&tab[kBhMax * n_keys + k], s_tab[kBhMax * n_keys + k]);
            atomicMin(&tab[kBhMin * n_keys + k], s_tab[kBhMin * n_keys + k]);
            atomicAdd(&tab[kBhSum * n_keys + k], s_tab[kBhSum * n_keys + k]);
        }
    }
}

// Exclusive scan of the bucket counts into the bucket starts (one warp).
__global__ void best_hit_bucket_scan_kernel(unsigned long long *tab, uint32_t n_keys) {
    const uint32_t lane = threadIdx.x & 31;
    unsigned long long carry = 0;
    for (uint32_t b = 0; b < n_keys; b += 32) {
        const unsigned long long v = b + lane < n_keys ? tab[kBhCount * n_keys + b + lane] : 0ull;
        unsigned long long incl = v;
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long o = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= (uint32_t)d) incl += o;
        }
        if (b + lane < n_keys) tab[kBhStart * n_keys + b + lane] = carry + incl - v;
        carry += __shfl_sync(0xffffffffu, incl, 31);
    }
}

// Index lists: read i goes to list[start[key] + rank]; the lanes of a warp that share a key take one atomic.
__global__ void __launch_bounds__(256) best_hit_bucket_scatter_kernel(const uint32_t *__restrict__ key, uint64_t n,
                                                                      uint32_t n_keys, unsigned long long *__restrict__ tab,
                                                                      uint32_t *__restrict__ list) {
    const uint32_t lane = threadIdx.x & 31;
    for (uint64_t b = (uint64_t)blockIdx.x * blockDim.x; b < n; b += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t i = b + threadIdx.x;
        const uint32_t k = i < n ? key[i] : ~0u;
        const uint32_t peers = __match_any_sync(0xffffffffu, k);
        if (k == ~0u) continue;
        const uint32_t leader = __ffs(peers) - 1;
        unsigned long long pos = 0;
        if (lane == leader) pos = atomicAdd(&tab[kBhCursor * n_keys + k], (unsigned long long)__popc(peers));
        pos = __shfl_sync(peers, pos, leader);
        list[tab[kBhStart * n_keys + k] + pos + __popc(peers & ((1u << lane) - 1))] = (uint32_t)i;
    }
}

// Length of each listed read, in list order (the compact batches' offsets are one scan of these).
__global__ void best_hit_list_len_kernel(const uint32_t *__restrict__ list, uint64_t m, const uint64_t *__restrict__ off,
                                         uint32_t n_strands, uint32_t *__restrict__ len) {
    const uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= m) return;
    const uint64_t i = list[p];
    len[p] = (uint32_t)(off[n_strands * i + 1] - off[n_strands * i]);
}

// Copies a bucket's reads (list[0, count)) into a compact batch: sequence t is read list[t] on its winning strand
// (sequence n_strands i + strand of the staged batch), at offset loff[t] - loff[0].  One warp per read.
__global__ void __launch_bounds__(256) best_hit_gather_kernel(const uint8_t *__restrict__ seq, const uint64_t *__restrict__ off,
                                                              uint32_t n_strands, const uint8_t *__restrict__ strand,
                                                              const uint32_t *__restrict__ list, const uint64_t *__restrict__ loff,
                                                              uint64_t count, uint8_t *__restrict__ out_seq,
                                                              uint64_t *__restrict__ out_off) {
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t b0 = loff[0];
    for (uint64_t t = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < count; t += warps) {
        const uint64_t i = list[t], src = n_strands * i + (n_strands > 1 ? strand[i] : 0);
        const uint64_t a = off[src], len = off[src + 1] - a, b = loff[t] - b0;
        for (uint64_t k = lane; k < len; k += 32) out_seq[b + k] = seq[a + k];
        if (lane == 0) {
            out_off[t] = b;
            if (t + 1 == count) out_off[count] = loff[count] - b0;
        }
    }
}

// A bucket's alignment outputs, back to read order.  in32 / out32: score, ref_start, ref_end, query_start, query_end;
// in8 / out8: status, tier, hazard (in8[2] null: the 3-pass pipeline, hazard 0).  The read's CIGAR words move from the
// bucket's cig_out to acc at acc_base + cig_off[t] (when `copy`: the words fit the accumulation buffer); cig_count and
// cig_src record where they are.  One warp per read.
struct BestHitScatterParams {
    const uint32_t *in32[5];
    uint32_t *out32[5];
    const uint8_t *in8[3];
    uint8_t *out8[3];
    const uint32_t *list;
    uint64_t count;
    const uint64_t *cig_off;
    const uint32_t *cig_out;
    uint32_t *cig_count;
    uint64_t *cig_src;
    uint32_t *acc;
    uint64_t acc_base;
    bool copy;
};

__global__ void __launch_bounds__(256) best_hit_scatter_kernel(const BestHitScatterParams p) {
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    const uint32_t lane = threadIdx.x & 31;
    for (uint64_t t = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < p.count; t += warps) {
        const uint64_t i = p.list[t], a = p.cig_off[t], len = p.cig_off[t + 1] - a;
        if (lane < 5) p.out32[lane][i] = p.in32[lane][t];
        if (lane >= 8 && lane < 11) p.out8[lane - 8][i] = p.in8[lane - 8] ? p.in8[lane - 8][t] : 0;
        if (lane == 16) {
            p.cig_count[i] = (uint32_t)len;
            p.cig_src[i] = p.acc_base + a;
        }
        if (p.copy)
            for (uint64_t k = lane; k < len; k += 32) p.acc[p.acc_base + a + k] = p.cig_out[a + k];
    }
}

// The final CIGAR stream in read order: read i's words from acc[src[i], +count[i]) to out[off[i], ...).  One warp per read.
__global__ void __launch_bounds__(256) best_hit_cigar_gather_kernel(const uint32_t *__restrict__ acc,
                                                                    const uint64_t *__restrict__ src,
                                                                    const uint32_t *__restrict__ count, uint64_t n,
                                                                    const uint64_t *__restrict__ off,
                                                                    uint32_t *__restrict__ out) {
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    const uint32_t lane = threadIdx.x & 31;
    for (uint64_t i = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += warps) {
        const uint64_t a = src[i], len = count[i], b = off[i];
        for (uint64_t k = lane; k < len; k += 32) out[b + k] = acc[a + k];
    }
}

}  // namespace zoe_cuda
