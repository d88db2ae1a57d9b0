// sw_3pass.cuh -- third pass of zoe's 3-pass local alignment (src/alignment/sw/three_pass.rs:21-104): given the
// score and the bounding box from the ranges pipeline (sw_ranges.cuh = sw_simd_score_ranges, striped.rs:355-388),
// produce the CIGAR without a full traceback matrix:
//   * no-gaps shortcut (three_pass.rs:39-59): equal range lengths and the diagonal's weights add up to the score;
//   * otherwise sw_banded_align (src/alignment/sw/banded.rs:40-133) on the box with band width |dr - dq| + 1,
//     doubled until the banded score equals the pass-1 score (three_pass.rs:66-79);
//   * otherwise sw_scalar_align on the box (three_pass.rs:81-84, src/alignment/sw/scalar.rs:173-271).
// One thread owns one pair and runs zoe's loops literally, so tie-breaks, flag bytes and the walk are zoe's by
// construction.  Scratch is BAND sized, not box sized: the band attempts run in rounds (every unresolved pair tries its
// current width; a pair whose banded score falls short re-enters the next round with twice the width and a scratch slice
// sized for it), so a 5 kb x 5 kb box of a long read costs rows x (2 bw + 1) flag bytes and a ring of 2 bw + 2 (H, E)
// entries -- about 1 MB -- instead of 25 MB.  Short reads (config 3) finish in round 0 with the ring in shared memory.
#pragma once
#include "sw_align.cuh"

namespace zoe_cuda {

constexpr uint32_t kTpNoDp = 0xffffffffu;    // pair emits no CIGAR (not Some)
constexpr uint32_t kTpNoGaps = 0xfffffffeu;  // pair took the no-gaps shortcut: its CIGAR follows from the ranges

struct ThreePassParams {
    const uint8_t *rseq;        // streamed batch, raw bytes
    const uint64_t *roff;
    const uint8_t *pbytes;      // profiled sequences, raw bytes
    const uint32_t *coff;
    uint32_t n_cseq;
    const int8_t *weights;      // S*S, zoe's weights[ref_idx][query_idx]
    int S;
    const uint8_t *lut;
    int go, ge;                 // zoe's signed gap weights (<= 0)
    int invert;                 // 1: SeqSrc::Query(streamed) -> Alignment::invert (output.rs:396-425)
    uint64_t pair_first;        // chunk = global pair ids [pair_first, pair_first + n_pairs)
    uint32_t n_pairs;
    uint32_t *score;            // per pair, from the ranges pipeline (final orientation)
    uint8_t *status;
    uint32_t *ref_start, *ref_end, *query_start, *query_end;
    uint32_t *cig_count;
    uint32_t *dp_pair;          // [n_pairs] slot -> global pair id
    unsigned long long *dp_off; // [n_pairs] slot -> byte offset of the pair's scratch of the CURRENT round inside `blob`
    unsigned long long *dp_off_next;  // ... of the NEXT round (a failing attempt plans its retry; both kernels of a round
    uint32_t *dp_bw_next;             // read the current arrays only, so neither sees the other's retries)
    unsigned long long *dp_cig_off;  // [n_pairs] slot -> byte offset of the pair's back-filled CIGAR inside `cig_blob`
    uint32_t *dp_cap;           // [n_pairs] slot -> CIGAR scratch capacity (words)
    uint32_t *dp_bw;            // [n_pairs] slot -> band width of the current round (0 = sw_scalar_align on the whole box)
    uint32_t *dp_slot;          // [n_pairs] chunk-local pair -> slot, kTpNoDp or kTpNoGaps
    uint8_t *blob;              // per round: [ring / row of (H, E)][flag bytes of the band / the box]
    uint8_t *cig_blob;          // per chunk: back-filled CIGARs of the DP pairs
    const uint32_t *list;       // slots of this round
    uint32_t *next_list;        // slots that re-enter the next round
    uint32_t warp_wcap;         // row cells + 2 tp_band_warp_kernel can hold this round (0: it is not launched)
    unsigned long long *ctr;    // per classification: [0] DP pairs, [1] scratch bytes of round 0, [2] CIGAR bytes,
                                // [5] no-gaps pairs; per round: [3] pairs of the next round, [4] their scratch bytes;
                                // per call: [6] banded, [7] scalar fallbacks, [8] banded attempts, [9] running CIGAR base,
                                // [10] walks outside the band storage (zoe would panic), [11] CIGAR scratch overflows,
                                // [12] widest row (cells) among the LARGE pairs of the round being planned
};

__host__ __device__ inline unsigned long long tp_align16(unsigned long long x) { return (x + 15ull) & ~15ull; }
__host__ __device__ inline uint32_t tp_cig_cap(uint32_t rn, uint32_t qn) { return 2u * (rn < qn ? rn : qn) + 8u; }
constexpr uint32_t kTpRing = 32, kTpThreads = 64;
// (H, E) entries a banded attempt keeps: a power-of-two ring covering the band (in shared memory up to kTpRing)
__host__ __device__ inline uint32_t tp_ring_size(uint32_t bw) {
    uint32_t r = kTpRing;
    while (r < 2 * bw + 2) r *= 2;
    return r;
}
// scratch of one attempt: bw > 0: ring + band flags (rows x (2 bw + 1)); bw == 0: full (H, E) row + box flags
__host__ __device__ inline unsigned long long tp_need(uint32_t bw, uint32_t rn, uint32_t qn) {
    if (bw == 0) return tp_align16(8ull * qn) + tp_align16((unsigned long long)rn * qn);
    return tp_align16(8ull * tp_ring_size(bw)) + tp_align16((unsigned long long)rn * (2ull * bw + 1));
}
// Which pairs does the warp kernel take?  Wide bands (their (H, E) ring would live in global memory: one thread walking
// 5 000 rows x 257 cells through L2 took 2.8 s of config 4's 3.4 s) and large scalar boxes.
__host__ __device__ inline bool tp_is_large(uint32_t bw, uint32_t rn, uint32_t qn) {
    return bw != 0 ? tp_ring_size(bw) > kTpRing : (unsigned long long)rn * qn > 65536ull;
}
// cells of one row the recurrence visits: banded 2 bw + 1 (plus the entering column's slot), scalar qn
__host__ __device__ inline uint32_t tp_row_cells(uint32_t bw, uint32_t qn) { return bw != 0 ? 2 * bw + 2 : qn; }


struct TpBox {
    uint32_t seq, cj;
    uint32_t n, m;            // streamed / profiled lengths
    uint32_t rs, re, qs, qe;  // un-inverted: rows (streamed) [rs,re), columns (profiled) [qs,qe)
};

__device__ inline TpBox tp_box(const ThreePassParams &t, uint64_t gid) {
    TpBox b;
    b.seq = (uint32_t)(gid / t.n_cseq);
    b.cj = (uint32_t)(gid % t.n_cseq);
    b.n = (uint32_t)(t.roff[b.seq + 1] - t.roff[b.seq]);
    b.m = t.coff[b.cj + 1] - t.coff[b.cj];
    if (t.invert) {  // ranges_finalize_kernel swapped them
        b.rs = t.query_start[gid];
        b.re = t.query_end[gid];
        b.qs = t.ref_start[gid];
        b.qe = t.ref_end[gid];
    } else {
        b.rs = t.ref_start[gid];
        b.re = t.ref_end[gid];
        b.qs = t.query_start[gid];
        b.qe = t.query_end[gid];
    }
    return b;
}

// Pass 3a: the no-gaps shortcut, and scratch allocation for the pairs that need a DP.
__global__ void __launch_bounds__(256) tp_classify_kernel(const ThreePassParams t) {
    __shared__ uint8_t s_lut[256];
    __shared__ int8_t s_w[32 * 32];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_lut[i] = t.lut[i];
    for (int i = threadIdx.x; i < t.S * t.S; i += blockDim.x) s_w[i] = t.weights[i];
    __syncthreads();
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= t.n_pairs) return;
    const uint64_t gid = t.pair_first + k;
    t.cig_count[gid] = 0;
    t.dp_slot[k] = kTpNoDp;
    if (t.status[gid] != 0) return;
    const TpBox b = tp_box(t, gid);
    if (b.qe <= b.qs) {  // query_range.is_empty() -> Unmapped (three_pass.rs:37-38)
        t.status[gid] = 2;
        t.score[gid] = 0;
        t.ref_start[gid] = t.ref_end[gid] = t.query_start[gid] = t.query_end[gid] = 0;
        return;
    }
    const uint32_t qn = b.qe - b.qs, rn = b.re - b.rs;
    if (qn == rn) {
        const uint8_t *R = t.rseq + t.roff[b.seq] + b.rs;
        const uint8_t *P = t.pbytes + t.coff[b.cj] + b.qs;
        long long sum = 0;
        for (uint32_t i = 0; i < qn; ++i) sum += s_w[(int)s_lut[R[i]] * t.S + s_lut[P[i]]];
        if (sum >= 0 && (unsigned long long)sum == (unsigned long long)t.score[gid]) {
            // AlignmentStates::new_no_gaps (state.rs:201-208); inverted: S(ref_start) M S(ref_len - ref_end)
            const uint32_t lead = t.invert ? b.rs : b.qs, trail = t.invert ? (b.n - b.re) : (b.m - b.qe);
            t.cig_count[gid] = 1u + (lead ? 1u : 0u) + (trail ? 1u : 0u);
            t.dp_slot[k] = kTpNoGaps;
            atomicAdd(&t.ctr[5], 1ULL);
            return;
        }
    }
    // a DP pair: a back-filled CIGAR row for the whole call, and the scratch of its first attempt (three_pass.rs:66-70:
    // band width |rn - qn| + 1 if that is a real band, else the scalar alignment of the whole box)
    const uint32_t cap = tp_cig_cap(rn, qn);
    uint32_t bw = (rn > qn ? rn - qn : qn - rn) + 1;
    if (bw > (qn - 1) / 2) bw = 0;
    const uint32_t slot = (uint32_t)atomicAdd(&t.ctr[0], 1ULL);
    t.dp_pair[slot] = (uint32_t)(gid - t.pair_first);
    t.dp_cap[slot] = cap;
    t.dp_bw[slot] = bw;
    t.dp_cig_off[slot] = atomicAdd(&t.ctr[2], tp_align16(4ull * cap));
    t.dp_off[slot] = atomicAdd(&t.ctr[1], tp_need(bw, rn, qn));
    t.next_list[slot] = slot;  // round 0 visits every DP pair
    if (tp_is_large(bw, rn, qn)) atomicMax(&t.ctr[12], (unsigned long long)tp_row_cells(bw, qn));
    t.dp_slot[k] = slot;
}

// zoe's scalar / banded recurrence over the box, flags into `fl`.  BANDED: src/alignment/sw/banded.rs:55-125 (rows keep
// the columns [r - bw, r + bw], flag row stride 2 bw + 1); otherwise src/alignment/sw/scalar.rs:190-262.
// Returns the best score; (r_end, c_end) = its first occurrence in row-major order; rows_done = rows the loop visited.
// h_row / e_row: BANDED keeps them in a ring, he[(c & ring_mask) * he_stride] -- a row only touches the columns of its
// band, the band moves right by one column per row, and a column that left the band is never read again, so the ring
// holds everything zoe's full-length vectors would be asked for; the column entering the band is (re)initialised to zoe's
// initial (0, gap_open) first.  Bands up to 15 use a ring in shared memory (stride = threads of the CTA: 4.4 -> 1 ms on
// config 3), wider ones a ring in the pair's scratch.  The scalar recurrence keeps the full row (ring_mask = ~0).
template <bool BANDED>
__device__ inline int32_t tp_fill(const uint8_t *R, uint32_t rn, const uint8_t *P, uint32_t qn, const uint8_t *s_lut,
                                  const int8_t *s_w, int S, int32_t go, int32_t ge, uint32_t bw, int2 *he, uint32_t ring_mask,
                                  uint32_t he_stride, uint8_t *fl, uint32_t *r_end, uint32_t *c_end, uint32_t *rows_done) {
    auto HE = [&](uint32_t c) -> int2 & { return he[(size_t)(c & ring_mask) * he_stride]; };
    if (BANDED) {
        for (uint32_t c = 0; c < min(bw, qn); ++c) HE(c) = make_int2(0, go);  // row 0's band except its entering column
    } else {
        for (uint32_t c = 0; c < qn; ++c) HE(c) = make_int2(0, go);  // h_row = 0, e_row = gap_open
    }
    int32_t best = 0, h_store = 0;
    uint32_t br = 0, bc = 0, r = 0;
    const uint32_t bfw = 2 * bw + 1;
    for (; r < rn; ++r) {
        const int8_t *wrow = s_w + (int)s_lut[R[r]] * S;
        int32_t f = go;
        int32_t h = BANDED ? h_store : 0;
        const uint32_t start_col = BANDED ? (r > bw ? r - bw : 0u) : 0u;
        const uint32_t end_col = BANDED ? min(r + bw + 1, qn) : qn;
        if (BANDED && r + bw < qn) HE(r + bw) = make_int2(0, go);  // the column entering the band
        if (BANDED) {
            if (start_col >= end_col) break;
            if (start_col + bw == r) h_store = max(max(h + (int32_t)wrow[s_lut[P[start_col]]], HE(start_col).y), 0);
        }
        uint8_t *frow = fl + (size_t)r * (BANDED ? bfw : qn) - (BANDED ? start_col : 0u);
        for (uint32_t c = start_col; c < end_col; ++c) {
            const int2 prev = HE(c);  // (H[r-1][c], E[r][c])
            int32_t e = prev.y;
            h += (int32_t)wrow[s_lut[P[c]]];
            h = max(max(h, e), max(f, 0));
            if (h > best) {
                best = h;
                br = r;
                bc = c;
            }
            uint32_t flag = (e == h ? 1u : 0u) | (f == h ? 4u : 0u);
            if (h == 0) flag = 16u;
            const int32_t ho = h + go;
            e = max(e + ge, ho);
            f = max(f + ge, ho);
            if (ho != go) flag |= (e > ho ? 2u : 0u) | (f > ho ? 8u : 0u);
            frow[c] = (uint8_t)flag;
            HE(c) = make_int2(h, e);
            h = prev.x;
        }
    }
    *r_end = br;
    *c_end = bc;
    *rows_done = r;
    return best;
}

// BackTrackable::to_alignment (backtrack.rs:290-342) over the row-major matrix (:408-411) or the band storage
// (BandedBacktrackMatrix::move_to, :628-633: cursor = r * (2 bw + 1) + c - r.saturating_sub(bw)), then zoe's soft-clip
// arithmetic (three_pass.rs:89-105) and, for SeqSrc::Query(streamed), Alignment::invert.  One thread.
__device__ inline void tp_walk_and_emit(const ThreePassParams &t, const TpBox &b, uint64_t gid, bool banded, uint32_t bw,
                                        uint32_t rows_done, uint32_t r_end, uint32_t c_end, const uint8_t *fl, uint32_t *cig,
                                        uint32_t cap) {
    const uint32_t qn = b.qe - b.qs, rn = b.re - b.rs;
    const long long bfw = 2ll * bw + 1, band_len = (long long)rn * bfw;
    bool oob = false;
    auto cell = [&](uint32_t r, uint32_t c) -> uint32_t {
        if (!banded) return fl[(size_t)r * qn + c];
        const long long skipped = r > bw ? (long long)(r - bw) : 0;
        const long long idx = (long long)r * bfw + ((long long)c - skipped);
        if ((long long)c < skipped || idx < 0 || idx >= band_len) {
            oob = true;
            return 16u;
        }
        // cells the fill loop never visited are zero in zoe's vec![0u8; ..]
        const uint32_t rr = (uint32_t)(idx / bfw), bc = (uint32_t)(idx % bfw);
        const uint32_t sc = rr > bw ? rr - bw : 0u, ec = min(rr + bw + 1, qn);
        if (rr >= rows_done || sc >= ec || bc >= ec - sc) return 0u;
        return fl[idx];
    };

    CigarBack cg;
    cg.init(cig, cap);
    const uint32_t OP_UP = t.invert ? 1u /*I*/ : 2u /*D*/, OP_LEFT = t.invert ? 2u : 1u;
    uint32_t r = r_end + 1, c = c_end + 1;
    const uint32_t r_end1 = r, c_end1 = c;
    // un-inverted: three_pass.rs:96 soft_clip(query.len() - adjusted_query_range.end) after to_alignment's own
    // soft clip of the sub-query's tail (backtrack.rs:305); inverted: invert() drops every S and clips by the
    // (adjusted) reference range of the un-inverted alignment = the streamed rows (output.rs:399-416)
    if (t.invert) {
        cg.push(4u, b.n - (r_end1 + b.rs));
    } else {
        cg.push(4u, b.m - (c_end1 + b.qs));
        cg.push(4u, qn - c_end1);
    }
    uint32_t cur = cell(r_end, c_end);
    int op = 0;  // 0 none, 1 D(up), 2 I(left), 3 M
    while (!(cur & 16u) && r > 0 && c > 0) {
        if (op == 1 && (cur & 2u)) {
            r -= 1;
        } else if (op == 2 && (cur & 8u)) {
            c -= 1;
        } else if (cur & 1u) {
            op = 1;
            r -= 1;
        } else if (cur & 4u) {
            op = 2;
            c -= 1;
        } else {
            op = 3;
            r -= 1;
            c -= 1;
        }
        cg.push(op == 1 ? OP_UP : (op == 2 ? OP_LEFT : 0u), 1);
        cur = cell(r > 0 ? r - 1 : 0, c > 0 ? c - 1 : 0);
    }
    if (t.invert) {
        cg.push(4u, r + b.rs);
    } else {
        cg.push(4u, c);          // to_alignment's 5' soft clip of the sub-query
        cg.push(4u, c + b.qs);   // three_pass.rs:95 prepend_soft_clip(adjusted_query_range.start)
    }
    cg.flush();
    if (cg.overflow) atomicAdd(&t.ctr[11], 1ULL);
    if (oob) atomicAdd(&t.ctr[10], 1ULL);
    t.cig_count[gid] = cg.n;
    // three_pass.rs:89-105: ranges of the sub-alignment shifted into the full sequences
    const uint32_t ar0 = r + b.rs, ar1 = r_end1 + b.rs, aq0 = c + b.qs, aq1 = c_end1 + b.qs;
    t.ref_start[gid] = t.invert ? aq0 : ar0;
    t.ref_end[gid] = t.invert ? aq1 : ar1;
    t.query_start[gid] = t.invert ? ar0 : aq0;
    t.query_end[gid] = t.invert ? ar1 : aq1;
}

// Pass 3b, one round: one thread per listed pair tries its current band width (or, width 0, the scalar alignment of the
// whole box).  A banded score short of the pass-1 score sends the pair to the next round with twice the width
// (three_pass.rs:71-79) or, beyond (qn - 1) / 2, with the scalar alignment (:81-84).
__global__ void __launch_bounds__(kTpThreads) tp_dp_kernel(const ThreePassParams t, uint32_t n_dp) {
    __shared__ uint8_t s_lut[256];
    __shared__ int8_t s_w[32 * 32];
    __shared__ int2 s_ring[kTpRing * kTpThreads];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_lut[i] = t.lut[i];
    for (int i = threadIdx.x; i < t.S * t.S; i += blockDim.x) s_w[i] = t.weights[i];
    __syncthreads();
    const uint32_t li = blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= n_dp) return;
    const uint32_t slot = t.list[li];
    const uint64_t gid = t.pair_first + t.dp_pair[slot];
    const TpBox b = tp_box(t, gid);
    const uint32_t qn = b.qe - b.qs, rn = b.re - b.rs;
    const uint8_t *R = t.rseq + t.roff[b.seq] + b.rs;
    const uint8_t *P = t.pbytes + t.coff[b.cj] + b.qs;
    const uint32_t cap = t.dp_cap[slot];
    uint32_t *cig = reinterpret_cast<uint32_t *>(t.cig_blob + t.dp_cig_off[slot]);
    const uint32_t bw = t.dp_bw[slot];
    if (tp_is_large(bw, rn, qn) && tp_row_cells(bw, qn) + 2 <= t.warp_wcap) return;  // tp_band_warp_kernel's pair
    uint8_t *base = t.blob + t.dp_off[slot];
    const int32_t score = (int32_t)t.score[gid];

    uint32_t r_end = 0, c_end = 0, rows_done = 0;
    const bool banded = bw != 0;
    if (banded) {
        atomicAdd(&t.ctr[8], 1ULL);
        const uint32_t ring = tp_ring_size(bw);
        uint8_t *fl = base + tp_align16(8ull * ring);
        const int32_t s = ring <= kTpRing
                              ? tp_fill<true>(R, rn, P, qn, s_lut, s_w, t.S, t.go, t.ge, bw, s_ring + threadIdx.x, kTpRing - 1,
                                              kTpThreads, fl, &r_end, &c_end, &rows_done)
                              : tp_fill<true>(R, rn, P, qn, s_lut, s_w, t.S, t.go, t.ge, bw, reinterpret_cast<int2 *>(base),
                                              ring - 1, 1, fl, &r_end, &c_end, &rows_done);
        if (!(s > 0 && s == score)) {  // widen the band, or give up on bands
            const uint32_t max_bw = (qn - 1) / 2;
            const uint32_t nbw = 2 * bw <= max_bw ? 2 * bw : 0u;
            t.dp_bw_next[slot] = nbw;
            t.dp_off_next[slot] = atomicAdd(&t.ctr[4], tp_need(nbw, rn, qn));
            t.next_list[atomicAdd(&t.ctr[3], 1ULL)] = slot;
            if (tp_is_large(nbw, rn, qn)) atomicMax(&t.ctr[12], (unsigned long long)tp_row_cells(nbw, qn));
            return;
        }
        atomicAdd(&t.ctr[6], 1ULL);
    } else {
        tp_fill<false>(R, rn, P, qn, s_lut, s_w, t.S, t.go, t.ge, 0, reinterpret_cast<int2 *>(base), 0xffffffffu, 1,
                       base + tp_align16(8ull * qn), &r_end, &c_end, &rows_done);
        atomicAdd(&t.ctr[7], 1ULL);
    }
    const uint8_t *fl = banded ? base + tp_align16(8ull * tp_ring_size(bw)) : base + tp_align16(8ull * qn);

    tp_walk_and_emit(t, b, gid, banded, bw, rows_done, r_end, c_end, fl, cig, cap);
}

// Pass 3b for large boxes: one WARP per listed pair.  Rows are sequential, the cells of a row are spread over the lanes in
// chunks of 32 consecutive columns.  The along-row gap state F -- the only dependency inside a row -- is a max-plus
// prefix scan: F(c) = max(go + (c - start) * ge, max_{c' < c} (H0(c') + go + (c - c' - 1) * ge)) with
// H0 = max(diag + w, E, 0) the cell value before F is considered (a gap opened from a cell that F itself produced is never
// better than extending that gap, because gap_extend >= gap_open: validate_profile_args), so a row costs five shuffle
// steps per chunk instead of a serial walk.  Values, flag bytes, storage layout (row stride 2 bw + 1 / qn) and the
// row-major "first best cell" are those of zoe's loops (banded.rs:55-125, scalar.rs:190-262).
// Shared memory per warp: H of the previous row and E of this row, indexed by band offset (banded: the arrays shift by
// one column per row) or by column (scalar), one guard slot in front.
constexpr int kTpNeg = -(1 << 29);

__global__ void __launch_bounds__(512) tp_band_warp_kernel(const ThreePassParams t, uint32_t n_dp, uint32_t wcap) {
    extern __shared__ __align__(16) uint8_t tp_sm[];
    __shared__ uint8_t s_lut[256];
    __shared__ int8_t s_w[32 * 32];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_lut[i] = t.lut[i];
    for (int i = threadIdx.x; i < t.S * t.S; i += blockDim.x) s_w[i] = t.weights[i];
    __syncthreads();
    constexpr unsigned ALL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    int *Hp = reinterpret_cast<int *>(tp_sm) + (size_t)warp * 2 * wcap + 1;  // Hp[-1] .. Hp[wcap - 2]
    int *En = Hp + wcap;

    for (uint32_t li = blockIdx.x * wpb + warp; li < n_dp; li += gridDim.x * wpb) {
        const uint32_t slot = t.list[li];
        const uint64_t gid = t.pair_first + t.dp_pair[slot];
        const TpBox b = tp_box(t, gid);
        const uint32_t qn = b.qe - b.qs, rn = b.re - b.rs;
        const uint32_t bw = t.dp_bw[slot];
        if (!tp_is_large(bw, rn, qn) || tp_row_cells(bw, qn) + 2 > wcap) continue;  // the thread kernel's pairs (warp-uniform)
        const uint8_t *R = t.rseq + t.roff[b.seq] + b.rs;
        const uint8_t *P = t.pbytes + t.coff[b.cj] + b.qs;
        const bool banded = bw != 0;
        uint8_t *base = t.blob + t.dp_off[slot];
        uint8_t *fl = banded ? base + tp_align16(8ull * tp_ring_size(bw)) : base + tp_align16(8ull * qn);
        const int32_t go = t.go, ge = t.ge;  // <= 0
        const int ncell = (int)tp_row_cells(bw, qn);  // array slots in use
        __syncwarp();
        for (int i = lane - 1; i < ncell + 1 && i < (int)wcap - 1; i += 32) {
            Hp[i] = 0;   // h_row = 0
            En[i] = go;  // e_row = gap_open
        }
        __syncwarp();
        if (banded && lane == 0) atomicAdd(&t.ctr[8], 1ULL);

        const uint32_t rows_done = banded ? min(rn, qn + bw) : rn;
        const int shift = banded ? 1 : 0;       // the band moves one column to the right per row
        const uint32_t bfw = 2 * bw + 1;
        int best = 0;                            // this lane's best cell, row-major first occurrence
        uint32_t br = 0, bc = 0;
        for (uint32_t r = 0; r < rows_done; ++r) {
            const int8_t *wrow = s_w + (int)s_lut[R[r]] * t.S;
            const int c_first = banded ? (int)r - (int)bw : 0;  // column of array index 0
            const int start_col = max(c_first, 0);
            const int end_col = banded ? (int)min(r + bw + 1, qn) : (int)qn;
            uint8_t *frow = fl + (size_t)r * (banded ? bfw : qn) - start_col;
            const int i_lo = start_col - c_first, i_hi = end_col - c_first;  // array indices [i_lo, i_hi)
            int carry = go;      // F entering the first cell of the row
            int diag_carry = 0;  // scalar: H(r-1, c-1) of the next chunk's first cell (its slot is overwritten by then)
            for (int i0 = i_lo; i0 < i_hi; i0 += 32) {
                const int i = i0 + lane;
                const bool on = i < i_hi;
                const int c = c_first + i;
                int diag = 0, e = go, h0 = kTpNeg, own_old = 0;
                if (on) {
                    diag = Hp[i + shift - 1];
                    e = En[i + shift];
                    if (!banded) own_old = Hp[i];
                }
                if (!banded) {
                    if (lane == 0 && i0 > i_lo) diag = diag_carry;
                    diag_carry = __shfl_sync(ALL, own_old, 31);
                }
                if (on) h0 = max(max(diag + (int)wrow[s_lut[P[c]]], e), 0);
                // inclusive max-plus scan: X_i = max_{i' <= i in chunk} (h0_i' + go + (i - i') * ge) = F at cell i + 1
                int X = on ? h0 + go : kTpNeg;
#pragma unroll
                for (int sft = 1; sft < 32; sft <<= 1) {
                    const int y = __shfl_up_sync(ALL, X, sft);
                    if (lane >= sft) X = max(X, y + sft * ge);
                }
                const int Xprev = __shfl_up_sync(ALL, X, 1);
                const int f = max(lane > 0 ? Xprev : kTpNeg, carry + lane * ge);
                const int Xlast = __shfl_sync(ALL, X, 31);
                carry = max(Xlast, carry + 32 * ge);
                __syncwarp();  // every lane has read its inputs of this chunk before anyone overwrites them
                if (on) {
                    const int h = max(h0, f);
                    if (h > best) {
                        best = h;
                        br = r;
                        bc = (uint32_t)c;
                    }
                    uint32_t flag = (e == h ? 1u : 0u) | (f == h ? 4u : 0u);
                    if (h == 0) flag = 16u;
                    const int ho = h + go;
                    const int e2 = max(e + ge, ho), f2 = max(f + ge, ho);
                    if (ho != go) flag |= (e2 > ho ? 2u : 0u) | (f2 > ho ? 8u : 0u);
                    frow[c] = (uint8_t)flag;
                    Hp[i] = h;
                    En[i] = e2;
                }
            }
            __syncwarp();
        }
        // the pair's best cell: max value, then the smallest row, then the smallest column -- three reductions over full
        // 32-bit values, so every row and score of a box is exact (no packed key to truncate them)
        const int32_t s_best = __reduce_max_sync(ALL, best);
        const uint32_t r_end = __reduce_min_sync(ALL, best == s_best ? br : 0xFFFFFFFFu);
        const uint32_t c_end = __reduce_min_sync(ALL, best == s_best && br == r_end ? bc : 0xFFFFFFFFu);
        __threadfence_block();
        __syncwarp();
        if (lane == 0) {
            const int32_t score = (int32_t)t.score[gid];
            if (banded && !(s_best > 0 && s_best == score)) {  // widen the band, or give up on bands
                const uint32_t max_bw = (qn - 1) / 2;
                const uint32_t nbw = 2 * bw <= max_bw ? 2 * bw : 0u;
                t.dp_bw_next[slot] = nbw;
                t.dp_off_next[slot] = atomicAdd(&t.ctr[4], tp_need(nbw, rn, qn));
                t.next_list[atomicAdd(&t.ctr[3], 1ULL)] = slot;
                if (tp_is_large(nbw, rn, qn)) atomicMax(&t.ctr[12], (unsigned long long)tp_row_cells(nbw, qn));
            } else {
                atomicAdd(&t.ctr[banded ? 6 : 7], 1ULL);
                tp_walk_and_emit(t, b, gid, banded, bw, rows_done, s_best > 0 ? r_end : 0u, s_best > 0 ? c_end : 0u, fl,
                                 reinterpret_cast<uint32_t *>(t.cig_blob + t.dp_cig_off[slot]), t.dp_cap[slot]);
            }
        }
        __syncwarp();
    }
}

// Pass 3c: CIGARs into the compacted output stream (offsets from the cigar_*scan* kernels of sw_align.cuh).
__global__ void __launch_bounds__(256) tp_gather_kernel(const ThreePassParams t, const uint64_t *out_off, uint32_t *out,
                                                        uint64_t out_cap) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= t.n_pairs) return;
    const uint32_t slot = t.dp_slot[k];
    if (slot == kTpNoDp) return;
    const uint64_t gid = t.pair_first + k;
    const uint64_t o = out_off[gid];
    const uint32_t cnt = t.cig_count[gid];
    if (o + cnt > out_cap) return;  // the caller reports ZOE_CUDA_E_CIGAR_CAP from the total
    const TpBox b = tp_box(t, gid);
    if (slot == kTpNoGaps) {
        const uint32_t lead = t.invert ? b.rs : b.qs, trail = t.invert ? (b.n - b.re) : (b.m - b.qe);
        uint32_t i = 0;
        if (lead) out[o + i++] = (lead << 4) | 4u;
        out[o + i++] = ((b.qe - b.qs) << 4) | 0u;
        if (trail) out[o + i++] = (trail << 4) | 4u;
        return;
    }
    const uint32_t cap = t.dp_cap[slot];
    const uint32_t *src = reinterpret_cast<const uint32_t *>(t.cig_blob + t.dp_cig_off[slot]) + (cap - min(cnt, cap));
    for (uint32_t i = 0; i < min(cnt, cap); ++i) out[o + i] = src[i];
}

}  // namespace zoe_cuda
