// sw_align.cuh -- local alignment with traceback for sm_100a.
//
// Replaces zoe's sw_simd_align (src/alignment/sw/striped.rs:449-598) + BackTrackable::to_alignment
// (src/alignment/types/backtrack.rs:290-342) + Alignment::invert (src/alignment/types/output.rs:396-425).
//
// Three kernels:
//   sw_align_fill_kernel   the systolic DP of sw_score.cuh, additionally emitting five direction bits per
//                          cell and the lexicographically first best cell (max H, min r, min c --
//                          striped.rs:555-583).  The bits are the *canonical* ones of zoe's scalar twin
//                          (src/alignment/sw/scalar.rs:173-271), which zoe's own tests require the
//                          striped kernel to agree with (sw/test.rs:7-51).
//   sw_traceback_kernel    one thread per pair walks the bits with zoe's priority rules and writes
//                          ranges + CIGAR; it raises `hazard` when the walk consults a cell with
//                          E == H == F (H > 0), the only case where the CIGAR depends on the striped lane
//                          layout (DESIGN.md "tie hazards").
//   sw_align_exact_kernel  literal emulation of the striped algorithm (one warp = one SIMD vector,
//                          lane = thread) at the lane count of the pair's score tier, for hazard
//                          pairs and for gap_open == 0.  Bit-identical to zoe by construction.
//
// Flag bits (backtrack.rs:18-34): UP=1 (E==H), UP_EXT=2, LEFT=4 (F==H), LEFT_EXT=8, STOP=16.
// Cell (r, c): r indexes the streamed (batch) sequence = register rows, c the profiled sequence =
// swept columns.  E (UP) runs along r, F (LEFT) along c.
//
// Flag storage of the fill kernel, per (task, profiled sequence):
//   word(c, lane, w) at ((c * G + lane) * NW + w), NW = words per lane per column (multiple of 4);
//   the low/high 16-bit halves belong to the task's first/second sequence; each half holds three
//   consecutive rows of the lane, 5 bits each: row = lane*K + 3*w + slot, bits [5*slot, 5*slot+5).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "sw_score.cuh"

namespace zoe_cuda {

__host__ __device__ inline int align_words_per_lane(int K) { return (((K + 2) / 3) + 3) & ~3; }

struct AlignEnd {      // per pair, written by the fill kernel
    int32_t best;      // exact best score; -1 = needs the 32-bit kernel
    uint32_t r_end;    // 0-based row (streamed index) of the best cell
    uint32_t c_end;    // 0-based column (profiled index) of the best cell
    uint32_t aux;      // windowed pipeline only (sw_align_win.cuh): last pair holding the maximum, then the window start
};
constexpr uint32_t kNotBucketed = 0xffffffffu;  // aux of a pair that takes no part in the windowed pipeline

struct AlignParams {
    ScoreParams s;               // sequences, tables, scoring (s.best unused)
    AlignEnd *ends;              // [n_rseq * n_cseq]
    uint32_t *flags;             // flag words
    const uint64_t *flag_base;   // [n_cseq] word offset of each profiled sequence inside a task's region
    uint64_t task_stride;        // words per task
    uint32_t chunk_first;        // first batch-sequence index of this chunk (tasks are chunk-relative)
};

// ---------------------------------------------------------------------------------------------
// fill
// ---------------------------------------------------------------------------------------------
template <int G, int K, bool PACKED>
__global__ void __launch_bounds__(512) sw_align_fill_kernel(const AlignParams ap) {
    using O = Ops<PACKED>;
    const ScoreParams &p = ap.s;
    constexpr int K4 = (K + 3) / 4;
    constexpr int NW = (((K + 2) / 3) + 3) & ~3;
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(16) uint8_t smem[];

    const int tid = threadIdx.x;
    const int lig = tid % G;
    const int group_in_block = tid / G;
    const int groups_per_block = blockDim.x / G;

    const TaskSmem sm = carve_and_stage<G, K4>(smem, p, p.cols_in_smem != 0);
    uint4 *const tab = sm.tab;
    const uint8_t *cc = p.cols_in_smem ? sm.s_cc : p.ccodes;

    const uint32_t go_s = O::splat(p.go), neg_ge = O::splat(-p.ge), one_s = O::splat(1), c21 = O::splat(21);

    const uint32_t total_groups = gridDim.x * groups_per_block;
    const uint32_t trips = (p.n_tasks + total_groups - 1) / total_groups;
    const uint32_t first = blockIdx.x * groups_per_block + group_in_block;

    for (uint32_t trip = 0; trip < trips; ++trip) {
        const uint32_t task = first + trip * total_groups;
        const bool valid = task < p.n_tasks;
        uint32_t id_lo = 0xffffffffu, id_hi = 0xffffffffu;
        if (valid) {
            if (PACKED) {
                uint32_t a = 2 * task, b = 2 * task + 1;
                if (p.task_ids) {
                    id_lo = p.task_ids[a];
                    id_hi = (b < p.n_rseq) ? p.task_ids[b] : 0xffffffffu;
                } else {
                    id_lo = ap.chunk_first + a;
                    id_hi = (b < p.n_rseq) ? ap.chunk_first + b : 0xffffffffu;
                }
            } else {
                id_lo = p.task_ids ? p.task_ids[task] : ap.chunk_first + task;
            }
        }
        uint64_t off_lo = 0, off_hi = 0;
        int len_lo = 0, len_hi = 0;
        if (id_lo != 0xffffffffu) {
            off_lo = p.roff[id_lo];
            len_lo = (int)(p.roff[id_lo + 1] - off_lo);
        }
        if (PACKED && id_hi != 0xffffffffu) {
            off_hi = p.roff[id_hi];
            len_hi = (int)(p.roff[id_hi + 1] - off_hi);
        }

        build_task_table<G, K, PACKED>(sm, p, lig, (int64_t)off_lo, len_lo, (int64_t)off_hi, len_hi);

        uint32_t *task_flags = ap.flags + (size_t)task * ap.task_stride;

        for (uint32_t cj = 0; cj < p.n_cseq; ++cj) {
            const uint32_t c0 = p.coff[cj];
            const int L = (int)(p.coff[cj + 1] - c0);
            const uint8_t *cs = cc + c0;
            uint32_t *fl = task_flags + ap.flag_base[cj] + (size_t)lig * NW;

            uint32_t Hrow[K], Frow[K];
#pragma unroll
            for (int i = 0; i < K; ++i) {
                Hrow[i] = 0;
                Frow[i] = 0;
            }
            uint32_t h_last = 0, e_out = 0, h_up_prev = 0;
            int bv_lo = 0, bv_hi = 0, bi_lo = 0, bi_hi = 0, bj_lo = 0, bj_hi = 0;
            const int nsteps = L + G - 1;

            for (int step = 0; step < nsteps; ++step) {
                uint32_t h_in = __shfl_up_sync(FULL, h_last, 1, G);
                uint32_t e_in = __shfl_up_sync(FULL, e_out, 1, G);
                if (lig == 0) {
                    h_in = 0;
                    e_in = 0;
                }
                const int j = step - lig;
                if (j >= 0 && j < L) {
                    const int s = cs[j];
                    const uint4 *tp = tab + (size_t)s * (K4 * G) + lig;
                    uint32_t diag = h_up_prev;
                    uint32_t E = e_in;
                    uint32_t cm = 0, hprev = 0;
                    uint32_t words[NW];
#pragma unroll
                    for (int w = 0; w < NW; ++w) words[w] = 0;
#pragma unroll
                    for (int i4 = 0; i4 < K4; ++i4) {
                        const uint4 w4 = tp[i4 * G];
                        const uint32_t wv[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int i = i4 * 4 + q;
                            if (i < K) {
                                const uint32_t Fi = Frow[i];
                                uint32_t x = O::max3(E, Fi, go_s) - go_s;
                                uint32_t H = O::addmax(diag, wv[q], x);
                                diag = Hrow[i];
                                uint32_t Hg = H + go_s;
                                uint32_t nve = O::min2(Hg - E, one_s);    // 0 where E == H   (UP)
                                uint32_t nhe = O::min2(Hg - Fi, one_s);   // 0 where F == H   (LEFT)
                                uint32_t E2 = O::addmax(E, neg_ge, H);
                                uint32_t F2 = O::addmax(Fi, neg_ge, H);
                                uint32_t xv = O::min2(E2 - H, one_s);     // 1 where next-row E extends (UP_EXT)
                                uint32_t xh = O::min2(F2 - H, one_s);     // 1 where next-col F extends (LEFT_EXT)
                                uint32_t ns = O::min2(H, one_s);          // 0 where H == 0   (STOP)
                                uint32_t code = c21 + 2u * xv + 8u * xh - nve - 4u * nhe - 16u * ns;
                                words[i / 3] += code << (5 * (i % 3));
                                E = E2;
                                Frow[i] = F2;
                                Hrow[i] = H;
                                if (i & 1)
                                    cm = O::max3(cm, H, hprev);
                                else
                                    hprev = H;
                            }
                        }
                    }
                    if (K & 1) cm = O::max2(cm, hprev);
                    h_last = Hrow[K - 1];
                    e_out = E;
                    if (valid) {
#pragma unroll
                        for (int w = 0; w < NW; w += 4)
                            *reinterpret_cast<uint4 *>(fl + (size_t)j * (G * NW) + w) =
                                make_uint4(words[w], words[w + 1], words[w + 2], words[w + 3]);
                    }

                    // ---- best-cell bookkeeping: (max H, min r, min c), striped.rs:555-583 ----
                    const int cm_lo = PACKED ? (int)(int16_t)(cm & 0xffff) : (int)cm;
                    const int cm_hi = PACKED ? (int)(int16_t)(cm >> 16) : 0;
                    if (cm_lo > 0 && cm_lo >= bv_lo) {
                        int irow = K;
#pragma unroll
                        for (int i = K - 1; i >= 0; --i) {
                            int h = PACKED ? (int)(int16_t)(Hrow[i] & 0xffff) : (int)Hrow[i];
                            if (h == cm_lo) irow = i;
                        }
                        if (cm_lo > bv_lo || irow < bi_lo) {
                            bv_lo = cm_lo;
                            bi_lo = irow;
                            bj_lo = j;
                        }
                    }
                    if (PACKED && cm_hi > 0 && cm_hi >= bv_hi) {
                        int irow = K;
#pragma unroll
                        for (int i = K - 1; i >= 0; --i) {
                            int h = (int)(int16_t)(Hrow[i] >> 16);
                            if (h == cm_hi) irow = i;
                        }
                        if (cm_hi > bv_hi || irow < bi_hi) {
                            bv_hi = cm_hi;
                            bi_hi = irow;
                            bj_hi = j;
                        }
                    }
                }
                h_up_prev = h_in;
            }

            // ---- group reduction of (best, r, c): larger score, then smaller row, then smaller column ----
            unsigned long long key_lo = ((unsigned long long)(uint32_t)bv_lo << 40) |
                                        ((unsigned long long)(0xFFFFFu - (uint32_t)(lig * K + bi_lo)) << 20) |
                                        (unsigned long long)(0xFFFFFu - (uint32_t)bj_lo);
            unsigned long long key_hi = ((unsigned long long)(uint32_t)bv_hi << 40) |
                                        ((unsigned long long)(0xFFFFFu - (uint32_t)(lig * K + bi_hi)) << 20) |
                                        (unsigned long long)(0xFFFFFu - (uint32_t)bj_hi);
#pragma unroll
            for (int d = G / 2; d >= 1; d >>= 1) {
                unsigned long long o = __shfl_xor_sync(FULL, key_lo, d, G);
                key_lo = o > key_lo ? o : key_lo;
                o = __shfl_xor_sync(FULL, key_hi, d, G);
                key_hi = o > key_hi ? o : key_hi;
            }
            if (lig == 0 && valid) {
                if (id_lo != 0xffffffffu) {  // (aux belongs to the windowed pipeline: left alone)
                    AlignEnd *e = ap.ends + (size_t)id_lo * p.n_cseq + cj;
                    int b = (int)(key_lo >> 40);
                    e->best = (PACKED && b >= p.ovf_thresh) ? -1 : b;
                    e->r_end = 0xFFFFFu - (uint32_t)((key_lo >> 20) & 0xFFFFFu);
                    e->c_end = 0xFFFFFu - (uint32_t)(key_lo & 0xFFFFFu);
                }
                if (PACKED && id_hi != 0xffffffffu) {
                    AlignEnd *e = ap.ends + (size_t)id_hi * p.n_cseq + cj;
                    int b = (int)(key_hi >> 40);
                    e->best = (b >= p.ovf_thresh) ? -1 : b;
                    e->r_end = 0xFFFFFu - (uint32_t)((key_hi >> 20) & 0xFFFFFu);
                    e->c_end = 0xFFFFFu - (uint32_t)(key_hi & 0xFFFFFu);
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// traceback over the fill kernel's flag words
// ---------------------------------------------------------------------------------------------
struct TraceParams {
    const AlignEnd *ends;       // [n_rseq_total * n_cseq]
    const uint32_t *flags;
    const uint64_t *flag_base;  // [n_cseq]
    uint64_t task_stride;
    const uint64_t *roff;       // batch sequence offsets (lengths)
    const uint32_t *coff;       // profiled offsets (lengths)
    uint32_t n_cseq;
    uint32_t chunk_first;       // first batch sequence of the chunk (when seq_ids == nullptr)
    const uint32_t *seq_ids;    // optional slot -> batch sequence list (32-bit re-run)
    uint32_t n_slots;           // batch sequences covered by the flag buffer
    int32_t *best_arr;          // [pairs total] copy of the best score (-1 where the packed lanes overflowed)
    int G, K, NW, packed;
    int invert;                 // 1: SeqSrc::Query(streamed) -> Alignment::invert
    // outputs, indexed by global pair id = seq * n_cseq + cj
    uint32_t *score;
    uint8_t *status, *tier, *hazard;
    uint32_t *ref_start, *ref_end, *query_start, *query_end;
    uint32_t *cig_scratch;      // [pairs_in_chunk * cig_cap], filled from the back
    uint32_t *cig_count;        // [pairs total]
    uint32_t cig_cap;
    unsigned long long *counters;  // [5] exact-list length, [6] cigar overflow count, [8] packed overflows
    uint32_t *hazard_list;      // global pair ids that need the exact kernel
    int all_exact;              // gap_open == 0: every Some pair goes to the exact kernel
    TierPolicy tp;
};

// CIGAR builder writing backwards (the walk runs end -> start, the CIGAR is start -> end).
struct CigarBack {
    uint32_t *buf;   // one past the last slot is buf + cap
    uint32_t cap, n;
    uint32_t cur_op, cur_len;
    bool overflow;
    __device__ void init(uint32_t *b, uint32_t c) {
        buf = b;
        cap = c;
        n = 0;
        cur_op = 0xff;
        cur_len = 0;
        overflow = false;
    }
    __device__ void flush() {
        if (cur_len) {
            if (n < cap)
                buf[cap - 1 - n] = (cur_len << 4) | cur_op;
            else
                overflow = true;
            n++;
        }
        cur_len = 0;
    }
    __device__ void push(uint32_t op, uint32_t len) {  // AlignmentStates::add_ciglet, state.rs:142-152
        if (!len) return;
        if (op == cur_op) {
            cur_len += len;
        } else {
            flush();
            cur_op = op;
            cur_len = len;
        }
    }
};


// Emit zoe's Alignment from a completed walk.  (r, c) = 0-based start, (r_end1, c_end1) = exclusive
// ends, n / m = streamed / profiled lengths.  The walk pushed its ops already (un-inverted letters are
// swapped by the caller through `invert`).
__global__ void sw_traceback_kernel(const TraceParams t) {
    const uint32_t pairs = t.n_slots * t.n_cseq;
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= pairs) return;
    const uint32_t seq_local = k / t.n_cseq, cj = k % t.n_cseq;
    const uint32_t seq = t.seq_ids ? t.seq_ids[seq_local] : t.chunk_first + seq_local;
    const size_t gid = (size_t)seq * t.n_cseq + cj;
    const AlignEnd e = t.ends[gid];
    const uint32_t n = (uint32_t)(t.roff[seq + 1] - t.roff[seq]);
    const uint32_t m = t.coff[cj + 1] - t.coff[cj];
    t.hazard[gid] = 0;
    t.cig_count[gid] = 0;
    t.best_arr[gid] = e.best;
    if (e.best < 0) {  // packed lanes reached the overflow threshold: exact 32-bit score + literal kernel
        t.status[gid] = 0xFF;
        t.hazard[gid] = 1;
        atomicAdd(&t.counters[8], 1ULL);
        unsigned long long slot = atomicAdd(&t.counters[5], 1ULL);
        t.hazard_list[slot] = (uint32_t)gid | 0x80000000u;  // no exact end cell yet
        return;
    }
    if (e.best == 0 || n == 0) {
        t.score[gid] = 0;
        t.status[gid] = 2;  // Unmapped
        t.tier[gid] = t.tp.first;
        t.ref_start[gid] = t.ref_end[gid] = t.query_start[gid] = t.query_end[gid] = 0;
        return;
    }
    const uint8_t tier = tier_for(t.tp, (uint32_t)e.best);
    if (tier == 0) {  // beyond the widest allowed integer type: Overflowed (striped.rs:555-562)
        t.score[gid] = 0;
        t.status[gid] = 1;
        t.tier[gid] = t.tp.last;
        t.ref_start[gid] = t.ref_end[gid] = t.query_start[gid] = t.query_end[gid] = 0;
        return;
    }
    t.score[gid] = (uint32_t)e.best;
    t.status[gid] = 0;
    t.tier[gid] = tier;
    if (t.all_exact) {
        unsigned long long slot = atomicAdd(&t.counters[5], 1ULL);
        t.hazard_list[slot] = (uint32_t)gid;
        t.hazard[gid] = 1;
        return;
    }

    const uint32_t task = t.packed ? seq_local / 2 : seq_local;
    const uint32_t half = t.packed ? (seq_local & 1) : 0;
    const uint32_t *fl = t.flags + (size_t)task * t.task_stride + t.flag_base[cj];
    const int G = t.G, K = t.K, NW = t.NW;
    auto cell = [&](uint32_t r, uint32_t c) -> uint32_t {
        uint32_t lane = r / K, kk = r % K;
        uint32_t w = fl[((size_t)c * G + lane) * NW + kk / 3];
        return (w >> (16 * half + 5 * (kk % 3))) & 31u;
    };

    CigarBack cg;  // scratch rows are indexed by the chunk-local pair id (what cigar_gather_kernel expects)
    cg.init(t.cig_scratch + (size_t)(t.seq_ids ? gid - (size_t)t.chunk_first * t.n_cseq : k) * t.cig_cap, t.cig_cap);
    // letters: zoe's walk emits D for an UP move (consumes a streamed residue) and I for a LEFT move;
    // invert() swaps them.
    const uint32_t OP_UP = t.invert ? 1u /*I*/ : 2u /*D*/, OP_LEFT = t.invert ? 2u : 1u;

    uint32_t r = e.r_end + 1, c = e.c_end + 1;
    const uint32_t r_end1 = r, c_end1 = c;
    // trailing soft clip: un-inverted = profiled tail (backtrack.rs:305); inverted = streamed tail (output.rs:416)
    cg.push(4u, t.invert ? (n - r_end1) : (m - c_end1));
    uint32_t cur = cell(e.r_end, e.c_end);
    int op = 0;  // 0 none, 1 D(up), 2 I(left), 3 M
    bool hz = false;
    while (!(cur & 16u) && r > 0 && c > 0) {
        if ((cur & 1u) && (cur & 4u)) hz = true;
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
    cg.push(4u, t.invert ? r : c);  // leading soft clip
    cg.flush();

    if (hz) {
        unsigned long long slot = atomicAdd(&t.counters[5], 1ULL);
        t.hazard_list[slot] = (uint32_t)gid;
        t.hazard[gid] = 1;
        return;  // the exact kernel rewrites everything for this pair
    }
    if (cg.overflow) atomicAdd(&t.counters[6], 1ULL);
    t.cig_count[gid] = cg.n;
    if (t.invert) {  // ref_range <-> query_range (output.rs:418-419)
        t.ref_start[gid] = c;
        t.ref_end[gid] = c_end1;
        t.query_start[gid] = r;
        t.query_end[gid] = r_end1;
    } else {
        t.ref_start[gid] = r;
        t.ref_end[gid] = r_end1;
        t.query_start[gid] = c;
        t.query_end[gid] = c_end1;
    }
}

// ---------------------------------------------------------------------------------------------
// literal striped emulation: one warp per pair
// ---------------------------------------------------------------------------------------------
struct ExactParams {
    const uint32_t *pair_ids;   // the literal list: global pair ids (bit 31: "no exact end cell yet", ignored here)
    const uint32_t *pos_list;   // optional: positions into pair_ids to process (else 0 .. n_pairs)
    const uint32_t *n_pairs_dev;  // optional: device-side length of pos_list (else n_pairs)
    uint32_t n_pairs;
    const uint8_t *rseq;
    const uint64_t *roff;
    const uint8_t *pbytes;      // profiled sequences, raw bytes
    const uint32_t *coff;
    uint32_t n_cseq;
    const int8_t *weights;      // S*S zoe weights[ref_idx][query_idx]
    int S;
    const uint8_t *lut;
    int go, ge;                 // positive
    int lanes8, lanes16, lanes32;
    int invert;
    // scratch, per warp slot
    int32_t *hbuf;              // [slots][4][vcap]   load, store, e, max_row
    uint8_t *fbuf;              // [slots][fcap]      flag bytes n * nv * N
    uint64_t vcap, fcap;
    int rows_in_smem;
    // outputs (same arrays as TraceParams)
    const uint32_t *score_in;   // exact score from the fill pass (decides the tier)
    uint32_t *ref_start, *ref_end, *query_start, *query_end;
    uint32_t *cig_scratch;      // [n_pairs][cig_cap] (separate region)
    uint32_t *cig_count;
    uint32_t cig_cap;
    unsigned long long *counters;  // [6] cigar overflow, [7] score mismatch (internal check)
    TierPolicy tp;
};

// Values are kept in true (un-offset) form: zoe stores x + T::MIN and saturates, so saturation at MIN is a
// clamp at 0 here; saturation at MAX cannot happen because the tier was chosen from the exact score.
// SMEM: the H / E rows, the current flag row, the profiled indices and the weights live in shared memory.  A template
// parameter rather than a run-time choice so that every access in the hot loops is an LDS / STS with a 32-bit address:
// with the pointers selected at run time the compiler emitted generic LD / ST (and 64-bit address arithmetic) for all
// of them.
template <bool SMEM>
__global__ void __launch_bounds__(128) sw_align_exact_kernel(const ExactParams x) {
    const int warps_per_block = blockDim.x / 32;
    const uint32_t slot = blockIdx.x * warps_per_block + threadIdx.x / 32;
    const uint32_t n_slots = gridDim.x * warps_per_block;
    const int lane = threadIdx.x & 31;
    constexpr unsigned FULL = 0xffffffffu;

    const uint32_t n_pairs = x.n_pairs_dev ? *x.n_pairs_dev : x.n_pairs;
    for (uint32_t pq = slot; pq < n_pairs; pq += n_slots) {
        const uint32_t pi = x.pos_list ? x.pos_list[pq] : pq;  // position in the literal list = CIGAR scratch row
        const uint32_t gid = x.pair_ids[pi] & 0x7fffffffu;
        const uint32_t seq = gid / x.n_cseq, cj = gid % x.n_cseq;
        const uint8_t *R = x.rseq + x.roff[seq];
        const int n = (int)(x.roff[seq + 1] - x.roff[seq]);
        const uint8_t *P = x.pbytes + x.coff[cj];
        const int m = (int)(x.coff[cj + 1] - x.coff[cj]);
        const uint32_t want = x.score_in[gid];
        const uint8_t want_tier = tier_for(x.tp, want);
        // Overflowed in every allowed type: nothing to align (warp-uniform).  A packed overflow whose exact score then
        // fell beyond the widest type is listed too, with score 0 (tier_for(0) is the first tier, not "Overflowed").
        if (want == 0 || want_tier == 0) continue;
        const int N = want_tier == 8 ? x.lanes8 : (want_tier == 16 ? x.lanes16 : x.lanes32);
        const int nv = (m + N - 1) / N;
        // lane t owns SIMD lanes t and t+32 (N <= 64)
        const int NL = (N + 31) / 32;
        // H / E rows: shared memory when the profiled sequence is short enough (latency 30 vs ~600 cycles),
        // else the per-slot global scratch
        extern __shared__ __align__(16) int32_t ex_smem[];
        const uint32_t vcap = (uint32_t)x.vcap;
        int32_t *load = SMEM ? ex_smem + (threadIdx.x / 32) * 4 * vcap : x.hbuf + (size_t)slot * 4 * x.vcap;
        int32_t *store = load + vcap, *es = store + vcap, *max_row = es + vcap;
        uint8_t *bt = x.fbuf + (size_t)slot * x.fcap;
        // the flag bytes of the row being computed live in shared memory (the lazy-F pass reads and rewrites them);
        // a finished row is copied to the per-slot global scratch the traceback reads
        uint8_t *frow = SMEM ? reinterpret_cast<uint8_t *>(ex_smem + warps_per_block * 4 * vcap) + (threadIdx.x / 32) * 2 * vcap
                             : nullptr;
        // profiled symbol indices and the weight matrix staged in shared memory: the inner loop would otherwise
        // chain three global loads (residue -> index -> weight) per vector
        uint8_t *pidx = SMEM ? frow + vcap : nullptr;
        const int8_t *wmat = x.weights;
        if (SMEM) {
            int8_t *ws = reinterpret_cast<int8_t *>(ex_smem + warps_per_block * 4 * vcap) + warps_per_block * 2 * vcap +
                         (threadIdx.x / 32) * 4096;
            for (int i = lane; i < m; i += 32) pidx[i] = x.lut[P[i]];
            for (int i = lane; i < x.S * x.S; i += 32) ws[i] = x.weights[i];
            wmat = ws;
        }
        for (int i = lane; i < nv * N; i += 32) {
            load[i] = 0;
            store[i] = 0;
            es[i] = 0;
            max_row[i] = 0;
        }
        __syncwarp();
        int best = 0;
        int r_end = n - 1;
#ifdef ZOE_EXACT_PROFILE
        long long t_main = 0, t_lazy = 0, t_pub = 0, t_all0 = clock64(), tt;
#define EXACT_TICK(acc) { long long now_ = clock64(); acc += now_ - tt; tt = now_; }
#else
#define EXACT_TICK(acc)
#endif

        for (int r = 0; r < n; ++r) {
#ifdef ZOE_EXACT_PROFILE
            tt = clock64();
#endif
            const int ref_index = x.lut[R[r]];
            const int8_t *wrow = wmat + ref_index * x.S;
            int F[2] = {0, 0}, H[2], rowmax[2] = {0, 0};
            // H = store[nv-1].shift_elements_right(MIN)
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                int l = lane + 32 * q;
                H[q] = (q < NL && l < N && l > 0) ? store[(size_t)(nv - 1) * N + l - 1] : 0;
            }
            __syncwarp();
            if (r > 1 && r_end == r - 2) {
                int32_t *sw = max_row;
                max_row = load;
                load = sw;
            }
            {
                int32_t *sw = load;
                load = store;
                store = sw;
            }
            uint8_t *grow = bt + (size_t)r * nv * N;
            uint8_t *brow = SMEM ? frow : grow;
            for (int v = 0; v < nv; ++v) {
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    int l = lane + 32 * q;
                    if (q < NL && l < N) {
                        int cidx = v + l * nv;
                        int w = cidx < m ? (int)wrow[SMEM ? pidx[cidx] : x.lut[P[cidx]]] : 0;
                        int E = es[v * N + l];
                        int h = max(H[q] + w, 0);  // saturating_add, floor at MIN
                        h = max(max(h, E), F[q]);
                        uint8_t fl = 0;
                        rowmax[q] = max(rowmax[q], h);
                        if (E == h) fl |= 1;
                        if (F[q] == h) fl |= 4;
                        bool stopped = (h == 0);
                        store[v * N + l] = h;
                        int ho = max(h - x.go, 0);
                        E = max(max(E - x.ge, 0), ho);
                        F[q] = max(max(F[q] - x.ge, 0), ho);
                        if (E > ho) fl |= 2;
                        if (F[q] > ho) fl |= 8;
                        if (stopped) fl = 16;
                        brow[v * N + l] = fl;
                        es[v * N + l] = E;
                        H[q] = load[v * N + l];
                    }
                }
            }
            __syncwarp();
            EXACT_TICK(t_main)
            // lazy-F: striped.rs:528-553
            for (int pass = 0; pass < N; ++pass) {
                // F = F.shift_elements_right(MIN)
                int f0 = F[0], f1 = F[1];
                int up0 = __shfl_up_sync(FULL, f0, 1);
                int up1 = __shfl_up_sync(FULL, f1, 1);
                int last0 = __shfl_sync(FULL, f0, 31);
                F[0] = (lane == 0) ? 0 : up0;
                F[1] = (lane == 0) ? last0 : up1;
                bool broke = false;
                for (int v = 0; v < nv; ++v) {
                    bool trig = false;
                    int hs[2] = {0, 0};
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        int l = lane + 32 * q;
                        if (q < NL && l < N) {
                            hs[q] = store[v * N + l];
                            if (F[q] > max(hs[q] - x.go, 0)) trig = true;
                        }
                    }
                    if (!__any_sync(FULL, trig)) {
                        broke = true;
                        break;
                    }
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        int l = lane + 32 * q;
                        if (q < NL && l < N) {
                            int h = max(hs[q], F[q]);
                            store[v * N + l] = h;
                            uint8_t fl = brow[v * N + l];
                            bool stopped = (h == 0);
                            if (F[q] == h) fl = (uint8_t)((fl & 2) | 4);
                            int ho = max(h - x.go, 0);
                            F[q] = max(F[q] - x.ge, 0);
                            if (F[q] > ho) fl |= 8;
                            if (stopped) fl = 16;
                            brow[v * N + l] = fl;
                        }
                    }
                }
                if (broke) break;
            }
            __syncwarp();
            EXACT_TICK(t_lazy)
            if (SMEM) {  // publish the finished row
                const int nb = nv * N;
                if ((nb & 3) == 0) {
                    const uint32_t *src = reinterpret_cast<const uint32_t *>(frow);
                    uint32_t *dst = reinterpret_cast<uint32_t *>(grow);
                    for (int i = lane; i < nb / 4; i += 32) dst[i] = src[i];
                } else {
                    for (int i = lane; i < nb; i += 32) grow[i] = frow[i];
                }
                __syncwarp();
            }
            int rb = max(rowmax[0], rowmax[1]);
#pragma unroll
            for (int d = 16; d >= 1; d >>= 1) rb = max(rb, __shfl_xor_sync(FULL, rb, d));
            if (rb > best) {
                best = rb;
                r_end = r;
            }
            EXACT_TICK(t_pub)
        }
        __syncwarp();
#ifdef ZOE_EXACT_PROFILE
        if (lane == 0 && pq == 0)
            printf("exact profile: N %d nv %d rows %d main %lld lazy %lld publish+reduce %lld loop-total %lld cycles\n", N, nv, n,
                   t_main, t_lazy, t_pub, clock64() - t_all0);
#endif
        if (r_end == n - 1)
            max_row = store;
        else if (n >= 2 && r_end == n - 2)
            max_row = load;

        if (lane == 0) {
            int c_end = m - 1;
            for (int ci = 0; ci < m; ++ci) {
                int v = ci % nv, l = ci / nv;
                if (max_row[(size_t)v * N + l] == best) {
                    c_end = ci;
                    break;
                }
            }
            if ((uint32_t)best != want) atomicAdd(&x.counters[7], 1ULL);
            auto cell = [&](int rr, int cc) -> uint32_t {
                int v = cc % nv, l = (cc - v) / nv;
                return bt[((size_t)nv * rr + v) * N + l];
            };
            CigarBack cg;
            cg.init(x.cig_scratch + (size_t)pi * x.cig_cap, x.cig_cap);
            const uint32_t OP_UP = x.invert ? 1u : 2u, OP_LEFT = x.invert ? 2u : 1u;
            uint32_t r = (uint32_t)r_end + 1, c = (uint32_t)c_end + 1;
            const uint32_t r_end1 = r, c_end1 = c;
            cg.push(4u, x.invert ? ((uint32_t)n - r_end1) : ((uint32_t)m - c_end1));
            uint32_t cur = cell(r_end, c_end);
            int op = 0;
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
                cur = cell(r > 0 ? (int)r - 1 : 0, c > 0 ? (int)c - 1 : 0);
            }
            cg.push(4u, x.invert ? r : c);
            cg.flush();
            if (cg.overflow) atomicAdd(&x.counters[6], 1ULL);
            x.cig_count[gid] = cg.n;
            if (x.invert) {
                x.ref_start[gid] = c;
                x.ref_end[gid] = c_end1;
                x.query_start[gid] = r;
                x.query_end[gid] = r_end1;
            } else {
                x.ref_start[gid] = r;
                x.ref_end[gid] = r_end1;
                x.query_start[gid] = c;
                x.query_end[gid] = c_end1;
            }
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// CIGAR compaction: exclusive scan of counts happens on the host side of the library (cub-free, one
// small kernel per chunk keeps the code dependency-free); this kernel gathers the back-filled scratch.
// ---------------------------------------------------------------------------------------------
// Single-block exclusive scan of the chunk's CIGAR lengths, continuing from a running device-side base
// (so chunks chain without a host round trip).  out_off[first + i] = base + sum(count[first .. first+i)).
__global__ void cigar_scan_kernel(const uint32_t *count, uint64_t first, uint64_t n, uint64_t *out_off,
                                  unsigned long long *running_base) {
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_carry;
    if (threadIdx.x == 0) s_carry = *running_base;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint64_t base = 0; base < n; base += blockDim.x) {
        uint64_t i = base + threadIdx.x;
        unsigned long long v = (i < n) ? count[first + i] : 0ULL;
        unsigned long long incl = v;
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long o = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += o;
        }
        if (lane == 31) s_warp[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            unsigned long long w = (lane < (int)(blockDim.x >> 5)) ? s_warp[lane] : 0ULL;
            unsigned long long wi = w;
            for (int d = 1; d < 32; d <<= 1) {
                unsigned long long o = __shfl_up_sync(0xffffffffu, wi, d);
                if (lane >= d) wi += o;
            }
            s_warp[lane] = wi - w;  // exclusive warp offsets
            if (lane == 31) s_warp[31] = wi - w;
        }
        __syncthreads();
        unsigned long long excl = s_carry + s_warp[wid] + incl - v;
        if (i < n) out_off[first + i] = excl;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) s_carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        *running_base = s_carry;
        out_off[first + n] = s_carry;
    }
}

// Multi-block version of the same scan (large chunks): per-block sums -> scan of the sums (one block) -> per-block
// exclusive scan seeded with its base.  out_off / running_base semantics are those of cigar_scan_kernel.
__global__ void cigar_block_sum_kernel(const uint32_t *count, uint64_t first, uint64_t n, unsigned long long *block_sum) {
    __shared__ unsigned long long s_warp[32];
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long v = (i < n) ? count[first + i] : 0ULL;
    for (int d = 16; d >= 1; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x < 32) {
        unsigned long long w = (threadIdx.x < (blockDim.x >> 5)) ? s_warp[threadIdx.x] : 0ULL;
        for (int d = 16; d >= 1; d >>= 1) w += __shfl_xor_sync(0xffffffffu, w, d);
        if (threadIdx.x == 0) block_sum[blockIdx.x] = w;
    }
}

// exclusive scan of the block sums in place (single block), seeded with and updating the running base
__global__ void cigar_scan_sums_kernel(unsigned long long *block_sum, uint32_t n_blocks, unsigned long long *running_base,
                                       uint64_t *out_off_last) {
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_carry;
    if (threadIdx.x == 0) s_carry = *running_base;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint32_t base = 0; base < n_blocks; base += blockDim.x) {
        const uint32_t i = base + threadIdx.x;
        const unsigned long long v = (i < n_blocks) ? block_sum[i] : 0ULL;
        unsigned long long incl = v;
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long o = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += o;
        }
        if (lane == 31) s_warp[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            unsigned long long w = (lane < (int)(blockDim.x >> 5)) ? s_warp[lane] : 0ULL;
            unsigned long long wi = w;
            for (int d = 1; d < 32; d <<= 1) {
                unsigned long long o = __shfl_up_sync(0xffffffffu, wi, d);
                if (lane >= d) wi += o;
            }
            s_warp[lane] = wi - w;
        }
        __syncthreads();
        const unsigned long long excl = s_carry + s_warp[wid] + incl - v;
        if (i < n_blocks) block_sum[i] = excl;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) s_carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        *running_base = s_carry;
        *out_off_last = s_carry;
    }
}

__global__ void cigar_block_scan_kernel(const uint32_t *count, uint64_t first, uint64_t n, const unsigned long long *block_base,
                                        uint64_t *out_off) {
    __shared__ unsigned long long s_warp[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned long long v = (i < n) ? count[first + i] : 0ULL;
    unsigned long long incl = v;
    for (int d = 1; d < 32; d <<= 1) {
        unsigned long long o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
    }
    if (lane == 31) s_warp[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        unsigned long long w = (lane < (int)(blockDim.x >> 5)) ? s_warp[lane] : 0ULL;
        unsigned long long wi = w;
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long o = __shfl_up_sync(0xffffffffu, wi, d);
            if (lane >= d) wi += o;
        }
        s_warp[lane] = wi - w;
    }
    __syncthreads();
    if (i < n) out_off[first + i] = block_base[blockIdx.x] + s_warp[wid] + incl - v;
}

__global__ void cigar_gather_kernel(const uint32_t *scratch, uint32_t cig_cap, const uint32_t *pair_of_slot,
                                    uint32_t n_slots, uint32_t slot_first_pair, const uint32_t *count,
                                    const uint64_t *out_off, uint32_t *out, uint64_t out_cap,
                                    const uint8_t *skip) {
    const uint32_t slot = blockIdx.x;
    if (slot >= n_slots) return;
    const uint32_t gid = pair_of_slot ? (pair_of_slot[slot] & 0x7fffffffu) : slot_first_pair + slot;
    if (skip && skip[gid]) return;  // hazard pairs are gathered from the exact kernel's scratch
    const uint32_t cnt = count[gid];
    const uint64_t o = out_off[gid];
    const uint32_t *src = scratch + (size_t)slot * cig_cap + (cig_cap - min(cnt, cig_cap));
    for (uint32_t i = threadIdx.x; i < min(cnt, cig_cap); i += blockDim.x)
        if (o + i < out_cap) out[o + i] = src[i];
}

}  // namespace zoe_cuda
