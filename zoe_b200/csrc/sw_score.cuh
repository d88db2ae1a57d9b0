// sw_score.cuh -- score-only local alignment (affine gaps) for sm_100a.
//
// Replaces zoe's sw_simd_score (src/alignment/sw/striped.rs:65-142) plus the i8->i16->i32
// escalation chain of ProfileSets::sw_score_from_i8 (src/alignment/profile_set.rs:71-78).
// It is NOT a port of the striped algorithm: the striped layout exists to feed 128..512-bit CPU
// vectors; on the GPU the same recurrence is evaluated as a register-resident systolic array.
//
// Layout ("row" = register-resident sequence, "col" = sequence streamed through):
//   * a group of G lanes owns one task = two batch sequences (packed as the two signed 16-bit
//     halves of every 32-bit register) or one (32-bit mode);
//   * lane l of the group keeps rows [l*K, (l+1)*K) of H and of the along-column gap state in
//     registers, so the K-row inner loop is fully unrolled;
//   * columns (the profiled sequences, staged once per CTA in shared memory) are swept with a
//     one-column skew per lane; the row-boundary H and the along-row gap state hop to the next
//     lane with two __shfl_up_sync per step;
//   * the substitution scores come from a per-task table in shared memory,
//     tab[col_symbol][row/4][lane] = uint4 of four packed row scores, read with one conflict-free
//     128-bit load per four cells.
//
// Arithmetic (true, un-offset values; zoe's MIN-offset saturating arithmetic computes the same
// H, SURVEY.md 8(a) "Equivalent closed form"):
//     x  = max(E^, F^, go) - go            (E^ = E + go, F^ = F + go: the shifted gap states)
//     H  = max(Hdiag + W, x)               VIADDMNMX.S16x2
//     E^ = max(E^ - ge, H)                 VIADDMNMX.S16x2
//     F^ = max(F^ - ge, H)                 VIADDMNMX.S16x2
//     best = max(best, H, H')              VIMNMX3.S16x2 (two rows per instruction)
// i.e. 4.5 DPX/ALU instructions + 1 plain add per packed cell pair.  The subtraction is exact as a
// plain 32-bit add because max(..., go) - go >= 0 in both halves (no borrow crosses the halves).
//
// Overflow / escalation: the packed kernel is exact while every H < OVF_THRESH (= 32767 - max
// weight); a task whose best reaches the threshold is reported as "needs wide" and re-run by the
// 32-bit instantiation of the same kernel -- the GPU analogue of or_else_overflowed
// (src/alignment/types/output.rs:81-83).  The zoe tier label (8/16/32) is derived from the exact
// score (striped.rs:608-633: i8 holds 1..=254, i16 1..=65534).
#pragma once
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>

#include "tma_stage.cuh"

namespace zoe_cuda {

// Lane skew of the systolic sweep (columns between neighbouring lanes).  With a skew of 2 the value a lane needs from
// the lane above was produced two steps earlier and shuffled during the previous step, so consecutive steps of a
// lane are independent dependency chains and the shuffle latency is never exposed.
#ifndef ZOE_SCORE_SKEW
#define ZOE_SCORE_SKEW 2
#endif
constexpr int kSkew = ZOE_SCORE_SKEW;

// Running maximum on the FMA pipe: the packed scores are non-negative 16-bit integers, and below 0x7C00 their bit
// patterns order exactly like IEEE half-precision numbers, so HMNMX2 (half2 max, FMA pipe) can stand in for
// VIMNMX3.S16x2 (ALU pipe, the pipe that bounds the kernel).  The packed overflow threshold is lowered accordingly
// (kPackedLimit); a NaN pattern (>= 0x7C00) can never displace the running maximum, so detection stays exact.
// MEASURED AND REJECTED on B200 (cfg 2, 400k reads): results stay bit-exact, but HMNMX2 issues on the ALU pipe as
// well, so the ALU count rises from 4.59 to 5.07 per pair: 6.30 TCUPS against 6.84 with VIMNMX3.  Kept behind the
// switch as a record of the experiment.
#ifndef ZOE_SCORE_HMAX
#define ZOE_SCORE_HMAX 0
#endif
constexpr bool kHalfMax = ZOE_SCORE_HMAX != 0;
constexpr int kPackedLimit = kHalfMax ? 0x7C00 : 32767;  // packed lanes are exact while H < kPackedLimit - max weight

constexpr int kPadWeight = -16384;  // score of a padding row (never wins a max, never wraps)

// Which zoe integer types may report a score (src/alignment/sw/striped.rs:608-633): the chain starts at `first` bits and
// escalates up to `last` bits (ProfileSets::sw_*_from_i8 / _i16 / _i32, src/alignment/profile_set.rs:71-118; a
// standalone StripedProfile<T,N,S> is first == last).  lim* = the largest score the tier can report:
// signed T: 2*MAX (254 / 65534 / 2^32-2); unsigned T with a biased matrix: MAX - bias - 1.
struct TierPolicy {
    uint32_t lim8, lim16, lim32;
    uint8_t first, last;
};
__host__ __device__ inline uint8_t tier_for(const TierPolicy &tp, uint32_t score) {  // 0 = Overflowed
    if (tp.first <= 8 && score <= tp.lim8) return 8;
    if (tp.first <= 16 && tp.last >= 16 && score <= tp.lim16) return 16;
    if (tp.last >= 32 && score <= tp.lim32) return 32;
    return 0;
}

struct ScoreParams {
    const uint8_t *rseq;       // batch sequences, raw bytes (device)
    const uint64_t *roff;      // n_rseq + 1 offsets into rseq
    const uint32_t *task_ids;  // optional list of batch-sequence indices (wide re-run); else nullptr
    uint32_t n_tasks;          // packed: ceil(n_rseq / 2) (or list length / 2); 32-bit: count
    uint32_t n_rseq;
    const uint8_t *ccodes;     // column sequences as dense symbol codes (device)
    const uint32_t *coff;      // n_cseq + 1 offsets into ccodes
    const uint32_t *corder;    // optional visiting order of the column sequences (longest first)
    uint32_t n_cseq;
    uint32_t ccodes_bytes;     // total bytes of ccodes (staged in smem when it fits)
    int cols_in_smem;
    const int8_t *wk;          // [n_csym][S] weight of (column dense code, row symbol index)
    int n_csym;                // dense column-symbol count
    int S;
    const uint8_t *lut;        // 256: byte -> row symbol index
    int go, ge;                // positive penalties
    int ovf_thresh;            // packed mode only
    int32_t *best;             // [n_rseq * n_cseq] exact score, or -1 = needs the wide kernel
    uint32_t best_stride;      // row stride of `best` (0 = n_cseq) and first column: a launch may cover a sub-range of the
    uint32_t best_col0;        // profiled set (panels larger than the shared-memory staging area are swept group by group)
    uint32_t task_first;       // first task of this launch (a call may cover its tasks in two launches, the first one running
                               // while the second part of the batch is still being uploaded); n_tasks stays the END task
};

template <bool PACKED>
struct Ops;

template <>
struct Ops<true> {
    static __device__ __forceinline__ uint32_t addmax(uint32_t a, uint32_t b, uint32_t c) {
        return __viaddmax_s16x2(a, b, c);
    }
    static __device__ __forceinline__ uint32_t max3(uint32_t a, uint32_t b, uint32_t c) {
        return __vimax3_s16x2(a, b, c);
    }
    static __device__ __forceinline__ uint32_t max2(uint32_t a, uint32_t b) { return __vmaxs2(a, b); }
    static __device__ __forceinline__ uint32_t min2(uint32_t a, uint32_t b) { return __vmins2(a, b); }
    static __device__ __forceinline__ uint32_t splat(int v) {
        return (uint32_t)(v & 0xffff) | ((uint32_t)(v & 0xffff) << 16);
    }
};

template <>
struct Ops<false> {
    static __device__ __forceinline__ uint32_t addmax(uint32_t a, uint32_t b, uint32_t c) {
        return (uint32_t)__viaddmax_s32((int)a, (int)b, (int)c);
    }
    static __device__ __forceinline__ uint32_t max3(uint32_t a, uint32_t b, uint32_t c) {
        return (uint32_t)__vimax3_s32((int)a, (int)b, (int)c);
    }
    static __device__ __forceinline__ uint32_t max2(uint32_t a, uint32_t b) { return (uint32_t)max((int)a, (int)b); }
    static __device__ __forceinline__ uint32_t min2(uint32_t a, uint32_t b) { return (uint32_t)min((int)a, (int)b); }
    static __device__ __forceinline__ uint32_t splat(int v) { return (uint32_t)v; }
};

// Where the packed score kernel takes the gap penalties from.  A DPX instruction accepts a 32-bit immediate but no
// constant-bank or uniform-register operand, so a penalty known only at run time occupies a vector register in three of
// the four DPX instructions of every row (max3 with go, the two addmax with -ge).
//   GapRt         the penalties of ScoreParams, kept opaque in registers (any scoring)
//   GapImm<O, E>  go = O, ge = E compiled in: the DPX instructions take them as immediates
// With immediates ptxas emits the "- go" of a row as VIADD rather than IMAD.IADD.  Pinning it to IMAD (a mad.lo.u32
// with a multiplier of 1 ptxas cannot see) measured slower on B200, config 2: 281.1 against 279.9 ms per step.
struct GapRt {
    static constexpr bool kImm = false;
    static constexpr int GO = 0, GE = 0;
};
template <int GO_, int GE_>
struct GapImm {
    static constexpr bool kImm = true;
    static constexpr int GO = GO_, GE = GE_;
};

__device__ __forceinline__ uint32_t half2_max_bits(uint32_t a, uint32_t b) {
    uint32_t r;
    asm("max.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
    return r;
}

// Shared-memory footprint helpers (host + device).
__host__ __device__ inline int score_tab_bytes(int n_csym, int G, int K) { return n_csym * ((K + 3) / 4) * G * 16; }


// Shared-memory carve-up common to the kernels that keep a score table per task:
//   [one table per group][byte -> symbol LUT, 256][weights n_csym x S][profiled symbol codes]
struct TaskSmem {
    uint4 *tab;      // this group's table
    uint8_t *s_lut;
    int8_t *s_wk;
    uint8_t *s_cc;
    int tab_bytes;
};

// Carves the dynamic shared memory, loads the LUT and the weights, stages the profiled symbol codes (one TMA bulk
// copy per CTA) when `stage_cols`, and synchronises the CTA.  Must be called by every thread of the CTA.
// TPG = tables per group (2: the group sweeps two tasks side by side; `tab` is the first of the two, back to back).
template <int G, int K4, int TPG = 1>
__device__ __forceinline__ TaskSmem carve_and_stage(uint8_t *smem, const ScoreParams &p, bool stage_cols) {
    const int tid = threadIdx.x;
    const int group_in_block = tid / G, groups_per_block = blockDim.x / G;
    TaskSmem m;
    m.tab_bytes = p.n_csym * K4 * G * 16;
    m.tab = reinterpret_cast<uint4 *>(smem + (size_t)group_in_block * (TPG * m.tab_bytes));
    m.s_lut = smem + (size_t)groups_per_block * (TPG * m.tab_bytes);
    m.s_wk = reinterpret_cast<int8_t *>(m.s_lut + 256);
    m.s_cc = reinterpret_cast<uint8_t *>(m.s_wk) + ((p.n_csym * p.S + 15) & ~15);
    for (int i = tid; i < 256; i += blockDim.x) m.s_lut[i] = p.lut[i];
    for (int i = tid; i < p.n_csym * p.S; i += blockDim.x) m.s_wk[i] = p.wk[i];
    if (stage_cols) stage_with_tma(m.s_cc, p.ccodes, p.ccodes_bytes);
    __syncthreads();
    return m;
}

// Builds a task's score table: lane `lig` fills its own K rows for every column symbol.  Row r of the low / high
// half reads rseq[base + dir * r] for r < len (dir = -1: a reversed prefix), else the padding weight.
// tab[(s * K4 + i4) * G + lig] = the four packed weights of rows lig*K + 4*i4 .. +3 against column symbol s.
// STAGED (the score kernel): the sequence bytes come in with coalesced 128-bit loads (north_star (2)) -- the group stages
// the 16-byte words covering its two sequences in the (not yet written) table area, every lane then picks its K residues
// out of shared memory, maps them to symbol indices (four per register) and only then writes the table over the staging
// area.  !STAGED (pass A, pass B, the ends kernels): every lane fetches its own residues with byte loads at immediate
// offsets.  Measured on one B200, same box, builds without -split-compile, byte loads / 128-bit staged:
//   sw_score_kernel      cfg 1 0.656 / 0.604 ms per call, cfg 2 292.1 / 288.2 ms
//   sw_align_scan_kernel cfg 3 align 59.6 / 60.7 ms, ranges 56.9 / 58.6 ms (one table per 1704-column sweep: the two extra
//                        warp barriers and the larger code cost more than the loads they replace)
template <int G, int K, bool PACKED, bool STAGED = false>
__device__ __forceinline__ void build_task_table(const TaskSmem &m, const ScoreParams &p, int lig, int64_t base_lo, int len_lo,
                                                 int64_t base_hi, int len_hi, int dir = 1) {
    constexpr int K4 = (K + 3) / 4;
  if constexpr (!STAGED) {
    __syncwarp();
    for (int i4 = 0; i4 < K4; ++i4) {
        int sym_lo[4], sym_hi[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int i = i4 * 4 + q, r = lig * K + i;
            sym_lo[q] = (i < K && r < len_lo) ? (int)m.s_lut[p.rseq[base_lo + (int64_t)dir * r]] : -1;
            sym_hi[q] = (PACKED && i < K && r < len_hi) ? (int)m.s_lut[p.rseq[base_hi + (int64_t)dir * r]] : -1;
        }
        for (int s = 0; s < p.n_csym; ++s) {
            const int8_t *wrow = m.s_wk + s * p.S;
            uint32_t w[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int wl = sym_lo[q] >= 0 ? (int)wrow[sym_lo[q]] : kPadWeight;
                const int wh = sym_hi[q] >= 0 ? (int)wrow[sym_hi[q]] : kPadWeight;
                w[q] = PACKED ? ((uint32_t)(wl & 0xffff) | ((uint32_t)(wh & 0xffff) << 16)) : (uint32_t)wl;
            }
            m.tab[(s * K4 + i4) * G + lig] = make_uint4(w[0], w[1], w[2], w[3]);
        }
    }
    __syncwarp();
  } else {
    constexpr int RA = (G * K + 32 + 15) & ~15;  // staging bytes per sequence; 2 * RA <= one symbol's table slice (G*K >= 32)
    static_assert(2 * RA <= K4 * G * 16, "the staging area must fit the table of one column symbol");
    uint8_t *stg = reinterpret_cast<uint8_t *>(m.tab);
    __syncwarp();
    int sh_lo = 0, sh_hi = 0;
    {
        const int64_t a0 = dir > 0 ? base_lo : base_lo - (len_lo - 1);
        const int64_t a0a = a0 & ~(int64_t)15;
        sh_lo = (int)(a0 - a0a);
        const int nq = len_lo > 0 ? (sh_lo + len_lo + 15) >> 4 : 0;
        for (int q = lig; q < nq; q += G)
            reinterpret_cast<uint4 *>(stg)[q] = __ldg(reinterpret_cast<const uint4 *>(p.rseq + a0a) + q);
    }
    if (PACKED) {
        const int64_t a0 = dir > 0 ? base_hi : base_hi - (len_hi - 1);
        const int64_t a0a = a0 & ~(int64_t)15;
        sh_hi = (int)(a0 - a0a);
        const int nq = len_hi > 0 ? (sh_hi + len_hi + 15) >> 4 : 0;
        for (int q = lig; q < nq; q += G)
            reinterpret_cast<uint4 *>(stg + RA)[q] = __ldg(reinterpret_cast<const uint4 *>(p.rseq + a0a) + q);
    }
    __syncwarp();
    uint32_t symw_lo[K4], symw_hi[K4];  // four symbol indices per register, 0xff = padding row
#pragma unroll
    for (int i4 = 0; i4 < K4; ++i4) {
        uint32_t wl = 0, wh = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int i = i4 * 4 + q, r = lig * K + i;
            uint32_t sl = 0xffu, sh = 0xffu;
            if (i < K && r < len_lo) sl = m.s_lut[stg[sh_lo + (dir > 0 ? r : len_lo - 1 - r)]];
            if (PACKED && i < K && r < len_hi) sh = m.s_lut[stg[RA + sh_hi + (dir > 0 ? r : len_hi - 1 - r)]];
            wl |= sl << (8 * q);
            wh |= sh << (8 * q);
        }
        symw_lo[i4] = wl;
        symw_hi[i4] = wh;
    }
    __syncwarp();  // every lane has read the staging area: the table may overwrite it
#pragma unroll
    for (int i4 = 0; i4 < K4; ++i4) {
        for (int s = 0; s < p.n_csym; ++s) {
            const int8_t *wrow = m.s_wk + s * p.S;
            uint32_t w[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint32_t sl = (symw_lo[i4] >> (8 * q)) & 0xffu, sh = (symw_hi[i4] >> (8 * q)) & 0xffu;
                const int wl = sl != 0xffu ? (int)wrow[sl] : kPadWeight;
                const int wh = sh != 0xffu ? (int)wrow[sh] : kPadWeight;
                w[q] = PACKED ? ((uint32_t)(wl & 0xffff) | ((uint32_t)(wh & 0xffff) << 16)) : (uint32_t)wl;
            }
            m.tab[(s * K4 + i4) * G + lig] = make_uint4(w[0], w[1], w[2], w[3]);
        }
    }
    __syncwarp();
  }
}

// One column step of one systolic stream: K rows, fully unrolled.  `tp` points at this lane's uint4 of the
// column symbol's table row; (diag, E) enter from the lane above.
// H is kept in two register sets (P = step parity): column j-1 is read from set P, column j is written to
// set 1-P, so the loop-carried "diag = H[i]" needs no register moves.
#define ZOE_SCORE_ROW(ST, W)                                     \
    {                                                            \
        uint32_t x = O::max3(ST##E, ST##F[i], go_s) - go_s;      \
        uint32_t H = O::addmax(ST##diag, W, x);                  \
        ST##diag = ST##H[PO][i];                                 \
        ST##E = O::addmax(ST##E, neg_ge, H);                     \
        ST##F[i] = O::addmax(ST##F[i], neg_ge, H);               \
        ST##H[PN][i] = H;                                        \
        if (PACKED && kHalfMax) {                                \
            ST##best = half2_max_bits(ST##best, H);              \
        } else if (i & 1) {                                      \
            ST##best = O::max3(ST##best, H, ST##hp);             \
        } else {                                                 \
            ST##hp = H;                                          \
        }                                                        \
    }

// NS = number of column sequences swept concurrently by one group (1 or 2).  With NS = 2 every thread
// carries two independent H/E/F recurrences that share the task's score table, which doubles the
// instruction-level parallelism available to hide the 4-deep dependent chain per row (the ALU pipe, not the
// issue slots or the latency, then bounds the kernel).  Column sequences are visited in `corder`
// (longest first) so the two streams of a pair have similar lengths.
#ifndef ZOE_SCORE_PP
#define ZOE_SCORE_PP 1
#endif
#ifndef ZOE_SCORE2_THREADS
#define ZOE_SCORE2_THREADS 384
#endif
template <int G, int K, bool PACKED, int NS, class Gap = GapRt, bool PP = (ZOE_SCORE_PP && NS == 2 && K <= 19)>
__global__ void __launch_bounds__((NS == 2 && (PP || K > 20)) ? ZOE_SCORE2_THREADS : 512) sw_score_kernel(const ScoreParams p) {
    using O = Ops<PACKED>;
    constexpr int K4 = (K + 3) / 4;
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(16) uint8_t smem[];

    const int tid = threadIdx.x;
    const int lig = tid % G;                  // lane in group
    const int group_in_block = tid / G;
    const int groups_per_block = blockDim.x / G;

    const TaskSmem sm = carve_and_stage<G, K4>(smem, p, p.cols_in_smem != 0);
    uint4 *const tab = sm.tab;
    uint8_t *const s_cc = sm.s_cc;
    const int tab_bytes = sm.tab_bytes;
    const uint8_t *cc = p.cols_in_smem ? s_cc : p.ccodes;

    static_assert(!Gap::kImm || PACKED, "compiled-in gap penalties exist for the packed kernels only");
    uint32_t go_s = O::splat(Gap::kImm ? Gap::GO : p.go), neg_ge = O::splat(Gap::kImm ? -Gap::GE : -p.ge);
    const uint4 *tab_lane = tab + lig;
    // Loop invariants kept opaque so the compiler does not rematerialise them inside the hot loops (S2R + address
    // arithmetic); the table offset stays a 32-bit offset into the shared array so the loads remain LDS.128.
    uint32_t tab_lane_off = (uint32_t)group_in_block * (uint32_t)tab_bytes + (uint32_t)lig * 16u;
    // lane 0 receives zeros from "above": multiplying by an opaque 0/1 keeps that on the FMA pipe (a SEL would
    // take an ALU slot, and the ALU pipe is what bounds this kernel)
    uint32_t nz = lig != 0 ? 1u : 0u;
    if constexpr (Gap::kImm)
        asm volatile("" : "+r"(tab_lane_off), "+r"(nz));
    else
        asm volatile("" : "+r"(go_s), "+r"(neg_ge), "+r"(tab_lane_off), "+r"(nz));

    // Static round-robin task assignment: every group of a warp makes the same number of trips,
    // so the warp never diverges on the task loop (invalid trips run on empty sequences).
    const uint32_t total_groups = gridDim.x * groups_per_block;
    const uint32_t trips = (p.n_tasks - p.task_first + total_groups - 1) / total_groups;
    const uint32_t first = p.task_first + blockIdx.x * groups_per_block + group_in_block;

    for (uint32_t trip = 0; trip < trips; ++trip) {
        const uint32_t task = first + trip * total_groups;
        const bool valid = task < p.n_tasks;

        // ---- which batch sequences does this task hold? ----
        uint32_t id_lo = 0xffffffffu, id_hi = 0xffffffffu;
        if (valid) {
            if (PACKED) {
                uint32_t a = 2 * task, b = 2 * task + 1;
                if (p.task_ids) {
                    id_lo = p.task_ids[a];
                    id_hi = (b < p.n_rseq) ? p.task_ids[b] : 0xffffffffu;
                } else {
                    id_lo = a;
                    id_hi = (b < p.n_rseq) ? b : 0xffffffffu;
                }
            } else {
                id_lo = p.task_ids ? p.task_ids[task] : task;
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

        build_task_table<G, K, PACKED, true>(sm, p, lig, (int64_t)off_lo, len_lo, (int64_t)off_hi, len_hi);

        // ---- sweep the column sequences, NS at a time ----
        for (uint32_t ci = 0; ci < p.n_cseq; ci += NS) {
            const uint32_t cjA = p.corder ? p.corder[ci] : ci;
            const uint32_t cA0 = p.coff[cjA];
            const int LA = (int)(p.coff[cjA + 1] - cA0);
            const uint8_t *csA = cc + cA0;
            uint32_t cjB = 0;
            int LB = 0;
            const uint8_t *csB = cc;
            if (NS == 2 && ci + 1 < p.n_cseq) {
                cjB = p.corder ? p.corder[ci + 1] : ci + 1;
                const uint32_t cB0 = p.coff[cjB];
                LB = (int)(p.coff[cjB + 1] - cB0);
                csB = cc + cB0;
            }

            // the same column codes through a pointer the compiler knows is shared memory (steady loops only)
            const uint8_t *scA = s_cc + (csA - cc), *scB = s_cc + (csB - cc);

            constexpr int NP = PP ? 2 : 1;  // register sets of H (ping-pong or in place)
            uint32_t aH[NP][K], aF[K], bH[NP][NS == 2 ? K : 1], bF[NS == 2 ? K : 1];
#pragma unroll
            for (int i = 0; i < K; ++i) {
                aH[0][i] = aH[NP - 1][i] = 0;
                aF[i] = 0;
                if (NS == 2) {
                    bH[0][i] = bH[NP - 1][i] = 0;
                    bF[i] = 0;
                }
            }
            uint32_t abest = 0, ah_last = 0, ae_out = 0, ah_up_prev = 0;
            uint32_t bbest = 0, bh_last = 0, be_out = 0, bh_up_prev = 0;
            uint32_t a_pend_h = 0, a_pend_e = 0, b_pend_h = 0, b_pend_e = 0;  // kSkew == 2: shuffled one step ahead
            const int nsteps = max(LA, LB) + kSkew * (G - 1);
            // Values entering from the lane above.  Skew 1: shuffle the neighbour's outputs of this very step's
            // predecessor and use them at once.  Skew 2: use what was shuffled during the previous step, then shuffle
            // the neighbour's latest outputs for the next step -- nothing in this step waits for a shuffle.
            auto exchange = [&](uint32_t &ah_in, uint32_t &ae_in, uint32_t &bh_in, uint32_t &be_in, const bool with_b) {
                const uint32_t ah_sh = __shfl_up_sync(FULL, ah_last, 1, G), ae_sh = __shfl_up_sync(FULL, ae_out, 1, G);
                uint32_t bh_sh = 0, be_sh = 0;
                if (with_b) {
                    bh_sh = __shfl_up_sync(FULL, bh_last, 1, G);
                    be_sh = __shfl_up_sync(FULL, be_out, 1, G);
                }
                if (kSkew == 1) {
                    ah_in = ah_sh * nz;
                    ae_in = ae_sh * nz;
                    bh_in = bh_sh * nz;
                    be_in = be_sh * nz;
                } else {
                    ah_in = a_pend_h;
                    ae_in = a_pend_e;
                    bh_in = b_pend_h;
                    be_in = b_pend_e;
                    a_pend_h = ah_sh * nz;
                    a_pend_e = ae_sh * nz;
                    b_pend_h = bh_sh * nz;
                    b_pend_e = be_sh * nz;
                }
            };

            auto do_step = [&](auto parity, const int step) {
                constexpr int PO = PP ? decltype(parity)::value : 0;      // set holding column j-1
                constexpr int PN = PP ? 1 - decltype(parity)::value : 0;  // set receiving column j
                uint32_t ah_in, ae_in, bh_in, be_in;
                exchange(ah_in, ae_in, bh_in, be_in, NS == 2);
                const int j = step - kSkew * lig;
                const bool actA = j >= 0 && j < LA;
                const bool actB = NS == 2 && j >= 0 && j < LB;
                if (actA && actB) {
                    const uint4 *tpA = tab_lane + (size_t)csA[j] * (K4 * G);
                    const uint4 *tpB = tab_lane + (size_t)csB[j] * (K4 * G);
                    uint32_t adiag = ah_up_prev, aE = ae_in, ahp = 0;
                    uint32_t bdiag = bh_up_prev, bE = be_in, bhp = 0;
#pragma unroll
                    for (int i4 = 0; i4 < K4; ++i4) {
                        const uint4 wa4 = tpA[i4 * G], wb4 = tpB[i4 * G];
                        const uint32_t wa[4] = {wa4.x, wa4.y, wa4.z, wa4.w};
                        const uint32_t wb[4] = {wb4.x, wb4.y, wb4.z, wb4.w};
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int i = i4 * 4 + q;
                            if (i < K) {
                                ZOE_SCORE_ROW(a, wa[q])
                                if (NS == 2) ZOE_SCORE_ROW(b, wb[q])
                            }
                        }
                    }
                    if ((K & 1) && !(PACKED && kHalfMax)) {
                        abest = O::max2(abest, ahp);
                        if (NS == 2) bbest = O::max2(bbest, bhp);
                    }
                    ah_last = aH[PN][K - 1];
                    ae_out = aE;
                    if (NS == 2) {
                        bh_last = bH[PN][K - 1];
                        be_out = bE;
                    }
                } else if (actA) {
                    const uint4 *tpA = tab_lane + (size_t)csA[j] * (K4 * G);
                    uint32_t adiag = ah_up_prev, aE = ae_in, ahp = 0;
#pragma unroll
                    for (int i4 = 0; i4 < K4; ++i4) {
                        const uint4 wa4 = tpA[i4 * G];
                        const uint32_t wa[4] = {wa4.x, wa4.y, wa4.z, wa4.w};
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int i = i4 * 4 + q;
                            if (i < K) ZOE_SCORE_ROW(a, wa[q])
                        }
                    }
                    if ((K & 1) && !(PACKED && kHalfMax)) abest = O::max2(abest, ahp);
                    ah_last = aH[PN][K - 1];
                    ae_out = aE;
                } else if (actB) {
                    const uint4 *tpB = tab_lane + (size_t)csB[j] * (K4 * G);
                    uint32_t bdiag = bh_up_prev, bE = be_in, bhp = 0;
#pragma unroll
                    for (int i4 = 0; i4 < K4; ++i4) {
                        const uint4 wb4 = tpB[i4 * G];
                        const uint32_t wb[4] = {wb4.x, wb4.y, wb4.z, wb4.w};
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int i = i4 * 4 + q;
                            if (i < K) ZOE_SCORE_ROW(b, wb[q])
                        }
                    }
                    if ((K & 1) && !(PACKED && kHalfMax)) bbest = O::max2(bbest, bhp);
                    bh_last = bH[PN][K - 1];
                    be_out = bE;
                }
                ah_up_prev = ah_in;
                bh_up_prev = bh_in;
            };
            // Steady steps: every lane of the group has a column (steps G .. L-1), so no activity predicates, no
            // per-lane branches; the column codes come from shared memory (LDS with a 32-bit address).  `BOTH`
            // = both streams, else stream A alone (the longer sequence of the pair once B has run out).
            auto steady_step = [&](auto parity, auto both, const int step) {
                constexpr int PO = PP ? decltype(parity)::value : 0;
                constexpr int PN = PP ? 1 - decltype(parity)::value : 0;
                constexpr bool BOTH = NS == 2 && decltype(both)::value;
                uint32_t ah_in, ae_in, bh_in, be_in;
                exchange(ah_in, ae_in, bh_in, be_in, BOTH);
                const int j = step - kSkew * lig;
                const uint4 *tpA = reinterpret_cast<const uint4 *>(smem + tab_lane_off + (uint32_t)scA[j] * (uint32_t)(K4 * G * 16));
                const uint4 *tpB = tpA;
                if (BOTH) tpB = reinterpret_cast<const uint4 *>(smem + tab_lane_off + (uint32_t)scB[j] * (uint32_t)(K4 * G * 16));
                uint32_t adiag = ah_up_prev, aE = ae_in, ahp = 0;
                uint32_t bdiag = bh_up_prev, bE = be_in, bhp = 0;
#pragma unroll
                for (int i4 = 0; i4 < K4; ++i4) {
                    const uint4 wa4 = tpA[i4 * G];
                    uint4 wb4 = wa4;
                    if (BOTH) wb4 = tpB[i4 * G];
                    const uint32_t wa[4] = {wa4.x, wa4.y, wa4.z, wa4.w};
                    const uint32_t wb[4] = {wb4.x, wb4.y, wb4.z, wb4.w};
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int i = i4 * 4 + q;
                        if (i < K) {
                            ZOE_SCORE_ROW(a, wa[q])
                            if (BOTH) ZOE_SCORE_ROW(b, wb[q])
                        }
                    }
                }
                if ((K & 1) && !(PACKED && kHalfMax)) {
                    abest = O::max2(abest, ahp);
                    if (BOTH) bbest = O::max2(bbest, bhp);
                }
                ah_last = aH[PN][K - 1];
                ae_out = aE;
                ah_up_prev = ah_in;
                if (BOTH) {
                    bh_last = bH[PN][K - 1];
                    be_out = bE;
                    bh_up_prev = bh_in;
                }
            };
            using P0 = std::integral_constant<int, 0>;
            using P1 = std::integral_constant<int, 1>;
            // A lane's active steps are consecutive, so its parity alternates exactly while it is active; before
            // that both register sets are zero, after that they are never read again.
            // Five segments, one code copy each (the loop over segments is deliberately not unrolled):
            //   0 generic [0, kSkew*G)      lanes switch on one by one
            //   1 steady, both streams      every lane active in A and B
            //   2 generic                   the shorter stream drains
            //   3 steady, stream A alone    (the longer sequence of the pair)
            //   4 generic                   tail: lanes switch off one by one
            const bool fast = p.cols_in_smem && G % 2 == 0;
            const int Lmin = NS == 2 ? min(LA, LB) : LA;
            const bool solo = fast && NS == 2 && LA - Lmin > 3 * kSkew * G;
            int seg_end[5];
            seg_end[0] = fast ? min(kSkew * G, nsteps) : nsteps;
            seg_end[1] = Lmin - 1;                                  // steady loops run while step + 1 < L
            seg_end[2] = solo ? ((Lmin + kSkew * G) & ~1) : 0;
            seg_end[3] = solo ? LA - 1 : 0;
            seg_end[4] = nsteps;
            int step = 0;
#pragma unroll 1
            for (int seg = 0; seg < 5; ++seg) {
                const int end = seg_end[seg];
                if (seg == 1) {
                    if (fast)
                        for (; step < end; step += 2) {
                            steady_step(P0{}, std::true_type{}, step);
                            steady_step(P1{}, std::true_type{}, step + 1);
                        }
                } else if (seg == 3) {
                    if (NS == 2)
                        for (; step < end; step += 2) {
                            steady_step(P0{}, std::false_type{}, step);
                            steady_step(P1{}, std::false_type{}, step + 1);
                        }
                } else {
                    for (; step < end; ++step) {
                        if (step & 1)
                            do_step(P1{}, step);
                        else
                            do_step(P0{}, step);
                    }
                }
            }

            // ---- reduce the group's best and write the exact scores ----
#pragma unroll
            for (int d = G / 2; d >= 1; d >>= 1) {
                abest = O::max2(abest, __shfl_xor_sync(FULL, abest, d, G));
                if (NS == 2) bbest = O::max2(bbest, __shfl_xor_sync(FULL, bbest, d, G));
            }
            if (lig == 0 && valid) {
#pragma unroll
                for (int st = 0; st < NS; ++st) {
                    if (st == 1 && !(ci + 1 < p.n_cseq)) break;
                    const uint32_t best = st == 0 ? abest : bbest;
                    const uint32_t cj = st == 0 ? cjA : cjB;
                    const size_t bstride = p.best_stride ? p.best_stride : p.n_cseq, bcol = (size_t)p.best_col0 + cj;
                    if (PACKED) {
                        int b_lo = (int)(int16_t)(best & 0xffff), b_hi = (int)(int16_t)(best >> 16);
                        if (id_lo != 0xffffffffu)
                            p.best[(size_t)id_lo * bstride + bcol] = (b_lo >= p.ovf_thresh) ? -1 : b_lo;
                        if (id_hi != 0xffffffffu)
                            p.best[(size_t)id_hi * bstride + bcol] = (b_hi >= p.ovf_thresh) ? -1 : b_hi;
                    } else {
                        p.best[(size_t)id_lo * bstride + bcol] = (int)best;
                    }
                }
            }
        }
    }
}

}  // namespace zoe_cuda
