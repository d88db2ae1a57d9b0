// sw_score_rows.cuh -- score-only local alignment with the PROFILED sequence register-resident (sm_100a).
//
// Same contract as sw_score.cuh (zoe: sw_simd_score, src/alignment/sw/striped.rs:65-142, with the escalation of
// src/alignment/profile_set.rs:71-78).  sw_score_kernel keeps the streamed sequences in registers and needs one
// score table PER TASK (column symbols x rows x 4 B): 2.5 kB for a 150-nt read pair, but 25 kB for a pair of 300-aa
// queries against a 20-letter target, which leaves 4 warps per SM (BASELINE config 5: 0.29 of the roofline).
// The local-alignment score is symmetric under transposition, so here the roles are swapped:
//
//   * rows     = the profiled sequence (<= G*K = 1024 residues), K rows per lane in registers, the same rows for
//                every task, hence ONE score table per CTA: tab[streamed symbol][row/4][lane] = uint4 of four row
//                weights, each zero-extended to 32 bits;
//   * columns  = the streamed sequences; a task is two of them (the two 16-bit halves), whose column symbols differ,
//                so the packed weight is assembled per row as  w = w_hi * 65536 + w_lo  (one IMAD on the FMA pipe,
//                which has slack: the ALU pipe bounds the kernel);
//   * a group (warp) sweeps TWO tasks at once as independent dependency chains (the table is shared, so the second
//                chain costs registers only).
//
// Per packed cell pair: 3.5 DPX/ALU + 2 per-half adds (dW, H - go) + 1 FMA-pipe IMAD (weight assembly) + 0.5 LDS.128.  The sweep is as short as a
// streamed sequence (300 columns in config 5), so the lane skew (G-1 steps of ramp and tail) is a real cost here:
// skew 1 is used (the shuffle latency is covered by the second chain).
//
// Columns past the end of the shorter sequence of a task use a pad symbol whose weights are kPadWeight: such cells
// can only be reached through a gap from a real cell and therefore never exceed the true best (same argument as the
// padding rows of sw_score_kernel).
#pragma once
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>

#include "sw_score.cuh"

namespace zoe_cuda {

struct RowsParams {
    ScoreParams s;        // rseq/roff = streamed (columns here), ccodes/coff/wk = profiled (rows here)
    uint32_t cj;          // which profiled sequence this launch scores
    uint32_t max_rlen;    // longest streamed sequence (sizes the per-warp staging area)
};

// bytes of the CTA-wide table: (S + 1 pad symbol) x K4 x G uint4
__host__ __device__ inline size_t rows_tab_bytes(int S, int G, int K) { return (size_t)(S + 1) * ((K + 3) / 4) * G * 16; }
// per-warp staging: 2 chains x 2 halves x max_rlen streamed symbol indices (uint16)
__host__ __device__ inline size_t rows_stage_bytes(uint32_t max_rlen) { return (size_t)4 * ((max_rlen + 7) & ~7u) * 2; }

template <int G, int K>
__global__ void __launch_bounds__(K > 20 ? 256 : 384) sw_score_rows_kernel(const RowsParams rp) {
    constexpr bool PACKED = true;
    using O = Ops<true>;
    const ScoreParams &p = rp.s;
    constexpr int K4 = (K + 3) / 4;
    constexpr unsigned FULL = 0xffffffffu;
    static_assert(G == 32, "one task pair per warp");
    extern __shared__ __align__(16) uint8_t smem[];

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int warps_per_block = blockDim.x >> 5;
    const int lig = lane;

    // ---- shared memory: [table (S+1) x K4 x G uint4][per-warp column offsets] ----
    const uint32_t sym_stride = (uint32_t)(K4 * G * 16);  // bytes per streamed symbol
    const size_t tab_bytes = rows_tab_bytes(p.S, G, K);
    const uint32_t stage_len = (rp.max_rlen + 7) & ~7u;
    uint16_t *stage = reinterpret_cast<uint16_t *>(smem + tab_bytes) + (size_t)warp * 4 * stage_len;

    // ---- build the table once per CTA: tab[q][i4][l].e = weight(streamed symbol q, profiled row l*K + 4*i4 + e) ----
    const uint32_t c0 = p.coff[rp.cj];
    const int Lrows = (int)(p.coff[rp.cj + 1] - c0);
    for (int idx = tid; idx < (p.S + 1) * K4 * G * 4; idx += blockDim.x) {
        const int e = idx & 3, l = (idx >> 2) % G, i4 = ((idx >> 2) / G) % K4, q = (idx >> 2) / (G * K4);
        const int i = i4 * 4 + e, r = l * K + i;
        int w = kPadWeight;
        if (q < p.S && i < K && r < Lrows) w = (int)p.wk[(size_t)p.ccodes[c0 + r] * p.S + q];
        reinterpret_cast<uint32_t *>(smem)[idx] = (uint32_t)(w & 0xffff);
    }
    __syncthreads();

    uint32_t neg_go = O::splat(-p.go), neg_ge = O::splat(-p.ge);
    uint32_t lane_off = (uint32_t)lane * 16u;
    uint32_t nz = lane != 0 ? 1u : 0u;
    uint32_t sym_stride_r = sym_stride;  // opaque: symbol index -> table offset by an IMAD (FMA pipe), not a shift (ALU)
    asm volatile("" : "+r"(neg_go), "+r"(neg_ge), "+r"(lane_off), "+r"(nz), "+r"(sym_stride_r));
    const uint32_t pad_sym = (uint32_t)p.S;

    // a "task" = two streamed sequences (2t, 2t+1); a warp sweeps two tasks (chains a and b) per trip
    const uint32_t n_tasks = (p.n_rseq + 1) / 2;
    const uint32_t n_trips_total = (n_tasks + 1) / 2;
    const uint32_t total_warps = gridDim.x * warps_per_block;
    for (uint32_t trip = blockIdx.x * warps_per_block + warp; trip < n_trips_total; trip += total_warps) {
        uint32_t ids[4];
        int lens[4];
        uint64_t offs[4];
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            const uint64_t a = (uint64_t)4 * trip + h;
            uint32_t id = 0xffffffffu;
            if (a < p.n_rseq) id = p.task_ids ? p.task_ids[a] : (uint32_t)a;
            ids[h] = id;
            offs[h] = id != 0xffffffffu ? p.roff[id] : 0;
            lens[h] = id != 0xffffffffu ? (int)(p.roff[id + 1] - offs[h]) : 0;
        }
        const int LA = max(lens[0], lens[1]), LB = max(lens[2], lens[3]);

        // ---- stage the column symbols of the four sequences ----
        __syncwarp();
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            const int Lh = h < 2 ? LA : LB;
            for (int j = lane; j < Lh; j += 32) {
                uint32_t sym = pad_sym;
                if (j < lens[h]) sym = (uint32_t)p.lut[p.rseq[offs[h] + j]];
                stage[h * stage_len + j] = (uint16_t)sym;
            }
        }
        __syncwarp();
        const uint16_t *cA_lo = stage, *cA_hi = stage + stage_len, *cB_lo = stage + 2 * stage_len, *cB_hi = stage + 3 * stage_len;

        uint32_t aH[2][K], aF[K], bH[2][K], bF[K];
#pragma unroll
        for (int i = 0; i < K; ++i) {
            aH[0][i] = aH[1][i] = 0;
            aF[i] = 0;
            bH[0][i] = bH[1][i] = 0;
            bF[i] = 0;
        }
        uint32_t abest = 0, ah_last = 0, ae_out = 0, ah_up_prev = 0;
        uint32_t bbest = 0, bh_last = 0, be_out = 0, bh_up_prev = 0;
        const int nsteps = max(LA, LB) + (G - 1);

        // one column of one chain; STEADY = no activity test
        auto chain_col = [&](auto parity, auto which, const int j, const uint32_t h_in, const uint32_t e_in) {
            constexpr int PO = decltype(parity)::value, PN = 1 - PO;
            constexpr bool IS_A = decltype(which)::value == 0;
            const uint32_t off_lo = (uint32_t)(IS_A ? cA_lo[j] : cB_lo[j]) * sym_stride_r;
            const uint32_t off_hi = (uint32_t)(IS_A ? cA_hi[j] : cB_hi[j]) * sym_stride_r;
            const uint4 *tl = reinterpret_cast<const uint4 *>(smem + lane_off + off_lo);
            const uint4 *th = reinterpret_cast<const uint4 *>(smem + lane_off + off_hi);
            if (IS_A) {
                uint32_t adiag = ah_up_prev, aE = e_in, ahp = 0;
#pragma unroll
                for (int i4 = 0; i4 < K4; ++i4) {
                    const uint4 l4 = tl[i4 * G], h4 = th[i4 * G];
                    const uint32_t w[4] = {h4.x * 65536u + l4.x, h4.y * 65536u + l4.y, h4.z * 65536u + l4.z, h4.w * 65536u + l4.w};
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int i = i4 * 4 + q;
                        if (i < K) ZOE_SCORE_ROW(a, w[q])
                    }
                }
                if (K & 1) abest = O::max2(abest, ahp);
                ah_last = aH[PN][K - 1];
                ae_out = aE;
            } else {
                uint32_t bdiag = bh_up_prev, bE = e_in, bhp = 0;
#pragma unroll
                for (int i4 = 0; i4 < K4; ++i4) {
                    const uint4 l4 = tl[i4 * G], h4 = th[i4 * G];
                    const uint32_t w[4] = {h4.x * 65536u + l4.x, h4.y * 65536u + l4.y, h4.z * 65536u + l4.z, h4.w * 65536u + l4.w};
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int i = i4 * 4 + q;
                        if (i < K) ZOE_SCORE_ROW(b, w[q])
                    }
                }
                if (K & 1) bbest = O::max2(bbest, bhp);
                bh_last = bH[PN][K - 1];
                be_out = bE;
            }
            (void)h_in;
        };
        using C0 = std::integral_constant<int, 0>;
        using C1 = std::integral_constant<int, 1>;
        auto step_fn = [&](auto parity, auto steady, const int step) {
            const uint32_t ah_in = __shfl_up_sync(FULL, ah_last, 1) * nz, ae_in = __shfl_up_sync(FULL, ae_out, 1) * nz;
            const uint32_t bh_in = __shfl_up_sync(FULL, bh_last, 1) * nz, be_in = __shfl_up_sync(FULL, be_out, 1) * nz;
            const int j = step - lig;
            if (decltype(steady)::value || (j >= 0 && j < LA)) chain_col(parity, C0{}, j, ah_in, ae_in);
            if (decltype(steady)::value || (j >= 0 && j < LB)) chain_col(parity, C1{}, j, bh_in, be_in);
            ah_up_prev = ah_in;
            bh_up_prev = bh_in;
        };

        // segments: ramp (generic), steady while every lane of both chains has a column, tail (generic)
        const int Lmin = min(LA, LB);
        int step = 0;
        int seg_end[3] = {min(G, nsteps), Lmin - 1, nsteps};
#pragma unroll 1
        for (int seg = 0; seg < 3; ++seg) {
            const int end = seg_end[seg];
            if (seg == 1) {
                for (; step < end; step += 2) {
                    step_fn(C0{}, std::true_type{}, step);
                    step_fn(C1{}, std::true_type{}, step + 1);
                }
            } else {
                for (; step < end; ++step) {
                    if (step & 1)
                        step_fn(C1{}, std::false_type{}, step);
                    else
                        step_fn(C0{}, std::false_type{}, step);
                }
            }
        }

        // ---- reduce and write ----
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) {
            abest = O::max2(abest, __shfl_xor_sync(FULL, abest, d));
            bbest = O::max2(bbest, __shfl_xor_sync(FULL, bbest, d));
        }
        if (lane == 0) {
            const int v[4] = {(int)(int16_t)(abest & 0xffff), (int)(int16_t)(abest >> 16), (int)(int16_t)(bbest & 0xffff),
                              (int)(int16_t)(bbest >> 16)};
#pragma unroll
            for (int h = 0; h < 4; ++h)
                if (ids[h] != 0xffffffffu) p.best[(size_t)ids[h] * p.n_cseq + rp.cj] = (v[h] >= p.ovf_thresh) ? -1 : v[h];
        }
    }
}


// ---------------------------------------------------------------------------------------------
// Streaming variant: a warp sweeps its trips back to back instead of draining the systolic array after each one.
// With sweeps as short as 300 columns the lane skew costs 31 half-idle ramp steps plus 31 tail steps per trip (10 % of
// config 5); here lane l starts trip t's first column at the step after it finished trip t-1's last one, so only the
// very first ramp and the very last tail of a warp's whole stream are idle.
//   * a trip's length is max over its four sequences (pad symbols beyond a sequence's own end, as before);
//   * boundary steps (the first 32 steps of a trip): lane l is still in trip t-1 while step < l, crosses at step == l
//     (parks its per-trip maxima in shared memory, zeroes its H / F registers and the pending diagonal -- a zero gap
//     state is exact, see sw_score.cuh), and reads the column symbols of whichever trip it is in (two staging buffers
//     per warp);
//   * steady steps: every lane is in the current trip, no per-lane tests -- the same loop as above.
// Requires every streamed sequence to have at least 64 residues (the host falls back to sw_score_rows_kernel otherwise).
// ---------------------------------------------------------------------------------------------
__host__ __device__ inline size_t rows_stream_stage_bytes(uint32_t max_rlen) {
    return (size_t)8 * ((max_rlen + 7) & ~7u) * 2 + 64 * 4;  // two staging buffers + the parked maxima (32 lanes x 2 chains)
}

template <int G, int K>
__global__ void __launch_bounds__(K > 20 ? 256 : 384) sw_score_rows_stream_kernel(const RowsParams rp) {
    constexpr bool PACKED = true;
    using O = Ops<true>;
    const ScoreParams &p = rp.s;
    constexpr int K4 = (K + 3) / 4;
    constexpr unsigned FULL = 0xffffffffu;
    static_assert(G == 32, "one task pair per warp");
    extern __shared__ __align__(16) uint8_t smem[];

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int warps_per_block = blockDim.x >> 5;
    const int lig = lane;

    const uint32_t sym_stride = (uint32_t)(K4 * G * 16);
    const size_t tab_bytes = rows_tab_bytes(p.S, G, K);
    const uint32_t stage_len = (rp.max_rlen + 7) & ~7u;
    uint8_t *wbase = smem + tab_bytes + (size_t)warp * rows_stream_stage_bytes(rp.max_rlen);
    uint16_t *stage2 = reinterpret_cast<uint16_t *>(wbase);                              // [2][4][stage_len]
    uint32_t *parked = reinterpret_cast<uint32_t *>(wbase + (size_t)16 * stage_len);     // [32 lanes][2 chains]

    const uint32_t c0 = p.coff[rp.cj];
    const int Lrows = (int)(p.coff[rp.cj + 1] - c0);
    for (int idx = tid; idx < (p.S + 1) * K4 * G * 4; idx += blockDim.x) {
        const int e = idx & 3, l = (idx >> 2) % G, i4 = ((idx >> 2) / G) % K4, q = (idx >> 2) / (G * K4);
        const int i = i4 * 4 + e, r = l * K + i;
        int w = kPadWeight;
        if (q < p.S && i < K && r < Lrows) w = (int)p.wk[(size_t)p.ccodes[c0 + r] * p.S + q];
        reinterpret_cast<uint32_t *>(smem)[idx] = (uint32_t)(w & 0xffff);
    }
    __syncthreads();

    uint32_t neg_go = O::splat(-p.go), neg_ge = O::splat(-p.ge);
    uint32_t lane_off = (uint32_t)lane * 16u;
    uint32_t nz = lane != 0 ? 1u : 0u;
    uint32_t sym_stride_r = sym_stride;
    asm volatile("" : "+r"(neg_go), "+r"(neg_ge), "+r"(lane_off), "+r"(nz), "+r"(sym_stride_r));
    const uint32_t pad_sym = (uint32_t)p.S;

    const uint32_t n_tasks = (p.n_rseq + 1) / 2;
    const uint32_t n_trips_total = (n_tasks + 1) / 2;
    const uint32_t total_warps = gridDim.x * warps_per_block;

    uint32_t aH[2][K], aF[K], bH[2][K], bF[K];
#pragma unroll
    for (int i = 0; i < K; ++i) {
        aH[0][i] = aH[1][i] = 0;
        aF[i] = 0;
        bH[0][i] = bH[1][i] = 0;
        bF[i] = 0;
    }
    uint32_t abest = 0, ah_last = 0, ae_out = 0, ah_up_prev = 0;
    uint32_t bbest = 0, bh_last = 0, be_out = 0, bh_up_prev = 0;

    // one column of one chain, its symbols read from the staging buffer `sb` (trip-local column j)
    auto chain_col = [&](auto parity, auto which, const uint16_t *sb, const int j, const uint32_t e_in) {
        constexpr int PO = decltype(parity)::value, PN = 1 - PO;
        constexpr bool IS_A = decltype(which)::value == 0;
        const uint16_t *c_lo = sb + (IS_A ? 0 : 2) * stage_len, *c_hi = c_lo + stage_len;
        const uint32_t off_lo = (uint32_t)c_lo[j] * sym_stride_r, off_hi = (uint32_t)c_hi[j] * sym_stride_r;
        const uint4 *tl = reinterpret_cast<const uint4 *>(smem + lane_off + off_lo);
        const uint4 *th = reinterpret_cast<const uint4 *>(smem + lane_off + off_hi);
        if (IS_A) {
            uint32_t adiag = ah_up_prev, aE = e_in, ahp = 0;
#pragma unroll
            for (int i4 = 0; i4 < K4; ++i4) {
                const uint4 l4 = tl[i4 * G], h4 = th[i4 * G];
                const uint32_t w[4] = {h4.x * 65536u + l4.x, h4.y * 65536u + l4.y, h4.z * 65536u + l4.z, h4.w * 65536u + l4.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int i = i4 * 4 + q;
                    if (i < K) ZOE_SCORE_ROW(a, w[q])
                }
            }
            if (K & 1) abest = O::max2(abest, ahp);
            ah_last = aH[PN][K - 1];
            ae_out = aE;
        } else {
            uint32_t bdiag = bh_up_prev, bE = e_in, bhp = 0;
#pragma unroll
            for (int i4 = 0; i4 < K4; ++i4) {
                const uint4 l4 = tl[i4 * G], h4 = th[i4 * G];
                const uint32_t w[4] = {h4.x * 65536u + l4.x, h4.y * 65536u + l4.y, h4.z * 65536u + l4.z, h4.w * 65536u + l4.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int i = i4 * 4 + q;
                    if (i < K) ZOE_SCORE_ROW(b, w[q])
                }
            }
            if (K & 1) bbest = O::max2(bbest, bhp);
            bh_last = bH[PN][K - 1];
            be_out = bE;
        }
    };
    using C0 = std::integral_constant<int, 0>;
    using C1 = std::integral_constant<int, 1>;

    // boundary / ramp / tail step: local step k of the current trip; a lane is in the current trip when k >= lane,
    // else still in the previous one (column Lprev + k - lane)
    auto generic_step = [&](auto parity, const int k, const bool have_cur, const bool have_prev, const int Lprev,
                            const uint16_t *sb_cur, const uint16_t *sb_prev) {
        const uint32_t ah_in = __shfl_up_sync(FULL, ah_last, 1) * nz, ae_in = __shfl_up_sync(FULL, ae_out, 1) * nz;
        const uint32_t bh_in = __shfl_up_sync(FULL, bh_last, 1) * nz, be_in = __shfl_up_sync(FULL, be_out, 1) * nz;
        const int jn = k - lig;
        const bool in_cur = have_cur && jn >= 0;
        if (in_cur && jn == 0) {  // crossing into the current trip
            parked[2 * lane] = abest;
            parked[2 * lane + 1] = bbest;
            abest = bbest = 0;
#pragma unroll
            for (int i = 0; i < K; ++i) {
                aH[0][i] = aH[1][i] = 0;
                aF[i] = 0;
                bH[0][i] = bH[1][i] = 0;
                bF[i] = 0;
            }
            ah_up_prev = bh_up_prev = 0;
        }
        // one pass over the columns for the whole warp: each lane reads the trip it is in
        if (in_cur || (have_prev && jn < 0)) {
            const uint16_t *sb = in_cur ? sb_cur : sb_prev;
            const int j = in_cur ? jn : Lprev + jn;
            chain_col(parity, C0{}, sb, j, ae_in);
            chain_col(parity, C1{}, sb, j, be_in);
        }
        ah_up_prev = ah_in;
        bh_up_prev = bh_in;
    };
    auto steady_step = [&](auto parity, const int k, const uint16_t *sb_cur) {
        const uint32_t ah_in = __shfl_up_sync(FULL, ah_last, 1) * nz, ae_in = __shfl_up_sync(FULL, ae_out, 1) * nz;
        const uint32_t bh_in = __shfl_up_sync(FULL, bh_last, 1) * nz, be_in = __shfl_up_sync(FULL, be_out, 1) * nz;
        const int j = k - lig;
        chain_col(parity, C0{}, sb_cur, j, ae_in);
        chain_col(parity, C1{}, sb_cur, j, be_in);
        ah_up_prev = ah_in;
        bh_up_prev = bh_in;
    };

    uint32_t pids[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
    bool have_prev = false;
    int Lprev = 0, buf = 0;
    uint32_t gs = 0;  // global step of this warp: its parity selects the ping-pong register set
    for (uint32_t trip = blockIdx.x * warps_per_block + warp;; trip += total_warps) {
        const bool have_cur = trip < n_trips_total;
        if (!have_cur && !have_prev) break;
        uint32_t ids[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
        int Lcur = 0;
        uint16_t *sb_cur = stage2 + (size_t)buf * 4 * stage_len;
        const uint16_t *sb_prev = stage2 + (size_t)(buf ^ 1) * 4 * stage_len;
        if (have_cur) {
            int lens[4];
            uint64_t offs[4];
#pragma unroll
            for (int h = 0; h < 4; ++h) {
                const uint64_t a = (uint64_t)4 * trip + h;
                uint32_t id = 0xffffffffu;
                if (a < p.n_rseq) id = p.task_ids ? p.task_ids[a] : (uint32_t)a;
                ids[h] = id;
                offs[h] = id != 0xffffffffu ? p.roff[id] : 0;
                lens[h] = id != 0xffffffffu ? (int)(p.roff[id + 1] - offs[h]) : 0;
            }
            Lcur = max(max(lens[0], lens[1]), max(lens[2], lens[3]));
            // ---- stage the column symbols of the four sequences (the other buffer still serves trip t-1's tail) ----
#pragma unroll
            for (int h = 0; h < 4; ++h)
                for (int j = lane; j < Lcur; j += 32) {
                    uint32_t sym = pad_sym;
                    if (j < lens[h]) sym = (uint32_t)p.lut[p.rseq[offs[h] + j]];
                    sb_cur[h * stage_len + j] = (uint16_t)sym;
                }
            __syncwarp();
        }

        // ---- boundary segment: 32 steps (every lane has crossed by step 31), plus one when the steady loop would
        //      otherwise start on an odd global step; without a current trip it is the 31-step tail of the stream ----
        int k = 0;
        const int nb = have_cur ? 32 : 31;
        for (; k < nb || (have_cur && (gs & 1)); ++k, ++gs) {
            if (gs & 1)
                generic_step(C1{}, k, have_cur, have_prev, Lprev, sb_cur, sb_prev);
            else
                generic_step(C0{}, k, have_cur, have_prev, Lprev, sb_cur, sb_prev);
        }
        if (!have_cur) {  // end of the stream: park the last trip's maxima
            parked[2 * lane] = abest;
            parked[2 * lane + 1] = bbest;
        }
        if (have_prev) {  // every lane has parked trip t-1's maxima: reduce and write
            __syncwarp();
            uint32_t va = parked[2 * lane], vb = parked[2 * lane + 1];
#pragma unroll
            for (int d = 16; d >= 1; d >>= 1) {
                va = O::max2(va, __shfl_xor_sync(FULL, va, d));
                vb = O::max2(vb, __shfl_xor_sync(FULL, vb, d));
            }
            if (lane == 0) {
                const int v[4] = {(int)(int16_t)(va & 0xffff), (int)(int16_t)(va >> 16), (int)(int16_t)(vb & 0xffff),
                                  (int)(int16_t)(vb >> 16)};
#pragma unroll
                for (int h = 0; h < 4; ++h)
                    if (pids[h] != 0xffffffffu) p.best[(size_t)pids[h] * p.n_cseq + rp.cj] = (v[h] >= p.ovf_thresh) ? -1 : v[h];
            }
            __syncwarp();
        }
        if (!have_cur) break;

        // ---- steady segment: every lane is inside the current trip ----
        for (; k + 1 < Lcur; k += 2, gs += 2) {
            steady_step(C0{}, k, sb_cur);
            steady_step(C1{}, k + 1, sb_cur);
        }
        for (; k < Lcur; ++k, ++gs) {
            if (gs & 1)
                generic_step(C1{}, k, true, false, 0, sb_cur, sb_prev);
            else
                generic_step(C0{}, k, true, false, 0, sb_cur, sb_prev);
        }
#pragma unroll
        for (int h = 0; h < 4; ++h) pids[h] = ids[h];
        have_prev = true;
        Lprev = Lcur;
        buf ^= 1;
    }
}

}  // namespace zoe_cuda
