// sw_score_long.cuh -- score-only local alignment for long streamed sequences (rows > 1024), sm_100a.
//
// Same recurrence and packed DPX arithmetic as sw_score.cuh (zoe: sw_simd_score,
// src/alignment/sw/striped.rs:65-142), for the ONT-read-vs-genome shape (BASELINE config 4): one warp
// owns a task (two sequences packed in the 16-bit halves), the rows are cut into chunks of up to
// 32 lanes x K rows that the warp sweeps one after the other over all columns; the H / E values leaving
// a chunk's last row are parked in a per-warp boundary row in global memory (8 bytes per column,
// L2-resident) and picked up as the top boundary of the next chunk:
//     * bottom boundary: lane 31 stores (H, E) of its last row, one 8-byte store per column (E = the true gap state
//       of sw_score.cuh; the next chunk's lane 0 takes it as its incoming E);
//     * top boundary: all lanes prefetch the next 32 columns with one coalesced 256-byte load, and
//       lane 0 receives its column's entry by __shfl_sync -- the load latency never sits on the systolic
//       critical path.
// The last (partial) chunk only executes the 4-row blocks it needs (a warp-uniform branch), so the
// padding waste is < 128 rows per task.  Tasks are sorted longest-first on the host and handed out through
// an atomic queue, so warps stay balanced although lengths vary 5x.
#pragma once
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>

#include "sw_score.cuh"

namespace zoe_cuda {

struct LongParams {
    ScoreParams s;           // s.task_ids is required (length-sorted sequence ids), s.n_rseq = list length
    uint2 *boundary;         // [warp slots][max_L]
    uint32_t max_L;
    unsigned int *queue;     // dynamic task counter (zeroed before launch)
};

// Lane skew of this kernel.  Measured on cfg 4 (20k reads): skew 1 = 5.79 TCUPS, skew 2 = 5.57 -- unlike the two-stream
// score kernel, the extra pending registers cost more here than the hidden shuffle latency gains.
constexpr int kSkewLong = 1;

template <int K, bool PACKED>
__global__ void __launch_bounds__(512) sw_score_long_kernel(const LongParams lp) {
    using O = Ops<PACKED>;
    const ScoreParams &p = lp.s;
    constexpr int G = 32;
    constexpr int K4 = K / 4;
    static_assert(K % 4 == 0, "K must be a multiple of 4");
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(16) uint8_t smem[];

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int warps_per_block = blockDim.x >> 5;

    const int tab_bytes = p.n_csym * K4 * G * 16;
    uint4 *tab = reinterpret_cast<uint4 *>(smem + (size_t)warp * tab_bytes);
    uint8_t *s_lut = smem + (size_t)warps_per_block * tab_bytes;
    int8_t *s_wk = reinterpret_cast<int8_t *>(s_lut + 256);
    uint8_t *s_cc = reinterpret_cast<uint8_t *>(s_wk) + ((p.n_csym * p.S + 15) & ~15);
    for (int i = tid; i < 256; i += blockDim.x) s_lut[i] = p.lut[i];
    for (int i = tid; i < p.n_csym * p.S; i += blockDim.x) s_wk[i] = p.wk[i];
    if (p.cols_in_smem) stage_with_tma(s_cc, p.ccodes, p.ccodes_bytes);  // one TMA bulk copy per CTA
    __syncthreads();
    const uint8_t *cc = p.cols_in_smem ? s_cc : p.ccodes;

    uint32_t neg_go = O::splat(-p.go), neg_ge = O::splat(-p.ge);
    // loop invariants kept opaque (no rematerialisation in the hot loop); table offset as a 32-bit shared offset
    uint32_t tab_lane_off = (uint32_t)warp * (uint32_t)tab_bytes + (uint32_t)lane * 16u;
    uint32_t nz = lane != 0 ? 1u : 0u;  // lane 0 takes its inputs from the previous chunk's boundary row instead
    asm volatile("" : "+r"(neg_go), "+r"(neg_ge), "+r"(tab_lane_off), "+r"(nz));
    uint2 *bnd = lp.boundary + (size_t)(blockIdx.x * warps_per_block + warp) * lp.max_L;

    for (;;) {
        uint32_t task = 0;
        if (lane == 0) task = atomicAdd(lp.queue, 1u);
        task = __shfl_sync(FULL, task, 0);
        if (task >= p.n_tasks) break;

        uint32_t id_lo, id_hi = 0xffffffffu;
        if (PACKED) {
            id_lo = p.task_ids[2 * task];
            if (2 * task + 1 < p.n_rseq) id_hi = p.task_ids[2 * task + 1];
        } else {
            id_lo = p.task_ids[task];
        }
        const uint64_t off_lo = p.roff[id_lo];
        const int len_lo = (int)(p.roff[id_lo + 1] - off_lo);
        uint64_t off_hi = 0;
        int len_hi = 0;
        if (PACKED && id_hi != 0xffffffffu) {
            off_hi = p.roff[id_hi];
            len_hi = (int)(p.roff[id_hi + 1] - off_hi);
        }
        const int nmax = max(len_lo, len_hi);
        const int R = G * K;
        const int nchunks = max(1, (nmax + R - 1) / R);

        for (uint32_t cj = 0; cj < p.n_cseq; ++cj) {
            const uint32_t c0 = p.coff[cj];
            const int L = (int)(p.coff[cj + 1] - c0);
            const uint8_t *cs = cc + c0;
            const uint8_t *scs = s_cc + c0;  // the same codes through a pointer known to be shared memory
            uint32_t best = 0;

            for (int ch = 0; ch < nchunks; ++ch) {
                const int row0 = ch * R;
                const int rows_left = nmax - row0;
                const int k4_eff = min(K4, max(1, (rows_left + 4 * G - 1) / (4 * G)));
                const int k_eff = 4 * k4_eff;
                const bool has_top = ch > 0, has_bottom = ch + 1 < nchunks;

                // ---- score table of this chunk: lane l owns rows row0 + l*k_eff + [0, k_eff) ----
                __syncwarp();
                for (int s = 0; s < p.n_csym; ++s) {
                    const int8_t *wrow = s_wk + s * p.S;
                    for (int i4 = 0; i4 < k4_eff; ++i4) {
                        uint32_t w[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int r = row0 + lane * k_eff + i4 * 4 + q;
                            int wl = kPadWeight, wh = kPadWeight;
                            if (r < len_lo) wl = wrow[s_lut[p.rseq[off_lo + r]]];
                            if (PACKED && r < len_hi) wh = wrow[s_lut[p.rseq[off_hi + r]]];
                            w[q] = PACKED ? ((uint32_t)(wl & 0xffff) | ((uint32_t)(wh & 0xffff) << 16)) : (uint32_t)wl;
                        }
                        tab[(s * K4 + i4) * G + lane] = make_uint4(w[0], w[1], w[2], w[3]);
                    }
                }
                __syncwarp();

                // H in two register sets (ping-pong by step parity): no register moves for the diagonal
                uint32_t H[2][K], F[K];
#pragma unroll
                for (int i = 0; i < K; ++i) {
                    H[0][i] = H[1][i] = 0;
                    F[i] = 0;
                }
                uint32_t h_last = 0, e_out = 0, h_up_prev = 0;
                uint2 cur = make_uint2(0, 0), nxt = make_uint2(0, 0);
                if (has_top && lane < L) cur = __ldcg(bnd + lane);
                // lane skew of 2 (as in sw_score.cuh): what a lane needs from the lane above was produced two steps
                // earlier and shuffled during the previous step, so consecutive steps are independent chains
                uint32_t pend_h = 0, pend_e = 0;
                const int nsteps = L + kSkewLong * (G - 1);
                const uint32_t top_on = has_top ? 1u - nz : 0u;  // 1 on lane 0 of a chunk that has a chunk above it

                // one column: FULLK = all K rows (a full chunk), else only the first k4_eff 4-row blocks
                auto column = [&](auto parity, auto fullk, const int j, const uint32_t h_in, const uint32_t e_in, const uint32_t code) {
                    constexpr int PO = decltype(parity)::value, PN = 1 - PO;
                    constexpr bool FULLK = decltype(fullk)::value;
                    const uint4 *tp = reinterpret_cast<const uint4 *>(smem + tab_lane_off + code * (uint32_t)(K4 * G * 16));
                    uint32_t diag = h_up_prev;
                    uint32_t E = e_in;
#pragma unroll
                    for (int i4 = 0; i4 < K4; ++i4) {
                        if (FULLK || i4 < k4_eff) {
                            const uint4 w4 = tp[i4 * G];
                            const uint32_t w[4] = {w4.x, w4.y, w4.z, w4.w};
                            uint32_t hp = 0;
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                const int i = i4 * 4 + q;
                                // the recurrence of ZOE_SCORE_ROW (sw_score.cuh)
                                const uint32_t dW = O::add(diag, w[q]);
                                const uint32_t Hn = O::max3z(dW, E, F[i]);
                                const uint32_t Hg = O::add(Hn, neg_go);
                                diag = H[PO][i];
                                E = O::addmax(E, neg_ge, Hg);
                                F[i] = O::addmax(F[i], neg_ge, Hg);
                                H[PN][i] = Hn;
                                if (q & 1)
                                    best = O::max3(best, dW, hp);
                                else
                                    hp = dW;
                            }
                            h_last = H[PN][i4 * 4 + 3];
                        }
                    }
                    e_out = E;
                    if (has_bottom && lane == G - 1) bnd[j] = make_uint2(h_last, e_out);
                };
                // inputs of this step: from the lane above, or (lane 0) from the boundary row of the chunk above
                auto inputs = [&](const int step, uint32_t &h_in, uint32_t &e_in) {
                    if (has_top && (step & 31) == 0) {
                        const int idx = step + 32 + lane;
                        nxt = (idx < L) ? __ldcg(bnd + idx) : make_uint2(0, 0);
                    }
                    const uint32_t h_sh = __shfl_up_sync(FULL, h_last, 1), e_sh = __shfl_up_sync(FULL, e_out, 1);
                    const uint32_t h_top = __shfl_sync(FULL, cur.x, step & 31), e_top = __shfl_sync(FULL, cur.y, step & 31);
                    if (kSkewLong == 1) {
                        h_in = h_sh * nz + h_top * top_on;
                        e_in = e_sh * nz + e_top * top_on;
                    } else {  // lane 0's boundary entry belongs to THIS step's column (lane 0: j == step)
                        h_in = pend_h * nz + h_top * top_on;
                        e_in = pend_e * nz + e_top * top_on;
                        pend_h = h_sh;
                        pend_e = e_sh;
                    }
                    if ((step & 31) == 31) cur = nxt;
                };
                using P0 = std::integral_constant<int, 0>;
                using P1 = std::integral_constant<int, 1>;
                auto generic_step = [&](auto parity, const int step) {
                    uint32_t h_in, e_in;
                    inputs(step, h_in, e_in);
                    const int j = step - kSkewLong * lane;
                    if (j >= 0 && j < L) column(parity, std::false_type{}, j, h_in, e_in, (uint32_t)cs[j]);
                    h_up_prev = h_in;
                };
                // a steady step inside a 32-step block: inputs without the per-step prefetch / hand-over tests
                auto block_step = [&](auto parity, const int step, const int k) {
                    const uint32_t h_sh = __shfl_up_sync(FULL, h_last, 1), e_sh = __shfl_up_sync(FULL, e_out, 1);
                    const uint32_t h_top = __shfl_sync(FULL, cur.x, k), e_top = __shfl_sync(FULL, cur.y, k);
                    const uint32_t h_in = h_sh * nz + h_top * top_on, e_in = e_sh * nz + e_top * top_on;
                    const int j = step - kSkewLong * lane;
                    column(parity, std::true_type{}, j, h_in, e_in, (uint32_t)scs[j]);
                    h_up_prev = h_in;
                };
                auto steady_step = [&](auto parity, auto fullk, const int step) {
                    uint32_t h_in, e_in;
                    inputs(step, h_in, e_in);
                    const int j = step - kSkewLong * lane;
                    column(parity, fullk, j, h_in, e_in, (uint32_t)scs[j]);
                    h_up_prev = h_in;
                };

                // segments: ramp [0, G) generic; steady while step + 1 < L (every lane has a column); tail generic
                const bool fast = p.cols_in_smem != 0;
                const bool fullk = k4_eff == K4;
                int seg_end[3] = {fast ? min(kSkewLong * G, nsteps) : nsteps, L - 1, nsteps};
                int step = 0;
#pragma unroll 1
                for (int seg = 0; seg < 3; ++seg) {
                    const int end = seg_end[seg];
                    if (seg == 1) {
                        if (fast && fullk) {
                            // whole blocks of 32 steps (the steady segment starts at step 32): the boundary-row prefetch
                            // and the hand-over cur <- nxt happen once per block, outside the two-step body, instead of
                            // being tested in every step (5.04 -> 4.9 ALU-pipe instructions per cell pair)
                            for (; step + 32 <= end; step += 32) {
                                if (has_top) {
                                    const int idx = step + 32 + lane;
                                    nxt = (idx < L) ? __ldcg(bnd + idx) : make_uint2(0, 0);
                                }
#pragma unroll 1
                                for (int k = 0; k < 32; k += 2) {
                                    block_step(P0{}, step + k, k);
                                    block_step(P1{}, step + k + 1, k + 1);
                                }
                                cur = nxt;
                            }
                            for (; step < end; step += 2) {
                                steady_step(P0{}, std::true_type{}, step);
                                steady_step(P1{}, std::true_type{}, step + 1);
                            }
                        } else if (fast) {
                            for (; step < end; step += 2) {
                                steady_step(P0{}, std::false_type{}, step);
                                steady_step(P1{}, std::false_type{}, step + 1);
                            }
                        }
                    } else {
                        for (; step < end; ++step) {
                            if (step & 1)
                                generic_step(P1{}, step);
                            else
                                generic_step(P0{}, step);
                        }
                    }
                }
                __syncwarp();
            }

#pragma unroll
            for (int d = 16; d >= 1; d >>= 1) best = O::max2(best, __shfl_xor_sync(FULL, best, d));
            if (lane == 0) {
                if (PACKED) {
                    int b_lo = (int)(int16_t)(best & 0xffff), b_hi = (int)(int16_t)(best >> 16);
                    p.best[(size_t)id_lo * p.n_cseq + cj] = (b_lo >= p.ovf_thresh) ? -1 : b_lo;
                    if (id_hi != 0xffffffffu) p.best[(size_t)id_hi * p.n_cseq + cj] = (b_hi >= p.ovf_thresh) ? -1 : b_hi;
                } else {
                    p.best[(size_t)id_lo * p.n_cseq + cj] = (int)best;
                }
            }
        }
    }
}

}  // namespace zoe_cuda
