// sw_exact_fast.cuh -- throughput version of the literal striped emulation (sm_100a).
//
// Same contract as sw_align_exact_kernel (sw_align.cuh): zoe's sw_simd_align (src/alignment/sw/striped.rs:449-598) run
// at the lane count N of the pair's score tier, flag for flag, so that CIGAR tie-breaks that depend on the striped lane
// layout come out as zoe's.  The old kernel spends 2-5 ms per 150 x 1704 pair (one warp per pair, every access a
// dependent load, flags of the whole matrix through global memory); a workload with a few per cent of tie hazards
// (small weights, cheap gaps) then pays more for the literal pairs than for everything else.  Differences here:
//
//   * thread = SIMD lane, but a warp carries 32 / N pairs (N = 16: two, N = 8: four), and a CTA up to 24 pairs, each
//     with its H row, E row, current flag row (and, for multi-sequence panels, its profiled symbol indices) in shared
//     memory as 16-bit / 8-bit values: 6 bytes per profiled residue instead of 18;
//   * one H buffer instead of zoe's load / store pair (row r-1's value is read into a register one step before it is
//     overwritten), no max_row copy: the end cell is known from the canonical pass (H is layout independent), or, for
//     the pairs that never had one (packed overflow), tracked per row;
//   * the main loop is software pipelined: the loads of vector v+1 are issued before the stores of vector v;
//   * only the flags the walk can reach leave the SM: rows 0..r_end, columns [c_lo, c_end] with c_lo from the score
//     bound on column-only moves (the same bound the window pipeline uses) -- about 150 x 170 bytes instead of 150 x 1704;
//   * the walk runs in a second kernel, one thread per pair, so its dependent loads overlap across thousands of pairs
//     instead of stalling a DP warp.
//
// Values are true (un-offset) scores: zoe keeps x + T::MIN and saturates, which is a clamp at 0 here; saturation at MAX
// cannot happen because the tier was chosen from the exact score.  Tiers 8 and 16 only (values < 65535 fit the 16-bit
// rows) with N <= 32; everything else stays with sw_align_exact_kernel.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "sw_align.cuh"

namespace zoe_cuda {

constexpr uint32_t kEndUnknown = 0x80000000u;  // hazard_list entry flag: the pair has no exact end cell yet

struct ExactFastParams {
    const uint32_t *list;         // positions into hazard_list of this launch's pairs
    uint32_t list_count;          // pairs of this round
    const uint32_t *hazard_list;  // global pair id | kEndUnknown
    const uint8_t *rseq;
    const uint64_t *roff;
    const uint8_t *pbytes;        // profiled sequences, raw bytes
    const uint32_t *coff;
    uint32_t n_cseq;
    const int8_t *weights;        // S*S zoe weights[ref_idx][query_idx]
    int S;
    const uint8_t *lut;
    int go, ge;                   // positive
    int maxw;
    int N;                        // SIMD lanes of this tier (power of two, <= 32)
    uint32_t vcap;                // shared-memory row capacity per pair (elements), >= nv * N for every profiled sequence
    int invert;
    AlignEnd *ends;               // in: exact end cell (known-end launches); out: exact end cell (FULL launches)
    const uint32_t *score_in;     // exact score (decides the tier; checked against the recomputed value)
    uint8_t *fbuf;                // [round slot][fcap] flag bytes, row stride wcap
    uint64_t fcap;
    uint32_t wcap;
    // walk outputs (same arrays as TraceParams)
    uint32_t *ref_start, *ref_end, *query_start, *query_end;
    uint32_t *cig_scratch;        // [hazard_list position][cig_cap]
    uint32_t *cig_count;
    uint32_t cig_cap;
    unsigned long long *counters; // [6] cigar overflow, [7] score mismatch (internal check)
    uint32_t *retry_list;         // walks that left their flag window go back to sw_align_exact_kernel (hazard_list positions)
    uint32_t *retry_count;
};

// Rows and columns of flags the walk of a pair can reach.  With the end cell known: rows 0..r_end; the walk follows
// one alignment of score S over n_r = r_end + 1 rows, whose column-only moves I satisfy
// S <= n_r * maxw - go - (I - 1) * ge (one gap run is the cheapest way to spend them), so it stays right of
// c_end + 1 - (n_r + I + 1).  Unknown end: everything.
__host__ __device__ inline void exact_window(bool end_known, uint32_t r_end, uint32_t c_end, uint32_t score, uint32_t n,
                                             uint32_t m, int maxw, int go, int ge, uint32_t &n_rows, uint32_t &c_lo,
                                             uint32_t &width) {
    if (!end_known) {
        n_rows = n;
        c_lo = 0;
        width = m;
        return;
    }
    n_rows = r_end + 1;
    c_lo = 0;
    if (ge > 0) {
        const long long num = (long long)n_rows * maxw - go - (long long)score;
        const long long imax = num >= 0 ? 1 + num / ge : 0;
        const long long need = (long long)n_rows + imax + 1;
        if ((long long)c_end + 1 > need) c_lo = (uint32_t)((long long)c_end + 1 - need);
    }
    width = c_end - c_lo + 1;
}

// Shared memory per CTA: [groups x (H u16[vcap], E u16[vcap], flags u8[vcap], (pidx u8[vcap]), F per lane i32[N])]
//                        [shared pidx u8[vcap] when n_cseq == 1][weights (S+1) x (S+1) i8][lut 256]
// The group stride is 2N bytes past a multiple of 128, so the 32 / N groups of a warp hit disjoint banks.
__host__ __device__ inline size_t exact_fast_group_bytes(uint32_t vcap, bool pidx_shared, int N) {
    return (((size_t)vcap * (pidx_shared ? 5 : 6) + 4 + 4 * (size_t)N + 127) & ~(size_t)127) + (N < 32 ? 2 * (size_t)N : 0);
}
__host__ __device__ inline size_t exact_fast_fixed_bytes(uint32_t vcap, int S, bool pidx_shared) {
    return (pidx_shared ? (size_t)vcap : 0) + (size_t)((S + 1) * (S + 1) + 15) / 16 * 16 + 256;
}

// Lane-major row layout: element (vector v, SIMD lane l) of a row lives at l * nvp + v, nvp = vectors per lane padded to
// twice an odd number -- the lanes of a warp then hit distinct banks in the main loop (thread = lane, same v), and one
// lane's vectors are contiguous for the lazy-F pass (threads = consecutive v of ONE lane).
__host__ __device__ inline int exact_fast_nvp(int nv) {
    int p = nv + (nv & 1);
    if (((p >> 1) & 1) == 0) p += 2;
    return p;
}

// N (SIMD lanes of the tier: 8, 16 or 32) is a template parameter: index arithmetic by shifts, constant shuffle widths.
template <bool FULL, int N>
__global__ void __launch_bounds__(512) sw_exact_fast_kernel(const ExactFastParams x) {
    extern __shared__ __align__(16) uint8_t xs[];
    constexpr unsigned ALL = 0xffffffffu;
    const int lig = threadIdx.x & (N - 1);
    const int group = threadIdx.x / N, groups = blockDim.x / N;
    const int lane = threadIdx.x & 31;
    const int gbase_lane = lane & ~(N - 1);  // first warp lane of this group
    const unsigned gmask = (N == 32 ? ALL : ((1u << N) - 1u)) << gbase_lane;
    const bool pidx_shared = x.n_cseq == 1;
    const uint32_t vcap = x.vcap;
    const int S1 = x.S + 1;

    uint8_t *gbase = xs + (size_t)group * exact_fast_group_bytes(vcap, pidx_shared, N);
    uint16_t *hrow = reinterpret_cast<uint16_t *>(gbase);
    uint16_t *es = hrow + vcap;
    uint8_t *frow = reinterpret_cast<uint8_t *>(es + vcap);
    uint8_t *fixed = xs + (size_t)groups * exact_fast_group_bytes(vcap, pidx_shared, N);
    uint8_t *pidx = pidx_shared ? fixed : frow + vcap;
    int *fsh = reinterpret_cast<int *>(gbase + (((size_t)vcap * (pidx_shared ? 5 : 6) + 3) & ~(size_t)3));  // lazy-F: F per lane
    int8_t *wtab = reinterpret_cast<int8_t *>(fixed + (pidx_shared ? vcap : 0));
    uint8_t *s_lut = reinterpret_cast<uint8_t *>(wtab) + ((S1 * S1 + 15) / 16) * 16;

    // weights with one extra all-zero row / column: the profile pads residues beyond the sequence with weight 0
    for (int i = threadIdx.x; i < S1 * S1; i += blockDim.x) {
        const int a = i / S1, b = i % S1;
        wtab[i] = (a < x.S && b < x.S) ? x.weights[a * x.S + b] : 0;
    }
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_lut[i] = x.lut[i];
    if (pidx_shared) {  // one profiled sequence: its striped symbol indices are the same for every pair of the CTA
        const int m = (int)(x.coff[1] - x.coff[0]);
        const int nv = (m + N - 1) / N, nvp = exact_fast_nvp(nv);
        for (int i = threadIdx.x; i < nvp * N; i += blockDim.x) {
            const int l = i / nvp, v = i % nvp, c = l * nv + v;
            pidx[i] = (v < nv && c < m) ? x.lut[x.pbytes[x.coff[0] + c]] : (uint8_t)x.S;
        }
    }
    __syncthreads();

    const uint32_t total_groups = gridDim.x * groups;
    const uint32_t trips = (x.list_count + total_groups - 1) / total_groups;
    const uint32_t first = blockIdx.x * groups + group;

    for (uint32_t trip = 0; trip < trips; ++trip) {
        const uint32_t slot = first + trip * total_groups;  // round slot = index into this round's list
        const bool valid = slot < x.list_count;
        uint32_t pos = 0, gid = 0;
        int n = 0, m = 0, nv = 0;
        const uint8_t *R = x.rseq, *P = x.pbytes;
        uint32_t want = 0, r_end_in = 0, c_end_in = 0;
        if (valid) {
            pos = x.list[slot];
            gid = x.hazard_list[pos] & ~kEndUnknown;
            const uint32_t seq = gid / x.n_cseq, cj = gid % x.n_cseq;
            R = x.rseq + x.roff[seq];
            n = (int)(x.roff[seq + 1] - x.roff[seq]);
            P = x.pbytes + x.coff[cj];
            m = (int)(x.coff[cj + 1] - x.coff[cj]);
            nv = (m + N - 1) / N;
            want = x.score_in[gid];
            if (!FULL) {
                const AlignEnd e = x.ends[gid];
                r_end_in = e.r_end;
                c_end_in = e.c_end;
            }
        }
        const int nvp = exact_fast_nvp(nv);
        uint32_t n_rows, c_lo, width;
        exact_window(!FULL, r_end_in, c_end_in, want, (uint32_t)n, (uint32_t)m, x.maxw, x.go, x.ge, n_rows, c_lo, width);
        if (!valid) n_rows = 0;
        // loop bounds are warp-uniform (the groups of a warp advance in lock step, idle where they have nothing to do)
        const int rows_w = (int)__reduce_max_sync(ALL, n_rows);
        const int nv_w = (int)__reduce_max_sync(ALL, (unsigned)nv);

        if (valid)
            for (int i = lig; i < nvp * N; i += N) {
                hrow[i] = 0;
                es[i] = 0;
                if (!pidx_shared) {
                    const int l = i / nvp, v = i % nvp, c = l * nv + v;
                    pidx[i] = (v < nv && c < m) ? s_lut[P[c]] : (uint8_t)x.S;
                }
            }
        // first window column of this lane and its striped coordinates (the same for every row)
        uint8_t *fdst = x.fbuf + (size_t)slot * x.fcap;
        const int t0 = lig;  // window offsets t0, t0 + N, ...
        int pv0 = 0, pl0 = 0;
        if (valid && nv > 0) {
            const int c0 = (int)c_lo + t0;
            pl0 = c0 / nv;
            pv0 = c0 - pl0 * nv;
        }
        __syncwarp();

        int best = 0, r_best = n > 0 ? n - 1 : 0, c_best = m > 0 ? m - 1 : 0;  // FULL: zoe's defaults (striped.rs:476, 573)
        const int go = x.go, ge = x.ge;
        const int mybase = lig * nvp;  // this lane's segment of every row

        for (int r = 0; r < rows_w; ++r) {
            const bool row_on = r < (int)n_rows;
            const int8_t *wrow = wtab + (row_on ? (int)s_lut[R[r]] : x.S) * S1;
            // H = store[nv-1].shift_elements_right(MIN): the final H of row r-1 at column l*nv - 1
            int Hd = (row_on && lig > 0) ? (int)hrow[mybase - nvp + nv - 1] : 0;
            __syncwarp();
            int F = 0, rowmax = 0;
            // software pipeline: the symbol index is fetched two vectors ahead, weight / E / previous H one vector ahead,
            // all before vector v is stored -- no load sits on the F -> H -> F chain
            int w_n = 0, E_n = 0, Hp_n = 0, pi_n = x.S;
            if (row_on && nv > 0) {
                w_n = wrow[pidx[mybase]];
                E_n = es[mybase];
                Hp_n = hrow[mybase];
                pi_n = pidx[mybase + 1];  // padded: always readable
            }
#pragma unroll 4
            for (int v = 0; v < nv_w; ++v) {
                const bool on = row_on && v < nv;
                const int w = w_n, E = E_n, Hp = Hp_n;
                const int idx = mybase + v;
                if (row_on && v + 1 < nv) {
                    w_n = wrow[pi_n];
                    E_n = es[idx + 1];
                    Hp_n = hrow[idx + 1];
                    pi_n = pidx[idx + 2];  // nvp >= nv + 1 keeps idx + 2 inside the lane's padded segment
                }
                if (on) {
                    const int h = __vimax3_s32(Hd + w, E, F);             // saturating_add floors at MIN = 0 <= E, F
                    const int ho = __viaddmax_s32(h, -go, 0);
                    const int E2 = __viaddmax_s32(E, -ge, ho);
                    const int F2 = __viaddmax_s32(F, -ge, ho);
                    uint32_t fl = (uint32_t)(E == h) | ((uint32_t)(F == h) << 2) | ((uint32_t)(E2 > ho) << 1) |
                                  ((uint32_t)(F2 > ho) << 3);
                    if (h == 0) fl = 16u;
                    rowmax = max(rowmax, h);
                    hrow[idx] = (uint16_t)h;
                    es[idx] = (uint16_t)E2;
                    frow[idx] = (uint8_t)fl;
                    F = F2;
                    Hd = Hp;
                }
            }
            __syncwarp();
            // ---- lazy-F (striped.rs:528-553).  Within a pass, lane L's F only decays: F_L(v) = max(F_L(0) - v * ge, 0),
            //      independent of H, and every vector is visited once.  So every (lane, vector) test
            //      "F_L(v) > H - gap_open" of a pass is known up front, a lane whose F enters the pass at 0 can never
            //      pass it, and the only coupling is the stopping rule: the pass ends at the first vector where NO lane
            //      passes.  The work of a pass is therefore spread over the group's threads by VECTOR (thread t takes
            //      v = t, t + N, ...) for the few lanes with F > 0 only -- typically one or two of N -- instead of every
            //      lane walking every vector:  1) test, 2) stop = first vector nobody passes (min over threads),
            //      3) update the cells before `stop` that zoe would change.  A cell changes iff F >= H there:
            //      H = max(H, F); LEFT corrected / set where F == H; LEFT_EXT where F - ge > H - go; STOP where H == MIN. ----
            {
                bool live = row_on && nv > 0;
                int pass = 0;
                while (__any_sync(ALL, live)) {
                    // F = F.shift_elements_right(MIN); every thread of the group can read every lane's F
                    const int Fs = __shfl_up_sync(ALL, F, 1, N);
                    const int Fl = lig == 0 ? 0 : Fs;
                    fsh[lig] = Fl;
                    const unsigned act = (__ballot_sync(ALL, live && Fl > 0) & gmask) >> gbase_lane;  // lanes that can still improve cells
                    __syncwarp();
                    // 1) + 2) own vectors in ascending order: the first one where no active lane passes the test
                    int stop = nv;
                    if (live) {
                        for (int v = lig; v < nv; v += N) {
                            bool hit = false;
                            for (unsigned a = act; a && !hit; a &= a - 1) {
                                const int L = __ffs(a) - 1;
                                hit = max(fsh[L] - v * ge, 0) > __viaddmax_s32((int)hrow[L * nvp + v], -go, 0);
                            }
                            if (!hit) {
                                stop = v;
                                break;
                            }
                        }
                    }
                    for (int d = N / 2; d >= 1; d >>= 1) stop = min(stop, __shfl_xor_sync(ALL, stop, d, N));
                    // 3) update the visited cells of the active lanes
                    if (live) {
                        for (unsigned a = act; a; a &= a - 1) {
                            const int L = __ffs(a) - 1;
                            const int FL = fsh[L];
                            const int lb = L * nvp;
                            for (int v = lig; v < stop; v += N) {
                                const int Fk = max(FL - v * ge, 0);
                                const int h = hrow[lb + v];
                                if (Fk >= h) {
                                    uint32_t fl = frow[lb + v];
                                    fl = (fl & 2u) | 4u;  // simd_correct_and_set_left (F == max(H, F))
                                    if (max(Fk - ge, 0) > __viaddmax_s32(Fk, -go, 0)) fl |= 8u;
                                    if (Fk == 0) fl = 16u;
                                    hrow[lb + v] = (uint16_t)Fk;
                                    frow[lb + v] = (uint8_t)fl;
                                } else if (max(Fk - ge, 0) > __viaddmax_s32(h, -go, 0)) {
                                    frow[lb + v] |= 8u;   // F < H, but F - ge still beats H - go: LEFT_EXT
                                }
                            }
                        }
                    }
                    __syncwarp();
                    if (live) {
                        if (stop < nv || act == 0) {
                            live = false;  // break 'lazy_f (no active lane: the very first test fails)
                        } else {
                            F = max(Fl - nv * ge, 0);  // what this pass leaves; the next pass shifts it
                            if (++pass == N) live = false;
                        }
                    }
                }
            }
            __syncwarp();
            // ---- row maximum; FULL: best cell so far = (max H, min r, min c) (striped.rs:555-583) ----
            int rb = rowmax;
            if (FULL || __any_sync(ALL, row_on && r == (int)r_end_in))
                for (int d = N / 2; d >= 1; d >>= 1) rb = max(rb, __shfl_xor_sync(ALL, rb, d, N));
            if (FULL) {
                const bool improved = row_on && rb > best;
                if (__any_sync(ALL, improved)) {
                    int cmin = 0x7fffffff;
                    if (improved) {
                        for (int v = 0; v < nv; ++v)
                            if ((int)hrow[mybase + v] == rb) {
                                const int c = lig * nv + v;
                                if (c < m) cmin = c;
                                break;
                            }
                    }
                    for (int d = N / 2; d >= 1; d >>= 1) cmin = min(cmin, __shfl_xor_sync(ALL, cmin, d, N));
                    if (improved) {
                        best = rb;
                        r_best = r;
                        c_best = cmin != 0x7fffffff ? cmin : m - 1;
                    }
                }
            } else if (row_on && r == (int)r_end_in && lig == 0) {
                const int v = (int)c_end_in % nv, l = (int)c_end_in / nv;
                if ((uint32_t)hrow[l * nvp + v] != want || (uint32_t)rb != want) atomicAdd(&x.counters[7], 1ULL);
            }
            // ---- publish the reachable part of the finished flag row ----
            if (row_on) {
                uint8_t *dst = fdst + (size_t)r * x.wcap;
                int pv = pv0, pl = pl0;
#pragma unroll 4
                for (int t = t0; t < (int)width; t += N) {
                    dst[t] = frow[pl * nvp + pv];
                    pv += N;
                    while (pv >= nv) {
                        pv -= nv;
                        ++pl;
                    }
                }
            }
            __syncwarp();
        }
        if (FULL && valid && lig == 0) {
            if ((uint32_t)best != want) atomicAdd(&x.counters[7], 1ULL);
            AlignEnd e;
            e.best = best;
            e.r_end = (uint32_t)r_best;
            e.c_end = (uint32_t)c_best;
            e.aux = kNotBucketed;
            x.ends[gid] = e;
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// One CTA per pair: the latency version, for short literal lists (a lone hazard pair in a 125k-read shard kept the whole
// GPU waiting 1.9 ms for one warp).  Warp L owns SIMD lane L; its nv vectors are spread over the warp's 32 threads in
// chunks of 32 consecutive vectors.  The only dependency inside a lane's main pass, F, is a max-plus prefix scan:
//     F(v) = max(0, max_{v' < v} (sat(H0(v') - go) - (v - v' - 1) * ge)),   H0 = max(Hdiag + w, E, 0)
// (a gap opened from a cell that F itself produced never beats extending that gap: gap_open >= gap_extend), so a row
// costs a few five-step warp scans instead of nv serial steps.  H rows are double buffered (the main pass reads row r-1,
// writes row r); the lazy-F pass is the cell-parallel one of sw_exact_fast_kernel with the stopping rule taken over the
// whole CTA.  Values and flags are those of the serial loops; the same walk kernel follows.  End cell known only.
// Shared memory (lane-major, as above): H x 2 and E as u16, flags, symbol indices and "some lane passes here" marks as
// u8, the F leaving every lane, two control words, weights, byte -> symbol map.
// ---------------------------------------------------------------------------------------------
__host__ __device__ inline size_t exact_cta_smem_bytes(uint32_t vcap, int S, int N) {
    return (((size_t)vcap * 9 + 3) & ~(size_t)3) + 4 * (size_t)N + 64 + (size_t)((S + 1) * (S + 1) + 15) / 16 * 16 + 256;
}

template <int N>
__global__ void __launch_bounds__(N * 32) sw_exact_cta_kernel(const ExactFastParams x) {
    extern __shared__ __align__(16) uint8_t xs[];
    constexpr unsigned ALL = 0xffffffffu;
    constexpr int NEG = -(1 << 29);
    const int tid = threadIdx.x, lane = tid & 31, L = tid >> 5;  // L = the SIMD lane this warp owns
    const uint32_t vcap = x.vcap;
    const int S1 = x.S + 1;
    uint16_t *hbuf0 = reinterpret_cast<uint16_t *>(xs);
    uint16_t *hbuf1 = hbuf0 + vcap;
    uint16_t *es = hbuf1 + vcap;
    uint8_t *frow = reinterpret_cast<uint8_t *>(es + vcap);
    uint8_t *pidx = frow + vcap;
    uint8_t *anyhit = pidx + vcap;
    int *fsh = reinterpret_cast<int *>(xs + (((size_t)vcap * 9 + 3) & ~(size_t)3));  // F leaving each lane's segment
    int *ctl = fsh + N;                                                               // [0] stop, [1] some lane is active
    int8_t *wtab = reinterpret_cast<int8_t *>(ctl + 16);
    uint8_t *s_lut = reinterpret_cast<uint8_t *>(wtab) + ((S1 * S1 + 15) / 16) * 16;
    for (int i = tid; i < S1 * S1; i += blockDim.x) {
        const int a = i / S1, b = i % S1;
        wtab[i] = (a < x.S && b < x.S) ? x.weights[a * x.S + b] : 0;
    }
    for (int i = tid; i < 256; i += blockDim.x) s_lut[i] = x.lut[i];
    __syncthreads();

    for (uint32_t slot = blockIdx.x; slot < x.list_count; slot += gridDim.x) {
        const uint32_t pos = x.list[slot];
        const uint32_t gid = x.hazard_list[pos] & ~kEndUnknown;
        const uint32_t seq = gid / x.n_cseq, cj = gid % x.n_cseq;
        const uint8_t *R = x.rseq + x.roff[seq];
        const int n = (int)(x.roff[seq + 1] - x.roff[seq]);
        const uint8_t *P = x.pbytes + x.coff[cj];
        const int m = (int)(x.coff[cj + 1] - x.coff[cj]);
        const int nv = (m + N - 1) / N, nvp = exact_fast_nvp(nv);
        const uint32_t want = x.score_in[gid];
        const AlignEnd e_in = x.ends[gid];
        uint32_t n_rows, c_lo, width;
        exact_window(true, e_in.r_end, e_in.c_end, want, (uint32_t)n, (uint32_t)m, x.maxw, x.go, x.ge, n_rows, c_lo, width);
        __syncthreads();
        for (int i = tid; i < nvp * N; i += blockDim.x) {
            const int l = i / nvp, v = i % nvp, c = l * nv + v;
            hbuf0[i] = 0;
            hbuf1[i] = 0;
            es[i] = 0;
            pidx[i] = (v < nv && c < m) ? s_lut[P[c]] : (uint8_t)x.S;
        }
        __syncthreads();
        uint8_t *fdst = x.fbuf + (size_t)slot * x.fcap;
        const int go = x.go, ge = x.ge;
        const int lb = L * nvp;
        uint16_t *hprev = hbuf0, *hcur = hbuf1;

        for (int r = 0; r < (int)n_rows; ++r) {
            const int8_t *wrow = wtab + (int)s_lut[R[r]] * S1;
            // ---- main pass of lane L: chunks of 32 vectors, F by a max-plus scan ----
            int carry = 0;  // F entering the chunk's first vector (F starts the row at MIN = 0)
            for (int v0 = 0; v0 < nv; v0 += 32) {
                const int v = v0 + lane;
                const bool on = v < nv;
                int h0 = NEG, E = 0;
                if (on) {
                    // H = store[v-1] of row r-1; vector 0 takes the last vector of lane L-1 (shift_elements_right)
                    const int Hd = v > 0 ? (int)hprev[lb + v - 1] : (L > 0 ? (int)hprev[lb - nvp + nv - 1] : 0);
                    E = es[lb + v];
                    h0 = max(max(Hd + (int)wrow[pidx[lb + v]], E), 0);
                }
                int X = on ? max(h0 - go, 0) : NEG;  // what this vector hands to the next one: sat(H0 - go)
#pragma unroll
                for (int sft = 1; sft < 32; sft <<= 1) {
                    const int y = __shfl_up_sync(ALL, X, sft);
                    if (lane >= sft) X = max(X, y - sft * ge);
                }
                const int Xprev = __shfl_up_sync(ALL, X, 1);
                const int F = max(max(lane > 0 ? Xprev : NEG, carry - lane * ge), 0);
                carry = max(max(__shfl_sync(ALL, X, 31), carry - 32 * ge), 0);
                if (on) {
                    const int h = max(h0, F);
                    const int ho = __viaddmax_s32(h, -go, 0);
                    const int E2 = __viaddmax_s32(E, -ge, ho);
                    const int F2 = __viaddmax_s32(F, -ge, ho);
                    uint32_t fl = (uint32_t)(E == h) | ((uint32_t)(F == h) << 2) | ((uint32_t)(E2 > ho) << 1) |
                                  ((uint32_t)(F2 > ho) << 3);
                    if (h == 0) fl = 16u;
                    hcur[lb + v] = (uint16_t)h;
                    es[lb + v] = (uint16_t)E2;
                    frow[lb + v] = (uint8_t)fl;
                    if (v == nv - 1) fsh[L] = F2;  // F leaving the lane's last vector
                }
            }
            __syncthreads();
            // ---- lazy-F (striped.rs:528-553): see sw_exact_fast_kernel; the stopping rule spans the whole CTA ----
            for (int pass = 0; pass < N; ++pass) {
                const int Fl = L > 0 ? fsh[L - 1] : 0;  // F.shift_elements_right(MIN)
                const bool active = Fl > 0;
                for (int i = tid; i < nv; i += blockDim.x) anyhit[i] = 0;
                if (tid == 0) ctl[1] = 0;
                __syncthreads();
                if (active) {
                    if (lane == 0) ctl[1] = 1;
                    for (int v = lane; v < nv; v += 32)
                        if (max(Fl - v * ge, 0) > __viaddmax_s32((int)hcur[lb + v], -go, 0)) anyhit[v] = 1;
                }
                __syncthreads();
                if (ctl[1] == 0) break;  // no lane carries an F: the first test fails (uniform)
                if (L == 0) {            // first vector where no lane passes
                    int stop = nv;
                    for (int v0 = 0; v0 < nv && stop == nv; v0 += 32) {
                        const int v = v0 + lane;
                        const unsigned miss = __ballot_sync(ALL, v < nv && anyhit[v] == 0);
                        if (miss) stop = v0 + __ffs(miss) - 1;
                    }
                    if (lane == 0) ctl[0] = stop;
                }
                __syncthreads();
                const int stop = ctl[0];
                if (active) {
                    for (int v = lane; v < stop; v += 32) {
                        const int Fk = max(Fl - v * ge, 0);
                        const int h = hcur[lb + v];
                        if (Fk >= h) {
                            uint32_t fl = frow[lb + v];
                            fl = (fl & 2u) | 4u;  // simd_correct_and_set_left (F == max(H, F))
                            if (max(Fk - ge, 0) > __viaddmax_s32(Fk, -go, 0)) fl |= 8u;
                            if (Fk == 0) fl = 16u;
                            hcur[lb + v] = (uint16_t)Fk;
                            frow[lb + v] = (uint8_t)fl;
                        } else if (max(Fk - ge, 0) > __viaddmax_s32(h, -go, 0)) {
                            frow[lb + v] |= 8u;  // F < H, but F - ge still beats H - go: LEFT_EXT
                        }
                    }
                }
                __syncthreads();  // every warp has read fsh[L - 1] and ctl
                if (stop < nv) break;
                if (lane == 0) fsh[L] = max(Fl - nv * ge, 0);  // what this pass leaves; the next pass shifts it
                __syncthreads();
            }
            __syncthreads();
            // ---- consistency at the end row, then publish the reachable part of the finished flag row ----
            if (r == (int)e_in.r_end && tid == 0) {
                const int v = (int)e_in.c_end % nv, l = (int)e_in.c_end / nv;
                if ((uint32_t)hcur[l * nvp + v] != want) atomicAdd(&x.counters[7], 1ULL);
            }
            uint8_t *dst = fdst + (size_t)r * x.wcap;
            for (int t = tid; t < (int)width; t += blockDim.x) {
                const int c = (int)c_lo + t, l = c / nv, v = c - l * nv;
                dst[t] = frow[l * nvp + v];
            }
            uint16_t *sw = hprev;
            hprev = hcur;
            hcur = sw;
            __syncthreads();
        }
    }
}

// zoe's walk (backtrack.rs:290-342) over the published flags: one thread per pair of the round.
__global__ void sw_exact_walk_kernel(const ExactFastParams x, int full) {
    const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= x.list_count) return;
    const uint32_t pos = x.list[slot];
    const uint32_t gid = x.hazard_list[pos] & ~kEndUnknown;
    const uint32_t seq = gid / x.n_cseq, cj = gid % x.n_cseq;
    const uint32_t n = (uint32_t)(x.roff[seq + 1] - x.roff[seq]);
    const uint32_t m = x.coff[cj + 1] - x.coff[cj];
    const AlignEnd e = x.ends[gid];
    uint32_t n_rows, c_lo, width;
    exact_window(!full, e.r_end, e.c_end, x.score_in[gid], n, m, x.maxw, x.go, x.ge, n_rows, c_lo, width);
    const uint8_t *fl = x.fbuf + (size_t)slot * x.fcap;
    auto cell = [&](uint32_t rr, uint32_t cc) -> uint32_t { return fl[(size_t)rr * x.wcap + (cc - c_lo)]; };

    CigarBack cg;
    cg.init(x.cig_scratch + (size_t)pos * x.cig_cap, x.cig_cap);
    const uint32_t OP_UP = x.invert ? 1u : 2u, OP_LEFT = x.invert ? 2u : 1u;
    uint32_t r = e.r_end + 1, c = e.c_end + 1;
    const uint32_t r_end1 = r, c_end1 = c;
    cg.push(4u, x.invert ? (n - r_end1) : (m - c_end1));
    uint32_t cur = cell(e.r_end, e.c_end);
    int op = 0;
    bool left_window = false;
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
        if (r == 0 || c == 0) break;  // zoe reads cell(max(r-1,0), max(c-1,0)) and then leaves the loop
        if (c - 1 < c_lo) {
            left_window = true;
            break;
        }
        cur = cell(r - 1, c - 1);
    }
    if (left_window) {  // cannot happen while the score bound holds; kept as a safety net, not as a code path
        x.retry_list[atomicAdd(x.retry_count, 1u)] = pos;
        return;
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

// Splits the literal list by what can run where: [0] tier 8, end known; [1] tier 16, end known; [2] tier 8, end unknown;
// [3] tier 16, end unknown; [4] everything else that needs an alignment (tier 32, lane counts beyond a warp, rows that
// do not fit shared memory) -> sw_align_exact_kernel.  Entries are positions into hazard_list (= the pair's row in the
// literal kernels' CIGAR scratch).  Pairs beyond the widest allowed type need nothing.
struct ExactPartitionParams {
    const uint32_t *hazard_list;
    uint32_t n;
    const uint32_t *score;
    TierPolicy tp;
    int fast8, fast16;   // the fast kernel can take this tier
    uint32_t *lists;     // 5 x n
    uint32_t *counts;    // [5]
};

__global__ void exact_partition_kernel(const ExactPartitionParams q) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= q.n) return;
    const uint32_t ent = q.hazard_list[i];
    const uint32_t gid = ent & ~kEndUnknown;
    const uint8_t tier = tier_for(q.tp, q.score[gid]);
    // score 0: a packed overflow whose exact score fell beyond the widest allowed type (Overflowed, like tier 0)
    if (tier == 0 || q.score[gid] == 0) return;
    int which = 4;
    if (tier == 8 && q.fast8) which = (ent & kEndUnknown) ? 2 : 0;
    if (tier == 16 && q.fast16) which = (ent & kEndUnknown) ? 3 : 1;
    const uint32_t slot = atomicAdd(&q.counts[which], 1u);
    q.lists[(size_t)which * q.n + slot] = i;
}

}  // namespace zoe_cuda
