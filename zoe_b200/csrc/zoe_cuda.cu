// zoe_cuda.cu -- the C-ABI shared library (include/zoe_cuda.h): context, scoring, profiled
// sequences, batch drivers, sharding over devices.  Kernels live in sw_score.cuh / sw_align.cuh.
//
// No CPU fallback exists in this file by design: every result returned through this ABI was
// computed by a CUDA kernel below.
#include "../../include/zoe_cuda.h"

#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <utility>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <atomic>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "sw_align.cuh"
#include "sw_align_win.cuh"
#include "sw_exact_fast.cuh"
#include "sw_score.cuh"
#include "sw_score_long.cuh"
#include "sw_ends_long.cuh"
#include "sw_score_rows.cuh"
#include "sw_ranges.cuh"
#include "sw_3pass.cuh"
#include "sneaky_snake.cuh"
#include "strands.cuh"
#include "best_hit.cuh"
#include "paired.cuh"

using namespace zoe_cuda;

namespace {

// ---------------------------------------------------------------------------------------------
// small utilities
// ---------------------------------------------------------------------------------------------
struct DebugTimer {  // host-side phase timing, printed when ZOE_CUDA_DEBUG is set
    bool on = getenv("ZOE_CUDA_DEBUG") != nullptr;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    void lap(const char *what) {
        if (!on) return;
        auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[zoe_cuda] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T *as() const {
        return reinterpret_cast<T *>(p);
    }
};

struct Device {
    int id = 0;
    int sm_count = 0;
    size_t free_at_create = 0;  // cudaMemGetInfo is slow (tens of ms on a 180 GB part): asked once
    cudaStream_t stream = nullptr;
    // per-profiled-sequence base offsets (flag_base / ckpt_base) are a function of the profiled set, the kernel's (G, K) and
    // the checkpoint spacing: uploaded once and reused (a pageable-memory copy synchronises the stream: 0.4 ms per call)
    uint64_t flb_epoch = 0, ckb_epoch = 0;
    int flb_G = 0, flb_K = 0, ckb_G = 0, ckb_K = 0, ckb_cb = -1;
    bool ckpt_base_cached(uint64_t epoch, int G, int K, int cb) const { return ckb_epoch == epoch && ckb_G == G && ckb_K == K && ckb_cb == cb; }
    void ckpt_base_mark(uint64_t epoch, int G, int K, int cb) { ckb_epoch = epoch; ckb_G = G; ckb_K = K; ckb_cb = cb; }
    // split upload (end-to-end calls): the first 1/8 of the sequences, then the rest, on `copy_stream`; the first kernel of
    // the call runs on the first part while the second is still arriving
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_first = nullptr, ev_copied = nullptr;
    bool copy_pending = false;
    uint64_t seq_split = 0;  // sequences [0, seq_split) of the shard are in the first part (even)
    cudaStream_t aux_stream = nullptr;  // align: the pin sweep of the ambiguous pairs runs beside the main window fill
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr, ev_k0 = nullptr, ev_k1 = nullptr;
    // scoring + profiled (replicated on every device)
    DevBuf ccodes, coff, wk, lut, corder;
    DevBuf ccodes_g, coff_g, corder_g;  // profiled set regrouped for panels beyond the shared-memory staging area
    // batch state
    DevBuf rseq, roff, best, score, status, tier, wide_ids, counters;
    // align state
    DevBuf pbytes, ends, flags, flag_base, ref_start, ref_end, query_start, query_end, hazard, hazard_list;
    DevBuf cig_scratch, cig_count, cig_off, cig_out, ex_hbuf, ex_fbuf, ex_cig, weights, ex_lists, ex_counts, ex_fast_fbuf;
    // windowed align path (sw_align_win.cuh)
    DevBuf ckpt, ckpt_base, win_hist, win_bucket, win_items, win_nitems, win_pitems, win_pnitems, win_amb;
    DevBuf starts;  // ranges: reverse-pass results
    DevBuf cig_bsum;  // CIGAR scan: per-block sums
    DevBuf sn_refs, sn_roff, sn_qry, sn_qoff, sn_out;  // SneakySnake filter batch (sneaky_snake.cuh)
    DevBuf tp_pair, tp_off, tp_cap, tp_slot, tp_blob, tp_ctr, tp_cigoff, tp_bw, tp_list, tp_cig;  // 3-pass: DP work lists + scratch (sw_3pass.cuh)
    uint64_t cig_total = 0;
    // long-row score path
    DevBuf long_ids, long_bnd, long_queue;
    // both-strand search (strands.cuh): the doubled batch is built here and swapped into rseq / roff; the selected
    // strand's per-pair outputs are gathered into the sel_* buffers and swapped into the ones the fetch paths read
    DevBuf xs_seq, xs_off, strand, sel32[5], sel8[3], sel_cig_count, sel_cig_off, sel_cig_out, sel_ctr;
    // best-hit search (best_hit.cuh): the staged batch moves to bh_seq / bh_off while each bucket's compact batch is
    // gathered into rseq / roff; bh_out* / bh_hit / bh_strand / bh_runner are the per-read outputs of the shard, bh_acc
    // collects the buckets' CIGAR words
    DevBuf bh_seq, bh_off, bh_key, bh_tab, bh_list, bh_llen, bh_loff, bh_hit, bh_strand, bh_runner, bh_out32[5], bh_out8[3];
    DevBuf bh_cig_count, bh_cig_src, bh_acc, bh_cig_off, bh_cig;
    // paired-end best-hit search (paired.cuh): the per-pair outputs (the per-mate ones are the bh_* buffers)
    DevBuf pr_hit, pr_proper, pr_tlen;
    uint64_t n_first = 0, n_count = 0;  // shard of the streamed batch owned by this device
    uint64_t rseq_bytes = 0;
    bool timed_kernel = false;
};

// Scorings (gap open, gap extend; positive penalties) whose packed score kernels are compiled with the penalties as
// immediates (GapImm, sw_score.cuh); any other scoring runs the kernels that read them from ScoreParams.  Every pair adds
// 28 kernels to the build.  (10, 1) is the scoring of all five benchmark configurations.
struct GapPair {
    int go, ge;
};
constexpr GapPair kGapImmPairs[] = {{10, 1}};
constexpr int kNumGapImm = sizeof(kGapImmPairs) / sizeof(kGapImmPairs[0]);
using ScoreFn = void (*)(const ScoreParams);
using GapImmFns = std::array<ScoreFn, kNumGapImm>;
template <int G, int K, int NS, size_t... I>
constexpr GapImmFns gap_imm_fns(std::index_sequence<I...>) {
    return {sw_score_kernel<G, K, true, NS, GapImm<kGapImmPairs[I].go, kGapImmPairs[I].ge>>...};
}
int gap_imm_index(int go, int ge) {
    for (int i = 0; i < kNumGapImm; ++i)
        if (kGapImmPairs[i].go == go && kGapImmPairs[i].ge == ge) return i;
    return -1;
}

struct KernelEntry {
    int G, K;
    void (*packed)(const ScoreParams);
    void (*wide)(const ScoreParams);
    void (*fill)(const AlignParams);
    void (*packed2)(const ScoreParams);  // two column sequences per sweep
    void (*scan)(const WinParams);       // windowed align, pass A
    void (*winfill)(const WinParams);    // windowed align, pass B
    void (*ends)(const EndsParams);      // score + end cell (ranges), packed
    void (*ends_wide)(const EndsParams); // ... 32-bit
    void (*scan_g)(const WinParams);     // pass A with the profiled symbol codes read from global memory (sets > 96 KB)
    void (*pin)(const WinParams);        // windowed align: exact best cell of the pairs whose maximum recurs
    void (*scan_rev)(const WinParams);   // ranges: reverse pass (score-rate scan + in-kernel pin)
    void (*scan2)(const WinParams);      // pass A, two tasks per group (K <= 20), codes in shared memory / ...
    void (*scan2_g)(const WinParams);    // ... codes from global memory
    GapImmFns packed_imm, packed2_imm;   // packed / packed2 with the penalties of kGapImmPairs[i] compiled in
};

// the two-task pass A exists for K <= 20 (two H / F register sets per thread); a rejected experiment (see pick_scan2):
// compiled only with -DZOE_CUDA_WITH_SCAN2 (28 large instantiations, a fifth of the build time)
#ifndef ZOE_CUDA_WITH_SCAN2
#define ZOE_CUDA_WITH_SCAN2 0
#endif
template <int G, int K, bool ON>
struct Scan2 {
    static constexpr void (*smem())(const WinParams) { return sw_align_scan2_kernel<G, K, true>; }
    static constexpr void (*gmem())(const WinParams) { return sw_align_scan2_kernel<G, K, false>; }
};
template <int G, int K>
struct Scan2<G, K, false> {
    static constexpr void (*smem())(const WinParams) { return nullptr; }
    static constexpr void (*gmem())(const WinParams) { return nullptr; }
};

#define ZK(G, K) \
    KernelEntry {                                                                                          \
        G, K, sw_score_kernel<G, K, true, 1>, sw_score_kernel<G, K, false, 1>, sw_align_fill_kernel<G, K, true>, \
            sw_score_kernel<G, K, true, 2>, sw_align_scan_kernel<G, K>, sw_align_winfill_kernel<G, K>,     \
            sw_ends_kernel<G, K, true>, sw_ends_kernel<G, K, false>, sw_align_scan_kernel<G, K, false>,     \
            sw_align_winfill_kernel<G, K, false>, sw_align_scan_kernel<G, K, true, true>,                   \
            Scan2<G, K, (ZOE_CUDA_WITH_SCAN2 != 0) && (K <= 20)>::smem(),                                  \
            Scan2<G, K, (ZOE_CUDA_WITH_SCAN2 != 0) && (K <= 20)>::gmem(),                                  \
            gap_imm_fns<G, K, 1>(std::make_index_sequence<kNumGapImm>{}),                                   \
            gap_imm_fns<G, K, 2>(std::make_index_sequence<kNumGapImm>{})                                    \
    }

// Row capacity G*K of each instantiation; the host picks the tightest fit for the longest
// sequence of a batch.  G = 8 serves short reads (150 nt -> 8 x 19), G = 32 the longest rows
// a single pass can hold (1024).
const KernelEntry kScoreKernels[] = {
    ZK(8, 4),  ZK(8, 8),   ZK(8, 13),  ZK(8, 16),  ZK(8, 19),  ZK(8, 24),  ZK(8, 32),
    ZK(16, 19), ZK(16, 24), ZK(16, 32), ZK(32, 10), ZK(32, 20), ZK(32, 24), ZK(32, 32),
};
constexpr int kNumScoreKernels = sizeof(kScoreKernels) / sizeof(kScoreKernels[0]);
constexpr int kMaxRowsSinglePass = 32 * 32;
// Pass A of the windowed pipeline (sw_align_scan_kernel) keeps step-pair indices in 16-bit halves: L + G - 1 <= 131071.
// Longer profiled sequences take the full-matrix align pipeline / sw_ends_kernel, whose keys hold 20-bit columns.
constexpr uint32_t kScanMaxCols = 131072 - 64;
constexpr uint32_t kEndsMaxCols = (1u << 20) - 64;

struct LaunchPlan {
    int threads = 0, blocks_per_sm = 0;
    size_t smem = 0;
    int cols_in_smem = 0;
};
struct PlanKey {
    const void *fn;
    size_t cc_bytes;
    int tabs_per_group;
    bool operator<(const PlanKey &o) const {
        if (fn != o.fn) return fn < o.fn;
        if (cc_bytes != o.cc_bytes) return cc_bytes < o.cc_bytes;
        return tabs_per_group < o.tabs_per_group;
    }
};

}  // namespace

struct zoe_cuda_ctx {
    std::vector<Device> devs;
    std::map<PlanKey, LaunchPlan> plans;  // launch configurations, valid for the current scoring + profiled set
    uint64_t profiled_epoch = 1;          // bumped by set_profiled: invalidates what the devices cached about the set
    // One extra stream + buffer set per GPU: zoe_cuda_sw_score_batch alternates sub-batches between devs[k] and alt[k]
    // so that the H2D copy of sub-batch i+1 and the D2H copy of sub-batch i-1 overlap the kernels of sub-batch i.
    std::vector<Device> alt;
    bool alt_used = false;  // the last call spread its work over both
    std::string err;
    // scoring
    bool have_scoring = false;
    int S = 0;
    std::vector<int8_t> weights;  // S*S, zoe's weights[ref_idx][query_idx]
    uint8_t lut[256];
    int go = 0, ge = 0;  // positive penalties
    bool no_gap_imm = false;  // ZOE_CUDA_NO_GAP_IMM: always the run-time-penalty score kernels (A/B runs, tests)
    int profiled_is_query = 0;
    int max_weight = 0;
    int lanes[3] = {32, 16, 8};
    int bias = 0;                     // |min(0, smallest weight)|: to_biased_matrix, src/data/matrices/mod.rs:448-491
    int first_bits = 8, last_bits = 32, is_unsigned = 0;
    TierPolicy tp{254u, 65534u, 4294967294u, 8, 32};
    // profiled
    bool have_profiled = false;
    uint32_t n_prof = 0;
    std::vector<uint8_t> prof_bytes;
    std::vector<uint64_t> prof_off;
    std::vector<uint8_t> ccodes;
    std::vector<uint32_t> coff, corder;
    std::vector<int8_t> wk;
    int n_csym = 0;
    uint32_t max_prof_len = 0;
    // Panels whose symbol codes exceed the shared-memory staging area (kColsSmemLimit) are swept group by group by the
    // score kernel: contiguous runs of profiled sequences that fit, each with its own 16-byte aligned copy of the codes.
    struct ColGroup {
        uint32_t j0, n;             // profiled sequences [j0, j0 + n)
        uint32_t byte_start, bytes; // into ccodes_g
        uint32_t coff_start;        // into coff_g (n + 1 entries, relative to byte_start) and corder_g (n entries)
    };
    std::vector<ColGroup> groups;
    std::vector<uint8_t> ccodes_g;
    std::vector<uint32_t> coff_g, corder_g;
    // staged batch (host view)
    uint64_t staged_n = 0;
    uint32_t staged_max_len = 0;
    uint32_t staged_min_len = 0;
    uint64_t staged_cells = 0;
    bool staged = false;
    std::vector<uint32_t> staged_len;  // per streamed sequence (only kept when the long-row path is needed)
    uint64_t flag_budget_bytes = 0;  // 0 = auto (a fraction of free device memory)
    int align_mode = 0;              // 0 = auto, 1 = full-matrix flags, 2 = checkpointed window
    int win_cb_log2 = 6;             // checkpoint spacing (columns), log2 (64: measured best on cfg 3, 70.3 vs 73.6 ms at 128)
    uint32_t win_slack = 16;         // columns kept left of the shortest possible walk ...
    bool win_slack_set = false;      // ... when the caller set it (zoe_cuda_set_align_options); else chosen per scoring
    // measurements
    float last_total_ms = 0.f, last_dp_ms = 0.f;
    std::atomic<uint32_t> last_launches{0};
    zoe_cuda_stats stats{};
    std::mutex mu;  // guards err / stats / last_dp_ms when the devices of one call are driven by parallel host threads
};

namespace {

int fail(zoe_cuda_ctx *ctx, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) {
        std::lock_guard<std::mutex> lk(ctx->mu);
        ctx->err = buf;
    }
    return code;
}

#define CU(ctx, call)                                                                              \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return fail(ctx, ZOE_CUDA_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                        __FILE__, __LINE__);                                                       \
    } while (0)

// Largest score each allowed integer type can report (striped.rs:608-633): signed T holds best - MIN < MAX - MIN, i.e.
// score <= 2*MAX; unsigned T with a biased matrix needs best + bias + 1 not to overflow, i.e. score <= MAX - bias - 1.
void refresh_tier_policy(zoe_cuda_ctx *ctx) {
    TierPolicy &tp = ctx->tp;
    if (ctx->is_unsigned) {
        const uint32_t b = (uint32_t)ctx->bias;
        tp.lim8 = 255u - b - 1u;
        tp.lim16 = 65535u - b - 1u;
        tp.lim32 = 4294967295u - b - 1u;
    } else {
        tp.lim8 = 254u;
        tp.lim16 = 65534u;
        tp.lim32 = 4294967294u;
    }
    tp.first = (uint8_t)ctx->first_bits;
    tp.last = (uint8_t)ctx->last_bits;
}

// zoe: validate_profile_args, src/alignment/profile.rs:32-44
int validate_profile_args(uint64_t len, int gap_open, int gap_extend) {
    if (len == 0) return ZOE_CUDA_E_EMPTY_SEQUENCE;
    if (gap_open < -127 || gap_open > 0) return ZOE_CUDA_E_GAP_OPEN_RANGE;
    if (gap_extend < -127 || gap_extend > 0) return ZOE_CUDA_E_GAP_EXTEND_RANGE;
    if (gap_extend < gap_open) return ZOE_CUDA_E_BAD_GAP_WEIGHTS;
    return 0;
}

// score/status/tier from the exact best score: src/alignment/sw/striped.rs:608-633 applied along
// the escalation chain of src/alignment/profile_set.rs:71-78.
__global__ void finalize_scores_kernel(const int32_t *best, uint64_t n, uint32_t *score, uint8_t *status,
                                       uint8_t *tier, unsigned long long *counters, const TierPolicy tp) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long c8 = 0, c16 = 0, c32 = 0, cun = 0, cov = 0;
    if (i < n) {
        int32_t b = best[i];
        uint32_t s = (uint32_t)b;
        uint8_t st = ZOE_CUDA_SOME, t = tp.first;
        if (b <= 0) {
            s = 0;
            st = ZOE_CUDA_UNMAPPED;  // Unmapped does not escalate: it is decided in the first tier of the chain
            cun = 1;
        } else {
            t = tier_for(tp, s);
            if (t == 8) {
                c8 = 1;
            } else if (t == 16) {
                c16 = 1;
            } else if (t == 32) {
                c32 = 1;
            } else {  // beyond the widest allowed integer type
                s = 0;
                st = ZOE_CUDA_OVERFLOWED;
                t = tp.last;
                cov = 1;
            }
        }
        score[i] = s;
        status[i] = st;
        tier[i] = t;
    }
    // warp-aggregate the counters
    for (int d = 16; d >= 1; d >>= 1) {
        c8 += __shfl_xor_sync(0xffffffffu, c8, d);
        c16 += __shfl_xor_sync(0xffffffffu, c16, d);
        c32 += __shfl_xor_sync(0xffffffffu, c32, d);
        cun += __shfl_xor_sync(0xffffffffu, cun, d);
        cov += __shfl_xor_sync(0xffffffffu, cov, d);
    }
    if ((threadIdx.x & 31) == 0) {
        if (c8) atomicAdd(&counters[0], c8);
        if (c16) atomicAdd(&counters[1], c16);
        if (c32) atomicAdd(&counters[2], c32);
        if (cun) atomicAdd(&counters[3], cun);
        if (cov) atomicAdd(&counters[13], cov);
    }
}

// Collect the batch sequences that have at least one pair flagged "needs wide" (-1).
__global__ void collect_wide_kernel(const int32_t *best, uint32_t n_rseq, uint32_t n_cseq, uint32_t *ids,
                                    unsigned long long *counters) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rseq) return;
    bool any = false;
    for (uint32_t j = 0; j < n_cseq; ++j) any |= (best[(size_t)i * n_cseq + j] == -1);
    if (any) {
        unsigned long long slot = atomicAdd(&counters[4], 1ULL);
        ids[slot] = i;
    }
}

// Integer max-plus issue-rate microbenchmarks (roofline denominator).
template <int KIND>
__global__ void __launch_bounds__(256) dpx_peak_kernel(uint32_t *out, int iters, uint32_t seed) {
    uint32_t a[8], b[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        a[i] = seed * (threadIdx.x + 1) + i;
        b[i] = seed + i * 7u;
    }
    const uint32_t c = seed ^ 0x00030003u, g = 0x000a000au;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (KIND == 0) {
                a[i] = __viaddmax_s16x2(a[i], c, b[i]);
                b[i] = __viaddmax_s16x2(b[i], c, a[i]);
            } else if (KIND == 2) {
                // half2 max on the integer bit patterns: which pipe does HMNMX2 use?
                __half2 ha = *reinterpret_cast<__half2 *>(&a[i]), hb = *reinterpret_cast<__half2 *>(&b[i]);
                ha = __hmax2(ha, hb);
                hb = __hmax2(hb, *reinterpret_cast<const __half2 *>(&c));
                a[i] = *reinterpret_cast<uint32_t *>(&ha) + 1u;
                b[i] = *reinterpret_cast<uint32_t *>(&hb) ^ a[i];
            } else if (KIND == 3) {
                // 4 DPX + 1 half2 max + 1 add per cell pair
                uint32_t x = __vimax3_s16x2(a[i], b[i], g) - g;
                uint32_t h = __viaddmax_s16x2(a[(i + 1) & 7], c, x);
                a[i] = __viaddmax_s16x2(a[i], c, h);
                b[i] = __viaddmax_s16x2(b[i], c, h);
                __half2 hm = __hmax2(*reinterpret_cast<__half2 *>(&a[(i + 3) & 7]), *reinterpret_cast<__half2 *>(&h));
                a[(i + 3) & 7] = *reinterpret_cast<uint32_t *>(&hm);
            } else {
                // the score kernel's per-cell-pair mix: 1 max3 + 1 add + 3 addmax + 0.5 max3
                uint32_t x = __vimax3_s16x2(a[i], b[i], g) - g;
                uint32_t h = __viaddmax_s16x2(a[(i + 1) & 7], c, x);
                a[i] = __viaddmax_s16x2(a[i], c, h);
                b[i] = __viaddmax_s16x2(b[i], c, h);
                if (i & 1) a[(i + 3) & 7] = __vimax3_s16x2(a[(i + 3) & 7], h, x);
            }
        }
    }
    uint32_t r = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) r ^= a[i] ^ b[i];
    if (r == 0x12345678u) out[threadIdx.x] = r;
}

const KernelEntry *pick_score_kernel(uint32_t max_len, int n_csym) {
    const KernelEntry *bestk = nullptr;
    for (int i = 0; i < kNumScoreKernels; ++i) {
        const KernelEntry &k = kScoreKernels[i];
        if ((uint32_t)(k.G * k.K) < max_len) continue;
        if (!bestk) {
            bestk = &k;
            continue;
        }
        int rows = k.G * k.K, brow = bestk->G * bestk->K;
        // tightest row capacity wins; on ties a large alphabet (big per-task table) prefers the
        // wider group (more threads per table), a small one the narrower group (less skew).
        if (rows < brow || (rows == brow && ((n_csym > 8) ? (k.G > bestk->G) : (k.G < bestk->G)))) bestk = &k;
    }
    return bestk;
}

constexpr size_t kColsSmemLimit = 96 * 1024;  // profiled symbol codes staged per CTA (leaves room for the task tables)

size_t score_smem_bytes(const zoe_cuda_ctx *ctx, const KernelEntry &k, int threads, int cols_in_smem, size_t cc_bytes,
                        int tabs_per_group = 1) {
    size_t tab = (size_t)score_tab_bytes(ctx->n_csym, k.G, k.K) * (threads / k.G) * tabs_per_group;
    size_t s = tab + 256 + (((size_t)ctx->n_csym * ctx->S + 15) & ~(size_t)15);
    if (cols_in_smem) s += (cc_bytes + 15) & ~(size_t)15;
    return s;
}

// cc_bytes: symbol-code bytes the launch covers (default: the whole profiled set)
template <class Fn>
int plan_launch(zoe_cuda_ctx *ctx, const KernelEntry &k, Fn fn, LaunchPlan *plan, size_t cc_bytes = ~(size_t)0,
                int tabs_per_group = 1) {
    if (cc_bytes == ~(size_t)0) cc_bytes = ctx->ccodes.size();
    // occupancy queries and attribute changes cost tens of microseconds each: a plan is computed once per (kernel,
    // profiled bytes) and reused until the scoring / profiled set changes (small batches are launch-bound otherwise)
    const PlanKey key{(const void *)fn, cc_bytes, tabs_per_group};
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        auto it = ctx->plans.find(key);
        if (it != ctx->plans.end()) {
            *plan = it->second;
            return 0;
        }
    }
    int best_warps = 0;
    LaunchPlan bp;
    cudaFuncAttributes fa{};
    if (cudaFuncGetAttributes(&fa, fn) != cudaSuccess) {
        cudaGetLastError();
        fa.maxThreadsPerBlock = 1024;
    }
    for (int cols_in_smem = 1; cols_in_smem >= 0; --cols_in_smem) {
        if (cols_in_smem && cc_bytes > kColsSmemLimit) continue;
        static const int env_max_threads = getenv("ZOE_CUDA_MAX_THREADS") ? atoi(getenv("ZOE_CUDA_MAX_THREADS")) : 1024;
        for (int threads : {640, 576, 512, 448, 384, 352, 320, 288, 256, 224, 192, 160, 128, 96, 64, 32}) {
            if (threads < k.G || threads % k.G || threads > fa.maxThreadsPerBlock || threads > env_max_threads) continue;
            size_t smem = score_smem_bytes(ctx, k, threads, cols_in_smem, cc_bytes, tabs_per_group);
            if (smem > 227 * 1024) continue;
            int nb = 0;
            cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) {
                cudaGetLastError();
                continue;
            }
            e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, threads, smem);
            if (e != cudaSuccess) {
                cudaGetLastError();
                continue;
            }
            int warps = nb * threads / 32;
            if (warps > best_warps) {
                best_warps = warps;
                bp.threads = threads;
                bp.blocks_per_sm = nb;
                bp.smem = smem;
                bp.cols_in_smem = cols_in_smem;
            }
        }
        if (best_warps > 0) break;  // prefer staging the columns in shared memory when possible
    }
    if (best_warps == 0)
        return fail(ctx, ZOE_CUDA_E_UNSUPPORTED, "no launch configuration fits shared memory (alphabet %d, G=%d K=%d)",
                    ctx->n_csym, k.G, k.K);
    *plan = bp;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        ctx->plans[key] = bp;
    }
    return 0;
}

// The shape of a persistent launch over `units` tasks.  Warps are bound to one of the SM's four schedulers, so the time
// of a grid trip goes with ceil(warps per SM / 4), not with the warps: 18 warps (576 threads) run exactly as long as 20
// (measured: config 3, 62 500 tasks, 9.43 ms either way), and only a multiple of four warps fewer helps.  A small batch
// whose last trip is mostly empty (62 500 tasks on 148 x 80 groups: 5.3, hence 6 trips of 5 warps per scheduler = 30) may
// be cheaper with fewer, narrower trips (7 trips of 4 = 28).  More warps hide more latency than this model knows (1M
// reads: 640 threads beat 512 although 43 x 5 > 53 x 4), so the shape changes only for a predicted gain of 5 % or more.
// [Also measured: spreading config 1's 5 000 tasks over 250 CTAs of 160 threads instead of 114 of 352 -- same warps per
// scheduler, more CTAs staging the columns: 0.672 against 0.632 ms.  Not done.]
struct GridShape {
    uint32_t blocks, threads;
};
GridShape balance_grid(const Device &d, const LaunchPlan &plan, int G, uint32_t units) {
    const uint32_t gpb = (uint32_t)plan.threads / (uint32_t)G, bps = (uint32_t)std::max(plan.blocks_per_sm, 1);
    GridShape g{std::min<uint32_t>((uint32_t)d.sm_count * bps, (units + gpb - 1) / gpb), (uint32_t)plan.threads};
    static const bool off = getenv("ZOE_CUDA_NO_BALANCE") != nullptr, dbg = getenv("ZOE_CUDA_DEBUG_GRID") != nullptr;
    if (!off && units != 0 && bps == 1 && (128 % G) == 0) {
        const uint32_t sms = (uint32_t)d.sm_count;
        auto cost = [&](uint32_t threads) {
            const uint32_t per_trip = sms * (threads / (uint32_t)G);
            return (uint64_t)((units + per_trip - 1) / per_trip) * ((threads / 32 + 3) / 4);
        };
        uint64_t best = cost((uint32_t)plan.threads) * 100;
        for (uint32_t t = ((uint32_t)plan.threads - 1) / 128 * 128; t >= 512; t -= 128)  // >= 16 warps: latency hiding
            if (cost(t) * 105 <= best) {
                best = cost(t) * 105;
                g.threads = t;
            }
        const uint32_t gpb2 = g.threads / (uint32_t)G;
        g.blocks = std::min<uint32_t>(sms, (units + gpb2 - 1) / gpb2);
    }
    if (dbg) fprintf(stderr, "[zoe_cuda] grid: %u units, plan %d x %d per SM -> %u CTAs of %u threads\n", units, plan.threads,
                     plan.blocks_per_sm, g.blocks, g.threads);
    return g;
}

// Pass A of the windowed pipelines with two tasks per group (two dependency chains per thread).  MEASURED AND REJECTED on
// cfg 3 (1M reads): 67.7 ms against 64.8 ms with the one-task kernel -- two score tables per group leave 11 warps per SM
// instead of 16 (22 chains against 16), and the 168-register build spills.  Kept behind ZOE_CUDA_SCAN2 as a record.
void pick_scan2(zoe_cuda_ctx *ctx, const KernelEntry &k, void (**scan_fn)(const WinParams), LaunchPlan *plan, int *tpg) {
    static const bool off = getenv("ZOE_CUDA_SCAN2") == nullptr;
    void (*fn2)(const WinParams) = plan->cols_in_smem ? k.scan2 : k.scan2_g;
    if (off || !fn2) return;
    LaunchPlan p2;
    if (plan_launch(ctx, k, fn2, &p2, ~(size_t)0, 2) != 0) return;
    if (p2.cols_in_smem != plan->cols_in_smem) return;
    if (2 * p2.blocks_per_sm * p2.threads <= plan->blocks_per_sm * plan->threads) return;
    *scan_fn = fn2;
    *plan = p2;
    *tpg = 2;
}

int upload_scoring_and_profiled(zoe_cuda_ctx *ctx) {
    std::vector<Device *> all;
    for (Device &d : ctx->devs) all.push_back(&d);
    for (Device &d : ctx->alt) all.push_back(&d);
    for (Device *dp : all) {
        Device &d = *dp;
        CU(ctx, cudaSetDevice(d.id));
        CU(ctx, d.ccodes.reserve(ctx->ccodes.size()));
        CU(ctx, d.coff.reserve(ctx->coff.size() * sizeof(uint32_t)));
        CU(ctx, d.wk.reserve(ctx->wk.size()));
        CU(ctx, d.lut.reserve(256));
        CU(ctx, cudaMemcpyAsync(d.ccodes.p, ctx->ccodes.data(), ctx->ccodes.size(), cudaMemcpyHostToDevice, d.stream));
        CU(ctx, cudaMemcpyAsync(d.coff.p, ctx->coff.data(), ctx->coff.size() * sizeof(uint32_t), cudaMemcpyHostToDevice,
                                d.stream));
        CU(ctx, cudaMemcpyAsync(d.wk.p, ctx->wk.data(), ctx->wk.size(), cudaMemcpyHostToDevice, d.stream));
        CU(ctx, cudaMemcpyAsync(d.lut.p, ctx->lut, 256, cudaMemcpyHostToDevice, d.stream));
        CU(ctx, d.corder.reserve(ctx->corder.size() * sizeof(uint32_t)));
        CU(ctx, cudaMemcpyAsync(d.corder.p, ctx->corder.data(), ctx->corder.size() * sizeof(uint32_t), cudaMemcpyHostToDevice,
                                d.stream));
        if (!ctx->groups.empty()) {
            CU(ctx, d.ccodes_g.reserve(ctx->ccodes_g.size()));
            CU(ctx, d.coff_g.reserve(ctx->coff_g.size() * sizeof(uint32_t)));
            CU(ctx, d.corder_g.reserve(ctx->corder_g.size() * sizeof(uint32_t)));
            CU(ctx, cudaMemcpyAsync(d.ccodes_g.p, ctx->ccodes_g.data(), ctx->ccodes_g.size(), cudaMemcpyHostToDevice, d.stream));
            CU(ctx, cudaMemcpyAsync(d.coff_g.p, ctx->coff_g.data(), ctx->coff_g.size() * sizeof(uint32_t), cudaMemcpyHostToDevice,
                                    d.stream));
            CU(ctx, cudaMemcpyAsync(d.corder_g.p, ctx->corder_g.data(), ctx->corder_g.size() * sizeof(uint32_t),
                                    cudaMemcpyHostToDevice, d.stream));
        }
        CU(ctx, d.pbytes.reserve(ctx->prof_bytes.size()));
        CU(ctx, d.weights.reserve(ctx->weights.size()));
        CU(ctx, cudaMemcpyAsync(d.pbytes.p, ctx->prof_bytes.data(), ctx->prof_bytes.size(), cudaMemcpyHostToDevice,
                                d.stream));
        CU(ctx, cudaMemcpyAsync(d.weights.p, ctx->weights.data(), ctx->weights.size(), cudaMemcpyHostToDevice,
                                d.stream));
        CU(ctx, cudaStreamSynchronize(d.stream));
    }
    return 0;
}

// The host-side derivation of a profiled set (offsets validated by the caller; max_len its longest sequence): symbol
// codes, visiting order, dense symbol table, wk and the column groups, then the upload to every device.  Invalidates the
// launch plans and everything the devices cached about the previous set.
int install_profiled(zoe_cuda_ctx *ctx, const uint8_t *concat, const uint64_t *offsets, uint32_t n, uint32_t max_len) {
    const uint64_t total = offsets[n] - offsets[0];
    ctx->plans.clear();
    ctx->profiled_epoch++;
    ctx->n_prof = n;
    ctx->max_prof_len = max_len;
    ctx->prof_bytes.assign(concat + offsets[0], concat + offsets[n]);
    ctx->prof_off.resize(n + 1);
    ctx->coff.resize(n + 1);
    for (uint32_t j = 0; j <= n; ++j) {
        ctx->prof_off[j] = offsets[j] - offsets[0];
        ctx->coff[j] = (uint32_t)ctx->prof_off[j];
    }
    // visiting order for the two-stream score kernel: longest first, so paired sweeps have similar lengths
    ctx->corder.resize(n);
    for (uint32_t j = 0; j < n; ++j) ctx->corder[j] = j;
    std::stable_sort(ctx->corder.begin(), ctx->corder.end(), [&](uint32_t a, uint32_t b) {
        return ctx->coff[a + 1] - ctx->coff[a] > ctx->coff[b + 1] - ctx->coff[b];
    });
    // dense column-symbol codes: only the symbols that occur in the profiled set get a table row
    int dense[64];
    for (int i = 0; i < 64; ++i) dense[i] = -1;
    std::vector<int> sym_of_dense;
    ctx->ccodes.resize(total);
    for (uint64_t i = 0; i < total; ++i) {
        int s = ctx->lut[ctx->prof_bytes[i]];
        if (dense[s] < 0) {
            dense[s] = (int)sym_of_dense.size();
            sym_of_dense.push_back(s);
        }
        ctx->ccodes[i] = (uint8_t)dense[s];
    }
    ctx->n_csym = (int)sym_of_dense.size();
    // wk[c][r] = weights[streamed symbol r][profiled symbol c]  (profile.rs:290-291: the profile row is
    // indexed by the streamed symbol, the lane by the profiled residue)
    ctx->wk.assign((size_t)ctx->n_csym * ctx->S, 0);
    for (int c = 0; c < ctx->n_csym; ++c)
        for (int r = 0; r < ctx->S; ++r) ctx->wk[(size_t)c * ctx->S + r] = ctx->weights[(size_t)r * ctx->S + sym_of_dense[c]];
    // regroup a panel that does not fit the staging area (see launch_score)
    ctx->groups.clear();
    ctx->ccodes_g.clear();
    ctx->coff_g.clear();
    ctx->corder_g.clear();
    if (total > kColsSmemLimit && n > 1) {
        uint32_t j = 0;
        while (j < n) {
            zoe_cuda_ctx::ColGroup g{};
            g.j0 = j;
            g.byte_start = (uint32_t)ctx->ccodes_g.size();
            g.coff_start = (uint32_t)ctx->corder_g.size();
            uint32_t bytes = 0;
            while (j < n && (bytes == 0 || bytes + (ctx->coff[j + 1] - ctx->coff[j]) <= kColsSmemLimit)) {
                ctx->coff_g.push_back(bytes);
                bytes += ctx->coff[j + 1] - ctx->coff[j];
                ++j;
            }
            ctx->coff_g.push_back(bytes);
            g.n = j - g.j0;
            g.bytes = bytes;
            ctx->ccodes_g.insert(ctx->ccodes_g.end(), ctx->ccodes.begin() + ctx->coff[g.j0], ctx->ccodes.begin() + ctx->coff[j]);
            ctx->ccodes_g.resize((ctx->ccodes_g.size() + 15) & ~(size_t)15, 0);  // next group starts 16-byte aligned (TMA)
            std::vector<uint32_t> order(g.n);
            for (uint32_t q = 0; q < g.n; ++q) order[q] = q;
            std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) {
                return ctx->coff[g.j0 + a + 1] - ctx->coff[g.j0 + a] > ctx->coff[g.j0 + b + 1] - ctx->coff[g.j0 + b];
            });
            ctx->corder_g.insert(ctx->corder_g.end(), order.begin(), order.end());
            ctx->groups.push_back(g);
        }
        ctx->ccodes_g.resize(ctx->ccodes_g.size() + 16, 0);
        if (ctx->groups.size() < 2) ctx->groups.clear();
    }
    return upload_scoring_and_profiled(ctx);
}

// Split [0, n) over the devices by contiguous index range (SURVEY.md 8(e)); no collective.
void shard(zoe_cuda_ctx *ctx, uint64_t n) {
    size_t nd = ctx->devs.size();
    for (size_t k = 0; k < nd; ++k) {
        uint64_t a = n * k / nd, b = n * (k + 1) / nd;
        ctx->devs[k].n_first = a;
        ctx->devs[k].n_count = b - a;
    }
}

__global__ void rebase_offsets_kernel(uint64_t *off, uint64_t n, uint64_t base) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) off[i] -= base;
}

// Validates a batch's offsets and widens [*min_len, *max_len] and *tot by its sequences' lengths.
int check_offsets(zoe_cuda_ctx *ctx, const uint64_t *offsets, uint64_t n, uint32_t *max_len, uint32_t *min_len,
                  uint64_t *tot) {
    for (uint64_t i = 0; i < n; ++i) {
        if (offsets[i + 1] < offsets[i]) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "offsets must be non-decreasing");
        uint64_t len = offsets[i + 1] - offsets[i];
        if (len > 0x7fffffffULL) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "sequence too long");
        *max_len = std::max<uint32_t>(*max_len, (uint32_t)len);
        *min_len = std::min<uint32_t>(*min_len, (uint32_t)len);
        *tot += len;
    }
    return 0;
}

// Validates a batch, records its global properties (count, longest / shortest sequence, cells) and shards it.
int prepare_batch(zoe_cuda_ctx *ctx, const uint8_t *concat, const uint64_t *offsets, uint64_t n) {
    if (!ctx->have_profiled) return fail(ctx, ZOE_CUDA_E_STATE, "set_profiled must be called before a batch");
    if (n > 0 && (!concat || !offsets)) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "null batch pointers");
    if (n >= 0x7fffffffULL) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "batch too large");
    uint32_t max_len = 0, min_len = n ? 0xffffffffu : 0u;
    uint64_t tot = 0;
    int rc = check_offsets(ctx, offsets, n, &max_len, &min_len, &tot);
    if (rc) return rc;
    ctx->staged_min_len = min_len;
    uint64_t prof_total = ctx->prof_off[ctx->n_prof];
    ctx->staged_n = n;
    ctx->staged_max_len = max_len;
    ctx->staged_len.clear();
    if (max_len > (uint32_t)kMaxRowsSinglePass) {
        ctx->staged_len.resize(n);
        for (uint64_t i = 0; i < n; ++i) ctx->staged_len[i] = (uint32_t)(offsets[i + 1] - offsets[i]);
    }
    ctx->staged_cells = tot * prof_total;
    ctx->staged = false;
    ctx->alt_used = false;
    shard(ctx, n);
    return 0;
}

// Uploads the sequences [d.n_first, d.n_first + d.n_count) of the batch to `d` (async on d.stream).
// Everything but the first launch of a call's first kernel needs the whole batch.
int ensure_resident(zoe_cuda_ctx *ctx, Device &d) {
    if (!d.copy_pending) return 0;
    CU(ctx, cudaStreamWaitEvent(d.stream, d.ev_copied, 0));
    d.copy_pending = false;
    return 0;
}

// Tasks (pairs of sequences) the first launch of a split call covers: whole trips of the persistent grid, so the extra
// launch adds no partial wave; 0 = do not split.
uint32_t first_part_tasks(const Device &d, uint32_t n_tasks, uint32_t total_groups) {
    if (!d.copy_pending || total_groups == 0) return 0;
    uint32_t t = (uint32_t)(d.seq_split / 2);
    if (t >= total_groups) t -= t % total_groups;
    return (t == 0 || t >= n_tasks) ? 0 : t;
}

// split: upload the first 1/8 of the sequences, let d.stream go on, upload the rest behind it on the copy stream.  The first
// kernel of the call (sw_score_kernel or pass A: persistent grids that take tasks in index order) is launched twice -- on
// the tasks of the first part at once, on the others once everything has arrived -- so the copy engine works beside the
// kernel instead of in front of it (config 3: 3.3 ms of a 70 ms call).  [An earlier version polled a "bytes arrived" word
// inside the kernels: the extra control flow cost the two-stream score kernel 67 register moves per 76 cell pairs in its
// steady loop, 292 -> 318 ms on config 2; measured and dropped.]
int reserve_batch_outputs(zoe_cuda_ctx *ctx, Device &d);
int stage_device(zoe_cuda_ctx *ctx, Device &d, const uint8_t *concat, const uint64_t *offsets, bool record_begin = true,
                 bool split = false) {
    CU(ctx, cudaSetDevice(d.id));
    if (record_begin) CU(ctx, cudaEventRecord(d.ev_begin, d.stream));
    d.copy_pending = false;
    if (d.n_count == 0) return 0;
    uint64_t b0 = offsets[d.n_first], b1 = offsets[d.n_first + d.n_count];
    d.rseq_bytes = b1 - b0;
    CU(ctx, d.rseq.reserve(d.rseq_bytes + 16));
    CU(ctx, d.roff.reserve((d.n_count + 1) * sizeof(uint64_t)));
    // (queued before the sequences: copies drain in issue order, and the first launch needs the offsets)
    // the shard's offsets go up as the caller holds them (one copy straight from the caller's buffer, which
    // outlives the call) and are rebased to the shard's first byte on the device
    CU(ctx, cudaMemcpyAsync(d.roff.p, offsets + d.n_first, (d.n_count + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice,
                            d.stream));
    if (b0) {
        rebase_offsets_kernel<<<(uint32_t)((d.n_count + 256) / 256), 256, 0, d.stream>>>(d.roff.as<uint64_t>(),
                                                                                         d.n_count + 1, b0);
        CU(ctx, cudaGetLastError());
    }
    // Only for shards of 64 MB and more: a 19-MB shard (125 k reads, one of eight) is uploaded in 0.4 ms, and splitting its
    // first kernel into a full-width trip plus a second launch costs more than that (end to end 9.70 ms split, 9.36 ms
    // single upload with one trip-balanced launch); at 150 MB the split gains 1.4 ms.  ZOE_CUDA_SPLIT_UPLOAD_MIN_MB: tests.
    uint64_t split_min_mb = 64;
    if (const char *e = getenv("ZOE_CUDA_SPLIT_UPLOAD_MIN_MB")) split_min_mb = (uint64_t)std::max(atoi(e), 1);
    split = split && d.rseq_bytes >= (split_min_mb << 20) && d.n_count >= 4096 && !getenv("ZOE_CUDA_NO_SPLIT_UPLOAD");
    if (split) {
        if (!d.copy_stream) {
            CU(ctx, cudaStreamCreateWithFlags(&d.copy_stream, cudaStreamNonBlocking));
            CU(ctx, cudaEventCreateWithFlags(&d.ev_first, cudaEventDisableTiming));
            CU(ctx, cudaEventCreateWithFlags(&d.ev_copied, cudaEventDisableTiming));
        }
        // 1/8 of the shard, but at least one trip of the widest persistent grid (96 groups per SM, two sequences per
        // group): a first launch that fills only part of the grid costs more than the copy it hides
        d.seq_split = std::min<uint64_t>(std::max<uint64_t>(d.n_count / 8, (uint64_t)d.sm_count * 96 * 2), d.n_count / 2) & ~1ull;
        const uint64_t bs = offsets[d.n_first + d.seq_split];
        if (bs < b0 || bs > b1) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "offsets must be non-decreasing");
        CU(ctx, cudaStreamWaitEvent(d.copy_stream, d.ev_begin, 0));
        if (bs > b0) CU(ctx, cudaMemcpyAsync(d.rseq.p, concat + b0, bs - b0, cudaMemcpyHostToDevice, d.copy_stream));
        CU(ctx, cudaEventRecord(d.ev_first, d.copy_stream));
        if (b1 > bs)
            CU(ctx, cudaMemcpyAsync((uint8_t *)d.rseq.p + (bs - b0), concat + bs, b1 - bs, cudaMemcpyHostToDevice, d.copy_stream));
        CU(ctx, cudaEventRecord(d.ev_copied, d.copy_stream));
        CU(ctx, cudaStreamWaitEvent(d.stream, d.ev_first, 0));
        d.copy_pending = true;
    } else if (d.rseq_bytes) {
        CU(ctx, cudaMemcpyAsync(d.rseq.p, concat + b0, d.rseq_bytes, cudaMemcpyHostToDevice, d.stream));
    }
    return reserve_batch_outputs(ctx, d);
}

// The score pass's per-pair buffers for the device's shard.
int reserve_batch_outputs(zoe_cuda_ctx *ctx, Device &d) {
    size_t pairs = (size_t)d.n_count * ctx->n_prof;
    CU(ctx, d.best.reserve(pairs * sizeof(int32_t)));
    CU(ctx, d.score.reserve(pairs * sizeof(uint32_t)));
    CU(ctx, d.status.reserve(pairs));
    CU(ctx, d.tier.reserve(pairs));
    CU(ctx, d.wide_ids.reserve((d.n_count + 1) * sizeof(uint32_t)));
    CU(ctx, d.counters.reserve(16 * sizeof(unsigned long long)));
    return 0;
}

int stage_on_devices(zoe_cuda_ctx *ctx, const uint8_t *concat, const uint64_t *offsets, uint64_t n, bool split = false) {
    // The upload only needs the shard boundaries, so it is queued first (after the cheap checks) and the pass over all
    // offsets -- validation, longest / shortest sequence, cells: 0.9 ms of host time for 1M reads -- runs while the copy
    // engine works.  A batch that fails validation is reported after the copies have drained.
    if (!ctx->have_profiled) return fail(ctx, ZOE_CUDA_E_STATE, "set_profiled must be called before a batch");
    if (n > 0 && (!concat || !offsets)) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "null batch pointers");
    if (n >= 0x7fffffffULL) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "batch too large");
    bool early = n > 0;
    if (early) {
        shard(ctx, n);
        for (Device &d : ctx->devs)  // shard boundaries must be ordered or nothing is queued early
            if (d.n_count && offsets[d.n_first + d.n_count] < offsets[d.n_first]) early = false;
    }
    int rc = 0;
    if (early)
        for (Device &d : ctx->devs) {
            rc = stage_device(ctx, d, concat, offsets, true, split);
            if (rc) return rc;
        }
    rc = prepare_batch(ctx, concat, offsets, n);
    if (rc) {
        for (Device &d : ctx->devs) {
            cudaSetDevice(d.id);
            cudaStreamSynchronize(d.stream);
        }
        return rc;
    }
    if (!early)
        for (Device &d : ctx->devs) {
            rc = stage_device(ctx, d, concat, offsets, true, split);
            if (rc) return rc;
        }
    ctx->staged = true;
    return 0;
}

int launch_score(zoe_cuda_ctx *ctx, Device &d, const KernelEntry &k, bool packed, const uint32_t *task_ids,
                 uint32_t n_ids) {
    ScoreParams p{};
    p.rseq = d.rseq.as<uint8_t>();
    p.roff = d.roff.as<uint64_t>();
    p.task_ids = task_ids;
    uint32_t n_seq = task_ids ? n_ids : (uint32_t)d.n_count;
    p.n_rseq = n_seq;
    p.n_tasks = packed ? (n_seq + 1) / 2 : n_seq;
    p.wk = d.wk.as<int8_t>();
    p.n_csym = ctx->n_csym;
    p.S = ctx->S;
    p.lut = d.lut.as<uint8_t>();
    p.go = ctx->go;
    p.ge = ctx->ge;
    p.ovf_thresh = kPackedLimit - std::max(ctx->max_weight, 0) - 1;
    p.best = d.best.as<int32_t>();
    p.best_stride = ctx->n_prof;
    if (p.n_tasks == 0) return ensure_resident(ctx, d);
    if (task_ids) {  // a re-run of listed sequences: no streamed upload can still be pending, but make sure
        int rc0 = ensure_resident(ctx, d);
        if (rc0) return rc0;
    }

    // one launch over the whole profiled set, or (panels beyond the staging area) one launch per group of profiled
    // sequences whose codes fit shared memory: the steady-state loops read the column codes from shared memory
    // (5.8 -> 6.9 TCUPS on a 131-kb panel); every launch re-reads the streamed batch, which is tiny next to the sweep
    const size_t n_launches = ctx->groups.empty() ? 1 : ctx->groups.size();
    const int imm = ctx->no_gap_imm ? -1 : gap_imm_index(ctx->go, ctx->ge);
    for (size_t gi = 0; gi < n_launches; ++gi) {
        uint32_t n_cseq = ctx->n_prof;
        size_t cc_bytes = ctx->ccodes.size();
        if (!ctx->groups.empty()) {
            const zoe_cuda_ctx::ColGroup &g = ctx->groups[gi];
            n_cseq = g.n;
            cc_bytes = g.bytes;
            p.ccodes = d.ccodes_g.as<uint8_t>() + g.byte_start;
            p.coff = d.coff_g.as<uint32_t>() + g.coff_start + gi;  // group gi's n + 1 offsets follow gi earlier "+1"s
            p.best_col0 = g.j0;
        } else {
            p.ccodes = d.ccodes.as<uint8_t>();
            p.coff = d.coff.as<uint32_t>();
            p.best_col0 = 0;
        }
        const bool two_streams = packed && n_cseq >= 2 && !getenv("ZOE_CUDA_ONE_STREAM");
        void (*fn)(const ScoreParams) = packed ? (two_streams ? k.packed2 : k.packed) : k.wide;
        if (packed && imm >= 0) fn = two_streams ? k.packed2_imm[imm] : k.packed_imm[imm];
        LaunchPlan plan;
        int rc = plan_launch(ctx, k, fn, &plan, cc_bytes);
        if (rc) return rc;
        p.corder = nullptr;
        if (two_streams)
            p.corder = ctx->groups.empty() ? d.corder.as<uint32_t>() : d.corder_g.as<uint32_t>() + ctx->groups[gi].coff_start;
        p.n_cseq = n_cseq;
        p.ccodes_bytes = (uint32_t)cc_bytes;
        p.cols_in_smem = plan.cols_in_smem;
        CU(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem));
        uint32_t groups_per_block = plan.threads / k.G;
        uint32_t max_blocks = (uint32_t)(d.sm_count * plan.blocks_per_sm);
        uint32_t need_blocks = (p.n_tasks + groups_per_block - 1) / groups_per_block;
        uint32_t blocks = std::min(max_blocks, need_blocks);
        // a call whose upload is still running covers the tasks of the first part now, the others once all has arrived
        const uint32_t t_end = p.n_tasks, t_a = first_part_tasks(d, p.n_tasks, blocks * groups_per_block);
        p.task_first = 0;
        if (t_a) {
            p.n_tasks = t_a;
            fn<<<blocks, plan.threads, plan.smem, d.stream>>>(p);
            CU(ctx, cudaGetLastError());
            ctx->last_launches++;
            p.task_first = t_a;
            p.n_tasks = t_end;
        }
        rc = ensure_resident(ctx, d);
        if (rc) return rc;
        const GridShape gs = balance_grid(d, plan, k.G, p.n_tasks - p.task_first);
        fn<<<gs.blocks, gs.threads, plan.smem, d.stream>>>(p);
        CU(ctx, cudaGetLastError());
        ctx->last_launches++;
        p.task_first = 0;
    }
    return 0;
}


// ---------------------------------------------------------------------------------------------
// shared-rows score path: the profiled sequence is register-resident (large alphabets, sw_score_rows.cuh)
// ---------------------------------------------------------------------------------------------
struct RowsEntry {
    int K;
    void (*fn)(const RowsParams);
};
// streaming variants (trips swept back to back; every streamed sequence >= 64 residues), same K list
const RowsEntry kRowsStreamKernels[] = {
    {8, sw_score_rows_stream_kernel<32, 8>},   {12, sw_score_rows_stream_kernel<32, 12>}, {16, sw_score_rows_stream_kernel<32, 16>},
    {18, sw_score_rows_stream_kernel<32, 18>}, {20, sw_score_rows_stream_kernel<32, 20>}, {24, sw_score_rows_stream_kernel<32, 24>},
    {28, sw_score_rows_stream_kernel<32, 28>}, {32, sw_score_rows_stream_kernel<32, 32>},
};
const RowsEntry kRowsKernels[] = {
    {8, sw_score_rows_kernel<32, 8>},   {12, sw_score_rows_kernel<32, 12>}, {16, sw_score_rows_kernel<32, 16>},
    {18, sw_score_rows_kernel<32, 18>}, {20, sw_score_rows_kernel<32, 20>}, {24, sw_score_rows_kernel<32, 24>},
    {28, sw_score_rows_kernel<32, 28>}, {32, sw_score_rows_kernel<32, 32>},
};

bool rows_path_applies(const zoe_cuda_ctx *ctx) {
    if (getenv("ZOE_CUDA_NO_ROWS_KERNEL")) return false;
    // a per-task table of n_csym x rows x 4 B starves sw_score_kernel of occupancy for large alphabets; the
    // transposed kernel needs the profiled sequences to fit one pass and a bounded staging area per warp
    return ctx->n_csym > 8 && ctx->max_prof_len <= 1024 && ctx->staged_max_len <= 1024 && ctx->staged_max_len >= 64;
}

int launch_score_rows(zoe_cuda_ctx *ctx, Device &d) {
    if (int rc0 = ensure_resident(ctx, d)) return rc0;
    const RowsEntry *k = nullptr;
    const bool stream = ctx->staged_min_len >= 64 && !getenv("ZOE_CUDA_NO_ROWS_STREAM");
    for (const RowsEntry &e : (stream ? kRowsStreamKernels : kRowsKernels))
        if ((uint32_t)(32 * e.K) >= ctx->max_prof_len) {
            k = &e;
            break;
        }
    if (!k) return fail(ctx, ZOE_CUDA_E_UNSUPPORTED, "profiled sequence too long for the shared-rows kernel");
    RowsParams rp{};
    ScoreParams &p = rp.s;
    p.rseq = d.rseq.as<uint8_t>();
    p.roff = d.roff.as<uint64_t>();
    p.task_ids = nullptr;
    p.n_rseq = (uint32_t)d.n_count;
    p.n_tasks = (p.n_rseq + 1) / 2;
    p.ccodes = d.ccodes.as<uint8_t>();
    p.coff = d.coff.as<uint32_t>();
    p.n_cseq = ctx->n_prof;
    p.wk = d.wk.as<int8_t>();
    p.n_csym = ctx->n_csym;
    p.S = ctx->S;
    p.lut = d.lut.as<uint8_t>();
    p.go = ctx->go;
    p.ge = ctx->ge;
    p.ovf_thresh = 32767 - std::max(ctx->max_weight, 0) - 1;
    p.best = d.best.as<int32_t>();
    rp.max_rlen = ctx->staged_max_len;
    const size_t tab = rows_tab_bytes(ctx->S, 32, k->K);
    const size_t stage = stream ? rows_stream_stage_bytes(rp.max_rlen) : rows_stage_bytes(rp.max_rlen);
    int best_warps = 0, best_threads = 0, best_blocks = 0;
    size_t best_smem = 0;
    cudaFuncAttributes fa{};
    CU(ctx, cudaFuncGetAttributes(&fa, k->fn));
    for (int threads : {384, 256, 128, 64}) {
        if (threads > fa.maxThreadsPerBlock) continue;
        const size_t smem = tab + stage * (threads / 32);
        if (smem > 227 * 1024) continue;
        if (cudaFuncSetAttribute(k->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
            cudaGetLastError();
            continue;
        }
        int nb = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k->fn, threads, smem) != cudaSuccess) {
            cudaGetLastError();
            continue;
        }
        if (nb * threads / 32 > best_warps) {
            best_warps = nb * threads / 32;
            best_threads = threads;
            best_blocks = nb;
            best_smem = smem;
        }
    }
    if (!best_warps) return fail(ctx, ZOE_CUDA_E_UNSUPPORTED, "shared-rows kernel does not fit shared memory");
    CU(ctx, cudaFuncSetAttribute(k->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)best_smem));
    const uint32_t trips = (p.n_tasks + 1) / 2, wpb = best_threads / 32;
    const uint32_t blocks = std::min<uint32_t>((uint32_t)(d.sm_count * best_blocks), (trips + wpb - 1) / wpb);
    for (uint32_t cj = 0; cj < ctx->n_prof; ++cj) {
        rp.cj = cj;
        k->fn<<<blocks, best_threads, best_smem, d.stream>>>(rp);
        CU(ctx, cudaGetLastError());
        ctx->last_launches++;
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------
// long-row score path (rows > kMaxRowsSinglePass): chunked sweeps with a boundary row per warp
// ---------------------------------------------------------------------------------------------
constexpr int kLongK = 24;  // rows per lane per chunk: 32 x 24 = 768 rows, 16 warps per SM at DNA alphabet size

template <bool PACKED>
int launch_score_long(zoe_cuda_ctx *ctx, Device &d, const uint32_t *d_ids, uint32_t n_ids) {
    auto fn = sw_score_long_kernel<kLongK, PACKED>;
    const size_t tab_per_warp = (size_t)ctx->n_csym * (kLongK / 4) * 32 * 16;
    const size_t fixed = 256 + (((size_t)ctx->n_csym * ctx->S + 15) & ~(size_t)15);
    int best_warps = 0, best_threads = 0, best_blocks = 0, best_cols = 0;
    size_t best_smem = 0;
    for (int cols_in_smem = 1; cols_in_smem >= 0 && best_warps == 0; --cols_in_smem) {
        if (cols_in_smem && ctx->ccodes.size() > kColsSmemLimit) continue;
        for (int threads : {512, 384, 256, 128, 64, 32}) {
            size_t smem = tab_per_warp * (threads / 32) + fixed + (cols_in_smem ? ((ctx->ccodes.size() + 15) & ~(size_t)15) : 0);
            if (smem > 227 * 1024) continue;
            if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
                cudaGetLastError();
                continue;
            }
            int nb = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, threads, smem) != cudaSuccess) {
                cudaGetLastError();
                continue;
            }
            if (nb * threads / 32 > best_warps) {
                best_warps = nb * threads / 32;
                best_threads = threads;
                best_blocks = nb;
                best_smem = smem;
                best_cols = cols_in_smem;
            }
        }
    }
    if (!best_warps) return fail(ctx, ZOE_CUDA_E_UNSUPPORTED, "long-row kernel does not fit shared memory (alphabet %d)", ctx->n_csym);
    LongParams lp{};
    ScoreParams &p = lp.s;
    p.rseq = d.rseq.as<uint8_t>();
    p.roff = d.roff.as<uint64_t>();
    p.task_ids = d_ids;
    p.n_rseq = n_ids;
    p.n_tasks = PACKED ? (n_ids + 1) / 2 : n_ids;
    p.ccodes = d.ccodes.as<uint8_t>();
    p.coff = d.coff.as<uint32_t>();
    p.n_cseq = ctx->n_prof;
    p.ccodes_bytes = (uint32_t)ctx->ccodes.size();
    p.cols_in_smem = best_cols;
    p.wk = d.wk.as<int8_t>();
    p.n_csym = ctx->n_csym;
    p.S = ctx->S;
    p.lut = d.lut.as<uint8_t>();
    p.go = ctx->go;
    p.ge = ctx->ge;
    p.ovf_thresh = 32767 - std::max(ctx->max_weight, 0) - 1;
    p.best = d.best.as<int32_t>();
    if (p.n_tasks == 0) return 0;
    const uint32_t warps_per_block = best_threads / 32;
    uint32_t blocks = std::min<uint32_t>((uint32_t)(d.sm_count * best_blocks), (p.n_tasks + warps_per_block - 1) / warps_per_block);
    CU(ctx, d.long_bnd.reserve((size_t)blocks * warps_per_block * ctx->max_prof_len * sizeof(uint2)));
    CU(ctx, d.long_queue.reserve(sizeof(unsigned int)));
    CU(ctx, cudaMemsetAsync(d.long_queue.p, 0, sizeof(unsigned int), d.stream));
    lp.boundary = d.long_bnd.as<uint2>();
    lp.max_L = ctx->max_prof_len;
    lp.queue = d.long_queue.as<unsigned int>();
    CU(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)best_smem));
    fn<<<blocks, best_threads, best_smem, d.stream>>>(lp);
    CU(ctx, cudaGetLastError());
    ctx->last_launches++;
    return 0;
}

int run_score_long_on_device(zoe_cuda_ctx *ctx, Device &d) {
    if (int rc0 = ensure_resident(ctx, d)) return rc0;
    // longest-first order, so that (a) the two halves of a packed task have similar lengths and (b) the
    // atomic queue hands out the big tasks first
    std::vector<uint32_t> order(d.n_count);
    for (uint64_t i = 0; i < d.n_count; ++i) order[i] = (uint32_t)i;
    const uint32_t *len = ctx->staged_len.data() + d.n_first;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return len[a] > len[b]; });
    CU(ctx, d.long_ids.reserve(order.size() * sizeof(uint32_t)));
    CU(ctx, cudaMemcpyAsync(d.long_ids.p, order.data(), order.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, d.stream));
    CU(ctx, cudaStreamSynchronize(d.stream));
    uint64_t bound = (uint64_t)std::min<uint32_t>(ctx->staged_max_len, ctx->max_prof_len) * (uint64_t)std::max(ctx->max_weight, 0);
    const bool packed_ok = bound < 60000;
    CU(ctx, cudaEventRecord(d.ev_k0, d.stream));
    int rc;
    if (packed_ok) {
        rc = launch_score_long<true>(ctx, d, d.long_ids.as<uint32_t>(), (uint32_t)d.n_count);
        if (rc) return rc;
        if (bound >= (uint64_t)(32767 - ctx->max_weight - 1)) {
            uint32_t threads = 256, blocks = (uint32_t)((d.n_count + threads - 1) / threads);
            collect_wide_kernel<<<blocks, threads, 0, d.stream>>>(d.best.as<int32_t>(), (uint32_t)d.n_count, ctx->n_prof,
                                                                  d.wide_ids.as<uint32_t>(), d.counters.as<unsigned long long>());
            CU(ctx, cudaGetLastError());
            ctx->last_launches++;
            unsigned long long n_wide = 0;
            CU(ctx, cudaMemcpyAsync(&n_wide, d.counters.as<unsigned long long>() + 4, sizeof(n_wide), cudaMemcpyDeviceToHost, d.stream));
            CU(ctx, cudaStreamSynchronize(d.stream));
            if (n_wide) {
                rc = launch_score_long<false>(ctx, d, d.wide_ids.as<uint32_t>(), (uint32_t)n_wide);
                if (rc) return rc;
                {
                    std::lock_guard<std::mutex> lk(ctx->mu);
                    ctx->stats.rerun_wide += n_wide * ctx->n_prof;
                }
            }
        }
    } else {
        rc = launch_score_long<false>(ctx, d, d.long_ids.as<uint32_t>(), (uint32_t)d.n_count);
        if (rc) return rc;
    }
    CU(ctx, cudaEventRecord(d.ev_k1, d.stream));
    d.timed_kernel = true;
    return 0;
}

// The score pipeline on one device, all asynchronous on d.stream.
int run_score_on_device(zoe_cuda_ctx *ctx, Device &d, bool reset_counters = true) {
    if (d.n_count == 0) return 0;
    CU(ctx, cudaSetDevice(d.id));
    size_t pairs = (size_t)d.n_count * ctx->n_prof;
    if (reset_counters) CU(ctx, cudaMemsetAsync(d.counters.p, 0, 16 * sizeof(unsigned long long), d.stream));
    if (ctx->staged_max_len > (uint32_t)kMaxRowsSinglePass) {
        int rc = run_score_long_on_device(ctx, d);
        if (rc) return rc;
        uint32_t threads = 256;
        uint32_t blocks = (uint32_t)((pairs + threads - 1) / threads);
        finalize_scores_kernel<<<blocks, threads, 0, d.stream>>>(d.best.as<int32_t>(), pairs, d.score.as<uint32_t>(),
                                                                 d.status.as<uint8_t>(), d.tier.as<uint8_t>(),
                                                                 d.counters.as<unsigned long long>(), ctx->tp);
        CU(ctx, cudaGetLastError());
        ctx->last_launches++;
        return 0;
    }
    const KernelEntry *k = pick_score_kernel(std::max<uint32_t>(ctx->staged_max_len, 1), ctx->n_csym);
    if (!k) return fail(ctx, ZOE_CUDA_E_UNSUPPORTED, "no kernel for length %u", ctx->staged_max_len);
    // Static bound: can any packed 16-bit lane reach the overflow threshold?
    uint64_t bound = (uint64_t)std::min<uint32_t>(ctx->staged_max_len, ctx->max_prof_len) *
                     (uint64_t)std::max(ctx->max_weight, 0);
    bool packed_ok = bound < 60000;  // above this nearly everything would be re-run: go wide directly
    CU(ctx, cudaEventRecord(d.ev_k0, d.stream));
    int rc;
    if (packed_ok) {
        rc = rows_path_applies(ctx) ? launch_score_rows(ctx, d) : launch_score(ctx, d, *k, true, nullptr, 0);
        if (rc) return rc;
        if (bound >= (uint64_t)(kPackedLimit - ctx->max_weight - 1)) {
            // escalation: re-run the flagged sequences at 32 bits (or_else_overflowed, output.rs:81-83)
            uint32_t threads = 256, blocks = (uint32_t)((d.n_count + threads - 1) / threads);
            collect_wide_kernel<<<blocks, threads, 0, d.stream>>>(d.best.as<int32_t>(), (uint32_t)d.n_count,
                                                                  ctx->n_prof, d.wide_ids.as<uint32_t>(),
                                                                  d.counters.as<unsigned long long>());
            CU(ctx, cudaGetLastError());
            ctx->last_launches++;
            unsigned long long n_wide = 0;
            CU(ctx, cudaMemcpyAsync(&n_wide, d.counters.as<unsigned long long>() + 4, sizeof(n_wide),
                                    cudaMemcpyDeviceToHost, d.stream));
            CU(ctx, cudaStreamSynchronize(d.stream));
            if (n_wide) {
                rc = launch_score(ctx, d, *k, false, d.wide_ids.as<uint32_t>(), (uint32_t)n_wide);
                if (rc) return rc;
                {
                    std::lock_guard<std::mutex> lk(ctx->mu);
                    ctx->stats.rerun_wide += n_wide * ctx->n_prof;
                }
            }
        }
    } else {
        rc = launch_score(ctx, d, *k, false, nullptr, 0);
        if (rc) return rc;
    }
    CU(ctx, cudaEventRecord(d.ev_k1, d.stream));
    d.timed_kernel = true;
    {
        uint32_t threads = 256;
        uint32_t blocks = (uint32_t)((pairs + threads - 1) / threads);
        finalize_scores_kernel<<<blocks, threads, 0, d.stream>>>(d.best.as<int32_t>(), pairs, d.score.as<uint32_t>(),
                                                                 d.status.as<uint8_t>(), d.tier.as<uint8_t>(),
                                                                 d.counters.as<unsigned long long>(), ctx->tp);
        CU(ctx, cudaGetLastError());
        ctx->last_launches++;
    }
    return 0;
}


// ---------------------------------------------------------------------------------------------
// align pipeline (one device): chunks of batch sequences -> fill -> traceback -> exact -> compaction
// ---------------------------------------------------------------------------------------------
__global__ void apply_wide_scores_kernel(const uint32_t *list, uint32_t n, const int32_t *best, uint32_t *score,
                                         uint8_t *status, uint8_t *tier, const TierPolicy tp) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t gid = list[i] & 0x7fffffffu;
    if (status[gid] != 0xFF) return;
    int32_t b = best[gid];
    const uint8_t t = b > 0 ? tier_for(tp, (uint32_t)b) : tp.first;
    score[gid] = (b > 0 && t) ? (uint32_t)b : 0u;
    status[gid] = b > 0 ? (t ? ZOE_CUDA_SOME : ZOE_CUDA_OVERFLOWED) : ZOE_CUDA_UNMAPPED;
    tier[gid] = t ? t : tp.last;
}

__global__ void collect_wide_range_kernel(const int32_t *best, uint32_t first, uint32_t count, uint32_t n_cseq,
                                          uint32_t *ids, unsigned long long *counters) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    uint32_t seq = first + i;
    bool any = false;
    for (uint32_t j = 0; j < n_cseq; ++j) any |= (best[(size_t)seq * n_cseq + j] == -1);
    if (any) {
        unsigned long long slot = atomicAdd(&counters[4], 1ULL);
        ids[slot] = seq;
    }
}

__global__ void count_status_kernel(const uint8_t *tier, const uint8_t *status, uint64_t n,
                                    unsigned long long *counters) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long c8 = 0, c16 = 0, c32 = 0, cun = 0, cov = 0;
    if (i < n) {
        if (status[i] == ZOE_CUDA_SOME) {
            const uint8_t t = tier[i];
            if (t == 8) c8 = 1; else if (t == 16) c16 = 1; else c32 = 1;
        } else if (status[i] == ZOE_CUDA_OVERFLOWED) {
            cov = 1;
        } else {
            cun = 1;
        }
    }
    for (int d = 16; d >= 1; d >>= 1) {
        c8 += __shfl_xor_sync(0xffffffffu, c8, d);
        c16 += __shfl_xor_sync(0xffffffffu, c16, d);
        c32 += __shfl_xor_sync(0xffffffffu, c32, d);
        cun += __shfl_xor_sync(0xffffffffu, cun, d);
        cov += __shfl_xor_sync(0xffffffffu, cov, d);
    }
    if ((threadIdx.x & 31) == 0) {
        if (c8) atomicAdd(&counters[0], c8);
        if (c16) atomicAdd(&counters[1], c16);
        if (c32) atomicAdd(&counters[2], c32);
        if (cun) atomicAdd(&counters[3], cun);
        if (cov) atomicAdd(&counters[13], cov);
    }
}

// Long-row align: every mapped pair of the chunk goes to the literal kernels, with the exact end cell the long-row
// ranges pipeline found (status / score / tier are already final).
__global__ void collect_mapped_kernel(const AlignEnd *ends, const uint8_t *status, uint32_t first_pair, uint32_t n_pairs,
                                      int32_t *best_arr, uint8_t *hazard, uint32_t *cig_count, uint32_t *hazard_list,
                                      unsigned long long *counters) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_pairs) return;
    const uint32_t gid = first_pair + k;
    best_arr[gid] = ends[gid].best;
    cig_count[gid] = 0;
    const bool mapped = status[gid] == ZOE_CUDA_SOME;
    hazard[gid] = mapped ? 1 : 0;
    if (mapped) hazard_list[atomicAdd(&counters[5], 1ULL)] = gid;
}

int run_ranges_long_on_device(zoe_cuda_ctx *ctx, Device &d);

int run_align_on_device(zoe_cuda_ctx *ctx, Device &d, uint64_t cigar_cap_words) {
    d.cig_total = 0;
    if (d.n_count == 0) return 0;
    CU(ctx, cudaSetDevice(d.id));
    // Streamed sequences beyond one pass of the register-resident kernels: zoe's sw_simd_align takes any length (and
    // documents its O(mn) memory as unsuitable for long pairs, striped.rs:410-413).  Here: score + exact end cell from the
    // chunked-row pipeline, then the literal striped kernels for every mapped pair -- correct, not fast; the memory-light
    // 3-pass alignment is the path meant for long reads.
    const bool long_mode = ctx->staged_max_len > (uint32_t)kMaxRowsSinglePass;
    if (long_mode) {
        int rc0 = run_ranges_long_on_device(ctx, d);
        if (rc0) return rc0;
    }
    const KernelEntry *k = pick_score_kernel(std::min<uint32_t>(std::max<uint32_t>(ctx->staged_max_len, 1), kMaxRowsSinglePass), ctx->n_csym);
    if (!k) return fail(ctx, ZOE_CUDA_E_UNSUPPORTED, "no kernel for length %u", ctx->staged_max_len);
    const int NW = align_words_per_lane(k->K);
    const uint32_t n_prof = ctx->n_prof;
    const size_t pairs = (size_t)d.n_count * n_prof;
    if (pairs >= 0x7fffffffULL) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "too many pairs for one align call");  // 31-bit pair ids

    // ---- which align pipeline? (DESIGN.md 4.3) ----
    // The checkpointed-window pipeline pays when the profiled sequences are much longer than the walk can
    // be; gap_open == 0 sends every pair to the literal kernel anyway, so only the scores matter there.
    int cb_log2 = ctx->win_cb_log2;
    while ((1 << cb_log2) < k->G) ++cb_log2;  // a checkpoint is a step boundary with every lane active
    const uint32_t CB = 1u << cb_log2;
    // window capacity in columns: the walk's reach + the distance to the previous checkpoint + the lane skew
    // Columns kept left of the shortest possible walk.  Unless the caller chose one: 16, or 128 when gaps are cheap next
    // to a match (open + extend <= 2 x the largest weight) -- unrelated reads then align as long gappy chains, and a walk
    // that leaves its window costs a literal-kernel run (tie-heavy scoring 4/-2/-3/-1, 200k reads: 38 % of the walks
    // left a 16-column slack, 0.08 % a 128-column one; 141 -> 95 ms).
    const uint32_t win_slack = ctx->win_slack_set ? ctx->win_slack
                                                  : ((ctx->go + ctx->ge <= 2 * std::max(ctx->max_weight, 0)) ? 128u : 16u);
    const uint32_t wmax = std::min<uint32_t>(ctx->max_prof_len, std::max<uint32_t>(ctx->staged_max_len, 1) + win_slack + CB) + k->G;
    if (ctx->max_prof_len > kEndsMaxCols)
        return fail(ctx, ZOE_CUDA_E_UNSUPPORTED, "profiled sequences longer than %u are not supported by the align path", kEndsMaxCols);
    const bool window_ok = ctx->go != 0 && ctx->max_prof_len <= kScanMaxCols;
    bool use_window = window_ok && (uint64_t)ctx->max_prof_len >= 2ull * wmax;
    if (ctx->align_mode == 1) use_window = false;
    if (long_mode) use_window = false;
    if (!use_window)
        if (int rc0 = ensure_resident(ctx, d)) return rc0;
    if (ctx->align_mode == 2) use_window = window_ok;
    if (const char *e = getenv("ZOE_CUDA_ALIGN_MODE")) {
        if (!strcmp(e, "full")) use_window = false;
        if (!strcmp(e, "window")) use_window = window_ok;
    }

    // flag layout of one task: every profiled sequence back to back (full-matrix pipeline), or one window
    std::vector<uint64_t> flag_base(n_prof), ckpt_base(n_prof);
    uint64_t task_stride = 0, ckpt_task_stride = 0;
    const int CKW = ckpt_words_per_lane(k->K);
    uint32_t nblk = 1;
    for (uint32_t j = 0; j < n_prof; ++j) {
        const uint64_t L = ctx->coff[j + 1] - ctx->coff[j];
        flag_base[j] = task_stride;
        task_stride += L * k->G * NW;
        ckpt_base[j] = ckpt_task_stride;
        ckpt_task_stride += ((L - 1) >> cb_log2) * (uint64_t)CKW * k->G;  // words
        nblk = std::max<uint32_t>(nblk, (uint32_t)((L - 1) >> cb_log2) + 1);
    }
    const uint32_t n_keys = n_prof * nblk;
    const uint64_t win_task_stride = (uint64_t)wmax * k->G * NW;  // words per pass-B task
    // chunk size from the flag-memory budget
    DebugTimer dbg0;
    const size_t free_b = d.free_at_create;
    uint64_t budget = ctx->flag_budget_bytes ? ctx->flag_budget_bytes : (uint64_t)(free_b * 0.55);
    budget = std::min<uint64_t>(budget, (uint64_t)48 << 30);
    // bytes per pass-A task (two sequences): full = all flags; window = checkpoints + one window per pair
    const uint32_t cig_cap = 2 * std::min<uint32_t>(std::max<uint32_t>(ctx->staged_max_len, 1), ctx->max_prof_len) + 4;
    const uint64_t per_task_bytes = long_mode ? (uint64_t)n_prof * cig_cap * 4 * 2 * 2  // the literal kernels' CIGAR rows only
                                    : use_window ? (ckpt_task_stride * 4 + (uint64_t)n_prof * win_task_stride * 4)
                                                 : task_stride * 4;
    uint64_t tasks_cap = std::max<uint64_t>(1, budget / std::max<uint64_t>(per_task_bytes, 1));
    uint64_t chunk_seqs = std::min<uint64_t>(d.n_count, tasks_cap * 2);
    if (chunk_seqs > 1) chunk_seqs &= ~1ULL;

    const bool flb_cached = d.flb_epoch == ctx->profiled_epoch && d.flb_G == k->G && d.flb_K == k->K;
    const bool ckb_cached = d.ckpt_base_cached(ctx->profiled_epoch, k->G, k->K, cb_log2);
    if (!flb_cached || !ckb_cached) {
        CU(ctx, d.flag_base.reserve(n_prof * sizeof(uint64_t)));
        CU(ctx, d.ckpt_base.reserve(n_prof * sizeof(uint64_t)));
        CU(ctx, cudaMemcpyAsync(d.flag_base.p, flag_base.data(), n_prof * sizeof(uint64_t), cudaMemcpyHostToDevice, d.stream));
        CU(ctx, cudaMemcpyAsync(d.ckpt_base.p, ckpt_base.data(), n_prof * sizeof(uint64_t), cudaMemcpyHostToDevice, d.stream));
        CU(ctx, cudaStreamSynchronize(d.stream));
        d.flb_epoch = ctx->profiled_epoch;
        d.flb_G = k->G;
        d.flb_K = k->K;
        d.ckpt_base_mark(ctx->profiled_epoch, k->G, k->K, cb_log2);
    }
    dbg0.lap("align: flag_base upload");
    CU(ctx, d.ends.reserve(pairs * sizeof(AlignEnd)));
    if (use_window) {
        const uint64_t max_items = chunk_seqs * n_prof + n_keys + 2;  // every bucket rounds up to even
        CU(ctx, d.flags.reserve((max_items / 2 + 1) * win_task_stride * 4));
        CU(ctx, d.ckpt.reserve(std::max<uint64_t>(((chunk_seqs + 1) / 2) * ckpt_task_stride * 4, 16)));
        CU(ctx, d.win_hist.reserve(n_keys * sizeof(uint32_t)));
        CU(ctx, d.win_bucket.reserve((n_keys + 1) * sizeof(uint32_t)));
        CU(ctx, d.win_items.reserve(max_items * sizeof(uint32_t)));
        CU(ctx, d.win_nitems.reserve(sizeof(uint32_t)));
        CU(ctx, d.win_pitems.reserve(max_items * sizeof(uint32_t)));
        CU(ctx, d.win_pnitems.reserve(sizeof(uint32_t)));
        CU(ctx, d.win_amb.reserve(chunk_seqs * n_prof + 16));
        if (!d.aux_stream) {
            CU(ctx, cudaStreamCreateWithFlags(&d.aux_stream, cudaStreamNonBlocking));
            CU(ctx, cudaEventCreateWithFlags(&d.ev_fork, cudaEventDisableTiming));
            CU(ctx, cudaEventCreateWithFlags(&d.ev_join, cudaEventDisableTiming));
        }
    } else if (!long_mode) {
        CU(ctx, d.flags.reserve(((chunk_seqs + 1) / 2) * task_stride * 4));
    }
    for (DevBuf *b : {&d.ref_start, &d.ref_end, &d.query_start, &d.query_end, &d.cig_count, &d.best, &d.score})
        CU(ctx, b->reserve(pairs * sizeof(uint32_t)));
    CU(ctx, d.status.reserve(pairs));
    CU(ctx, d.tier.reserve(pairs));
    CU(ctx, d.hazard.reserve(pairs));
    CU(ctx, d.hazard_list.reserve((size_t)chunk_seqs * n_prof * sizeof(uint32_t)));
    CU(ctx, d.cig_scratch.reserve(long_mode ? 16 : (size_t)chunk_seqs * n_prof * cig_cap * sizeof(uint32_t)));
    CU(ctx, d.cig_off.reserve((pairs + 1) * sizeof(uint64_t)));
    CU(ctx, d.cig_out.reserve(std::max<uint64_t>(cigar_cap_words, 1) * sizeof(uint32_t)));
    CU(ctx, d.wide_ids.reserve((d.n_count + 1) * sizeof(uint32_t)));
    CU(ctx, d.counters.reserve(16 * sizeof(unsigned long long)));
    CU(ctx, cudaMemsetAsync(d.counters.p, 0, 16 * sizeof(unsigned long long), d.stream));
    unsigned long long *ctr = d.counters.as<unsigned long long>();
    dbg0.lap("align: reserves");
    { DebugTimer t; if (t.on) fprintf(stderr, "[zoe_cuda] align: chunk_seqs %llu task_stride %llu words, cig_cap %u\n", (unsigned long long)chunk_seqs, (unsigned long long)task_stride, cig_cap); }

    DebugTimer dbg;
    LaunchPlan plan, plan_b;
    // pass A comes in two instantiations: profiled symbol codes staged in shared memory, or (sets > 96 KB) read from
    // global memory; plan_launch tells which one fits
    int rc = long_mode ? 0 : (use_window ? plan_launch(ctx, *k, k->scan, &plan) : plan_launch(ctx, *k, k->fill, &plan));
    if (rc) return rc;
    if (long_mode) plan.threads = k->G;  // no fill launch below; keeps the block arithmetic defined
    void (*scan_fn)(const WinParams) = k->scan;
    if (use_window && !plan.cols_in_smem) {
        scan_fn = k->scan_g;
        rc = plan_launch(ctx, *k, scan_fn, &plan);
        if (rc) return rc;
    }
    int scan_tpg = 1;  // tasks a group sweeps side by side in pass A
    if (use_window) pick_scan2(ctx, *k, &scan_fn, &plan, &scan_tpg);
    LaunchPlan plan_p;
    if (use_window) {
        rc = plan_launch(ctx, *k, k->winfill, &plan_b);
        if (rc) return rc;
        rc = plan_launch(ctx, *k, k->pin, &plan_p);
        if (rc) return rc;
        CU(ctx, cudaFuncSetAttribute(k->pin, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan_p.smem));
        CU(ctx, cudaFuncSetAttribute(scan_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem));
        CU(ctx, cudaFuncSetAttribute(k->winfill, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan_b.smem));
    } else if (!long_mode) {
        CU(ctx, cudaFuncSetAttribute(k->fill, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem));
    }
    dbg.lap("align: plan");
    // ZOE_CUDA_ALL_EXACT: every pair through the literal kernel (testing / timing; results are identical by design)
    const bool all_exact = (ctx->go == 0) || getenv("ZOE_CUDA_ALL_EXACT") != nullptr;
    const int invert = ctx->profiled_is_query ? 0 : 1;
    float dp_ms_total = 0.f;

    for (uint64_t c0 = 0; c0 < d.n_count; c0 += chunk_seqs) {
        const uint32_t cn = (uint32_t)std::min<uint64_t>(chunk_seqs, d.n_count - c0);
        // ---- fill ----
        AlignParams ap{};
        ScoreParams &p = ap.s;
        p.rseq = d.rseq.as<uint8_t>();
        p.roff = d.roff.as<uint64_t>();
        p.task_ids = nullptr;
        p.n_rseq = cn;
        p.n_tasks = (cn + 1) / 2;
        p.ccodes = d.ccodes.as<uint8_t>();
        p.coff = d.coff.as<uint32_t>();
        p.n_cseq = n_prof;
        p.ccodes_bytes = (uint32_t)ctx->ccodes.size();
        p.cols_in_smem = plan.cols_in_smem;
        p.wk = d.wk.as<int8_t>();
        p.n_csym = ctx->n_csym;
        p.S = ctx->S;
        p.lut = d.lut.as<uint8_t>();
        p.go = ctx->go;
        p.ge = ctx->ge;
        p.ovf_thresh = 32767 - std::max(ctx->max_weight, 0) - 1 - ctx->go;
        p.best = nullptr;
        ap.ends = d.ends.as<AlignEnd>();
        ap.flags = d.flags.as<uint32_t>();
        ap.flag_base = d.flag_base.as<uint64_t>();
        ap.task_stride = task_stride;
        ap.chunk_first = (uint32_t)c0;
        uint32_t groups_per_block = plan.threads / k->G;
        uint32_t blocks = std::min<uint32_t>((uint32_t)(d.sm_count * plan.blocks_per_sm),
                                             (p.n_tasks + groups_per_block - 1) / groups_per_block);
        if (!use_window && !long_mode) {
            CU(ctx, cudaEventRecord(d.ev_k0, d.stream));
            k->fill<<<blocks, plan.threads, plan.smem, d.stream>>>(ap);
            CU(ctx, cudaGetLastError());
            CU(ctx, cudaEventRecord(d.ev_k1, d.stream));
            ctx->last_launches++;
        }

        // ---- traceback ----
        CU(ctx, cudaMemsetAsync(ctr + 4, 0, 2 * sizeof(unsigned long long), d.stream));  // [4] wide seqs, [5] exact list
        CU(ctx, cudaMemsetAsync(ctr + 8, 0, sizeof(unsigned long long), d.stream));      // [8] packed overflows (per chunk)
        TraceParams t{};
        t.ends = ap.ends;
        t.flags = ap.flags;
        t.flag_base = ap.flag_base;
        t.task_stride = task_stride;
        t.roff = p.roff;
        t.coff = p.coff;
        t.n_cseq = n_prof;
        t.chunk_first = (uint32_t)c0;
        t.seq_ids = nullptr;
        t.n_slots = cn;
        t.best_arr = d.best.as<int32_t>();
        t.G = k->G;
        t.K = k->K;
        t.NW = NW;
        t.packed = 1;
        t.invert = invert;
        t.score = d.score.as<uint32_t>();
        t.status = d.status.as<uint8_t>();
        t.tier = d.tier.as<uint8_t>();
        t.hazard = d.hazard.as<uint8_t>();
        t.ref_start = d.ref_start.as<uint32_t>();
        t.ref_end = d.ref_end.as<uint32_t>();
        t.query_start = d.query_start.as<uint32_t>();
        t.query_end = d.query_end.as<uint32_t>();
        t.cig_scratch = d.cig_scratch.as<uint32_t>();
        t.cig_count = d.cig_count.as<uint32_t>();
        t.cig_cap = cig_cap;
        t.counters = ctr;
        t.hazard_list = d.hazard_list.as<uint32_t>();
        t.all_exact = all_exact ? 1 : 0;
        t.tp = ctx->tp;
        // ---- literal striped emulation for hazard / overflow / gap_open == 0 pairs (the first n_exact entries of
        //      hazard_list).  Tiers 8 / 16 with at most 32 lanes whose rows fit shared memory run in
        //      sw_exact_fast_kernel + sw_exact_walk_kernel, in rounds sized by the scratch budget; the rest (tier 32,
        //      64-lane presets, very long profiled sequences) in sw_align_exact_kernel. ----
        auto launch_exact = [&](uint32_t n_exact, cudaStream_t stream) -> int {
            const uint32_t n_rows_max = std::max<uint32_t>(ctx->staged_max_len, 1);
            const uint64_t ex_budget = std::max<uint64_t>(std::min<uint64_t>(budget / 4, (uint64_t)4 << 30), (uint64_t)64 << 20);
            CU(ctx, d.ex_cig.reserve((size_t)n_exact * cig_cap * sizeof(uint32_t)));
            CU(ctx, d.ex_lists.reserve((size_t)5 * n_exact * sizeof(uint32_t)));
            CU(ctx, d.ex_counts.reserve(8 * sizeof(uint32_t)));
            CU(ctx, cudaMemsetAsync(d.ex_counts.p, 0, 8 * sizeof(uint32_t), stream));
            // can the fast kernel hold a pair of this tier?  (lanes <= 32, one group's rows within the shared memory)
            const bool pidx_shared = n_prof == 1;
            auto fast_plan = [&](int N, uint32_t *vcap_out, int *groups_out, size_t *smem_out) -> bool {
                if ((N != 8 && N != 16 && N != 32) || getenv("ZOE_CUDA_EXACT_SLOW")) return false;
                const uint32_t vcap = ((uint32_t)N * (uint32_t)exact_fast_nvp((int)((ctx->max_prof_len + N - 1) / N)) + 31u) & ~31u;
                const size_t gb = exact_fast_group_bytes(vcap, pidx_shared, N), fx = exact_fast_fixed_bytes(vcap, ctx->S, pidx_shared);
                const size_t lim = 200 * 1024;
                if (gb * (32 / N) + fx > lim) return false;
                int groups = (int)std::min<size_t>((lim - fx) / gb, (size_t)(512 / N));
                groups -= groups % (32 / N);  // whole warps
                *vcap_out = vcap;
                *groups_out = groups;
                *smem_out = gb * groups + fx;
                return groups > 0;
            };
            uint32_t vcap8 = 0, vcap16 = 0;
            int groups8 = 0, groups16 = 0;
            size_t smem8 = 0, smem16 = 0;
            const bool fast8 = fast_plan(ctx->lanes[0], &vcap8, &groups8, &smem8);
            const bool fast16 = fast_plan(ctx->lanes[1], &vcap16, &groups16, &smem16);
            ExactPartitionParams q{};
            q.hazard_list = d.hazard_list.as<uint32_t>();
            q.n = n_exact;
            q.score = t.score;
            q.tp = ctx->tp;
            q.fast8 = fast8;
            q.fast16 = fast16;
            q.lists = d.ex_lists.as<uint32_t>();
            q.counts = d.ex_counts.as<uint32_t>();
            exact_partition_kernel<<<(n_exact + 255) / 256, 256, 0, stream>>>(q);
            CU(ctx, cudaGetLastError());
            ctx->last_launches++;
            uint32_t cnt[5] = {0, 0, 0, 0, 0};
            CU(ctx, cudaMemcpyAsync(cnt, d.ex_counts.p, sizeof(cnt), cudaMemcpyDeviceToHost, stream));
            CU(ctx, cudaStreamSynchronize(stream));
            bool any_fast = false;
            for (int which = 0; which < 4; ++which) {
                if (cnt[which] == 0) continue;
                any_fast = true;
                const bool full = which >= 2;
                const int N = (which & 1) ? ctx->lanes[1] : ctx->lanes[0];
                const uint32_t vcap = (which & 1) ? vcap16 : vcap8;
                const int groups = (which & 1) ? groups16 : groups8;
                const size_t smem = (which & 1) ? smem16 : smem8;
                // flag window capacity of one pair: the widest window any pair of this launch can have
                uint32_t wcap = ctx->max_prof_len;
                if (!full && ctx->ge > 0) {
                    const uint64_t imax = 1 + ((uint64_t)n_rows_max * (uint64_t)std::max(ctx->max_weight, 0)) / (uint64_t)ctx->ge;
                    wcap = (uint32_t)std::min<uint64_t>(wcap, (uint64_t)n_rows_max + imax + 2);
                }
                wcap = (wcap + 15u) & ~15u;
                const uint64_t fcap = (uint64_t)n_rows_max * wcap;
                const uint32_t round = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(cnt[which], ex_budget / fcap));
                CU(ctx, d.ex_fast_fbuf.reserve((size_t)round * fcap));
                ExactFastParams x{};
                x.hazard_list = d.hazard_list.as<uint32_t>();
                x.rseq = p.rseq;
                x.roff = p.roff;
                x.pbytes = d.pbytes.as<uint8_t>();
                x.coff = p.coff;
                x.n_cseq = n_prof;
                x.weights = d.weights.as<int8_t>();
                x.S = ctx->S;
                x.lut = p.lut;
                x.go = ctx->go;
                x.ge = ctx->ge;
                x.maxw = std::max(ctx->max_weight, 0);
                x.N = N;
                x.vcap = vcap;
                x.invert = invert;
                x.ends = d.ends.as<AlignEnd>();
                x.score_in = t.score;
                x.fbuf = d.ex_fast_fbuf.as<uint8_t>();
                x.fcap = fcap;
                x.wcap = wcap;
                x.ref_start = t.ref_start;
                x.ref_end = t.ref_end;
                x.query_start = t.query_start;
                x.query_end = t.query_end;
                x.cig_scratch = d.ex_cig.as<uint32_t>();
                x.cig_count = t.cig_count;
                x.cig_cap = cig_cap;
                x.counters = ctr;
                x.retry_list = d.ex_lists.as<uint32_t>() + (size_t)4 * n_exact;
                x.retry_count = d.ex_counts.as<uint32_t>() + 4;
                void (*fn)(const ExactFastParams) = nullptr;
                switch (N) {
                    case 8: fn = full ? sw_exact_fast_kernel<true, 8> : sw_exact_fast_kernel<false, 8>; break;
                    case 16: fn = full ? sw_exact_fast_kernel<true, 16> : sw_exact_fast_kernel<false, 16>; break;
                    case 32: fn = full ? sw_exact_fast_kernel<true, 32> : sw_exact_fast_kernel<false, 32>; break;
                    default: break;
                }
                if (!fn) return fail(ctx, ZOE_CUDA_E_STATE, "internal error: no literal kernel for %d lanes", N);
                // short lists with known end cells: one CTA per pair (latency), else one group of N threads per pair
                void (*fn_cta)(const ExactFastParams) = N == 8 ? sw_exact_cta_kernel<8> : (N == 16 ? sw_exact_cta_kernel<16> : sw_exact_cta_kernel<32>);
                const size_t cta_smem = exact_cta_smem_bytes(vcap, ctx->S, N);
                const int cta_env = getenv("ZOE_CUDA_EXACT_CTA") ? atoi(getenv("ZOE_CUDA_EXACT_CTA")) : -1;  // 0 never, 1 always
                const bool use_cta = !full && cta_smem <= 200 * 1024 &&
                                     (cta_env == 1 || (cta_env != 0 && cnt[which] <= 4u * (uint32_t)d.sm_count));
                if (use_cta) CU(ctx, cudaFuncSetAttribute(fn_cta, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cta_smem));
                CU(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                for (uint32_t r0 = 0; r0 < cnt[which]; r0 += round) {
                    x.list = d.ex_lists.as<uint32_t>() + (size_t)which * n_exact + r0;
                    x.list_count = std::min<uint32_t>(round, cnt[which] - r0);
                    if (use_cta) {
                        fn_cta<<<std::min<uint32_t>(x.list_count, 2u * (uint32_t)d.sm_count), N * 32, cta_smem, stream>>>(x);
                    } else {
                        const uint32_t blocks = std::min<uint32_t>((uint32_t)d.sm_count, (x.list_count + groups - 1) / groups);
                        fn<<<blocks, groups * N, smem, stream>>>(x);
                    }
                    CU(ctx, cudaGetLastError());
                    sw_exact_walk_kernel<<<(x.list_count + 127) / 128, 128, 0, stream>>>(x, full ? 1 : 0);
                    CU(ctx, cudaGetLastError());
                    ctx->last_launches += 2;
                }
            }
            uint32_t n_slow = cnt[4];
            if (any_fast) {  // walks that left their window were appended to the slow list (none, unless the bound is wrong)
                CU(ctx, cudaMemcpyAsync(&n_slow, d.ex_counts.as<uint32_t>() + 4, sizeof(n_slow), cudaMemcpyDeviceToHost, stream));
                CU(ctx, cudaStreamSynchronize(stream));
            }
            if (n_slow == 0) return 0;
            const uint64_t vcap = ((uint64_t)ctx->max_prof_len + 64 + 3) & ~3ull;  // multiple of 4: rows stay word-aligned
            const uint64_t fcap = (uint64_t)n_rows_max * vcap;
            // per-slot scratch of the literal kernel: the flag matrix and four H / E rows; as many slots as the budget
            // allows (the kernel loops over the list), at least one block
            uint32_t slots = std::min<uint32_t>(n_slow, (uint32_t)d.sm_count * 16);
            slots = (uint32_t)std::min<uint64_t>(slots, std::max<uint64_t>(ex_budget / (fcap + 16 * vcap), 1));
            slots = (slots + 3u) & ~3u;
            CU(ctx, d.ex_hbuf.reserve((size_t)slots * 4 * vcap * sizeof(int32_t)));
            CU(ctx, d.ex_fbuf.reserve((size_t)slots * fcap));
            ExactParams x{};
            x.pair_ids = d.hazard_list.as<uint32_t>();
            x.pos_list = d.ex_lists.as<uint32_t>() + (size_t)4 * n_exact;
            x.n_pairs_dev = nullptr;
            x.n_pairs = n_slow;
            x.rseq = p.rseq;
            x.roff = p.roff;
            x.pbytes = d.pbytes.as<uint8_t>();
            x.coff = p.coff;
            x.n_cseq = n_prof;
            x.weights = d.weights.as<int8_t>();
            x.S = ctx->S;
            x.lut = p.lut;
            x.go = ctx->go;
            x.ge = ctx->ge;
            x.lanes8 = ctx->lanes[0];
            x.lanes16 = ctx->lanes[1];
            x.lanes32 = ctx->lanes[2];
            x.invert = invert;
            x.hbuf = d.ex_hbuf.as<int32_t>();
            x.fbuf = d.ex_fbuf.as<uint8_t>();
            x.vcap = vcap;
            x.fcap = fcap;
            x.score_in = t.score;
            x.ref_start = t.ref_start;
            x.ref_end = t.ref_end;
            x.query_start = t.query_start;
            x.query_end = t.query_end;
            x.cig_scratch = d.ex_cig.as<uint32_t>();
            x.cig_count = t.cig_count;
            x.cig_cap = cig_cap;
            x.counters = ctr;
            x.tp = ctx->tp;
            // four warps per block when their H/E rows fit in shared memory, else global scratch
            // per warp: H/E rows + the current flag row + profiled symbol indices + the weight matrix (<= 64 x 64)
            const size_t rows_bytes = (size_t)4 * vcap * sizeof(int32_t) + 2 * vcap + 4096;
            x.rows_in_smem = rows_bytes * 4 <= 200 * 1024 ? 1 : 0;
            const size_t ex_smem = x.rows_in_smem ? rows_bytes * 4 : 0;
            if (ex_smem > 48 * 1024)
                CU(ctx, cudaFuncSetAttribute(sw_align_exact_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ex_smem));
            if (x.rows_in_smem)
                sw_align_exact_kernel<true><<<slots / 4, 128, ex_smem, stream>>>(x);
            else
                sw_align_exact_kernel<false><<<slots / 4, 128, 0, stream>>>(x);
            CU(ctx, cudaGetLastError());
            ctx->last_launches++;
            return 0;
        };
        const uint32_t cpairs = cn * n_prof;
        if (long_mode) {
            collect_mapped_kernel<<<(cpairs + 255) / 256, 256, 0, d.stream>>>(d.ends.as<AlignEnd>(), d.status.as<uint8_t>(),
                                                                              (uint32_t)(c0 * n_prof), cpairs, t.best_arr, t.hazard,
                                                                              t.cig_count, t.hazard_list, ctr);
            CU(ctx, cudaGetLastError());
            ctx->last_launches++;
        } else if (!use_window) {
            sw_traceback_kernel<<<(cpairs + 127) / 128, 128, 0, d.stream>>>(t);
            CU(ctx, cudaGetLastError());
            ctx->last_launches++;
        } else {
            // ---- checkpointed-window pipeline: scan -> classify -> bucket -> scatter -> window fill -> walk ----
            WinParams wp{};
            wp.s = p;
            wp.ends = ap.ends;
            wp.chunk_first = (uint32_t)c0;
            wp.ckpt = d.ckpt.as<uint32_t>();
            wp.ckpt_base = d.ckpt_base.as<uint64_t>();
            wp.ckpt_task_stride = ckpt_task_stride;
            wp.cb_log2 = cb_log2;
            wp.slack = win_slack;
            wp.nblk = nblk;
            wp.hist = d.win_hist.as<uint32_t>();
            wp.bucket_start = d.win_bucket.as<uint32_t>();
            wp.items = d.win_items.as<uint32_t>();
            wp.n_items = d.win_nitems.as<uint32_t>();
            wp.flags = d.flags.as<uint32_t>();
            wp.win_task_stride = win_task_stride;
            wp.wmax = wmax;
            wp.counters = ctr;
            const uint64_t max_items = (uint64_t)cpairs + n_keys + 2;
            CU(ctx, cudaEventRecord(d.ev_k0, d.stream));
            {
                const uint32_t gpa = plan.threads / k->G, units = (p.n_tasks + scan_tpg - 1) / scan_tpg;
                const uint32_t nba = std::min<uint32_t>((uint32_t)(d.sm_count * plan.blocks_per_sm), (units + gpa - 1) / gpa);
                // split upload: pass A on the sequences of the first part now, on the others once all has arrived (the
                // second launch continues the chunk: checkpoints are indexed by chunk-relative task)
                const uint32_t t_a = (c0 == 0 && scan_tpg == 1) ? first_part_tasks(d, p.n_tasks, nba * gpa) : 0;
                if (t_a) {
                    WinParams wa = wp;
                    wa.s.n_rseq = 2 * t_a;
                    wa.s.n_tasks = t_a;
                    scan_fn<<<nba, plan.threads, plan.smem, d.stream>>>(wa);
                    CU(ctx, cudaGetLastError());
                    ctx->last_launches++;
                    if (int rc0 = ensure_resident(ctx, d)) return rc0;
                    wa.chunk_first = wp.chunk_first + 2 * t_a;
                    wa.s.n_rseq = cn - 2 * t_a;
                    wa.s.n_tasks = (wa.s.n_rseq + 1) / 2;
                    wa.ckpt = wp.ckpt + (size_t)t_a * ckpt_task_stride;
                    const GridShape gs = balance_grid(d, plan, k->G, wa.s.n_tasks);
                    scan_fn<<<gs.blocks, gs.threads, plan.smem, d.stream>>>(wa);
                } else {
                    if (int rc0 = ensure_resident(ctx, d)) return rc0;
                    const GridShape gs = scan_tpg == 1 ? balance_grid(d, plan, k->G, units) : GridShape{nba, (uint32_t)plan.threads};
                    scan_fn<<<gs.blocks, gs.threads, plan.smem, d.stream>>>(wp);
                }
            }
            CU(ctx, cudaGetLastError());
            ClassifyParams cp{};
            cp.ends = ap.ends;
            cp.roff = p.roff;
            cp.coff = p.coff;
            cp.n_cseq = n_prof;
            cp.chunk_first = (uint32_t)c0;
            cp.n_slots = cn;
            cp.K = k->K;
            cp.cb_log2 = cb_log2;
            cp.slack = win_slack;
            cp.maxw = std::max(ctx->max_weight, 0);
            cp.go = ctx->go;
            cp.ge = ctx->ge;
            cp.nblk = nblk;
            cp.all_exact = all_exact ? 1 : 0;
            cp.tp = ctx->tp;
            cp.hist = wp.hist;
            cp.best_arr = t.best_arr;
            cp.score = t.score;
            cp.status = t.status;
            cp.tier = t.tier;
            cp.hazard = t.hazard;
            cp.ref_start = t.ref_start;
            cp.ref_end = t.ref_end;
            cp.query_start = t.query_start;
            cp.query_end = t.query_end;
            cp.cig_count = t.cig_count;
            cp.counters = ctr;
            cp.hazard_list = t.hazard_list;
            // counting sort of the selected pairs by (profiled sequence, checkpoint block) into `items`
            cp.amb = d.win_amb.as<uint8_t>();
            auto bucket = [&](int pin_stage, int subset, uint32_t *items, uint32_t *n_items) -> int {
                cp.pin_stage = pin_stage;
                cp.subset = subset;
                CU(ctx, cudaMemsetAsync(d.win_hist.p, 0, n_keys * sizeof(uint32_t), d.stream));
                CU(ctx, cudaMemsetAsync(items, 0xff, max_items * sizeof(uint32_t), d.stream));
                win_classify_kernel<<<(cpairs + 255) / 256, 256, 0, d.stream>>>(cp);
                CU(ctx, cudaGetLastError());
                win_bucket_scan_kernel<<<1, 1024, 0, d.stream>>>(wp.hist, n_keys, wp.bucket_start, n_items);
                CU(ctx, cudaGetLastError());
                win_scatter_kernel<<<(cpairs + 255) / 256, 256, 0, d.stream>>>(cp, wp.bucket_start, items);
                CU(ctx, cudaGetLastError());
                ctx->last_launches += 3;
                return 0;
            };
            TraceWinParams tw{};
            tw.t = t;
            tw.items = wp.items;
            tw.n_items = wp.n_items;
            tw.wflags = wp.flags;
            tw.win_task_stride = win_task_stride;
            tw.cb_log2 = cb_log2;
            tw.slack = win_slack;
            // Small chunks: the pin sweep (second stream) must fit on an SM beside a window-fill CTA -- shared memory AND
            // registers (a 512-thread fill CTA holds 61k of the 64k registers) -- so the fill runs with 384 threads and the
            // pin with 128, one CTA each per SM.
            const bool small_chunk = cpairs <= 400000u && plan_b.threads >= 384 && 384 % k->G == 0 && plan_p.threads >= 128 &&
                                     128 % k->G == 0 && !getenv("ZOE_CUDA_NO_PIN_OVERLAP");
            auto fill_and_walk = [&](bool beside_pin) -> int {  // window fill + walk of the pairs in wp.items
                WinParams wb = wp;
                wb.pin_mode = 0;
                wb.s.cols_in_smem = plan_b.cols_in_smem;
                const int fthreads = beside_pin ? 384 : plan_b.threads;
                const size_t fsmem = beside_pin ? score_smem_bytes(ctx, *k, fthreads, plan_b.cols_in_smem, ctx->ccodes.size()) : plan_b.smem;
                const uint32_t gpb = fthreads / k->G;
                const uint32_t nb = std::min<uint32_t>((uint32_t)(d.sm_count * (beside_pin ? 1 : plan_b.blocks_per_sm)),
                                                       (uint32_t)((max_items / 2 + gpb - 1) / gpb));
                k->winfill<<<nb, fthreads, fsmem, d.stream>>>(wb);
                CU(ctx, cudaGetLastError());
                sw_traceback_win_kernel<<<(uint32_t)((max_items + 127) / 128), 128, 0, d.stream>>>(tw);
                CU(ctx, cudaGetLastError());
                ctx->last_launches += 2;
                return 0;
            };
            // ---- pin stage: pairs whose maximum recurs in the winning lane get their exact best cell.  Few pairs, long
            //      sweeps: latency bound (1.6 ms whatever the batch size), so it runs on a second stream beside the
            //      window fill + walk of the unambiguous pairs; the pinned pairs follow in a second, short pass ----
            rc = bucket(1, 0, d.win_pitems.as<uint32_t>(), d.win_pnitems.as<uint32_t>());
            if (rc) return rc;
            CU(ctx, cudaEventRecord(d.ev_fork, d.stream));
            CU(ctx, cudaStreamWaitEvent(d.aux_stream, d.ev_fork, 0));
            {
                WinParams wq = wp;
                wq.pin_mode = 1;
                wq.items = d.win_pitems.as<uint32_t>();
                wq.n_items = d.win_pnitems.as<uint32_t>();
                wq.s.cols_in_smem = plan_p.cols_in_smem;
                const int pin_threads = small_chunk ? 128 : plan_p.threads;
                const size_t pin_smem = small_chunk ? score_smem_bytes(ctx, *k, pin_threads, plan_p.cols_in_smem, ctx->ccodes.size())
                                                    : plan_p.smem;
                const uint32_t gpb = pin_threads / k->G;
                const uint32_t nb = std::min<uint32_t>(small_chunk ? (uint32_t)d.sm_count : (uint32_t)(d.sm_count * plan_p.blocks_per_sm),
                                                       (uint32_t)((max_items / 2 + gpb - 1) / gpb));
                k->pin<<<nb, pin_threads, pin_smem, d.aux_stream>>>(wq);
                CU(ctx, cudaGetLastError());
                ctx->last_launches++;
            }
            CU(ctx, cudaEventRecord(d.ev_join, d.aux_stream));
            // ---- classification proper, window fill, walk: the unambiguous pairs, then the pinned ones ----
            rc = bucket(0, 1, wp.items, wp.n_items);
            if (rc) return rc;
            rc = fill_and_walk(small_chunk);
            if (rc) return rc;
            CU(ctx, cudaStreamWaitEvent(d.stream, d.ev_join, 0));
            rc = bucket(0, 2, wp.items, wp.n_items);
            if (rc) return rc;
            rc = fill_and_walk(false);
            if (rc) return rc;
            CU(ctx, cudaEventRecord(d.ev_k1, d.stream));
        }

        unsigned long long hc[5] = {0, 0, 0, 0, 0};  // ctr[4..8]
        CU(ctx, cudaMemcpyAsync(hc, ctr + 4, sizeof(hc), cudaMemcpyDeviceToHost, d.stream));
        CU(ctx, cudaStreamSynchronize(d.stream));
        {
            float ms = 0.f;
            CU(ctx, cudaEventElapsedTime(&ms, d.ev_k0, d.ev_k1));
            dp_ms_total += ms;
        }
        const uint32_t n_exact = (uint32_t)hc[1];
        dbg.lap("align: fill+traceback");
        if (getenv("ZOE_CUDA_DEBUG"))
            fprintf(stderr, "[zoe_cuda] chunk %llu: wide_seqs %llu exact %llu cig_ovf %llu mismatch %llu overflow %llu\n",
                    (unsigned long long)c0, hc[0], hc[1], hc[2], hc[3], hc[4]);
        if (hc[4] > 0 && n_exact > 0) {
            // packed overflow: exact scores from the 32-bit score kernel (or_else_overflowed, output.rs:81-83)
            collect_wide_range_kernel<<<(cn + 255) / 256, 256, 0, d.stream>>>(d.best.as<int32_t>(), (uint32_t)c0, cn, n_prof,
                                                                              d.wide_ids.as<uint32_t>(), ctr);
            CU(ctx, cudaGetLastError());
            unsigned long long n_wide = 0;
            CU(ctx, cudaMemcpyAsync(&n_wide, ctr + 4, sizeof(n_wide), cudaMemcpyDeviceToHost, d.stream));
            CU(ctx, cudaStreamSynchronize(d.stream));
            rc = launch_score(ctx, d, *k, false, d.wide_ids.as<uint32_t>(), (uint32_t)n_wide);
            if (rc) return rc;
            apply_wide_scores_kernel<<<(n_exact + 255) / 256, 256, 0, d.stream>>>(
                d.hazard_list.as<uint32_t>(), n_exact, d.best.as<int32_t>(), t.score, t.status, t.tier, ctx->tp);
            CU(ctx, cudaGetLastError());
            ctx->last_launches += 2;
            {
                std::lock_guard<std::mutex> lk(ctx->mu);
                ctx->stats.rerun_wide += hc[4];
            }
        }
        if (n_exact > 0) {
            rc = launch_exact(n_exact, d.stream);
            if (rc) return rc;
        }
        if (n_exact > 0) {
            std::lock_guard<std::mutex> lk(ctx->mu);
            ctx->stats.hazard += n_exact - hc[4];
        }
        // ---- CIGAR compaction, chained through the device-side running base ctr[9] ----
        if (cpairs >= (1u << 16)) {  // three short launches instead of one block walking a million counts
            const uint32_t nbk = (cpairs + 1023) / 1024;
            CU(ctx, d.cig_bsum.reserve((size_t)nbk * sizeof(unsigned long long)));
            cigar_block_sum_kernel<<<nbk, 1024, 0, d.stream>>>(t.cig_count, (uint64_t)c0 * n_prof, cpairs,
                                                               d.cig_bsum.as<unsigned long long>());
            CU(ctx, cudaGetLastError());
            cigar_scan_sums_kernel<<<1, 1024, 0, d.stream>>>(d.cig_bsum.as<unsigned long long>(), nbk, ctr + 9,
                                                             d.cig_off.as<uint64_t>() + (uint64_t)c0 * n_prof + cpairs);
            CU(ctx, cudaGetLastError());
            cigar_block_scan_kernel<<<nbk, 1024, 0, d.stream>>>(t.cig_count, (uint64_t)c0 * n_prof, cpairs,
                                                                d.cig_bsum.as<unsigned long long>(), d.cig_off.as<uint64_t>());
            CU(ctx, cudaGetLastError());
            ctx->last_launches += 2;
        } else {
            cigar_scan_kernel<<<1, 1024, 0, d.stream>>>(t.cig_count, (uint64_t)c0 * n_prof, cpairs, d.cig_off.as<uint64_t>(),
                                                        ctr + 9);
            CU(ctx, cudaGetLastError());
        }
        cigar_gather_kernel<<<cpairs, 32, 0, d.stream>>>(t.cig_scratch, cig_cap, nullptr, cpairs, (uint32_t)(c0 * n_prof),
                                                         t.cig_count, d.cig_off.as<uint64_t>(), d.cig_out.as<uint32_t>(),
                                                         cigar_cap_words, t.hazard);
        CU(ctx, cudaGetLastError());
        ctx->last_launches += 2;
        if (n_exact > 0) {
            cigar_gather_kernel<<<n_exact, 32, 0, d.stream>>>(d.ex_cig.as<uint32_t>(), cig_cap, d.hazard_list.as<uint32_t>(),
                                                              n_exact, 0, t.cig_count, d.cig_off.as<uint64_t>(),
                                                              d.cig_out.as<uint32_t>(), cigar_cap_words, nullptr);
            CU(ctx, cudaGetLastError());
            ctx->last_launches++;
        }
    }
    // tier histogram + totals
    CU(ctx, cudaMemsetAsync(ctr, 0, 4 * sizeof(unsigned long long), d.stream));
    count_status_kernel<<<(uint32_t)((pairs + 255) / 256), 256, 0, d.stream>>>(d.tier.as<uint8_t>(), d.status.as<uint8_t>(),
                                                                              pairs, ctr);
    CU(ctx, cudaGetLastError());
    ctx->last_launches++;
    unsigned long long tail[3] = {0, 0, 0};  // ctr[7] score mismatch, [8] overflow, [9] cigar total
    CU(ctx, cudaMemcpyAsync(tail, ctr + 7, sizeof(tail), cudaMemcpyDeviceToHost, d.stream));
    unsigned long long cig_ovf = 0, win_fb[2] = {0, 0};  // ctr[10] walks that left their window, [11] ambiguous ends
    CU(ctx, cudaMemcpyAsync(&cig_ovf, ctr + 6, sizeof(cig_ovf), cudaMemcpyDeviceToHost, d.stream));
    CU(ctx, cudaMemcpyAsync(win_fb, ctr + 10, sizeof(win_fb), cudaMemcpyDeviceToHost, d.stream));
    CU(ctx, cudaStreamSynchronize(d.stream));
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        ctx->stats.window_fallback += win_fb[0];
        ctx->stats.window_pinned += win_fb[1];
        ctx->stats.hazard -= std::min<uint64_t>(ctx->stats.hazard, win_fb[0]);
        ctx->last_dp_ms = std::max(ctx->last_dp_ms, dp_ms_total);
    }
    dbg.lap("align: compaction+tail");
    d.cig_total = tail[2];
    d.timed_kernel = false;  // several fill launches: report their sum instead of one event pair
    if (tail[0]) return fail(ctx, ZOE_CUDA_E_STATE, "internal error: literal kernel disagreed with the fill score on %llu pairs", tail[0]);
    if (cig_ovf) return fail(ctx, ZOE_CUDA_E_STATE, "internal error: CIGAR scratch overflow on %llu pairs", cig_ovf);
    return 0;
}

// ---------------------------------------------------------------------------------------------
// ranges pipeline for long streamed sequences (rows > kMaxRowsSinglePass) or key spaces too large for the bucketed
// reverse pass: sw_ends_long_kernel forward (score + exact end cell) -> mapped pairs -> sw_ends_long_kernel<REV> ->
// ranges_finalize_kernel.  zoe: sw_simd_score_ranges has no length limit (striped.rs:355-388).
// ---------------------------------------------------------------------------------------------
constexpr int kEndsLongK = 24;

template <bool PACKED, bool REV>
int launch_ends_long(zoe_cuda_ctx *ctx, Device &d, EndsLongParams lp, uint32_t n_tasks_bound, uint32_t max_rows) {
    auto fn = sw_ends_long_kernel<kEndsLongK, PACKED, REV>;
    const size_t tab_per_warp = (size_t)ctx->n_csym * (kEndsLongK / 4) * 32 * 16;
    const size_t fixed = 256 + (((size_t)ctx->n_csym * ctx->S + 15) & ~(size_t)15);
    const LaunchPlan *cached = nullptr;
    const PlanKey key{(const void *)fn, ctx->ccodes.size(), 0};
    LaunchPlan plan;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        auto it = ctx->plans.find(key);
        if (it != ctx->plans.end()) {
            plan = it->second;
            cached = &plan;
        }
    }
    if (!cached) {
        int best_warps = 0;
        cudaFuncAttributes fa{};
        CU(ctx, cudaFuncGetAttributes(&fa, fn));
        for (int cols_in_smem = 1; cols_in_smem >= 0 && best_warps == 0; --cols_in_smem) {
            if (cols_in_smem && ctx->ccodes.size() > kColsSmemLimit) continue;
            for (int threads : {512, 448, 384, 320, 256, 192, 128, 64, 32}) {
                if (threads > fa.maxThreadsPerBlock) continue;
                const size_t smem = tab_per_warp * (threads / 32) + fixed + (cols_in_smem ? ((ctx->ccodes.size() + 15) & ~(size_t)15) : 0);
                if (smem > 227 * 1024) continue;
                if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
                    cudaGetLastError();
                    continue;
                }
                int nb = 0;
                if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, threads, smem) != cudaSuccess) {
                    cudaGetLastError();
                    continue;
                }
                if (nb * threads / 32 > best_warps) {
                    best_warps = nb * threads / 32;
                    plan.threads = threads;
                    plan.blocks_per_sm = nb;
                    plan.smem = smem;
                    plan.cols_in_smem = cols_in_smem;
                }
            }
        }
        if (!best_warps) return fail(ctx, ZOE_CUDA_E_UNSUPPORTED, "long-row ends kernel does not fit shared memory (alphabet %d)", ctx->n_csym);
        std::lock_guard<std::mutex> lk(ctx->mu);
        ctx->plans[key] = plan;
    }
    if (n_tasks_bound == 0) return 0;
    const uint32_t wpb = plan.threads / 32;
    const uint32_t R = 32 * kEndsLongK;
    const uint32_t chunk_cap = std::max<uint32_t>(1, (max_rows + R - 1) / R - 1);  // bottom rows of all chunks but the last
    uint32_t blocks = std::min<uint32_t>((uint32_t)(d.sm_count * plan.blocks_per_sm), (n_tasks_bound + wpb - 1) / wpb);
    // boundary rows: [warp slot][chunk][column] x 8 bytes, bounded by the scratch budget (fewer blocks if need be)
    const uint64_t per_block = (uint64_t)wpb * chunk_cap * ctx->max_prof_len * sizeof(uint2);
    uint64_t budget = ctx->flag_budget_bytes ? ctx->flag_budget_bytes : (uint64_t)(d.free_at_create * 0.4);
    budget = std::min<uint64_t>(budget, (uint64_t)32 << 30);
    blocks = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(blocks, budget / std::max<uint64_t>(per_block, 1)));
    CU(ctx, d.long_bnd.reserve((size_t)blocks * per_block));
    CU(ctx, d.long_queue.reserve(sizeof(unsigned int)));
    CU(ctx, cudaMemsetAsync(d.long_queue.p, 0, sizeof(unsigned int), d.stream));
    lp.s.cols_in_smem = plan.cols_in_smem;
    lp.boundary = d.long_bnd.as<uint2>();
    lp.max_L = ctx->max_prof_len;
    lp.chunk_cap = chunk_cap;
    lp.queue = d.long_queue.as<unsigned int>();
    CU(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem));
    fn<<<blocks, plan.threads, plan.smem, d.stream>>>(lp);
    CU(ctx, cudaGetLastError());
    ctx->last_launches++;
    return 0;
}

int run_ranges_long_on_device(zoe_cuda_ctx *ctx, Device &d) {
    if (int rc0 = ensure_resident(ctx, d)) return rc0;
    const uint32_t n_prof = ctx->n_prof;
    const size_t pairs = (size_t)d.n_count * n_prof;
    if (pairs >= 0x7fffffffULL) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "too many pairs for one ranges call");
    // longest first: the two halves of a packed task have similar lengths, the queue hands out the big tasks first
    std::vector<uint32_t> order(d.n_count);
    for (uint64_t i = 0; i < d.n_count; ++i) order[i] = (uint32_t)i;
    if (!ctx->staged_len.empty()) {
        const uint32_t *len = ctx->staged_len.data() + d.n_first;
        std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return len[a] > len[b]; });
    }
    CU(ctx, d.long_ids.reserve(order.size() * sizeof(uint32_t)));
    CU(ctx, cudaMemcpyAsync(d.long_ids.p, order.data(), order.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, d.stream));
    CU(ctx, cudaStreamSynchronize(d.stream));
    CU(ctx, d.ends.reserve(pairs * sizeof(AlignEnd)));
    CU(ctx, d.starts.reserve(pairs * sizeof(AlignEnd)));
    for (DevBuf *b : {&d.ref_start, &d.ref_end, &d.query_start, &d.query_end, &d.score})
        CU(ctx, b->reserve(pairs * sizeof(uint32_t)));
    CU(ctx, d.status.reserve(pairs));
    CU(ctx, d.tier.reserve(pairs));
    CU(ctx, d.win_items.reserve((pairs + 2) * sizeof(uint32_t)));
    CU(ctx, d.win_nitems.reserve(sizeof(uint32_t)));
    CU(ctx, d.counters.reserve(16 * sizeof(unsigned long long)));
    CU(ctx, cudaMemsetAsync(d.counters.p, 0, 16 * sizeof(unsigned long long), d.stream));
    CU(ctx, cudaMemsetAsync(d.win_nitems.p, 0, sizeof(uint32_t), d.stream));
    unsigned long long *ctr = d.counters.as<unsigned long long>();
    // packed 16-bit lanes only when no pair can reach their limit and the step-pair indices fit 16 bits
    const uint64_t bound = (uint64_t)std::min<uint32_t>(ctx->staged_max_len, ctx->max_prof_len) * (uint64_t)std::max(ctx->max_weight, 0);
    const bool packed = bound < (uint64_t)(32767 - std::max(ctx->max_weight, 0) - 1 - ctx->go) && ctx->max_prof_len <= kScanMaxCols;

    EndsLongParams lp{};
    ScoreParams &p = lp.s;
    p.rseq = d.rseq.as<uint8_t>();
    p.roff = d.roff.as<uint64_t>();
    p.task_ids = d.long_ids.as<uint32_t>();
    p.n_rseq = (uint32_t)d.n_count;
    p.n_tasks = packed ? (p.n_rseq + 1) / 2 : p.n_rseq;
    p.ccodes = d.ccodes.as<uint8_t>();
    p.coff = d.coff.as<uint32_t>();
    p.n_cseq = n_prof;
    p.ccodes_bytes = (uint32_t)ctx->ccodes.size();
    p.wk = d.wk.as<int8_t>();
    p.n_csym = ctx->n_csym;
    p.S = ctx->S;
    p.lut = d.lut.as<uint8_t>();
    p.go = ctx->go;
    p.ge = ctx->ge;
    p.ovf_thresh = 0x7fffffff;  // packed lanes cannot overflow here (static bound above)
    lp.out = d.ends.as<AlignEnd>();
    lp.counters = ctr;
    CU(ctx, cudaEventRecord(d.ev_k0, d.stream));
    int rc = packed ? launch_ends_long<true, false>(ctx, d, lp, p.n_tasks, ctx->staged_max_len)
                    : launch_ends_long<false, false>(ctx, d, lp, p.n_tasks, ctx->staged_max_len);
    if (rc) return rc;

    RangesLongParams rl{};
    rl.ends = d.ends.as<AlignEnd>();
    rl.roff = p.roff;
    rl.order = d.long_ids.as<uint32_t>();
    rl.n_seq = (uint32_t)d.n_count;
    rl.n_cseq = n_prof;
    rl.score = d.score.as<uint32_t>();
    rl.status = d.status.as<uint8_t>();
    rl.tier = d.tier.as<uint8_t>();
    rl.ref_start = d.ref_start.as<uint32_t>();
    rl.ref_end = d.ref_end.as<uint32_t>();
    rl.query_start = d.query_start.as<uint32_t>();
    rl.query_end = d.query_end.as<uint32_t>();
    rl.items = d.win_items.as<uint32_t>();
    rl.n_items = d.win_nitems.as<uint32_t>();
    rl.tp = ctx->tp;
    const uint32_t pb = (uint32_t)((pairs + 255) / 256);
    ranges_long_classify_kernel<<<pb, 256, 0, d.stream>>>(rl);
    CU(ctx, cudaGetLastError());

    EndsLongParams lr = lp;
    lr.s.task_ids = nullptr;
    lr.items = d.win_items.as<uint32_t>();
    lr.n_tasks_dev = d.win_nitems.as<uint32_t>();
    lr.rev_in = d.ends.as<AlignEnd>();
    lr.rev_maxw = std::max(ctx->max_weight, 0);
    lr.out = d.starts.as<AlignEnd>();
    rc = packed ? launch_ends_long<true, true>(ctx, d, lr, (uint32_t)pairs, ctx->staged_max_len)
                : launch_ends_long<false, true>(ctx, d, lr, (uint32_t)pairs, ctx->staged_max_len);
    if (rc) return rc;
    CU(ctx, cudaEventRecord(d.ev_k1, d.stream));
    d.timed_kernel = true;

    RangesParams rp{};
    rp.ends = d.ends.as<AlignEnd>();
    rp.starts = d.starts.as<AlignEnd>();
    rp.roff = p.roff;
    rp.n_cseq = n_prof;
    rp.chunk_first = 0;
    rp.n_slots = (uint32_t)d.n_count;
    rp.score = d.score.as<uint32_t>();
    rp.status = d.status.as<uint8_t>();
    rp.tier = d.tier.as<uint8_t>();
    rp.ref_start = d.ref_start.as<uint32_t>();
    rp.ref_end = d.ref_end.as<uint32_t>();
    rp.query_start = d.query_start.as<uint32_t>();
    rp.query_end = d.query_end.as<uint32_t>();
    rp.counters = ctr;
    rp.invert = ctx->profiled_is_query ? 0 : 1;
    rp.tp = ctx->tp;
    ranges_finalize_kernel<<<pb, 256, 0, d.stream>>>(rp);
    CU(ctx, cudaGetLastError());
    count_status_kernel<<<pb, 256, 0, d.stream>>>(d.tier.as<uint8_t>(), d.status.as<uint8_t>(), pairs, ctr);
    CU(ctx, cudaGetLastError());
    ctx->last_launches += 3;
    unsigned long long mism = 0;
    CU(ctx, cudaMemcpyAsync(&mism, ctr + 7, sizeof(mism), cudaMemcpyDeviceToHost, d.stream));
    CU(ctx, cudaStreamSynchronize(d.stream));
    if (mism) return fail(ctx, ZOE_CUDA_E_STATE, "internal error: the long-row ranges passes disagreed on %llu pairs", mism);
    return 0;
}

// ---------------------------------------------------------------------------------------------
// ranges pipeline (one device): forward ends -> bucket by (profiled, c_end) -> reverse ends -> ranges
// ---------------------------------------------------------------------------------------------
int run_ranges_on_device(zoe_cuda_ctx *ctx, Device &d) {
    if (d.n_count == 0) return 0;
    CU(ctx, cudaSetDevice(d.id));
    // long rows, or a (profiled, end column) key space too large for the bucketed reverse pass: the chunked-row pipeline
    if (ctx->staged_max_len > (uint32_t)kMaxRowsSinglePass || (uint64_t)ctx->n_prof * ctx->max_prof_len > (1ull << 27) ||
        ctx->max_prof_len > kEndsMaxCols || getenv("ZOE_CUDA_RANGES_LONG"))
        return run_ranges_long_on_device(ctx, d);
    const bool scan_ok = ctx->max_prof_len <= kScanMaxCols && !getenv("ZOE_CUDA_RANGES_SLOW");
    const KernelEntry *k = pick_score_kernel(std::max<uint32_t>(ctx->staged_max_len, 1), ctx->n_csym);
    if (!k) return fail(ctx, ZOE_CUDA_E_UNSUPPORTED, "no kernel for length %u", ctx->staged_max_len);
    const uint32_t n_prof = ctx->n_prof;
    const size_t pairs = (size_t)d.n_count * n_prof;
    if (pairs >= 0x7fffffffULL) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "too many pairs for one ranges call");
    // packed 16-bit lanes only when no pair can reach their limit (otherwise everything runs at 32 bits)
    const uint64_t bound = (uint64_t)std::min<uint32_t>(ctx->staged_max_len, ctx->max_prof_len) * (uint64_t)std::max(ctx->max_weight, 0);
    const bool packed = bound < (uint64_t)(32767 - std::max(ctx->max_weight, 0) - 1 - ctx->go);
    void (*fn)(const EndsParams) = packed ? k->ends : k->ends_wide;
    LaunchPlan plan;
    int rc = plan_launch(ctx, *k, fn, &plan);
    if (rc) return rc;
    CU(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem));

    const uint32_t key_stride = ctx->max_prof_len;
    const uint64_t n_keys = (uint64_t)n_prof * key_stride;
    const uint64_t max_items = pairs + n_keys + 2;
    CU(ctx, d.ends.reserve(pairs * sizeof(AlignEnd)));
    CU(ctx, d.starts.reserve(pairs * sizeof(AlignEnd)));
    for (DevBuf *b : {&d.ref_start, &d.ref_end, &d.query_start, &d.query_end, &d.score})
        CU(ctx, b->reserve(pairs * sizeof(uint32_t)));
    CU(ctx, d.status.reserve(pairs));
    CU(ctx, d.tier.reserve(pairs));
    CU(ctx, d.win_hist.reserve(n_keys * sizeof(uint32_t)));
    CU(ctx, d.win_bucket.reserve((n_keys + 1) * sizeof(uint32_t)));
    CU(ctx, d.win_items.reserve(max_items * sizeof(uint32_t)));
    CU(ctx, d.win_nitems.reserve(sizeof(uint32_t)));
    CU(ctx, d.counters.reserve(16 * sizeof(unsigned long long)));
    CU(ctx, cudaMemsetAsync(d.counters.p, 0, 16 * sizeof(unsigned long long), d.stream));
    CU(ctx, cudaMemsetAsync(d.win_hist.p, 0, n_keys * sizeof(uint32_t), d.stream));
    CU(ctx, cudaMemsetAsync(d.win_items.p, 0xff, max_items * sizeof(uint32_t), d.stream));
    unsigned long long *ctr = d.counters.as<unsigned long long>();

    EndsParams ep{};
    ScoreParams &p = ep.s;
    p.rseq = d.rseq.as<uint8_t>();
    p.roff = d.roff.as<uint64_t>();
    p.n_rseq = (uint32_t)d.n_count;
    p.n_tasks = packed ? (p.n_rseq + 1) / 2 : p.n_rseq;
    p.ccodes = d.ccodes.as<uint8_t>();
    p.coff = d.coff.as<uint32_t>();
    p.n_cseq = n_prof;
    p.ccodes_bytes = (uint32_t)ctx->ccodes.size();
    p.cols_in_smem = plan.cols_in_smem;
    p.wk = d.wk.as<int8_t>();
    p.n_csym = ctx->n_csym;
    p.S = ctx->S;
    p.lut = d.lut.as<uint8_t>();
    p.go = ctx->go;
    p.ge = ctx->ge;
    p.ovf_thresh = 0x7fffffff;  // packed lanes cannot overflow here (static bound above)
    ep.chunk_first = 0;
    ep.items = nullptr;
    ep.n_items = nullptr;
    ep.ends_in = nullptr;
    ep.out = d.ends.as<AlignEnd>();
    const uint32_t gpb = plan.threads / k->G;
    const uint32_t max_blocks = (uint32_t)(d.sm_count * plan.blocks_per_sm);
    CU(ctx, cudaEventRecord(d.ev_k0, d.stream));
    if (packed && scan_ok) {
        // ---- forward pass, fast: the align pipeline's pass A (score-rate scan + checkpoints) followed by a pin sweep
        //      of every mapped pair from the checkpoint before its first best column pair (about CB/2 columns) ----
        int cb_log2 = ctx->win_cb_log2;
        while ((1 << cb_log2) < k->G) ++cb_log2;
        const int CKW = ckpt_words_per_lane(k->K);
        std::vector<uint64_t> ckpt_base(n_prof);
        uint64_t ckpt_task_stride = 0;
        uint32_t nblk = 1;
        for (uint32_t j = 0; j < n_prof; ++j) {
            const uint64_t L = ctx->coff[j + 1] - ctx->coff[j];
            ckpt_base[j] = ckpt_task_stride;
            ckpt_task_stride += ((L - 1) >> cb_log2) * (uint64_t)CKW * k->G;
            nblk = std::max<uint32_t>(nblk, (uint32_t)((L - 1) >> cb_log2) + 1);
        }
        const uint32_t pin_keys = n_prof * nblk;
        uint64_t budget = ctx->flag_budget_bytes ? ctx->flag_budget_bytes : (uint64_t)(d.free_at_create * 0.55);
        budget = std::min<uint64_t>(budget, (uint64_t)48 << 30);
        uint64_t chunk_seqs = std::min<uint64_t>(d.n_count, 2 * std::max<uint64_t>(1, budget / std::max<uint64_t>(ckpt_task_stride * 4, 1)));
        if (chunk_seqs > 1) chunk_seqs &= ~1ULL;
        LaunchPlan plan_a, plan_p;
        void (*scan_fn)(const WinParams) = k->scan;
        int rc2 = plan_launch(ctx, *k, scan_fn, &plan_a);
        if (rc2) return rc2;
        if (!plan_a.cols_in_smem) {
            scan_fn = k->scan_g;
            rc2 = plan_launch(ctx, *k, scan_fn, &plan_a);
            if (rc2) return rc2;
        }
        int scan_tpg = 1;
        pick_scan2(ctx, *k, &scan_fn, &plan_a, &scan_tpg);
        rc2 = plan_launch(ctx, *k, k->pin, &plan_p);
        if (rc2) return rc2;
        CU(ctx, cudaFuncSetAttribute(scan_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan_a.smem));
        CU(ctx, cudaFuncSetAttribute(k->pin, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan_p.smem));
        CU(ctx, d.ckpt.reserve(std::max<uint64_t>(((chunk_seqs + 1) / 2) * ckpt_task_stride * 4, 16)));
        if (!d.ckpt_base_cached(ctx->profiled_epoch, k->G, k->K, cb_log2)) {
            CU(ctx, d.ckpt_base.reserve(n_prof * sizeof(uint64_t)));
            CU(ctx, cudaMemcpyAsync(d.ckpt_base.p, ckpt_base.data(), n_prof * sizeof(uint64_t), cudaMemcpyHostToDevice, d.stream));
            CU(ctx, cudaStreamSynchronize(d.stream));
            d.ckpt_base_mark(ctx->profiled_epoch, k->G, k->K, cb_log2);
        }
        // (win_hist / win_bucket / win_items are sized for the larger key space of the reverse pass below)
        for (uint64_t c0 = 0; c0 < d.n_count; c0 += chunk_seqs) {
            const uint32_t cn = (uint32_t)std::min<uint64_t>(chunk_seqs, d.n_count - c0);
            const uint32_t cpairs = cn * n_prof;
            const uint64_t chunk_items = (uint64_t)cpairs + pin_keys + 2;
            WinParams wp{};
            wp.s = p;
            wp.s.n_rseq = cn;
            wp.s.n_tasks = (cn + 1) / 2;
            wp.s.cols_in_smem = plan_a.cols_in_smem;
            wp.ends = d.ends.as<AlignEnd>();
            wp.chunk_first = (uint32_t)c0;
            wp.ckpt = d.ckpt.as<uint32_t>();
            wp.ckpt_base = d.ckpt_base.as<uint64_t>();
            wp.ckpt_task_stride = ckpt_task_stride;
            wp.cb_log2 = cb_log2;
            wp.slack = ctx->win_slack;
            wp.nblk = nblk;
            wp.hist = d.win_hist.as<uint32_t>();
            wp.bucket_start = d.win_bucket.as<uint32_t>();
            wp.items = d.win_items.as<uint32_t>();
            wp.n_items = d.win_nitems.as<uint32_t>();
            wp.counters = ctr;
            const uint32_t gpa = plan_a.threads / k->G, units = (wp.s.n_tasks + scan_tpg - 1) / scan_tpg;
            {
                const uint32_t nba = std::min<uint32_t>((uint32_t)(d.sm_count * plan_a.blocks_per_sm), (units + gpa - 1) / gpa);
                const uint32_t t_a = (c0 == 0 && scan_tpg == 1) ? first_part_tasks(d, wp.s.n_tasks, nba * gpa) : 0;
                if (t_a) {  // split upload: see run_align_on_device
                    WinParams wa = wp;
                    wa.s.n_rseq = 2 * t_a;
                    wa.s.n_tasks = t_a;
                    scan_fn<<<nba, plan_a.threads, plan_a.smem, d.stream>>>(wa);
                    CU(ctx, cudaGetLastError());
                    ctx->last_launches++;
                    if (int rc0 = ensure_resident(ctx, d)) return rc0;
                    wa.chunk_first = wp.chunk_first + 2 * t_a;
                    wa.s.n_rseq = cn - 2 * t_a;
                    wa.s.n_tasks = (wa.s.n_rseq + 1) / 2;
                    wa.ckpt = wp.ckpt + (size_t)t_a * ckpt_task_stride;
                    const GridShape gs = balance_grid(d, plan_a, k->G, wa.s.n_tasks);
                    scan_fn<<<gs.blocks, gs.threads, plan_a.smem, d.stream>>>(wa);
                } else {
                    if (int rc0 = ensure_resident(ctx, d)) return rc0;
                    const GridShape gs = scan_tpg == 1 ? balance_grid(d, plan_a, k->G, units) : GridShape{nba, (uint32_t)plan_a.threads};
                    scan_fn<<<gs.blocks, gs.threads, plan_a.smem, d.stream>>>(wp);
                }
            }
            CU(ctx, cudaGetLastError());
            ClassifyParams cp{};
            cp.ends = d.ends.as<AlignEnd>();
            cp.roff = p.roff;
            cp.coff = p.coff;
            cp.n_cseq = n_prof;
            cp.chunk_first = (uint32_t)c0;
            cp.n_slots = cn;
            cp.K = k->K;
            cp.cb_log2 = cb_log2;
            cp.slack = ctx->win_slack;
            cp.maxw = std::max(ctx->max_weight, 0);
            cp.go = ctx->go;
            cp.ge = ctx->ge;
            cp.nblk = nblk;
            cp.all_exact = 0;
            cp.tp = ctx->tp;
            cp.hist = wp.hist;
            cp.counters = ctr;
            cp.pin_stage = 2;
            CU(ctx, cudaMemsetAsync(d.win_hist.p, 0, pin_keys * sizeof(uint32_t), d.stream));
            CU(ctx, cudaMemsetAsync(d.win_items.p, 0xff, chunk_items * sizeof(uint32_t), d.stream));
            win_classify_kernel<<<(cpairs + 255) / 256, 256, 0, d.stream>>>(cp);
            CU(ctx, cudaGetLastError());
            win_bucket_scan_kernel<<<1, 1024, 0, d.stream>>>(wp.hist, pin_keys, wp.bucket_start, wp.n_items);
            CU(ctx, cudaGetLastError());
            win_scatter_kernel<<<(cpairs + 255) / 256, 256, 0, d.stream>>>(cp, wp.bucket_start, wp.items);
            CU(ctx, cudaGetLastError());
            WinParams wq = wp;
            wq.pin_mode = 2;
            wq.s.cols_in_smem = plan_p.cols_in_smem;
            const uint32_t gpp = plan_p.threads / k->G;
            k->pin<<<std::min<uint32_t>((uint32_t)(d.sm_count * plan_p.blocks_per_sm), (uint32_t)((chunk_items / 2 + gpp - 1) / gpp)),
                     plan_p.threads, plan_p.smem, d.stream>>>(wq);
            CU(ctx, cudaGetLastError());
            ctx->last_launches += 5;
        }
        CU(ctx, cudaMemsetAsync(d.win_hist.p, 0, n_keys * sizeof(uint32_t), d.stream));
        CU(ctx, cudaMemsetAsync(d.win_items.p, 0xff, max_items * sizeof(uint32_t), d.stream));
    } else {
        if (int rc0 = ensure_resident(ctx, d)) return rc0;
        fn<<<std::min<uint32_t>(max_blocks, (p.n_tasks + gpb - 1) / gpb), plan.threads, plan.smem, d.stream>>>(ep);
        CU(ctx, cudaGetLastError());
    }

    RangesParams rp{};
    rp.ends = d.ends.as<AlignEnd>();
    rp.starts = d.starts.as<AlignEnd>();
    rp.roff = p.roff;
    rp.n_cseq = n_prof;
    rp.chunk_first = 0;
    rp.n_slots = (uint32_t)d.n_count;
    rp.key_stride = key_stride;
    rp.hist = d.win_hist.as<uint32_t>();
    rp.score = d.score.as<uint32_t>();
    rp.status = d.status.as<uint8_t>();
    rp.tier = d.tier.as<uint8_t>();
    rp.ref_start = d.ref_start.as<uint32_t>();
    rp.ref_end = d.ref_end.as<uint32_t>();
    rp.query_start = d.query_start.as<uint32_t>();
    rp.query_end = d.query_end.as<uint32_t>();
    rp.counters = ctr;
    rp.invert = ctx->profiled_is_query ? 0 : 1;
    rp.tp = ctx->tp;
    const uint32_t pb = (uint32_t)((pairs + 255) / 256);
    ranges_classify_kernel<<<pb, 256, 0, d.stream>>>(rp);
    CU(ctx, cudaGetLastError());
    win_bucket_scan_kernel<<<1, 1024, 0, d.stream>>>(rp.hist, (uint32_t)n_keys, d.win_bucket.as<uint32_t>(), d.win_nitems.as<uint32_t>());
    CU(ctx, cudaGetLastError());
    ranges_scatter_kernel<<<pb, 256, 0, d.stream>>>(rp, d.win_bucket.as<uint32_t>(), d.win_items.as<uint32_t>());
    CU(ctx, cudaGetLastError());

    const uint64_t max_tasks = packed ? max_items / 2 : max_items;
    LaunchPlan plan_r;
    bool fast_rev = packed && scan_ok;
    if (fast_rev) {
        int rc2 = plan_launch(ctx, *k, k->scan_rev, &plan_r);
        if (rc2) return rc2;
        fast_rev = plan_r.cols_in_smem != 0;  // the reverse instantiation reads the profiled codes from shared memory
    }
    if (fast_rev) {
        // ---- reverse pass, fast: pass A's recurrence and bookkeeping over the reversed, truncated sub-problems, the
        //      exact start cell pinned by re-sweeping the first columns inside the same kernel ----
        CU(ctx, cudaFuncSetAttribute(k->scan_rev, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan_r.smem));
        WinParams wr{};
        wr.s = p;
        wr.s.cols_in_smem = 1;
        wr.items = d.win_items.as<uint32_t>();
        wr.n_items = d.win_nitems.as<uint32_t>();
        wr.rev_in = d.ends.as<AlignEnd>();
        wr.rev_maxw = getenv("ZOE_CUDA_REV_FULL") ? 0x3fffffff / 2048 : std::max(ctx->max_weight, 0);  // env: sweep the whole prefix
        wr.rev_out = d.starts.as<AlignEnd>();
        wr.counters = ctr;
        wr.cb_log2 = ctx->win_cb_log2;
        const uint32_t gpr = plan_r.threads / k->G;
        k->scan_rev<<<std::min<uint32_t>((uint32_t)(d.sm_count * plan_r.blocks_per_sm), (uint32_t)((max_tasks + gpr - 1) / gpr)),
                      plan_r.threads, plan_r.smem, d.stream>>>(wr);
        CU(ctx, cudaGetLastError());
    } else {
        EndsParams er = ep;
        er.items = d.win_items.as<uint32_t>();
        er.n_items = d.win_nitems.as<uint32_t>();
        er.ends_in = d.ends.as<AlignEnd>();
        er.out = d.starts.as<AlignEnd>();
        fn<<<std::min<uint32_t>(max_blocks, (uint32_t)((max_tasks + gpb - 1) / gpb)), plan.threads, plan.smem, d.stream>>>(er);
        CU(ctx, cudaGetLastError());
    }
    CU(ctx, cudaEventRecord(d.ev_k1, d.stream));
    d.timed_kernel = true;
    ranges_finalize_kernel<<<pb, 256, 0, d.stream>>>(rp);
    CU(ctx, cudaGetLastError());
    count_status_kernel<<<pb, 256, 0, d.stream>>>(d.tier.as<uint8_t>(), d.status.as<uint8_t>(), pairs, ctr);
    CU(ctx, cudaGetLastError());
    ctx->last_launches += 7;
    unsigned long long mism = 0;
    CU(ctx, cudaMemcpyAsync(&mism, ctr + 7, sizeof(mism), cudaMemcpyDeviceToHost, d.stream));
    CU(ctx, cudaStreamSynchronize(d.stream));
    if (mism) return fail(ctx, ZOE_CUDA_E_STATE, "internal error: reverse pass disagreed with the forward score on %llu pairs", mism);
    return 0;
}

// ---------------------------------------------------------------------------------------------
// 3-pass alignment (one device): ranges pipeline (passes 1 + 2) -> no-gaps shortcut / banded / scalar DP on the
// bounding box (pass 3, sw_3pass.cuh) -> CIGAR compaction.  zoe: sw_align_3pass, src/alignment/sw/three_pass.rs:21-104.
// ---------------------------------------------------------------------------------------------
int run_3pass_on_device(zoe_cuda_ctx *ctx, Device &d, uint64_t cigar_cap_words) {
    d.cig_total = 0;
    if (d.n_count == 0) return 0;
    if (ctx->S > 32) return fail(ctx, ZOE_CUDA_E_UNSUPPORTED, "3-pass alignment supports alphabets up to 32 symbols");
    int rc = run_ranges_on_device(ctx, d);
    if (rc) return rc;
    CU(ctx, cudaSetDevice(d.id));
    const uint32_t n_prof = ctx->n_prof;
    const uint64_t pairs = (uint64_t)d.n_count * n_prof;
    uint64_t budget = ctx->flag_budget_bytes ? ctx->flag_budget_bytes : (uint64_t)(d.free_at_create * 0.4);
    budget = std::min<uint64_t>(budget, (uint64_t)32 << 30);
    uint64_t chunk_pairs = std::min<uint64_t>(pairs, 1ull << 24);
    CU(ctx, d.cig_count.reserve(pairs * sizeof(uint32_t)));
    CU(ctx, d.cig_off.reserve((pairs + 1) * sizeof(uint64_t)));
    CU(ctx, d.cig_out.reserve(std::max<uint64_t>(cigar_cap_words, 1) * sizeof(uint32_t)));
    CU(ctx, d.tp_pair.reserve(chunk_pairs * sizeof(uint32_t)));
    CU(ctx, d.tp_cap.reserve(chunk_pairs * sizeof(uint32_t)));
    CU(ctx, d.tp_slot.reserve(chunk_pairs * sizeof(uint32_t)));
    CU(ctx, d.tp_bw.reserve(2 * chunk_pairs * sizeof(uint32_t)));
    CU(ctx, d.tp_list.reserve(2 * chunk_pairs * sizeof(uint32_t)));
    CU(ctx, d.tp_off.reserve(2 * chunk_pairs * sizeof(unsigned long long)));
    CU(ctx, d.tp_cigoff.reserve(chunk_pairs * sizeof(unsigned long long)));
    CU(ctx, d.tp_ctr.reserve(16 * sizeof(unsigned long long)));
    CU(ctx, cudaMemsetAsync(d.tp_ctr.p, 0, 16 * sizeof(unsigned long long), d.stream));
    unsigned long long *ctr = d.tp_ctr.as<unsigned long long>();

    ThreePassParams t{};
    t.rseq = d.rseq.as<uint8_t>();
    t.roff = d.roff.as<uint64_t>();
    t.pbytes = d.pbytes.as<uint8_t>();
    t.coff = d.coff.as<uint32_t>();
    t.n_cseq = n_prof;
    t.weights = d.weights.as<int8_t>();
    t.S = ctx->S;
    t.lut = d.lut.as<uint8_t>();
    t.go = -ctx->go;
    t.ge = -ctx->ge;
    t.invert = ctx->profiled_is_query ? 0 : 1;
    t.score = d.score.as<uint32_t>();
    t.status = d.status.as<uint8_t>();
    t.ref_start = d.ref_start.as<uint32_t>();
    t.ref_end = d.ref_end.as<uint32_t>();
    t.query_start = d.query_start.as<uint32_t>();
    t.query_end = d.query_end.as<uint32_t>();
    t.cig_count = d.cig_count.as<uint32_t>();
    t.dp_pair = d.tp_pair.as<uint32_t>();
    t.dp_cap = d.tp_cap.as<uint32_t>();
    t.dp_slot = d.tp_slot.as<uint32_t>();
    t.dp_bw = d.tp_bw.as<uint32_t>();
    t.dp_off = d.tp_off.as<unsigned long long>();
    t.dp_cig_off = d.tp_cigoff.as<unsigned long long>();
    t.ctr = ctr;

    unsigned long long n_nogaps = 0;
    for (uint64_t p0 = 0; p0 < pairs;) {
        uint32_t cn = (uint32_t)std::min<uint64_t>(chunk_pairs, pairs - p0);
        unsigned long long work[13] = {0};  // [0] DP pairs, [1] round-0 scratch, [2] CIGAR bytes, [5] no-gaps pairs, [12] widest large row
        uint32_t *lists[2] = {d.tp_list.as<uint32_t>(), d.tp_list.as<uint32_t>() + chunk_pairs};
        uint32_t *bws[2] = {d.tp_bw.as<uint32_t>(), d.tp_bw.as<uint32_t>() + chunk_pairs};
        unsigned long long *offs[2] = {d.tp_off.as<unsigned long long>(), d.tp_off.as<unsigned long long>() + chunk_pairs};
        for (;;) {
            t.pair_first = p0;
            t.n_pairs = cn;
            t.next_list = lists[0];  // the classification lists round 0
            t.dp_bw = bws[0];
            t.dp_off = offs[0];
            CU(ctx, cudaMemsetAsync(ctr, 0, 6 * sizeof(unsigned long long), d.stream));
            CU(ctx, cudaMemsetAsync(ctr + 12, 0, sizeof(unsigned long long), d.stream));
            tp_classify_kernel<<<(cn + 255) / 256, 256, 0, d.stream>>>(t);
            CU(ctx, cudaGetLastError());
            ctx->last_launches++;
            CU(ctx, cudaMemcpyAsync(work, ctr, sizeof(work), cudaMemcpyDeviceToHost, d.stream));
            CU(ctx, cudaStreamSynchronize(d.stream));
            if (work[1] + work[2] <= budget || cn == 1) break;
            cn = std::max<uint32_t>(1, cn / 2);  // this chunk needs more scratch than the budget: split it
            chunk_pairs = cn;
        }
        n_nogaps += work[5];
        if (work[0] > 0) {
            // rounds: every unresolved pair tries its current band width; failures come back with twice the width
            CU(ctx, d.tp_cig.reserve(work[2] + 16));
            t.cig_blob = d.tp_cig.as<uint8_t>();
            uint32_t n_round = (uint32_t)work[0];
            unsigned long long bytes = work[1], wide = work[12];
            int cur = 0;
            for (int round = 0; n_round > 0; ++round) {
                if (round > 64) return fail(ctx, ZOE_CUDA_E_STATE, "internal error: 3-pass band rounds do not terminate");
                CU(ctx, d.tp_blob.reserve(bytes + 16));
                t.blob = d.tp_blob.as<uint8_t>();
                t.list = lists[cur];
                t.next_list = lists[cur ^ 1];
                t.dp_bw = bws[cur];
                t.dp_off = offs[cur];
                t.dp_bw_next = bws[cur ^ 1];
                t.dp_off_next = offs[cur ^ 1];
                // large boxes (wide bands, big scalar boxes): one warp per pair, two int rows per warp in shared memory
                uint32_t wcap = 0, warps = 0;
                if (wide > 0 && !getenv("ZOE_CUDA_TP_THREAD")) {
                    wcap = (uint32_t)std::min<unsigned long long>((wide + 2 + 31) & ~31ull, 24 * 1024);  // <= 192 KB per warp
                    warps = (uint32_t)std::min<size_t>(16, (200 * 1024) / ((size_t)wcap * 8));
                    if (warps == 0) wcap = 0;
                }
                t.warp_wcap = wcap;
                CU(ctx, cudaMemsetAsync(ctr + 3, 0, 2 * sizeof(unsigned long long), d.stream));
                CU(ctx, cudaMemsetAsync(ctr + 12, 0, sizeof(unsigned long long), d.stream));
                tp_dp_kernel<<<(n_round + kTpThreads - 1) / kTpThreads, kTpThreads, 0, d.stream>>>(t, n_round);
                CU(ctx, cudaGetLastError());
                ctx->last_launches++;
                if (wcap) {
                    const size_t smem = (size_t)warps * wcap * 8;
                    CU(ctx, cudaFuncSetAttribute(tp_band_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                    const uint32_t nb = std::min<uint32_t>((n_round + warps - 1) / warps, (uint32_t)d.sm_count * 8);
                    tp_band_warp_kernel<<<nb, warps * 32, smem, d.stream>>>(t, n_round, wcap);
                    CU(ctx, cudaGetLastError());
                    ctx->last_launches++;
                }
                unsigned long long nxt[10] = {0};
                CU(ctx, cudaMemcpyAsync(nxt, ctr + 3, sizeof(nxt), cudaMemcpyDeviceToHost, d.stream));
                CU(ctx, cudaStreamSynchronize(d.stream));
                n_round = (uint32_t)nxt[0];
                bytes = nxt[1];
                wide = nxt[9];
                cur ^= 1;
            }
        }
        // CIGAR compaction, chained through the device-side running base ctr[9]
        if (cn >= (1u << 16)) {
            const uint32_t nbk = (cn + 1023) / 1024;
            CU(ctx, d.cig_bsum.reserve((size_t)nbk * sizeof(unsigned long long)));
            cigar_block_sum_kernel<<<nbk, 1024, 0, d.stream>>>(t.cig_count, p0, cn, d.cig_bsum.as<unsigned long long>());
            CU(ctx, cudaGetLastError());
            cigar_scan_sums_kernel<<<1, 1024, 0, d.stream>>>(d.cig_bsum.as<unsigned long long>(), nbk, ctr + 9,
                                                             d.cig_off.as<uint64_t>() + p0 + cn);
            CU(ctx, cudaGetLastError());
            cigar_block_scan_kernel<<<nbk, 1024, 0, d.stream>>>(t.cig_count, p0, cn, d.cig_bsum.as<unsigned long long>(),
                                                                d.cig_off.as<uint64_t>());
            CU(ctx, cudaGetLastError());
            ctx->last_launches += 3;
        } else {
            cigar_scan_kernel<<<1, 1024, 0, d.stream>>>(t.cig_count, p0, cn, d.cig_off.as<uint64_t>(), ctr + 9);
            CU(ctx, cudaGetLastError());
            ctx->last_launches++;
        }
        tp_gather_kernel<<<(cn + 255) / 256, 256, 0, d.stream>>>(t, d.cig_off.as<uint64_t>(), d.cig_out.as<uint32_t>(),
                                                                 cigar_cap_words);
        CU(ctx, cudaGetLastError());
        ctx->last_launches++;
        p0 += cn;
    }
    unsigned long long tail[16];
    CU(ctx, cudaMemcpyAsync(tail, ctr, sizeof(tail), cudaMemcpyDeviceToHost, d.stream));
    CU(ctx, cudaStreamSynchronize(d.stream));
    d.cig_total = tail[9];
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        ctx->stats.tp_nogaps += n_nogaps;
        ctx->stats.tp_banded += tail[6];
        ctx->stats.tp_scalar += tail[7];
        ctx->stats.tp_band_attempts += tail[8];
    }
    if (tail[10]) return fail(ctx, ZOE_CUDA_E_STATE, "3-pass: %llu banded walks left the band storage (zoe would panic here)", tail[10]);
    if (tail[11]) return fail(ctx, ZOE_CUDA_E_STATE, "internal error: CIGAR scratch overflow on %llu pairs", tail[11]);
    return 0;
}

// Drives every device of the context with `fn`.  The align and ranges pipelines synchronise with the host between
// their stages, so with several devices in one process each device gets its own host thread (the streams alone
// would serialise the devices); a single device runs inline.
template <class Fn>
int for_each_device(zoe_cuda_ctx *ctx, Fn fn) {
    if (ctx->devs.size() == 1) return fn(ctx->devs[0]);
    std::vector<int> rcs(ctx->devs.size(), 0);
    std::vector<std::thread> th;
    for (size_t k = 0; k < ctx->devs.size(); ++k) th.emplace_back([&, k] { rcs[k] = fn(ctx->devs[k]); });
    for (std::thread &t : th) t.join();
    for (int rc : rcs)
        if (rc) return rc;
    return 0;
}

int sync_and_time(zoe_cuda_ctx *ctx) {
    float total = 0.f, dp = 0.f;
    std::vector<Device *> all;
    for (Device &d : ctx->devs) all.push_back(&d);
    if (ctx->alt_used)
        for (Device &d : ctx->alt) all.push_back(&d);
    for (Device *dp_ : all) {
        Device &d = *dp_;
        CU(ctx, cudaSetDevice(d.id));
        CU(ctx, cudaEventRecord(d.ev_end, d.stream));
        CU(ctx, cudaStreamSynchronize(d.stream));
        float t = 0.f;
        CU(ctx, cudaEventElapsedTime(&t, d.ev_begin, d.ev_end));
        total = std::max(total, t);
        if (d.timed_kernel) {
            CU(ctx, cudaEventElapsedTime(&t, d.ev_k0, d.ev_k1));
            dp = std::max(dp, t);
        }
    }
    ctx->last_total_ms = total;
    ctx->last_dp_ms = std::max(dp, ctx->last_dp_ms);
    return 0;
}

int gather_stats(zoe_cuda_ctx *ctx) {
    std::vector<Device *> all;
    for (Device &d : ctx->devs) all.push_back(&d);
    if (ctx->alt_used)
        for (Device &d : ctx->alt) all.push_back(&d);
    for (Device *dp_ : all) {
        Device &d = *dp_;
        if (d.n_count == 0 || !d.counters.p) continue;
        CU(ctx, cudaSetDevice(d.id));
        unsigned long long c[16];
        CU(ctx, cudaMemcpy(c, d.counters.p, sizeof(c), cudaMemcpyDeviceToHost));
        ctx->stats.tier8 += c[0];
        ctx->stats.tier16 += c[1];
        ctx->stats.tier32 += c[2];
        ctx->stats.unmapped += c[3];
        ctx->stats.overflowed += c[13];
    }
    ctx->stats.pairs = ctx->staged_n * ctx->n_prof;
    ctx->stats.cells = ctx->staged_cells;
    return 0;
}

void begin_call(zoe_cuda_ctx *ctx) {
    ctx->last_launches = 0;
    ctx->last_dp_ms = 0.f;
    ctx->stats = zoe_cuda_stats{};
    for (Device &d : ctx->devs) d.timed_kernel = false;
    for (Device &d : ctx->alt) d.timed_kernel = false;
}

// Copies the per-pair alignment outputs and the compacted CIGAR stream of every device into the caller's arrays
// (devices own contiguous index ranges; CIGAR offsets become global).  Shared by the align and 3-pass entry points.
int fetch_alignments(zoe_cuda_ctx *ctx, uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *ref_start,
                     uint32_t *ref_end, uint32_t *query_start, uint32_t *query_end, uint32_t *cigar, uint64_t *cigar_off,
                     uint64_t cigar_cap, uint8_t *hazard) {
    // CIGAR offsets: device-local running sums -> global offsets (devices own contiguous index ranges)
    uint64_t total = 0;
    for (Device &d : ctx->devs) total += d.cig_total;
    if (total > cigar_cap) {
        cigar_off[0] = total;
        sync_and_time(ctx);
        return fail(ctx, ZOE_CUDA_E_CIGAR_CAP, "CIGAR buffer too small: need %llu words, have %llu",
                    (unsigned long long)total, (unsigned long long)cigar_cap);
    }
    uint64_t base = 0;
    for (Device &d : ctx->devs) {
        if (d.n_count == 0) continue;
        CU(ctx, cudaSetDevice(d.id));
        size_t first = (size_t)d.n_first * ctx->n_prof, pairs = (size_t)d.n_count * ctx->n_prof;
        auto d2h = [&](void *dst, const DevBuf &src, size_t elem) -> cudaError_t {
            if (!dst) return cudaSuccess;
            return cudaMemcpyAsync((uint8_t *)dst + first * elem, src.p, pairs * elem, cudaMemcpyDeviceToHost, d.stream);
        };
        CU(ctx, d2h(score, d.score, 4));
        CU(ctx, d2h(status, d.status, 1));
        CU(ctx, d2h(tier, d.tier, 1));
        CU(ctx, d2h(ref_start, d.ref_start, 4));
        CU(ctx, d2h(ref_end, d.ref_end, 4));
        CU(ctx, d2h(query_start, d.query_start, 4));
        CU(ctx, d2h(query_end, d.query_end, 4));
        if (hazard) CU(ctx, d2h(hazard, d.hazard, 1));
        CU(ctx, cudaMemcpyAsync(cigar_off + first, d.cig_off.p, (pairs + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost,
                                d.stream));
        if (d.cig_total)
            CU(ctx, cudaMemcpyAsync(cigar + base, d.cig_out.p, d.cig_total * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                                    d.stream));
        CU(ctx, cudaStreamSynchronize(d.stream));
        if (base)
            for (size_t i = 0; i <= pairs; ++i) cigar_off[first + i] += base;
        base += d.cig_total;
    }
    return 0;
}

// Queues the D2H copies of a device's score outputs behind its kernels (score entry points).
int queue_score_d2h(zoe_cuda_ctx *ctx, Device &d, uint32_t *score, uint8_t *status, uint8_t *tier) {
    if (d.n_count == 0) return 0;
    CU(ctx, cudaSetDevice(d.id));
    size_t first = (size_t)d.n_first * ctx->n_prof, pairs = (size_t)d.n_count * ctx->n_prof;
    if (score)
        CU(ctx, cudaMemcpyAsync(score + first, d.score.p, pairs * sizeof(uint32_t), cudaMemcpyDeviceToHost, d.stream));
    if (status) CU(ctx, cudaMemcpyAsync(status + first, d.status.p, pairs, cudaMemcpyDeviceToHost, d.stream));
    if (tier) CU(ctx, cudaMemcpyAsync(tier + first, d.tier.p, pairs, cudaMemcpyDeviceToHost, d.stream));
    return 0;
}

// Queues the D2H copies of every device's ranges outputs (ranges entry points).
int queue_ranges_d2h(zoe_cuda_ctx *ctx, uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *ref_start,
                     uint32_t *ref_end, uint32_t *query_start, uint32_t *query_end) {
    for (Device &d : ctx->devs) {
        if (d.n_count == 0) continue;
        CU(ctx, cudaSetDevice(d.id));
        size_t first = (size_t)d.n_first * ctx->n_prof, pairs = (size_t)d.n_count * ctx->n_prof;
        auto d2h = [&](void *dst, const DevBuf &src, size_t elem) -> cudaError_t {
            if (!dst) return cudaSuccess;
            return cudaMemcpyAsync((uint8_t *)dst + first * elem, src.p, pairs * elem, cudaMemcpyDeviceToHost, d.stream);
        };
        CU(ctx, d2h(score, d.score, 4));
        CU(ctx, d2h(status, d.status, 1));
        CU(ctx, d2h(tier, d.tier, 1));
        CU(ctx, d2h(ref_start, d.ref_start, 4));
        CU(ctx, d2h(ref_end, d.ref_end, 4));
        CU(ctx, d2h(query_start, d.query_start, 4));
        CU(ctx, d2h(query_end, d.query_end, 4));
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------
// both-strand search (strands.cuh, DESIGN.md 4.8): stage -> strand expansion -> the unchanged pipelines on the doubled
// batch -> strand selection -> the unchanged fetch paths on the real shard
// ---------------------------------------------------------------------------------------------
// While a both-strand call runs its pipelines, the host bookkeeping describes the doubled, interleaved batch the
// expansion kernel built (count, cells, per-sequence lengths, every device's shard); the rest of the call sees the real
// batch.  The destructor restores the real batch, leaves nothing "staged" (the device holds a doubled batch), and on
// an error return drains every stream so that no copy from the caller's buffers is still in flight.
struct DoubledView {
    zoe_cuda_ctx *ctx;
    bool doubled = false, ok = false;
    std::vector<uint32_t> real_len;
    explicit DoubledView(zoe_cuda_ctx *c) : ctx(c) {}
    DoubledView(const DoubledView &) = delete;
    DoubledView &operator=(const DoubledView &) = delete;
    void enter() {
        ctx->staged_n *= 2;
        ctx->staged_cells *= 2;
        real_len.swap(ctx->staged_len);
        ctx->staged_len.resize(2 * real_len.size());
        for (size_t i = 0; i < real_len.size(); ++i) ctx->staged_len[2 * i] = ctx->staged_len[2 * i + 1] = real_len[i];
        for (Device &d : ctx->devs) {
            d.n_first *= 2;
            d.n_count *= 2;
        }
        doubled = true;
    }
    void leave() {
        if (!doubled) return;
        ctx->staged_n /= 2;
        ctx->staged_cells /= 2;
        ctx->staged_len.swap(real_len);
        for (Device &d : ctx->devs) {
            d.n_first /= 2;
            d.n_count /= 2;
        }
        doubled = false;
    }
    ~DoubledView() {
        leave();
        ctx->staged = false;
        if (ok) return;
        for (Device &d : ctx->devs) {
            cudaSetDevice(d.id);
            if (d.copy_stream) cudaStreamSynchronize(d.copy_stream);
            cudaStreamSynchronize(d.stream);
            d.copy_pending = false;
        }
    }
};

// Checks the doubled batch against the single-strand limits (sequences per call; with pair_limit, pairs per device for
// the align / ranges / 3-pass pipelines), before anything is queued.
int check_both_strands_limits(zoe_cuda_ctx *ctx, uint64_t n, bool pair_limit) {
    if (n >= 0x7fffffffULL / 2 + 1)
        return fail(ctx, ZOE_CUDA_E_BAD_ARG, "batch too large: a both-strand search doubles the batch, so it takes at most "
                    "%llu sequences (half the single-strand limit)", 0x7fffffffULL / 2);
    if (pair_limit && ctx->have_profiled) {
        shard(ctx, n);
        for (Device &d : ctx->devs)
            if (2 * d.n_count * ctx->n_prof >= 0x7fffffffULL)
                return fail(ctx, ZOE_CUDA_E_BAD_ARG, "too many pairs: a both-strand search doubles the pairs of a device "
                            "(%llu) past the %llu of one call; halve the batch",
                            (unsigned long long)(2 * d.n_count * ctx->n_prof), 0x7fffffffULL - 1);
    }
    return 0;
}

// Queues the strand expansion of the device's staged shard and swaps the doubled batch into rseq / roff.  The pair
// buffers staging sized for the real shard are grown for the doubled one.  paired: the shard is a pair shard staged by
// stage_pairs (its reads are the mates, interleaved by pair).
int expand_strands(zoe_cuda_ctx *ctx, Device &d, bool paired = false) {
    if (d.n_count == 0) return 0;
    CU(ctx, cudaSetDevice(d.id));
    CU(ctx, d.xs_seq.reserve(2 * d.rseq_bytes + 16));
    CU(ctx, d.xs_off.reserve((2 * d.n_count + 1) * sizeof(uint64_t)));
    const uint32_t blocks = (uint32_t)std::min<uint64_t>((d.n_count + 7) / 8, (uint64_t)d.sm_count * 16);
    if (paired) {
        const uint64_t np = d.n_count / 2;
        const ExpandPairs src{d.rseq.as<uint8_t>(), d.roff.as<uint64_t>(), d.roff.as<uint64_t>() + np + 1, np};
        strand_expand_kernel<<<blocks, 256, 0, d.stream>>>(src, d.n_count, d.xs_seq.as<uint8_t>(), d.xs_off.as<uint64_t>());
    } else {
        const ExpandSingle src{d.rseq.as<uint8_t>(), d.roff.as<uint64_t>()};
        strand_expand_kernel<<<blocks, 256, 0, d.stream>>>(src, d.n_count, d.xs_seq.as<uint8_t>(), d.xs_off.as<uint64_t>());
    }
    CU(ctx, cudaGetLastError());
    ctx->last_launches++;
    std::swap(d.rseq, d.xs_seq);
    std::swap(d.roff, d.xs_off);
    d.rseq_bytes *= 2;
    const size_t pairs = (size_t)2 * d.n_count * ctx->n_prof;
    CU(ctx, d.best.reserve(pairs * sizeof(int32_t)));
    CU(ctx, d.score.reserve(pairs * sizeof(uint32_t)));
    CU(ctx, d.status.reserve(pairs));
    CU(ctx, d.tier.reserve(pairs));
    CU(ctx, d.wide_ids.reserve((2 * d.n_count + 1) * sizeof(uint32_t)));
    return 0;
}

// Stages a both-strand batch (one upload: the expansion needs the whole shard), expands it on every device and switches
// the host bookkeeping to the doubled view.
int stage_both_strands(zoe_cuda_ctx *ctx, DoubledView &view, const uint8_t *concat, const uint64_t *offsets, uint64_t n,
                       bool pair_limit) {
    int rc = check_both_strands_limits(ctx, n, pair_limit);
    if (rc) return rc;
    rc = stage_on_devices(ctx, concat, offsets, n, /*split=*/false);
    if (rc) return rc;
    for (Device &d : ctx->devs) {
        rc = expand_strands(ctx, d);
        if (rc) return rc;
    }
    view.enter();
    return 0;
}

// Stages a paired batch: n pairs, mate 1 of pair i being sequence i of the first batch and mate 2 sequence i of the
// second.  The host view is the 2n mates interleaved by pair (read 2i + m is mate m of pair i), sharded over pairs so
// that no device splits a pair.  Each device gets its pair range of both batches with one upload per caller buffer
// (the expansion reads the whole shard: no split upload), mate-1 bytes then mate-2 bytes in rseq and the two offset
// arrays, each rebased to its own first byte, back to back in roff.  Then the strand expansion (ExpandPairs) and the
// doubled view, as stage_both_strands: the devices hold the quadrupled batch, sequence 4i + 2m + s.
int stage_pairs(zoe_cuda_ctx *ctx, DoubledView &view, const uint8_t *concat1, const uint64_t *offsets1,
                const uint8_t *concat2, const uint64_t *offsets2, uint64_t n) {
    if (!ctx->have_profiled) return fail(ctx, ZOE_CUDA_E_STATE, "set_profiled must be called before a batch");
    if (n > 0 && (!concat1 || !offsets1 || !concat2 || !offsets2)) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "null batch pointers");
    int rc = check_both_strands_limits(ctx, 2 * std::min<uint64_t>(n, 0x7fffffffULL), false);
    if (rc) return rc;
    uint32_t max_len = 0, min_len = n ? 0xffffffffu : 0u;
    uint64_t tot = 0;
    rc = check_offsets(ctx, offsets1, n, &max_len, &min_len, &tot);
    if (rc) return rc;
    rc = check_offsets(ctx, offsets2, n, &max_len, &min_len, &tot);
    if (rc) return rc;
    ctx->staged_n = 2 * n;
    ctx->staged_max_len = max_len;
    ctx->staged_min_len = min_len;
    ctx->staged_cells = tot * ctx->prof_off[ctx->n_prof];
    ctx->staged_len.clear();
    if (max_len > (uint32_t)kMaxRowsSinglePass) {
        ctx->staged_len.resize(2 * n);
        for (uint64_t i = 0; i < n; ++i) {
            ctx->staged_len[2 * i] = (uint32_t)(offsets1[i + 1] - offsets1[i]);
            ctx->staged_len[2 * i + 1] = (uint32_t)(offsets2[i + 1] - offsets2[i]);
        }
    }
    ctx->alt_used = false;
    shard(ctx, n);
    for (Device &d : ctx->devs) {
        const uint64_t a = d.n_first, np = d.n_count;
        d.n_first = 2 * a;
        d.n_count = 2 * np;
        CU(ctx, cudaSetDevice(d.id));
        CU(ctx, cudaEventRecord(d.ev_begin, d.stream));
        d.copy_pending = false;
        if (np == 0) continue;
        const uint64_t a1 = offsets1[a], b1 = offsets1[a + np], a2 = offsets2[a], b2 = offsets2[a + np];
        d.rseq_bytes = (b1 - a1) + (b2 - a2);
        CU(ctx, d.rseq.reserve(d.rseq_bytes + 16));
        CU(ctx, d.roff.reserve(2 * (np + 1) * sizeof(uint64_t)));
        uint64_t *off = d.roff.as<uint64_t>();
        CU(ctx, cudaMemcpyAsync(off, offsets1 + a, (np + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, d.stream));
        CU(ctx, cudaMemcpyAsync(off + np + 1, offsets2 + a, (np + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, d.stream));
        if (b1 > a1) CU(ctx, cudaMemcpyAsync(d.rseq.p, concat1 + a1, b1 - a1, cudaMemcpyHostToDevice, d.stream));
        if (b2 > a2)
            CU(ctx, cudaMemcpyAsync(d.rseq.as<uint8_t>() + (b1 - a1), concat2 + a2, b2 - a2, cudaMemcpyHostToDevice, d.stream));
        const uint32_t blocks = (uint32_t)((np + 256) / 256);
        for (int m = 0; m < 2; ++m) {
            const uint64_t b0 = m == 0 ? a1 : a2;
            if (b0 == 0) continue;
            rebase_offsets_kernel<<<blocks, 256, 0, d.stream>>>(off + m * (np + 1), np + 1, b0);
            CU(ctx, cudaGetLastError());
        }
        rc = reserve_batch_outputs(ctx, d);
        if (rc) return rc;
        rc = expand_strands(ctx, d, /*paired=*/true);
        if (rc) return rc;
    }
    ctx->staged = true;
    view.enter();
    return 0;
}

// Queues the exclusive scan of n 32-bit counts into off[0, n] (off[n] = the total, also left in *base, which is zeroed
// first): the CIGAR offset scan of the align pipeline.
int scan_counts(zoe_cuda_ctx *ctx, Device &d, const uint32_t *cnt, uint64_t n, uint64_t *off, unsigned long long *base) {
    CU(ctx, cudaMemsetAsync(base, 0, sizeof(unsigned long long), d.stream));
    if (n >= (1u << 16)) {
        const uint32_t nbk = (uint32_t)((n + 1023) / 1024);
        CU(ctx, d.cig_bsum.reserve((size_t)nbk * sizeof(unsigned long long)));
        cigar_block_sum_kernel<<<nbk, 1024, 0, d.stream>>>(cnt, 0, n, d.cig_bsum.as<unsigned long long>());
        CU(ctx, cudaGetLastError());
        cigar_scan_sums_kernel<<<1, 1024, 0, d.stream>>>(d.cig_bsum.as<unsigned long long>(), nbk, base, off + n);
        CU(ctx, cudaGetLastError());
        cigar_block_scan_kernel<<<nbk, 1024, 0, d.stream>>>(cnt, 0, n, d.cig_bsum.as<unsigned long long>(), off);
        CU(ctx, cudaGetLastError());
        ctx->last_launches += 3;
    } else {
        cigar_scan_kernel<<<1, 1024, 0, d.stream>>>(cnt, 0, n, off, base);
        CU(ctx, cudaGetLastError());
        ctx->last_launches++;
    }
    return 0;
}

enum class StrandOutputs { Score, Ranges, Align, ThreePass };

// Strand selection on one device (doubled view): gathers the selected strand's per-pair outputs into the buffers the
// fetch paths read and writes d.strand.  For the alignments, also the selected CIGAR lengths and their offsets
// (sel_cig_count -> sel_cig_off, the CIGAR offset scan of the align pipeline); *cig_need gets the selected total.
int select_strands(zoe_cuda_ctx *ctx, Device &d, StrandOutputs kind, uint64_t *cig_need) {
    *cig_need = 0;
    const uint64_t n_out = d.n_count / 2 * ctx->n_prof;
    if (n_out == 0) return 0;
    CU(ctx, cudaSetDevice(d.id));
    const bool cig = kind == StrandOutputs::Align || kind == StrandOutputs::ThreePass;
    StrandSelectParams p{};
    DevBuf *b32[5] = {&d.score, &d.ref_start, &d.ref_end, &d.query_start, &d.query_end};
    DevBuf *b8[3] = {&d.status, &d.tier, &d.hazard};
    p.n32 = kind == StrandOutputs::Score ? 1 : 5;
    p.n8 = kind == StrandOutputs::Align ? 3 : 2;
    for (int k = 0; k < p.n32; ++k) {
        CU(ctx, d.sel32[k].reserve(n_out * sizeof(uint32_t)));
        p.in32[k] = b32[k]->as<uint32_t>();
        p.out32[k] = d.sel32[k].as<uint32_t>();
    }
    for (int k = 0; k < p.n8; ++k) {
        CU(ctx, d.sel8[k].reserve(n_out));
        p.in8[k] = b8[k]->as<uint8_t>();
        p.out8[k] = d.sel8[k].as<uint8_t>();
    }
    CU(ctx, d.strand.reserve(n_out));
    p.strand = d.strand.as<uint8_t>();
    p.n_out = n_out;
    p.n_prof = ctx->n_prof;
    if (cig) {
        CU(ctx, d.sel_cig_count.reserve(n_out * sizeof(uint32_t)));
        p.cig_off = d.cig_off.as<uint64_t>();
        p.cig_count = d.sel_cig_count.as<uint32_t>();
    }
    strand_select_kernel<<<(uint32_t)((n_out + 255) / 256), 256, 0, d.stream>>>(p);
    CU(ctx, cudaGetLastError());
    ctx->last_launches++;
    for (int k = 0; k < p.n32; ++k) std::swap(*b32[k], d.sel32[k]);
    for (int k = 0; k < p.n8; ++k) std::swap(*b8[k], d.sel8[k]);
    if (!cig) return 0;
    CU(ctx, d.sel_cig_off.reserve((n_out + 1) * sizeof(uint64_t)));
    CU(ctx, d.sel_ctr.reserve(sizeof(unsigned long long)));
    unsigned long long *base = d.sel_ctr.as<unsigned long long>();
    int rc = scan_counts(ctx, d, d.sel_cig_count.as<uint32_t>(), n_out, d.sel_cig_off.as<uint64_t>(), base);
    if (rc) return rc;
    unsigned long long need = 0;
    CU(ctx, cudaMemcpyAsync(&need, base, sizeof(need), cudaMemcpyDeviceToHost, d.stream));
    CU(ctx, cudaStreamSynchronize(d.stream));
    *cig_need = need;
    return 0;
}

// Copies the selected strands' CIGAR words (select_strands ran) into a compact stream and swaps it and its offsets into
// the buffers fetch_alignments reads.  Needs every word of the doubled run in d.cig_out.
int gather_strand_cigars(zoe_cuda_ctx *ctx, Device &d, uint64_t total) {
    const uint64_t n_out = d.n_count / 2 * ctx->n_prof;
    d.cig_total = total;
    if (n_out == 0) return 0;
    CU(ctx, cudaSetDevice(d.id));
    CU(ctx, d.sel_cig_out.reserve(std::max<uint64_t>(total, 1) * sizeof(uint32_t)));
    if (total) {
        const uint32_t blocks = (uint32_t)std::min<uint64_t>((n_out + 7) / 8, (uint64_t)d.sm_count * 16);
        strand_cigar_gather_kernel<<<blocks, 256, 0, d.stream>>>(d.cig_out.as<uint32_t>(), d.cig_off.as<uint64_t>(),
                                                                 d.strand.as<uint8_t>(), n_out, ctx->n_prof,
                                                                 d.sel_cig_off.as<uint64_t>(), d.sel_cig_out.as<uint32_t>());
        CU(ctx, cudaGetLastError());
        ctx->last_launches++;
    }
    std::swap(d.cig_off, d.sel_cig_off);
    std::swap(d.cig_out, d.sel_cig_out);
    return 0;
}

// Copies every device's strand choices into the caller's array (real view).
int queue_strand_d2h(zoe_cuda_ctx *ctx, uint8_t *strand) {
    if (!strand) return 0;
    for (Device &d : ctx->devs) {
        if (d.n_count == 0) continue;
        CU(ctx, cudaSetDevice(d.id));
        CU(ctx, cudaMemcpyAsync(strand + (size_t)d.n_first * ctx->n_prof, d.strand.p, (size_t)d.n_count * ctx->n_prof,
                                cudaMemcpyDeviceToHost, d.stream));
    }
    return 0;
}

// The statistics of a both-strand call count the work done: gather_stats ran on the real view, its counters on the
// doubled batch.
int gather_both_strands_stats(zoe_cuda_ctx *ctx) {
    int rc = gather_stats(ctx);
    ctx->stats.pairs *= 2;
    ctx->stats.cells *= 2;
    return rc;
}

constexpr int kNotMixed = 1;
int align_split_long_short(zoe_cuda_ctx *ctx, bool both_strands, const uint8_t *streamed_concat, const uint64_t *offsets,
                           uint64_t n, uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *ref_start,
                           uint32_t *ref_end, uint32_t *query_start, uint32_t *query_end, uint32_t *cigar,
                           uint64_t *cigar_off, uint64_t cigar_cap, uint8_t *hazard, uint8_t *strand);

// The align and 3-pass both-strand entry points.  The doubled run gets its own device CIGAR capacity (the caller's
// capacity bounds the selected strands only); a run whose non-selected strands overflowed it is repeated once with the
// exact need.
int align_both_strands(zoe_cuda_ctx *ctx, bool three_pass, const uint8_t *streamed_concat, const uint64_t *offsets,
                       uint64_t n, uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *ref_start, uint32_t *ref_end,
                       uint32_t *query_start, uint32_t *query_end, uint32_t *cigar, uint64_t *cigar_off, uint64_t cigar_cap,
                       uint8_t *hazard, uint8_t *strand) {
    if (!cigar_off || (!cigar && cigar_cap)) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "null CIGAR outputs");
    begin_call(ctx);
    DoubledView view(ctx);
    int rc = check_both_strands_limits(ctx, n, true);
    if (rc) return rc;
    rc = stage_on_devices(ctx, streamed_concat, offsets, n, /*split=*/false);
    if (rc) return rc;
    if (!three_pass && n > 0 && ctx->staged_max_len > (uint32_t)kMaxRowsSinglePass &&
        ctx->staged_min_len <= (uint32_t)kMaxRowsSinglePass) {
        for (Device &d : ctx->devs) {
            CU(ctx, cudaSetDevice(d.id));
            CU(ctx, cudaStreamSynchronize(d.stream));
        }
        rc = align_split_long_short(ctx, true, streamed_concat, offsets, n, score, status, tier, ref_start, ref_end,
                                    query_start, query_end, cigar, cigar_off, cigar_cap, hazard, strand);
        if (rc != kNotMixed) {
            view.ok = rc == 0;
            return rc;
        }
    }
    for (Device &d : ctx->devs) {
        rc = expand_strands(ctx, d);
        if (rc) return rc;
    }
    view.enter();
    const StrandOutputs kind = three_pass ? StrandOutputs::ThreePass : StrandOutputs::Align;
    uint64_t dev_cap = 2 * cigar_cap + 1024;
    std::vector<uint64_t> need(ctx->devs.size());
    for (int attempt = 0;; ++attempt) {
        rc = for_each_device(ctx, [&](Device &d) {
            return three_pass ? run_3pass_on_device(ctx, d, dev_cap) : run_align_on_device(ctx, d, dev_cap);
        });
        if (rc) return rc;
        uint64_t total = 0, widest = 0;
        for (size_t k = 0; k < ctx->devs.size(); ++k) {
            rc = select_strands(ctx, ctx->devs[k], kind, &need[k]);
            if (rc) return rc;
            total += need[k];
            widest = std::max<uint64_t>(widest, ctx->devs[k].cig_total);
        }
        if (total > cigar_cap) {
            cigar_off[0] = total;
            return fail(ctx, ZOE_CUDA_E_CIGAR_CAP, "CIGAR buffer too small: the selected strands need %llu words, have %llu",
                        (unsigned long long)total, (unsigned long long)cigar_cap);
        }
        if (widest <= dev_cap) break;
        if (attempt > 0) return fail(ctx, ZOE_CUDA_E_STATE, "internal error: both-strand CIGAR capacity not met on the re-run");
        dev_cap = widest;
    }
    for (size_t k = 0; k < ctx->devs.size(); ++k) {
        rc = gather_strand_cigars(ctx, ctx->devs[k], need[k]);
        if (rc) return rc;
    }
    view.leave();
    rc = queue_strand_d2h(ctx, strand);
    if (rc) return rc;
    rc = fetch_alignments(ctx, score, status, tier, ref_start, ref_end, query_start, query_end, cigar, cigar_off, cigar_cap,
                          three_pass ? nullptr : hazard);
    if (rc) return rc;
    if (n == 0) cigar_off[0] = 0;
    rc = sync_and_time(ctx);
    if (rc) return rc;
    view.ok = true;
    return gather_both_strands_stats(ctx);
}

// A batch that mixes long (> 1024 residues) and short sequences is aligned in two parts: the short ones take the fast
// pipelines, the long ones the long-row path (run_align_on_device, long_mode); results are merged in the caller's order.
// Each part re-enters the entry point the caller used (single- or both-strand).  Returns kNotMixed, having done nothing,
// when the batch has only one kind.
int align_split_long_short(zoe_cuda_ctx *ctx, bool both_strands, const uint8_t *streamed_concat, const uint64_t *offsets,
                           uint64_t n, uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *ref_start,
                           uint32_t *ref_end, uint32_t *query_start, uint32_t *query_end, uint32_t *cigar,
                           uint64_t *cigar_off, uint64_t cigar_cap, uint8_t *hazard, uint8_t *strand) {
    std::vector<uint64_t> idx[2];  // [0] short, [1] long
    for (uint64_t i = 0; i < n; ++i) idx[offsets[i + 1] - offsets[i] > (uint64_t)kMaxRowsSinglePass ? 1 : 0].push_back(i);
    if (idx[0].empty() || idx[1].empty()) return kNotMixed;
    const uint32_t np = ctx->n_prof;
    struct Part {
        std::vector<uint8_t> buf;
        std::vector<uint64_t> off;
        std::vector<uint32_t> score, rs, re, qs, qe, cig;
        std::vector<uint8_t> status, tier, hz, sd;
        std::vector<uint64_t> coff;
    } part[2];
    zoe_cuda_stats total{};
    float total_ms = 0.f, dp_ms = 0.f;
    uint32_t launches = 0;
    uint64_t need = 0;
    int rc_cap = 0;
    for (int w = 0; w < 2; ++w) {
        Part &q = part[w];
        q.off.push_back(0);
        for (uint64_t i : idx[w]) {
            q.buf.insert(q.buf.end(), streamed_concat + offsets[i], streamed_concat + offsets[i + 1]);
            q.off.push_back(q.buf.size());
        }
        if (q.buf.empty()) q.buf.push_back(0);
        const size_t pairs = idx[w].size() * np;
        for (auto *v : {&q.score, &q.rs, &q.re, &q.qs, &q.qe}) v->assign(pairs, 0);
        for (auto *v : {&q.status, &q.tier, &q.hz, &q.sd}) v->assign(pairs, 0);
        q.coff.assign(pairs + 1, 0);
        q.cig.assign(std::max<uint64_t>(cigar_cap, 1), 0);
        int rc = both_strands
                     ? zoe_cuda_sw_align_both_strands_batch(ctx, q.buf.data(), q.off.data(), idx[w].size(), q.score.data(),
                                                            q.status.data(), q.tier.data(), q.rs.data(), q.re.data(),
                                                            q.qs.data(), q.qe.data(), q.cig.data(), q.coff.data(), cigar_cap,
                                                            q.hz.data(), q.sd.data())
                     : zoe_cuda_sw_align_batch(ctx, q.buf.data(), q.off.data(), idx[w].size(), q.score.data(), q.status.data(),
                                               q.tier.data(), q.rs.data(), q.re.data(), q.qs.data(), q.qe.data(), q.cig.data(),
                                               q.coff.data(), cigar_cap, q.hz.data());
        if (rc == ZOE_CUDA_E_CIGAR_CAP) {
            rc_cap = rc;
            need += q.coff[0];
            continue;
        }
        if (rc) return rc;
        need += q.coff[pairs];
        const zoe_cuda_stats &st = ctx->stats;
        total.pairs += st.pairs; total.cells += st.cells; total.tier8 += st.tier8; total.tier16 += st.tier16;
        total.tier32 += st.tier32; total.overflowed += st.overflowed; total.unmapped += st.unmapped;
        total.rerun_wide += st.rerun_wide; total.hazard += st.hazard; total.window_fallback += st.window_fallback;
        total.window_pinned += st.window_pinned;
        total_ms += ctx->last_total_ms;
        dp_ms += ctx->last_dp_ms;
        launches += ctx->last_launches.load();
    }
    if (rc_cap || need > cigar_cap) {
        cigar_off[0] = need;
        return fail(ctx, ZOE_CUDA_E_CIGAR_CAP, "CIGAR buffer too small: need at least %llu words, have %llu",
                    (unsigned long long)need, (unsigned long long)cigar_cap);
    }
    uint64_t pos = 0;
    size_t cursor[2] = {0, 0};
    for (uint64_t i = 0; i < n; ++i) {
        const int w = offsets[i + 1] - offsets[i] > (uint64_t)kMaxRowsSinglePass ? 1 : 0;
        const Part &q = part[w];
        const size_t src = cursor[w]++ * np, dst = (size_t)i * np;
        for (uint32_t j = 0; j < np; ++j) {
            if (score) score[dst + j] = q.score[src + j];
            if (status) status[dst + j] = q.status[src + j];
            if (tier) tier[dst + j] = q.tier[src + j];
            if (ref_start) ref_start[dst + j] = q.rs[src + j];
            if (ref_end) ref_end[dst + j] = q.re[src + j];
            if (query_start) query_start[dst + j] = q.qs[src + j];
            if (query_end) query_end[dst + j] = q.qe[src + j];
            if (hazard) hazard[dst + j] = q.hz[src + j];
            if (strand) strand[dst + j] = q.sd[src + j];
            cigar_off[dst + j] = pos;
            const uint64_t a = q.coff[src + j], b = q.coff[src + j + 1];
            if (b > a) memcpy(cigar + pos, q.cig.data() + a, (b - a) * sizeof(uint32_t));
            pos += b - a;
        }
    }
    cigar_off[(size_t)n * np] = pos;
    ctx->stats = total;
    ctx->last_total_ms = total_ms;
    ctx->last_dp_ms = dp_ms;
    ctx->last_launches = launches;
    ctx->staged = false;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// best-hit search (best_hit.cuh, DESIGN.md 4.9): the score pass over every candidate -> per-read selection -> for the
// align entry point, buckets of Some winners by (hit, length class), each aligned by the unchanged pipelines under a
// profiled view of its one sequence -> per-read outputs and one CIGAR stream in read order
// ---------------------------------------------------------------------------------------------
// The host state of a profiled set, set aside while a one-sequence view is installed.
struct PanelState {
    uint32_t n_prof = 0, max_prof_len = 0;
    int n_csym = 0;
    std::vector<uint8_t> prof_bytes, ccodes, ccodes_g;
    std::vector<uint64_t> prof_off;
    std::vector<uint32_t> coff, corder, coff_g, corder_g;
    std::vector<int8_t> wk;
    std::vector<zoe_cuda_ctx::ColGroup> groups;
    void swap_with(zoe_cuda_ctx *ctx) {
        std::swap(n_prof, ctx->n_prof);
        std::swap(max_prof_len, ctx->max_prof_len);
        std::swap(n_csym, ctx->n_csym);
        prof_bytes.swap(ctx->prof_bytes);
        ccodes.swap(ctx->ccodes);
        ccodes_g.swap(ctx->ccodes_g);
        prof_off.swap(ctx->prof_off);
        coff.swap(ctx->coff);
        corder.swap(ctx->corder);
        coff_g.swap(ctx->coff_g);
        corder_g.swap(ctx->corder_g);
        wk.swap(ctx->wk);
        groups.swap(ctx->groups);
    }
};

// Installs the profiled set {j} of the context's panel for one bucket, and restores the panel on leave() or on
// destruction, error or not.  Both directions derive and upload the set as zoe_cuda_set_profiled does (bump
// profiled_epoch, clear the plans).  The kernels are not pointed at a slice of the panel's buffers: the codes are
// staged by TMA from 16-byte-aligned starts, the dense symbol table and wk belong to the whole set, and flag_base /
// ckpt_base are cached against the epoch.
struct ProfiledView {
    zoe_cuda_ctx *ctx;
    bool active = false;
    PanelState panel;
    explicit ProfiledView(zoe_cuda_ctx *c) : ctx(c) {}
    ProfiledView(const ProfiledView &) = delete;
    ProfiledView &operator=(const ProfiledView &) = delete;
    int enter(uint32_t j) {
        if (!active) {
            panel.swap_with(ctx);
            active = true;
        }
        const uint64_t off[2] = {panel.prof_off[j], panel.prof_off[j + 1]};
        return install_profiled(ctx, panel.prof_bytes.data(), off, 1, (uint32_t)(off[1] - off[0]));
    }
    int leave() {
        if (!active) return 0;
        panel.swap_with(ctx);
        active = false;
        ctx->plans.clear();
        ctx->profiled_epoch++;
        return upload_scoring_and_profiled(ctx);
    }
    ~ProfiledView() { leave(); }
};

// Per-read selection on one device (real view; the score pass's results are resident in d.score / d.status / d.tier).
int select_best_hits(zoe_cuda_ctx *ctx, Device &d, uint32_t n_strands) {
    const uint64_t n = d.n_count;
    if (n == 0) return 0;
    CU(ctx, cudaSetDevice(d.id));
    for (DevBuf *b : {&d.bh_hit, &d.bh_runner, &d.bh_out32[0]}) CU(ctx, b->reserve(n * sizeof(uint32_t)));
    for (DevBuf *b : {&d.bh_strand, &d.bh_out8[0], &d.bh_out8[1]}) CU(ctx, b->reserve(n));
    BestHitSelectParams p{};
    p.score = d.score.as<uint32_t>();
    p.status = d.status.as<uint8_t>();
    p.tier = d.tier.as<uint8_t>();
    p.n = n;
    p.n_prof = ctx->n_prof;
    p.n_strands = n_strands;
    p.hit = d.bh_hit.as<uint32_t>();
    p.score_out = d.bh_out32[0].as<uint32_t>();
    p.runner_up = d.bh_runner.as<uint32_t>();
    p.strand = d.bh_strand.as<uint8_t>();
    p.status_out = d.bh_out8[0].as<uint8_t>();
    p.tier_out = d.bh_out8[1].as<uint8_t>();
    // a thread per read while a read's candidates fit one warp's width, a warp per read beyond
    if ((uint64_t)ctx->n_prof * n_strands <= 32) {
        const uint32_t blocks = (uint32_t)std::min<uint64_t>((n + 255) / 256, (uint64_t)d.sm_count * 8);
        best_hit_select_kernel<1><<<blocks, 256, 0, d.stream>>>(p);
    } else {
        const uint32_t blocks = (uint32_t)std::min<uint64_t>((n + 7) / 8, (uint64_t)d.sm_count * 16);
        best_hit_select_kernel<32><<<blocks, 256, 0, d.stream>>>(p);
    }
    CU(ctx, cudaGetLastError());
    ctx->last_launches++;
    return 0;
}

// Pair selection on one device (paired search, real view: the device's reads are the mates of its pairs): the winner
// of every pair to pr_hit and each mate's result under it to the per-read buffers select_best_hits fills.
int select_pairs(zoe_cuda_ctx *ctx, Device &d) {
    const uint64_t n = d.n_count, np = n / 2;
    if (n == 0) return 0;
    CU(ctx, cudaSetDevice(d.id));
    for (DevBuf *b : {&d.bh_hit, &d.bh_runner, &d.bh_out32[0]}) CU(ctx, b->reserve(n * sizeof(uint32_t)));
    for (DevBuf *b : {&d.bh_strand, &d.bh_out8[0], &d.bh_out8[1]}) CU(ctx, b->reserve(n));
    CU(ctx, d.pr_hit.reserve(np * sizeof(uint32_t)));
    PairSelectParams p{};
    p.score = d.score.as<uint32_t>();
    p.status = d.status.as<uint8_t>();
    p.tier = d.tier.as<uint8_t>();
    p.n_pairs = np;
    p.n_prof = ctx->n_prof;
    p.pair_hit = d.pr_hit.as<uint32_t>();
    p.hit = d.bh_hit.as<uint32_t>();
    p.score_out = d.bh_out32[0].as<uint32_t>();
    p.runner_up = d.bh_runner.as<uint32_t>();
    p.strand = d.bh_strand.as<uint8_t>();
    p.status_out = d.bh_out8[0].as<uint8_t>();
    p.tier_out = d.bh_out8[1].as<uint8_t>();
    // a thread per pair while a pair's 2 n_prof candidates fit one warp's width, a warp per pair beyond
    if ((uint64_t)ctx->n_prof * 2 <= 32) {
        const uint32_t blocks = (uint32_t)std::min<uint64_t>((np + 255) / 256, (uint64_t)d.sm_count * 8);
        pair_select_kernel<1><<<blocks, 256, 0, d.stream>>>(p);
    } else {
        const uint32_t blocks = (uint32_t)std::min<uint64_t>((np + 7) / 8, (uint64_t)d.sm_count * 16);
        pair_select_kernel<32><<<blocks, 256, 0, d.stream>>>(p);
    }
    CU(ctx, cudaGetLastError());
    ctx->last_launches++;
    return 0;
}

// tlen and proper of one device's pairs from its per-mate outputs (in mate order).
int finalize_pairs(zoe_cuda_ctx *ctx, Device &d, uint32_t min_insert, uint32_t max_insert) {
    const uint64_t np = d.n_count / 2;
    if (np == 0) return 0;
    CU(ctx, cudaSetDevice(d.id));
    CU(ctx, d.pr_proper.reserve(np));
    CU(ctx, d.pr_tlen.reserve(np * sizeof(int32_t)));
    PairFinalizeParams p{};
    p.status = d.bh_out8[0].as<uint8_t>();
    p.strand = d.bh_strand.as<uint8_t>();
    p.start = d.bh_out32[ctx->profiled_is_query ? 3 : 1].as<uint32_t>();
    p.end = d.bh_out32[ctx->profiled_is_query ? 4 : 2].as<uint32_t>();
    p.n_pairs = np;
    p.min_insert = min_insert;
    p.max_insert = max_insert;
    p.proper = d.pr_proper.as<uint8_t>();
    p.tlen = d.pr_tlen.as<int32_t>();
    const uint32_t blocks = (uint32_t)std::min<uint64_t>((np + 255) / 256, (uint64_t)d.sm_count * 8);
    pair_finalize_kernel<<<blocks, 256, 0, d.stream>>>(p);
    CU(ctx, cudaGetLastError());
    ctx->last_launches++;
    return 0;
}

// Buckets one device's Some winners (best_hit_bucket_*_kernel), zeroes the outputs of the reads no bucket aligns, and
// reads the bucket table back into tab (kBhStart + 1 rows of n_keys words).
int bucket_best_hits(zoe_cuda_ctx *ctx, Device &d, uint32_t n_strands, bool split_long, uint32_t n_keys,
                     std::vector<unsigned long long> &tab) {
    tab.assign((size_t)(kBhStart + 1) * n_keys, 0);
    const uint64_t n = d.n_count;
    if (n == 0) return 0;
    CU(ctx, cudaSetDevice(d.id));
    CU(ctx, d.bh_key.reserve(n * sizeof(uint32_t)));
    CU(ctx, d.bh_list.reserve(n * sizeof(uint32_t)));
    CU(ctx, d.bh_tab.reserve(((size_t)kBhTabRows * n_keys + 1) * sizeof(unsigned long long)));
    for (DevBuf *b : {&d.bh_out32[1], &d.bh_out32[2], &d.bh_out32[3], &d.bh_out32[4], &d.bh_cig_count}) {
        CU(ctx, b->reserve(n * sizeof(uint32_t)));
        CU(ctx, cudaMemsetAsync(b->p, 0, n * sizeof(uint32_t), d.stream));
    }
    CU(ctx, d.bh_out8[2].reserve(n));
    CU(ctx, cudaMemsetAsync(d.bh_out8[2].p, 0, n, d.stream));
    CU(ctx, d.bh_cig_src.reserve(n * sizeof(uint64_t)));
    unsigned long long *t = d.bh_tab.as<unsigned long long>();
    CU(ctx, cudaMemsetAsync(t, 0, ((size_t)kBhTabRows * n_keys + 1) * sizeof(unsigned long long), d.stream));
    CU(ctx, cudaMemsetAsync(t + (size_t)kBhMin * n_keys, 0xff, (size_t)n_keys * sizeof(unsigned long long), d.stream));
    const size_t smem = (size_t)4 * n_keys * sizeof(unsigned long long);
    const bool use_smem = smem <= 48 * 1024;
    const uint32_t blocks = (uint32_t)std::min<uint64_t>((n + 255) / 256, (uint64_t)d.sm_count * 4);
    best_hit_bucket_count_kernel<<<blocks, 256, use_smem ? smem : 0, d.stream>>>(
        d.bh_hit.as<uint32_t>(), d.bh_out8[0].as<uint8_t>(), d.roff.as<uint64_t>(), n_strands, n, split_long, n_keys,
        use_smem, d.bh_key.as<uint32_t>(), t);
    CU(ctx, cudaGetLastError());
    best_hit_bucket_scan_kernel<<<1, 32, 0, d.stream>>>(t, n_keys);
    CU(ctx, cudaGetLastError());
    best_hit_bucket_scatter_kernel<<<blocks, 256, 0, d.stream>>>(d.bh_key.as<uint32_t>(), n, n_keys, t,
                                                                 d.bh_list.as<uint32_t>());
    CU(ctx, cudaGetLastError());
    ctx->last_launches += 3;
    CU(ctx, cudaMemcpyAsync(tab.data(), t, tab.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, d.stream));
    CU(ctx, cudaStreamSynchronize(d.stream));
    // compact-batch offsets of every listed read, in list order (bucket b's batch: loff[start_b, start_b + count_b])
    uint64_t m = 0;
    for (uint32_t k = 0; k < n_keys; ++k) m += tab[(size_t)kBhCount * n_keys + k];
    CU(ctx, d.bh_llen.reserve(std::max<uint64_t>(m, 1) * sizeof(uint32_t)));
    CU(ctx, d.bh_loff.reserve((m + 1) * sizeof(uint64_t)));
    if (m) {
        best_hit_list_len_kernel<<<(uint32_t)((m + 255) / 256), 256, 0, d.stream>>>(
            d.bh_list.as<uint32_t>(), m, d.roff.as<uint64_t>(), n_strands, d.bh_llen.as<uint32_t>());
        CU(ctx, cudaGetLastError());
        ctx->last_launches++;
    }
    return scan_counts(ctx, d, d.bh_llen.as<uint32_t>(), m, d.bh_loff.as<uint64_t>(), t + (size_t)kBhTabRows * n_keys);
}

// Grows b to `bytes`, keeping its first `used` bytes.
int reserve_keep(zoe_cuda_ctx *ctx, Device &d, DevBuf &b, size_t used, size_t bytes) {
    if (bytes <= b.cap) return 0;
    DevBuf nb;
    CU(ctx, nb.reserve(bytes));
    if (used) CU(ctx, cudaMemcpyAsync(nb.p, b.p, used, cudaMemcpyDeviceToDevice, d.stream));
    CU(ctx, cudaStreamSynchronize(d.stream));
    b.release();
    b = nb;
    return 0;
}

// One bucket on one device, under the bucket's host view: gather its reads into rseq / roff, align them against the
// one profiled sequence, scatter the outputs to read order and move the CIGAR words to bh_acc at *acc_used.
int align_bucket(zoe_cuda_ctx *ctx, Device &d, bool three_pass, uint32_t n_strands, uint64_t start, uint64_t max_len,
                 uint64_t cigar_cap, uint64_t *acc_used) {
    if (d.n_count == 0) return 0;
    CU(ctx, cudaSetDevice(d.id));
    const uint64_t cnt = d.n_count;
    CU(ctx, d.rseq.reserve(d.rseq_bytes + 16));
    CU(ctx, d.roff.reserve((cnt + 1) * sizeof(uint64_t)));
    const uint32_t blocks = (uint32_t)std::min<uint64_t>((cnt + 7) / 8, (uint64_t)d.sm_count * 16);
    best_hit_gather_kernel<<<blocks, 256, 0, d.stream>>>(d.bh_seq.as<uint8_t>(), d.bh_off.as<uint64_t>(), n_strands,
                                                         d.bh_strand.as<uint8_t>(), d.bh_list.as<uint32_t>() + start,
                                                         d.bh_loff.as<uint64_t>() + start, cnt, d.rseq.as<uint8_t>(),
                                                         d.roff.as<uint64_t>());
    CU(ctx, cudaGetLastError());
    ctx->last_launches++;
    // The bucket's CIGARs are part of what the caller receives, so the caller's capacity bounds them; a bucket that
    // overflows it makes the call fail with ZOE_CUDA_E_CIGAR_CAP and needs no re-run.  (A pair's CIGAR has at most
    // rows + columns + 4 words: small buckets reserve no more.)
    const uint64_t cap = std::min<uint64_t>(cigar_cap, cnt * (max_len + ctx->max_prof_len + 4));
    int rc = three_pass ? run_3pass_on_device(ctx, d, cap) : run_align_on_device(ctx, d, cap);
    if (rc) return rc;
    const uint64_t words = d.cig_total;
    if (words > cap && cap < cigar_cap)
        return fail(ctx, ZOE_CUDA_E_STATE, "internal error: best-hit bucket CIGAR bound exceeded (%llu words)",
                    (unsigned long long)words);
    const bool copy = *acc_used + words <= cigar_cap;
    if (copy) {
        rc = reserve_keep(ctx, d, d.bh_acc, *acc_used * sizeof(uint32_t), std::max<uint64_t>(*acc_used + words, 1) * sizeof(uint32_t));
        if (rc) return rc;
    }
    BestHitScatterParams p{};
    DevBuf *in32[5] = {&d.score, &d.ref_start, &d.ref_end, &d.query_start, &d.query_end};
    DevBuf *in8[3] = {&d.status, &d.tier, &d.hazard};
    for (int k = 0; k < 5; ++k) {
        p.in32[k] = in32[k]->as<uint32_t>();
        p.out32[k] = d.bh_out32[k].as<uint32_t>();
    }
    for (int k = 0; k < 3; ++k) {
        p.in8[k] = (k == 2 && three_pass) ? nullptr : in8[k]->as<uint8_t>();
        p.out8[k] = d.bh_out8[k].as<uint8_t>();
    }
    p.list = d.bh_list.as<uint32_t>() + start;
    p.count = cnt;
    p.cig_off = d.cig_off.as<uint64_t>();
    p.cig_out = d.cig_out.as<uint32_t>();
    p.cig_count = d.bh_cig_count.as<uint32_t>();
    p.cig_src = d.bh_cig_src.as<uint64_t>();
    p.acc = d.bh_acc.as<uint32_t>();
    p.acc_base = *acc_used;
    p.copy = copy && words > 0;
    best_hit_scatter_kernel<<<blocks, 256, 0, d.stream>>>(p);
    CU(ctx, cudaGetLastError());
    ctx->last_launches++;
    *acc_used += words;
    return 0;
}

// What the paired entry points add to the best-hit search: the mate-2 batch, the insert bounds and the per-pair
// outputs (hit then has one entry per pair).
struct PairedArgs {
    const uint8_t *concat2;
    const uint64_t *offsets2;
    uint32_t min_insert, max_insert;
    uint8_t *proper;
    int32_t *tlen;
};

// The best-hit entry points.  align = false: score pass + selection only.  pair: the paired search, n pairs (concat /
// offsets are mate 1); it runs on both strands, selects per pair and finishes with the pair outputs.
int best_hit(zoe_cuda_ctx *ctx, bool align, bool both_strands, bool three_pass, const uint8_t *concat,
             const uint64_t *offsets, uint64_t n, const PairedArgs *pair, uint32_t *hit, uint8_t *strand,
             uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *runner_up, uint32_t *ref_start,
             uint32_t *ref_end, uint32_t *query_start, uint32_t *query_end, uint32_t *cigar, uint64_t *cigar_off,
             uint64_t cigar_cap, uint8_t *hazard) {
    if (align && (!cigar_off || (!cigar && cigar_cap))) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "null CIGAR outputs");
    if (pair && pair->min_insert > pair->max_insert)
        return fail(ctx, ZOE_CUDA_E_BAD_ARG, "min_insert (%u) > max_insert (%u)", pair->min_insert, pair->max_insert);
    begin_call(ctx);
    DoubledView view(ctx);  // (entered only with both strands; drains every stream on an error return)
    int rc = pair           ? stage_pairs(ctx, view, concat, offsets, pair->concat2, pair->offsets2, n)
             : both_strands ? stage_both_strands(ctx, view, concat, offsets, n, /*pair_limit=*/false)
                            : stage_on_devices(ctx, concat, offsets, n, /*split=*/false);
    if (rc) return rc;
    for (Device &d : ctx->devs) {
        rc = run_score_on_device(ctx, d);
        if (rc) return rc;
    }
    if (align) {
        // the score pass's counters (every candidate) are read before the align stage reuses them; gather_stats reads
        // them with a copy that does not wait for the library's streams
        for (Device &d : ctx->devs) {
            CU(ctx, cudaSetDevice(d.id));
            CU(ctx, cudaStreamSynchronize(d.stream));
        }
        rc = gather_stats(ctx);
        if (rc) return rc;
    }
    view.leave();
    const uint32_t S = both_strands || pair ? 2 : 1;
    for (Device &d : ctx->devs) {
        rc = pair ? select_pairs(ctx, d) : select_best_hits(ctx, d, S);
        if (rc) return rc;
    }
    const size_t nd = ctx->devs.size();
    std::vector<uint64_t> acc_used(nd, 0);
    if (align) {
        const bool split_long = !three_pass;
        const uint32_t P = ctx->n_prof, K = split_long ? 2 * P : P;
        std::vector<std::vector<unsigned long long>> tab(nd);
        std::vector<uint64_t> first(nd), count(nd);
        for (size_t k = 0; k < nd; ++k) {
            Device &d = ctx->devs[k];
            rc = bucket_best_hits(ctx, d, S, split_long, K, tab[k]);
            if (rc) return rc;
            first[k] = d.n_first;
            count[k] = d.n_count;
            std::swap(d.rseq, d.bh_seq);
            std::swap(d.roff, d.bh_off);
        }
        const uint64_t real_n = ctx->staged_n;
        std::vector<uint32_t> read_len;  // per read when a read is long (prepare_batch, stage_pairs)
        read_len.swap(ctx->staged_len);
        uint64_t aligned = 0, aligned_cells = 0;
        {
            ProfiledView pv(ctx);
            for (uint32_t key = 0; key < K; ++key) {
                uint64_t total = 0, residues = 0, longest = 0, shortest = ~0ull;
                auto at = [&](size_t k, int row) { return (uint64_t)tab[k][(size_t)row * K + key]; };
                for (size_t k = 0; k < nd; ++k) {
                    if (at(k, kBhCount) == 0) continue;
                    total += at(k, kBhCount);
                    residues += at(k, kBhSum);
                    longest = std::max<uint64_t>(longest, at(k, kBhMax));
                    shortest = std::min<uint64_t>(shortest, at(k, kBhMin));
                }
                if (total == 0) continue;  // a profiled sequence no read chose
                rc = pv.enter(split_long ? key / 2 : key);
                if (rc) return rc;
                // the host view of the bucket's batch: the devices' buckets back to back
                ctx->staged_n = total;
                ctx->staged_max_len = (uint32_t)longest;
                ctx->staged_min_len = (uint32_t)shortest;
                ctx->staged_cells = residues * ctx->max_prof_len;
                ctx->staged_len.clear();
                if (longest > (uint64_t)kMaxRowsSinglePass) ctx->staged_len.resize(total);
                uint64_t pos = 0;
                for (size_t k = 0; k < nd; ++k) {
                    Device &d = ctx->devs[k];
                    d.n_first = pos;
                    d.n_count = at(k, kBhCount);
                    d.rseq_bytes = at(k, kBhSum);
                    d.copy_pending = false;
                    if (!ctx->staged_len.empty() && d.n_count) {
                        // the long-row path orders its tasks by length: a long bucket's lengths come from the batch's
                        // per-read lengths (such reads are few)
                        std::vector<uint32_t> ids(d.n_count);
                        CU(ctx, cudaSetDevice(d.id));
                        CU(ctx, cudaMemcpy(ids.data(), d.bh_list.as<uint32_t>() + at(k, kBhStart), d.n_count * sizeof(uint32_t),
                                           cudaMemcpyDeviceToHost));
                        for (uint64_t t = 0; t < d.n_count; ++t) ctx->staged_len[pos + t] = read_len[first[k] + ids[t]];
                    }
                    pos += d.n_count;
                }
                rc = for_each_device(ctx, [&](Device &d) {
                    const size_t k = (size_t)(&d - ctx->devs.data());
                    return align_bucket(ctx, d, three_pass, S, at(k, kBhStart), at(k, kBhMax), cigar_cap, &acc_used[k]);
                });
                if (rc) return rc;
                aligned += total;
                aligned_cells += ctx->staged_cells;
            }
            rc = pv.leave();
            if (rc) return rc;
        }
        ctx->staged_n = real_n;
        for (size_t k = 0; k < nd; ++k) {
            ctx->devs[k].n_first = first[k];
            ctx->devs[k].n_count = count[k];
        }
        uint64_t need = 0;
        for (uint64_t u : acc_used) need += u;
        if (need > cigar_cap) {
            cigar_off[0] = need;
            sync_and_time(ctx);
            return fail(ctx, ZOE_CUDA_E_CIGAR_CAP, "CIGAR buffer too small: the best hits need %llu words, have %llu",
                        (unsigned long long)need, (unsigned long long)cigar_cap);
        }
        // the CIGAR stream in read order
        for (size_t k = 0; k < nd; ++k) {
            Device &d = ctx->devs[k];
            if (d.n_count == 0) continue;
            CU(ctx, cudaSetDevice(d.id));
            CU(ctx, d.bh_cig_off.reserve((d.n_count + 1) * sizeof(uint64_t)));
            CU(ctx, d.bh_cig.reserve(std::max<uint64_t>(acc_used[k], 1) * sizeof(uint32_t)));
            rc = scan_counts(ctx, d, d.bh_cig_count.as<uint32_t>(), d.n_count, d.bh_cig_off.as<uint64_t>(),
                             d.bh_tab.as<unsigned long long>() + (size_t)kBhTabRows * K);
            if (rc) return rc;
            if (acc_used[k]) {
                const uint32_t blocks = (uint32_t)std::min<uint64_t>((d.n_count + 7) / 8, (uint64_t)d.sm_count * 16);
                best_hit_cigar_gather_kernel<<<blocks, 256, 0, d.stream>>>(d.bh_acc.as<uint32_t>(), d.bh_cig_src.as<uint64_t>(),
                                                                          d.bh_cig_count.as<uint32_t>(), d.n_count,
                                                                          d.bh_cig_off.as<uint64_t>(), d.bh_cig.as<uint32_t>());
                CU(ctx, cudaGetLastError());
                ctx->last_launches++;
            }
        }
        ctx->stats.pairs += aligned;
        ctx->stats.cells += aligned_cells;
        if (pair)
            for (Device &d : ctx->devs) {
                rc = finalize_pairs(ctx, d, pair->min_insert, pair->max_insert);
                if (rc) return rc;
            }
    }
    // per-read outputs (and the CIGAR stream) to the caller
    uint64_t cig_base = 0;
    for (size_t k = 0; k < nd; ++k) {
        Device &d = ctx->devs[k];
        if (d.n_count == 0) continue;
        CU(ctx, cudaSetDevice(d.id));
        const size_t first = d.n_first, cnt = d.n_count;
        auto d2h = [&](void *dst, const DevBuf &src, size_t elem) -> cudaError_t {
            if (!dst) return cudaSuccess;
            return cudaMemcpyAsync((uint8_t *)dst + first * elem, src.p, cnt * elem, cudaMemcpyDeviceToHost, d.stream);
        };
        if (pair) {  // per-pair outputs: the device's pairs are its mates halved
            auto pair_d2h = [&](void *dst, const DevBuf &src, size_t elem) -> cudaError_t {
                if (!dst) return cudaSuccess;
                return cudaMemcpyAsync((uint8_t *)dst + first / 2 * elem, src.p, cnt / 2 * elem, cudaMemcpyDeviceToHost,
                                       d.stream);
            };
            CU(ctx, pair_d2h(hit, d.pr_hit, 4));
            if (align) {
                CU(ctx, pair_d2h(pair->proper, d.pr_proper, 1));
                CU(ctx, pair_d2h(pair->tlen, d.pr_tlen, 4));
            }
        } else {
            CU(ctx, d2h(hit, d.bh_hit, 4));
        }
        CU(ctx, d2h(strand, d.bh_strand, 1));
        CU(ctx, d2h(score, d.bh_out32[0], 4));
        CU(ctx, d2h(status, d.bh_out8[0], 1));
        CU(ctx, d2h(tier, d.bh_out8[1], 1));
        CU(ctx, d2h(runner_up, d.bh_runner, 4));
        if (!align) continue;
        CU(ctx, d2h(ref_start, d.bh_out32[1], 4));
        CU(ctx, d2h(ref_end, d.bh_out32[2], 4));
        CU(ctx, d2h(query_start, d.bh_out32[3], 4));
        CU(ctx, d2h(query_end, d.bh_out32[4], 4));
        CU(ctx, d2h(hazard, d.bh_out8[2], 1));
        CU(ctx, cudaMemcpyAsync(cigar_off + first, d.bh_cig_off.p, (cnt + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost,
                                d.stream));
        if (acc_used[k])
            CU(ctx, cudaMemcpyAsync(cigar + cig_base, d.bh_cig.p, acc_used[k] * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                                    d.stream));
        CU(ctx, cudaStreamSynchronize(d.stream));
        if (cig_base)
            for (size_t i = 0; i <= cnt; ++i) cigar_off[first + i] += cig_base;
        cig_base += acc_used[k];
    }
    if (align && n == 0) cigar_off[0] = 0;
    rc = sync_and_time(ctx);
    if (rc) return rc;
    view.ok = true;
    if (align) return 0;
    rc = gather_stats(ctx);  // (real view: pairs and cells of one strand)
    ctx->stats.pairs *= S;
    ctx->stats.cells *= S;
    return rc;
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int zoe_cuda_create(zoe_cuda_ctx **out, const int *device_ids, int n_devices) {
    if (!out) return ZOE_CUDA_E_BAD_ARG;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) return ZOE_CUDA_E_CUDA;  // no CPU fallback: fail loudly
    if (n_devices <= 0) n_devices = 1;
    if (n_devices > count) return ZOE_CUDA_E_BAD_ARG;
    zoe_cuda_ctx *ctx = new zoe_cuda_ctx();
    for (int i = 0; i < 256; ++i) ctx->lut[i] = 0;
    ctx->no_gap_imm = getenv("ZOE_CUDA_NO_GAP_IMM") != nullptr;
    for (int k = 0; k < n_devices; ++k) {
        Device d;
        d.id = device_ids ? device_ids[k] : k;
        if (d.id < 0 || d.id >= count || cudaSetDevice(d.id) != cudaSuccess ||
            cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, d.id) != cudaSuccess ||
            [&] { size_t tot = 0; return cudaMemGetInfo(&d.free_at_create, &tot); }() != cudaSuccess ||
            cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreate(&d.ev_begin) != cudaSuccess || cudaEventCreate(&d.ev_end) != cudaSuccess ||
            cudaEventCreate(&d.ev_k0) != cudaSuccess || cudaEventCreate(&d.ev_k1) != cudaSuccess) {
            delete ctx;
            return ZOE_CUDA_E_CUDA;
        }
        ctx->devs.push_back(d);
        Device l;  // second stream + buffer set on the same GPU (score-batch pipelining)
        l.id = d.id;
        l.sm_count = d.sm_count;
        l.free_at_create = d.free_at_create;
        if (cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreate(&l.ev_begin) != cudaSuccess || cudaEventCreate(&l.ev_end) != cudaSuccess ||
            cudaEventCreate(&l.ev_k0) != cudaSuccess || cudaEventCreate(&l.ev_k1) != cudaSuccess) {
            delete ctx;
            return ZOE_CUDA_E_CUDA;
        }
        ctx->alt.push_back(l);
    }
    *out = ctx;
    return 0;
}

void zoe_cuda_destroy(zoe_cuda_ctx *ctx) {
    if (!ctx) return;
    std::vector<Device *> all;
    for (Device &d : ctx->devs) all.push_back(&d);
    for (Device &d : ctx->alt) all.push_back(&d);
    for (Device *dp : all) {
        Device &d = *dp;
        cudaSetDevice(d.id);
        for (DevBuf *b : {&d.ccodes, &d.coff, &d.wk, &d.lut, &d.corder, &d.ccodes_g, &d.coff_g, &d.corder_g, &d.rseq, &d.roff, &d.best, &d.score, &d.status, &d.tier,
                          &d.wide_ids, &d.counters, &d.pbytes, &d.ends, &d.flags, &d.flag_base, &d.ref_start, &d.ref_end,
                          &d.query_start, &d.query_end, &d.hazard, &d.hazard_list, &d.cig_scratch, &d.cig_count,
                          &d.cig_off, &d.cig_out, &d.ex_hbuf, &d.ex_fbuf, &d.ex_cig, &d.ex_lists, &d.ex_counts, &d.ex_fast_fbuf, &d.weights, &d.tp_pair, &d.tp_off, &d.tp_cap, &d.tp_slot,
                          &d.tp_blob, &d.tp_ctr, &d.tp_cigoff, &d.tp_bw, &d.tp_list, &d.tp_cig, &d.sn_refs, &d.sn_roff, &d.sn_qry, &d.sn_qoff, &d.sn_out, &d.long_ids, &d.long_bnd,
                          &d.long_queue, &d.ckpt, &d.ckpt_base, &d.win_hist, &d.win_bucket, &d.win_items, &d.win_nitems, &d.win_pitems, &d.win_pnitems, &d.win_amb, &d.starts, &d.cig_bsum})
            b->release();
        for (DevBuf *b : {&d.xs_seq, &d.xs_off, &d.strand, &d.sel_cig_count, &d.sel_cig_off, &d.sel_cig_out, &d.sel_ctr})
            b->release();
        for (DevBuf &b : d.sel32) b.release();
        for (DevBuf &b : d.sel8) b.release();
        for (DevBuf *b : {&d.bh_seq, &d.bh_off, &d.bh_key, &d.bh_tab, &d.bh_list, &d.bh_llen, &d.bh_loff, &d.bh_hit,
                          &d.bh_strand, &d.bh_runner, &d.bh_cig_count, &d.bh_cig_src, &d.bh_acc, &d.bh_cig_off, &d.bh_cig})
            b->release();
        for (DevBuf &b : d.bh_out32) b.release();
        for (DevBuf &b : d.bh_out8) b.release();
        if (d.ev_begin) cudaEventDestroy(d.ev_begin);
        if (d.ev_end) cudaEventDestroy(d.ev_end);
        if (d.ev_k0) cudaEventDestroy(d.ev_k0);
        if (d.ev_k1) cudaEventDestroy(d.ev_k1);
        if (d.ev_fork) cudaEventDestroy(d.ev_fork);
        if (d.ev_join) cudaEventDestroy(d.ev_join);
        if (d.aux_stream) cudaStreamDestroy(d.aux_stream);
        if (d.copy_stream) cudaStreamDestroy(d.copy_stream);
        if (d.ev_first) cudaEventDestroy(d.ev_first);
        if (d.ev_copied) cudaEventDestroy(d.ev_copied);
        if (d.stream) cudaStreamDestroy(d.stream);
    }
    delete ctx;
}

const char *zoe_cuda_last_error(const zoe_cuda_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int zoe_cuda_set_scoring(zoe_cuda_ctx *ctx, const int8_t *weights, int S, const uint8_t byte_to_index[256],
                         int8_t gap_open, int8_t gap_extend, int profiled_is_query) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    if (!weights || !byte_to_index || S < 1 || S > 64) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "bad scoring arguments");
    int rc = validate_profile_args(1, gap_open, gap_extend);
    if (rc) return fail(ctx, rc, "invalid gap penalties (open %d, extend %d)", gap_open, gap_extend);
    for (int i = 0; i < 256; ++i)
        if (byte_to_index[i] >= S) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "byte_to_index[%d] out of range", i);
    ctx->S = S;
    ctx->weights.assign(weights, weights + (size_t)S * S);
    memcpy(ctx->lut, byte_to_index, 256);
    ctx->go = -(int)gap_open;
    ctx->ge = -(int)gap_extend;
    ctx->profiled_is_query = profiled_is_query ? 1 : 0;
    ctx->max_weight = *std::max_element(ctx->weights.begin(), ctx->weights.end());
    ctx->bias = std::max(0, -(int)*std::min_element(ctx->weights.begin(), ctx->weights.end()));
    refresh_tier_policy(ctx);
    ctx->plans.clear();
    ctx->have_scoring = true;
    ctx->have_profiled = false;
    ctx->staged = false;
    return 0;
}

int zoe_cuda_set_lanes(zoe_cuda_ctx *ctx, int lanes_i8, int lanes_i16, int lanes_i32) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    for (int l : {lanes_i8, lanes_i16, lanes_i32})
        if (l < 1 || l > 64 || (l & (l - 1))) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "lane counts must be powers of two <= 64");
    ctx->lanes[0] = lanes_i8;
    ctx->lanes[1] = lanes_i16;
    ctx->lanes[2] = lanes_i32;
    return 0;
}

int zoe_cuda_set_width_policy(zoe_cuda_ctx *ctx, int first_bits, int last_bits, int is_unsigned) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    auto ok = [](int b) { return b == 8 || b == 16 || b == 32; };
    if (!ok(first_bits) || !ok(last_bits) || first_bits > last_bits)
        return fail(ctx, ZOE_CUDA_E_BAD_ARG, "bad width policy (%d..%d bits)", first_bits, last_bits);
    ctx->first_bits = first_bits;
    ctx->last_bits = last_bits;
    ctx->is_unsigned = is_unsigned ? 1 : 0;
    refresh_tier_policy(ctx);
    return 0;
}

int zoe_cuda_set_align_options(zoe_cuda_ctx *ctx, int mode, int checkpoint_log2, int slack) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    if (mode < 0 || mode > 2 || checkpoint_log2 < 2 || checkpoint_log2 > 16 || slack < 1 || slack > (1 << 20))
        return fail(ctx, ZOE_CUDA_E_BAD_ARG, "bad align options (mode %d, checkpoint_log2 %d, slack %d)", mode, checkpoint_log2, slack);
    ctx->align_mode = mode;
    ctx->win_cb_log2 = checkpoint_log2;
    ctx->win_slack = (uint32_t)slack;
    ctx->win_slack_set = true;
    return 0;
}

int zoe_cuda_set_memory_budget(zoe_cuda_ctx *ctx, uint64_t scratch_bytes) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    ctx->flag_budget_bytes = scratch_bytes;  // 0 = automatic
    return 0;
}

int zoe_cuda_set_profiled(zoe_cuda_ctx *ctx, const uint8_t *concat, const uint64_t *offsets, uint32_t n) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    if (!ctx->have_scoring) return fail(ctx, ZOE_CUDA_E_STATE, "set_scoring must be called before set_profiled");
    if (n == 0 || !concat || !offsets) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "no profiled sequences");
    uint64_t total = offsets[n] - offsets[0];
    if (total > 0x7fffffffULL) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "profiled sequences too long");
    uint32_t max_len = 0;
    for (uint32_t j = 0; j < n; ++j) {
        if (offsets[j + 1] < offsets[j]) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "offsets must be non-decreasing");
        uint64_t len = offsets[j + 1] - offsets[j];
        // StripedProfile::new -> validate_profile_args: an empty profiled sequence is an error
        if (len == 0) return fail(ctx, ZOE_CUDA_E_EMPTY_SEQUENCE, "profiled sequence %u is empty", j);
        max_len = std::max<uint32_t>(max_len, (uint32_t)len);
    }
    int rc = install_profiled(ctx, concat, offsets, n, max_len);
    if (rc) return rc;
    ctx->have_profiled = true;
    ctx->staged = false;
    return 0;
}

int zoe_cuda_stage_streamed(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets, uint64_t n) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    begin_call(ctx);
    int rc = stage_on_devices(ctx, streamed_concat, offsets, n);
    if (rc) return rc;
    return sync_and_time(ctx);
}

int zoe_cuda_run_score_staged(zoe_cuda_ctx *ctx) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    if (!ctx->staged) return fail(ctx, ZOE_CUDA_E_STATE, "nothing staged");
    begin_call(ctx);
    for (Device &d : ctx->devs) {
        CU(ctx, cudaSetDevice(d.id));
        CU(ctx, cudaEventRecord(d.ev_begin, d.stream));
    }
    for (Device &d : ctx->devs) {
        int rc = run_score_on_device(ctx, d);
        if (rc) return rc;
    }
    int rc = sync_and_time(ctx);
    if (rc) return rc;
    return gather_stats(ctx);
}

int zoe_cuda_run_align_staged(zoe_cuda_ctx *ctx) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    if (!ctx->staged) return fail(ctx, ZOE_CUDA_E_STATE, "nothing staged");
    begin_call(ctx);
    for (Device &d : ctx->devs) {
        CU(ctx, cudaSetDevice(d.id));
        CU(ctx, cudaEventRecord(d.ev_begin, d.stream));
    }
    // generous device-side CIGAR capacity: 64 words per pair, at most 1 GB (typical CIGARs have <= 5 entries; cheap gaps
    // fragment them).  Nothing is fetched by this entry point: words beyond the capacity are dropped, not an error.
    int rc = for_each_device(ctx, [&](Device &d) {
        return run_align_on_device(ctx, d, std::min<uint64_t>((uint64_t)d.n_count * ctx->n_prof * 64 + 1024, (uint64_t)1 << 28));
    });
    if (rc) return rc;
    rc = sync_and_time(ctx);
    if (rc) return rc;
    return gather_stats(ctx);
}

int zoe_cuda_fetch_scores(zoe_cuda_ctx *ctx, uint32_t *score, uint8_t *status, uint8_t *tier) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    if (!ctx->staged) return fail(ctx, ZOE_CUDA_E_STATE, "nothing staged");
    for (Device &d : ctx->devs) {
        if (d.n_count == 0) continue;
        CU(ctx, cudaSetDevice(d.id));
        size_t first = (size_t)d.n_first * ctx->n_prof, pairs = (size_t)d.n_count * ctx->n_prof;
        if (score)
            CU(ctx, cudaMemcpyAsync(score + first, d.score.p, pairs * sizeof(uint32_t), cudaMemcpyDeviceToHost, d.stream));
        if (status) CU(ctx, cudaMemcpyAsync(status + first, d.status.p, pairs, cudaMemcpyDeviceToHost, d.stream));
        if (tier) CU(ctx, cudaMemcpyAsync(tier + first, d.tier.p, pairs, cudaMemcpyDeviceToHost, d.stream));
    }
    for (Device &d : ctx->devs) {
        CU(ctx, cudaSetDevice(d.id));
        CU(ctx, cudaStreamSynchronize(d.stream));
    }
    return 0;
}

int zoe_cuda_sw_score_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets, uint64_t n,
                            uint32_t *score, uint8_t *status, uint8_t *tier) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    begin_call(ctx);
    int rc = prepare_batch(ctx, streamed_concat, offsets, n);
    if (rc) return rc;
    auto d2h = [&](Device &d) { return queue_score_d2h(ctx, d, score, status, tier); };
    // Large batches are cut into sub-batches that alternate between the two streams of a GPU, so the H2D copy of the
    // next sub-batch and the D2H copy of the previous one overlap the kernels of the current one.  Not for the long-row
    // path (its copies are negligible next to its kernels) nor when packed lanes may overflow (the 32-bit re-run
    // synchronises with the host).
    constexpr int kSub = 4;
    const uint64_t bound = (uint64_t)std::min<uint32_t>(ctx->staged_max_len, ctx->max_prof_len) * (uint64_t)std::max(ctx->max_weight, 0);
    const uint64_t per_dev = n / std::max<size_t>(ctx->devs.size(), 1);
    // worth it only when the copies are a visible share of the step: each sub-batch is its own launch with its own
    // tail (cfg 2: copies 3 % of the step, one shot is faster; cfg 5: 40 %, pipelining gains 7 %)
    const double copy_s = ((double)(n ? offsets[n] - offsets[0] : 0) + (double)n * 8.0 + (double)n * ctx->n_prof * 6.0) / 25e9;
    const double kernel_s = (double)ctx->staged_cells / 6e12;
    const bool pipeline = per_dev >= (uint64_t)kSub * 65536 && ctx->staged_max_len <= (uint32_t)kMaxRowsSinglePass &&
                          bound < (uint64_t)(kPackedLimit - std::max(ctx->max_weight, 0) - 1) &&
                          (copy_s > 0.1 * kernel_s || getenv("ZOE_CUDA_PIPELINE")) && !getenv("ZOE_CUDA_NO_PIPELINE");
    if (!pipeline) {
        for (Device &d : ctx->devs) {
            rc = stage_device(ctx, d, streamed_concat, offsets, true, /*split=*/true);
            if (rc) return rc;
        }
        for (Device &d : ctx->devs) {
            rc = run_score_on_device(ctx, d);
            if (rc) return rc;
        }
        for (Device &d : ctx->devs) {
            rc = d2h(d);
            if (rc) return rc;
        }
        ctx->staged = true;
    } else {
        const size_t nd = ctx->devs.size();
        std::vector<uint64_t> first(nd), count(nd);
        for (size_t k = 0; k < nd; ++k) {
            first[k] = ctx->devs[k].n_first;
            count[k] = ctx->devs[k].n_count;
        }
        ctx->alt_used = true;
        for (int i = 0; i < kSub; ++i) {
            for (size_t k = 0; k < nd; ++k) {
                Device &lane = (i & 1) ? ctx->alt[k] : ctx->devs[k];
                // an even first index keeps the packed pairs (sequences 2t, 2t+1) of the one-shot run
                const uint64_t lo = (count[k] * i / kSub) & ~1ull, hi = i + 1 == kSub ? count[k] : ((count[k] * (i + 1) / kSub) & ~1ull);
                lane.n_first = first[k] + lo;
                lane.n_count = hi - lo;
                rc = stage_device(ctx, lane, streamed_concat, offsets, /*record_begin=*/i < 2);
                if (rc) return rc;
                rc = run_score_on_device(ctx, lane, /*reset_counters=*/i < 2);
                if (rc) return rc;
            }
            if (i > 0)
                for (size_t k = 0; k < nd; ++k) {
                    rc = d2h(((i - 1) & 1) ? ctx->alt[k] : ctx->devs[k]);
                    if (rc) return rc;
                }
        }
        for (size_t k = 0; k < nd; ++k) {
            rc = d2h(((kSub - 1) & 1) ? ctx->alt[k] : ctx->devs[k]);
            if (rc) return rc;
        }
        // the device buffers now hold sub-batches only: nothing is "staged" for the run_*_staged entry points
        ctx->staged = false;
    }
    rc = sync_and_time(ctx);
    if (rc) return rc;
    return gather_stats(ctx);
}

int zoe_cuda_sw_align_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets, uint64_t n,
                            uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *ref_start, uint32_t *ref_end,
                            uint32_t *query_start, uint32_t *query_end, uint32_t *cigar, uint64_t *cigar_off,
                            uint64_t cigar_cap, uint8_t *hazard) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    if (!cigar_off || (!cigar && cigar_cap)) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "null CIGAR outputs");
    begin_call(ctx);
    DebugTimer dbg;
    int rc = stage_on_devices(ctx, streamed_concat, offsets, n, /*split=*/true);
    if (rc) return rc;
    dbg.lap("align: stage");
    // A batch that mixes long (> 1024 residues) and short sequences is split (align_split_long_short).
    // Detected from the lengths the staging pass collects anyway (a separate pass that lists the indices of 1M reads
    // cost 3-4 ms of host time in front of every call); the upload already queued for the whole batch is drained and dropped.
    if (n > 0 && ctx->staged_max_len > (uint32_t)kMaxRowsSinglePass && ctx->staged_min_len <= (uint32_t)kMaxRowsSinglePass) {
        for (Device &d : ctx->devs) {
            cudaSetDevice(d.id);
            if (d.copy_stream) cudaStreamSynchronize(d.copy_stream);
            cudaStreamSynchronize(d.stream);
            d.copy_pending = false;
        }
        ctx->staged = false;
        rc = align_split_long_short(ctx, false, streamed_concat, offsets, n, score, status, tier, ref_start, ref_end,
                                    query_start, query_end, cigar, cigar_off, cigar_cap, hazard, nullptr);
        if (rc != kNotMixed) return rc;
    }
    rc = for_each_device(ctx, [&](Device &d) { return run_align_on_device(ctx, d, cigar_cap); });
    if (rc) return rc;
    dbg.lap("align: run_align_on_device");
    rc = fetch_alignments(ctx, score, status, tier, ref_start, ref_end, query_start, query_end, cigar, cigar_off, cigar_cap,
                          hazard);
    if (rc) return rc;
    if (n == 0) cigar_off[0] = 0;
    dbg.lap("align: d2h");
    rc = sync_and_time(ctx);
    if (rc) return rc;
    return gather_stats(ctx);
}

int zoe_cuda_sw_score_ranges_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets, uint64_t n,
                                   uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *ref_start, uint32_t *ref_end,
                                   uint32_t *query_start, uint32_t *query_end) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    begin_call(ctx);
    int rc = stage_on_devices(ctx, streamed_concat, offsets, n, /*split=*/true);
    if (rc) return rc;
    rc = for_each_device(ctx, [&](Device &d) { return run_ranges_on_device(ctx, d); });
    if (rc) return rc;
    rc = queue_ranges_d2h(ctx, score, status, tier, ref_start, ref_end, query_start, query_end);
    if (rc) return rc;
    rc = sync_and_time(ctx);
    if (rc) return rc;
    return gather_stats(ctx);
}

int zoe_cuda_run_ranges_staged(zoe_cuda_ctx *ctx) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    if (!ctx->staged) return fail(ctx, ZOE_CUDA_E_STATE, "nothing staged");
    begin_call(ctx);
    for (Device &d : ctx->devs) {
        CU(ctx, cudaSetDevice(d.id));
        CU(ctx, cudaEventRecord(d.ev_begin, d.stream));
    }
    int rc = for_each_device(ctx, [&](Device &d) { return run_ranges_on_device(ctx, d); });
    if (rc) return rc;
    rc = sync_and_time(ctx);
    if (rc) return rc;
    return gather_stats(ctx);
}

int zoe_cuda_sw_align_3pass_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets, uint64_t n,
                                  uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *ref_start, uint32_t *ref_end,
                                  uint32_t *query_start, uint32_t *query_end, uint32_t *cigar, uint64_t *cigar_off,
                                  uint64_t cigar_cap) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    if (!cigar_off || (!cigar && cigar_cap)) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "null CIGAR outputs");
    begin_call(ctx);
    int rc = stage_on_devices(ctx, streamed_concat, offsets, n, /*split=*/true);
    if (rc) return rc;
    rc = for_each_device(ctx, [&](Device &d) { return run_3pass_on_device(ctx, d, cigar_cap); });
    if (rc) return rc;
    rc = fetch_alignments(ctx, score, status, tier, ref_start, ref_end, query_start, query_end, cigar, cigar_off, cigar_cap,
                          nullptr);
    if (rc) return rc;
    if (n == 0) cigar_off[0] = 0;
    rc = sync_and_time(ctx);
    if (rc) return rc;
    return gather_stats(ctx);
}

int zoe_cuda_run_3pass_staged(zoe_cuda_ctx *ctx) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    if (!ctx->staged) return fail(ctx, ZOE_CUDA_E_STATE, "nothing staged");
    begin_call(ctx);
    for (Device &d : ctx->devs) {
        CU(ctx, cudaSetDevice(d.id));
        CU(ctx, cudaEventRecord(d.ev_begin, d.stream));
    }
    int rc = for_each_device(ctx, [&](Device &d) { return run_3pass_on_device(ctx, d, (uint64_t)d.n_count * ctx->n_prof * 8 + 1024); });
    if (rc) return rc;
    rc = sync_and_time(ctx);
    if (rc) return rc;
    return gather_stats(ctx);
}

int zoe_cuda_sw_score_both_strands_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets,
                                         uint64_t n, uint32_t *score, uint8_t *status, uint8_t *tier, uint8_t *strand) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    begin_call(ctx);
    DoubledView view(ctx);
    int rc = stage_both_strands(ctx, view, streamed_concat, offsets, n, /*pair_limit=*/false);
    if (rc) return rc;
    uint64_t no_cigar = 0;
    for (Device &d : ctx->devs) {
        rc = run_score_on_device(ctx, d);
        if (rc) return rc;
        rc = select_strands(ctx, d, StrandOutputs::Score, &no_cigar);
        if (rc) return rc;
    }
    view.leave();
    for (Device &d : ctx->devs) {
        rc = queue_score_d2h(ctx, d, score, status, tier);
        if (rc) return rc;
    }
    rc = queue_strand_d2h(ctx, strand);
    if (rc) return rc;
    rc = sync_and_time(ctx);
    if (rc) return rc;
    view.ok = true;
    return gather_both_strands_stats(ctx);
}

int zoe_cuda_sw_score_ranges_both_strands_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets,
                                                uint64_t n, uint32_t *score, uint8_t *status, uint8_t *tier,
                                                uint32_t *ref_start, uint32_t *ref_end, uint32_t *query_start,
                                                uint32_t *query_end, uint8_t *strand) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    begin_call(ctx);
    DoubledView view(ctx);
    int rc = stage_both_strands(ctx, view, streamed_concat, offsets, n, /*pair_limit=*/true);
    if (rc) return rc;
    rc = for_each_device(ctx, [&](Device &d) { return run_ranges_on_device(ctx, d); });
    if (rc) return rc;
    uint64_t no_cigar = 0;
    for (Device &d : ctx->devs) {
        rc = select_strands(ctx, d, StrandOutputs::Ranges, &no_cigar);
        if (rc) return rc;
    }
    view.leave();
    rc = queue_ranges_d2h(ctx, score, status, tier, ref_start, ref_end, query_start, query_end);
    if (rc) return rc;
    rc = queue_strand_d2h(ctx, strand);
    if (rc) return rc;
    rc = sync_and_time(ctx);
    if (rc) return rc;
    view.ok = true;
    return gather_both_strands_stats(ctx);
}

int zoe_cuda_sw_align_both_strands_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets,
                                         uint64_t n, uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *ref_start,
                                         uint32_t *ref_end, uint32_t *query_start, uint32_t *query_end, uint32_t *cigar,
                                         uint64_t *cigar_off, uint64_t cigar_cap, uint8_t *hazard, uint8_t *strand) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    return align_both_strands(ctx, false, streamed_concat, offsets, n, score, status, tier, ref_start, ref_end, query_start,
                              query_end, cigar, cigar_off, cigar_cap, hazard, strand);
}

int zoe_cuda_sw_align_3pass_both_strands_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets,
                                               uint64_t n, uint32_t *score, uint8_t *status, uint8_t *tier,
                                               uint32_t *ref_start, uint32_t *ref_end, uint32_t *query_start,
                                               uint32_t *query_end, uint32_t *cigar, uint64_t *cigar_off, uint64_t cigar_cap,
                                               uint8_t *strand) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    return align_both_strands(ctx, true, streamed_concat, offsets, n, score, status, tier, ref_start, ref_end, query_start,
                              query_end, cigar, cigar_off, cigar_cap, nullptr, strand);
}

int zoe_cuda_sw_score_best_hit_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets,
                                     uint64_t n, int both_strands, uint32_t *hit, uint8_t *strand, uint32_t *score,
                                     uint8_t *status, uint8_t *tier, uint32_t *runner_up) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    return best_hit(ctx, false, both_strands != 0, false, streamed_concat, offsets, n, nullptr, hit, strand, score, status, tier,
                    runner_up, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr);
}

int zoe_cuda_sw_align_best_hit_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets,
                                     uint64_t n, int both_strands, int three_pass, uint32_t *hit, uint8_t *strand,
                                     uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *runner_up,
                                     uint32_t *ref_start, uint32_t *ref_end, uint32_t *query_start, uint32_t *query_end,
                                     uint32_t *cigar, uint64_t *cigar_off, uint64_t cigar_cap, uint8_t *hazard) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    return best_hit(ctx, true, both_strands != 0, three_pass != 0, streamed_concat, offsets, n, nullptr, hit, strand, score, status,
                    tier, runner_up, ref_start, ref_end, query_start, query_end, cigar, cigar_off, cigar_cap, hazard);
}

int zoe_cuda_sw_score_paired_best_hit_batch(zoe_cuda_ctx *ctx, const uint8_t *mate1_concat, const uint64_t *mate1_offsets,
                                            const uint8_t *mate2_concat, const uint64_t *mate2_offsets, uint64_t n_pairs,
                                            uint32_t *hit, uint8_t *strand, uint32_t *score, uint8_t *status, uint8_t *tier,
                                            uint32_t *runner_up) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    const PairedArgs pair{mate2_concat, mate2_offsets, 0, ~0u, nullptr, nullptr};
    return best_hit(ctx, false, true, false, mate1_concat, mate1_offsets, n_pairs, &pair, hit, strand, score, status, tier,
                    runner_up, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr);
}

int zoe_cuda_sw_align_paired_best_hit_batch(zoe_cuda_ctx *ctx, const uint8_t *mate1_concat, const uint64_t *mate1_offsets,
                                            const uint8_t *mate2_concat, const uint64_t *mate2_offsets, uint64_t n_pairs,
                                            int three_pass, uint32_t min_insert, uint32_t max_insert, uint32_t *hit,
                                            uint8_t *proper, int *tlen, uint8_t *strand, uint32_t *score, uint8_t *status,
                                            uint8_t *tier, uint32_t *runner_up, uint32_t *ref_start, uint32_t *ref_end,
                                            uint32_t *query_start, uint32_t *query_end, uint32_t *cigar, uint64_t *cigar_off,
                                            uint64_t cigar_cap, uint8_t *hazard) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    const PairedArgs pair{mate2_concat, mate2_offsets, min_insert, max_insert, proper, tlen};
    return best_hit(ctx, true, true, three_pass != 0, mate1_concat, mate1_offsets, n_pairs, &pair, hit, strand, score,
                    status, tier, runner_up, ref_start, ref_end, query_start, query_end, cigar, cigar_off, cigar_cap, hazard);
}

int zoe_cuda_sneaky_snake_batch(zoe_cuda_ctx *ctx, const uint8_t *refs, const uint64_t *ref_offsets, const uint8_t *queries,
                                const uint64_t *query_offsets, uint64_t n, float threshold, uint8_t *out) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    if (n == 0) return 0;
    if (!ref_offsets || !query_offsets || !out) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "null argument");
    begin_call(ctx);
    // pairs are split over the context's devices by contiguous index range, like every other batch call
    const size_t nd = ctx->devs.size();
    for (Device &d : ctx->devs) {  // every device takes part in the timing, also one that gets no pairs
        CU(ctx, cudaSetDevice(d.id));
        CU(ctx, cudaEventRecord(d.ev_begin, d.stream));
    }
    for (size_t k = 0; k < nd; ++k) {
        Device &d = ctx->devs[k];
        const uint64_t lo = n * k / nd, hi = n * (k + 1) / nd, cnt = hi - lo;
        if (cnt == 0) continue;
        CU(ctx, cudaSetDevice(d.id));
        const uint64_t rb = ref_offsets[hi] - ref_offsets[lo], qb = query_offsets[hi] - query_offsets[lo];
        if ((rb && !refs) || (qb && !queries)) return fail(ctx, ZOE_CUDA_E_BAD_ARG, "null sequence buffer");
        CU(ctx, d.sn_refs.reserve(std::max<uint64_t>(rb, 1)));
        CU(ctx, d.sn_qry.reserve(std::max<uint64_t>(qb, 1)));
        CU(ctx, d.sn_roff.reserve((cnt + 1) * sizeof(uint64_t)));
        CU(ctx, d.sn_qoff.reserve((cnt + 1) * sizeof(uint64_t)));
        CU(ctx, d.sn_out.reserve(cnt));
        if (rb) CU(ctx, cudaMemcpyAsync(d.sn_refs.p, refs + ref_offsets[lo], rb, cudaMemcpyHostToDevice, d.stream));
        if (qb) CU(ctx, cudaMemcpyAsync(d.sn_qry.p, queries + query_offsets[lo], qb, cudaMemcpyHostToDevice, d.stream));
        CU(ctx, cudaMemcpyAsync(d.sn_roff.p, ref_offsets + lo, (cnt + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, d.stream));
        CU(ctx, cudaMemcpyAsync(d.sn_qoff.p, query_offsets + lo, (cnt + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, d.stream));
        SnakeParams sp{};
        // the offsets stay absolute; the kernel subtracts the shard's first offset
        sp.refs = d.sn_refs.as<uint8_t>();
        sp.ref_off = d.sn_roff.as<uint64_t>();
        sp.ref_base = ref_offsets[lo];
        sp.queries = d.sn_qry.as<uint8_t>();
        sp.qry_off = d.sn_qoff.as<uint64_t>();
        sp.qry_base = query_offsets[lo];
        sp.n = cnt;
        sp.threshold = threshold;
        sp.out = d.sn_out.as<uint8_t>();
        CU(ctx, cudaEventRecord(d.ev_k0, d.stream));
        // warp per pair when both sequences of every pair fit the staging area, else zoe's loops one thread per pair
        uint64_t longest = 0;
        for (uint64_t q = lo; q < hi; ++q)
            longest = std::max<uint64_t>(longest, std::max(ref_offsets[q + 1] - ref_offsets[q], query_offsets[q + 1] - query_offsets[q]));
        if (longest <= (uint64_t)kSnakeStage && !getenv("ZOE_CUDA_SNAKE_THREAD")) {
            const int wpb = 8;
            const size_t smem = (size_t)wpb * 2 * kSnakeStage;
            const uint32_t nb = (uint32_t)std::min<uint64_t>((cnt + wpb - 1) / wpb, (uint64_t)d.sm_count * 32);
            sneaky_snake_warp_kernel<<<nb, wpb * 32, smem, d.stream>>>(sp);
        } else {
            sneaky_snake_kernel<<<(uint32_t)((cnt + 127) / 128), 128, 0, d.stream>>>(sp);
        }
        CU(ctx, cudaGetLastError());
        CU(ctx, cudaEventRecord(d.ev_k1, d.stream));
        d.timed_kernel = true;
        ctx->last_launches++;
        CU(ctx, cudaMemcpyAsync(out + lo, d.sn_out.p, cnt, cudaMemcpyDeviceToHost, d.stream));
    }
    return sync_and_time(ctx);
}

int zoe_cuda_last_timing(const zoe_cuda_ctx *ctx, float *total_ms, float *dp_kernel_ms, uint32_t *kernel_launches) {
    if (!ctx) return ZOE_CUDA_E_BAD_ARG;
    if (total_ms) *total_ms = ctx->last_total_ms;
    if (dp_kernel_ms) *dp_kernel_ms = ctx->last_dp_ms;
    if (kernel_launches) *kernel_launches = ctx->last_launches.load();
    return 0;
}

int zoe_cuda_last_stats(const zoe_cuda_ctx *ctx, zoe_cuda_stats *out) {
    if (!ctx || !out) return ZOE_CUDA_E_BAD_ARG;
    *out = ctx->stats;
    return 0;
}

int zoe_cuda_dpx_peak(zoe_cuda_ctx *ctx, int kind, double *giga_lane_instr_per_s, float *ms_out) {
    if (!ctx || !giga_lane_instr_per_s) return ZOE_CUDA_E_BAD_ARG;
    Device &d = ctx->devs[0];
    CU(ctx, cudaSetDevice(d.id));
    const int iters = 4096, threads = 256, blocks = d.sm_count * 8;
    DevBuf out;
    CU(ctx, out.reserve(threads * sizeof(uint32_t)));
    float best_ms = 1e30f;
    for (int rep = 0; rep < 5; ++rep) {
        CU(ctx, cudaEventRecord(d.ev_k0, d.stream));
        if (kind == 0)
            dpx_peak_kernel<0><<<blocks, threads, 0, d.stream>>>(out.as<uint32_t>(), iters, 12345u + rep);
        else if (kind == 2)
            dpx_peak_kernel<2><<<blocks, threads, 0, d.stream>>>(out.as<uint32_t>(), iters, 12345u + rep);
        else if (kind == 3)
            dpx_peak_kernel<3><<<blocks, threads, 0, d.stream>>>(out.as<uint32_t>(), iters, 12345u + rep);
        else
            dpx_peak_kernel<1><<<blocks, threads, 0, d.stream>>>(out.as<uint32_t>(), iters, 12345u + rep);
        CU(ctx, cudaGetLastError());
        CU(ctx, cudaEventRecord(d.ev_k1, d.stream));
        CU(ctx, cudaStreamSynchronize(d.stream));
        float ms = 0.f;
        CU(ctx, cudaEventElapsedTime(&ms, d.ev_k0, d.ev_k1));
        if (rep > 0) best_ms = std::min(best_ms, ms);
    }
    out.release();
    // kind 0: 16 DPX instructions per inner iteration; kind 1: 8 cell pairs x 5.5 instructions
    // kind 2: 8 x (2 hmax2 + 2 integer ops); kind 3: 8 cell pairs x 6 instructions
    double instr_per_thread = (kind == 0) ? 16.0 * iters : (kind == 2 ? 32.0 * iters : (kind == 3 ? 48.0 * iters : 8.0 * 5.5 * iters));
    double lanes = (double)blocks * threads;
    *giga_lane_instr_per_s = instr_per_thread * lanes / (best_ms * 1e-3) / 1e9;
    if (ms_out) *ms_out = best_ms;
    return 0;
}

void *zoe_cuda_stream(zoe_cuda_ctx *ctx, int dev_index) {
    if (!ctx || dev_index < 0 || dev_index >= (int)ctx->devs.size()) return nullptr;
    return (void *)ctx->devs[dev_index].stream;
}

}  // extern "C"
