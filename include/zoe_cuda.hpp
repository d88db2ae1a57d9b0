// zoe_cuda.hpp -- header-only C++ mirror of zoe's Rust interface for the striped SW path, over the
// C ABI of include/zoe_cuda.h.  zoe is compiled code (Rust); no Rust toolchain exists in this image,
// so the host side above the C ABI is written in C++ with zoe's names, argument meaning and error
// behaviour (the Rust `cuda` backend a maintainer would add is shown in INTEGRATION.md):
//
//   zoe                                                         here
//   ---------------------------------------------------------   -----------------------------------
//   ProfileError            src/alignment/errors.rs:6-15        zoe::cuda::ProfileError (exception)
//   MaybeAligned<T>         src/alignment/types/output.rs:18-25 zoe::cuda::MaybeAligned<T>
//   Alignment<u32>          src/alignment/types/output.rs:264   zoe::cuda::Alignment
//   Ciglet / AlignmentStates src/data/types/cigar, types/state.rs std::vector<Ciglet>
//   SeqSrc                  src/alignment/mod.rs:157-162        zoe::cuda::SeqSrc
//   WeightMatrix<i8,S>      src/data/matrices/mod.rs:230-235    zoe::cuda::WeightMatrix
//   SharedProfiles::new_with_w{128,256,512}, sw_score_from_i8,
//   sw_align_from_i8        src/alignment/profile_set.rs        zoe::cuda::CudaProfiles (batched)
#pragma once
#include <cstdint>
#include <stdexcept>
#include <optional>
#include <string>
#include <utility>
#include <vector>

#include "zoe_cuda.h"

namespace zoe {
namespace cuda {

struct ProfileError : std::invalid_argument {
    enum Kind { EmptySequence, GapOpenOutOfRange, GapExtendOutOfRange, BadGapWeights } kind;
    ProfileError(Kind k, const std::string &msg) : std::invalid_argument(msg), kind(k) {}
};

struct CudaError : std::runtime_error {
    int code;
    CudaError(int c, const std::string &msg) : std::runtime_error(msg), code(c) {}
};

enum class Status : uint8_t { Some = ZOE_CUDA_SOME, Overflowed = ZOE_CUDA_OVERFLOWED, Unmapped = ZOE_CUDA_UNMAPPED };

template <class T>
struct MaybeAligned {
    Status status = Status::Unmapped;
    T value{};
    bool is_some() const { return status == Status::Some; }
    const T &unwrap() const {
        if (status != Status::Some) throw std::logic_error("called unwrap() on a non-Some MaybeAligned");
        return value;
    }
};

struct Ciglet {
    uint32_t inc;
    char op;  // one of M I D S
};

struct Alignment {
    uint32_t score = 0;
    std::pair<uint32_t, uint32_t> ref_range{0, 0}, query_range{0, 0};  // 0-based half-open
    std::vector<Ciglet> states;
    uint32_t ref_len = 0, query_len = 0;
    std::string cigar() const {
        std::string s;
        for (const Ciglet &c : states) s += std::to_string(c.inc) + c.op;
        return s;
    }
};

// zoe's ScoreAndRanges<u32> (src/alignment/types/output.rs): score + 0-based half-open ranges
struct ScoreAndRanges {
    uint32_t score = 0;
    std::pair<uint32_t, uint32_t> ref_range{0, 0}, query_range{0, 0};
};

enum class SeqSrc { Query, Reference };

// Which strand of a streamed sequence a both-strand result belongs to (zoe_cuda.h, both-strand search)
enum class Strand : uint8_t { Forward = 0, Reverse = 1 };

struct WeightMatrix {
    int S = 0;
    std::vector<int8_t> weights;  // S*S, weights[ref_idx][query_idx]
    uint8_t byte_to_index[256];
    // WeightMatrix::new (matrices/mod.rs:358-399) for the DNA profile map (dna.rs:177-178)
    static WeightMatrix new_dna_matrix(int8_t matching, int8_t mismatch, bool ignore_n = true) {
        WeightMatrix m;
        m.S = 5;
        m.weights.assign(25, mismatch);
        for (int i = 0; i < 5; ++i) m.weights[i * 5 + i] = matching;
        if (ignore_n)
            for (int i = 0; i < 5; ++i) m.weights[4 * 5 + i] = m.weights[i * 5 + 4] = 0;
        for (int i = 0; i < 256; ++i) m.byte_to_index[i] = 4;
        const char *keys = "ACGT";
        for (int i = 0; i < 4; ++i) {
            m.byte_to_index[(uint8_t)keys[i]] = (uint8_t)i;
            m.byte_to_index[(uint8_t)(keys[i] + 32)] = (uint8_t)i;
        }
        m.byte_to_index[(uint8_t)'U'] = m.byte_to_index[(uint8_t)'u'] = 3;
        return m;
    }
};

class CudaProfiles {
  public:
    // SharedProfiles::new_with_w256 (profile_set.rs:434-483) for every target; `streamed_are` says which role
    // the sequences later passed to sw_*_batch play (SeqSrc::Query(seq) => targets are references).
    static CudaProfiles new_with_w128(const std::vector<std::string> &t, const WeightMatrix &m, int8_t go, int8_t ge,
                                      SeqSrc streamed_are = SeqSrc::Query, int n_devices = 1) {
        return CudaProfiles(t, m, go, ge, 16, 8, 4, streamed_are, n_devices);
    }
    static CudaProfiles new_with_w256(const std::vector<std::string> &t, const WeightMatrix &m, int8_t go, int8_t ge,
                                      SeqSrc streamed_are = SeqSrc::Query, int n_devices = 1) {
        return CudaProfiles(t, m, go, ge, 32, 16, 8, streamed_are, n_devices);
    }
    static CudaProfiles new_with_w512(const std::vector<std::string> &t, const WeightMatrix &m, int8_t go, int8_t ge,
                                      SeqSrc streamed_are = SeqSrc::Query, int n_devices = 1) {
        return CudaProfiles(t, m, go, ge, 64, 32, 16, streamed_are, n_devices);
    }
    CudaProfiles(CudaProfiles &&o) noexcept : ctx_(o.ctx_), targets_(std::move(o.targets_)), streamed_are_(o.streamed_are_) {
        o.ctx_ = nullptr;
    }
    CudaProfiles(const CudaProfiles &) = delete;
    CudaProfiles &operator=(const CudaProfiles &) = delete;
    ~CudaProfiles() { zoe_cuda_destroy(ctx_); }

    size_t n_profiled() const { return targets_.size(); }

    // out[i * n_profiled + j] == profiles[j].sw_score_from_i8(&seqs[i])
    // Which zoe integer types may report a result: (8,32) = sw_*_from_i8 (default), (16,32) = ..._from_i16,
    // (32,32) = ..._from_i32 (profile_set.rs:71-179); first == last = a standalone StripedProfile<T,N,S>;
    // is_unsigned = the u8/u16/u32 profiles over the biased matrix (matrices/mod.rs:471-491).
    void set_width_policy(int first_bits, int last_bits, bool is_unsigned) {
        check(zoe_cuda_set_width_policy(ctx_, first_bits, last_bits, is_unsigned ? 1 : 0));
    }
    // Tuning only (never changes results): 0 auto, 1 full-matrix direction bits, 2 checkpointed window.
    void set_align_options(int mode, int checkpoint_log2 = 6, int slack = 16) {
        check(zoe_cuda_set_align_options(ctx_, mode, checkpoint_log2, slack));
    }

    // Upper bound on the device scratch of one align / ranges / 3-pass call (0 = automatic); results never depend on it.
    void set_memory_budget(uint64_t scratch_bytes) { check(zoe_cuda_set_memory_budget(ctx_, scratch_bytes)); }

    // out[i * n_profiled + j] == profiles[j].sw_score_ranges_from_i8(SeqSrc::X(&seqs[i])) (profile_set.rs:313-322)
    std::vector<MaybeAligned<ScoreAndRanges>> sw_score_ranges_batch(const std::vector<std::string> &seqs) {
        return ranges(seqs, nullptr);
    }

    std::vector<MaybeAligned<uint32_t>> sw_score_batch(const std::vector<std::string> &seqs) { return scores(seqs, nullptr); }

    // out[i * n_profiled + j] == profiles[j].sw_align_from_i8(SeqSrc::X(&seqs[i])) with X as given at construction
    std::vector<MaybeAligned<Alignment>> sw_align_batch(const std::vector<std::string> &seqs) { return align(seqs, false); }

    // out[i * n_profiled + j] == profiles[j].sw_align_from_i8_3pass(SeqSrc::X(&seqs[i])) (profile_set.rs:213-231)
    std::vector<MaybeAligned<Alignment>> sw_align_3pass_batch(const std::vector<std::string> &seqs) { return align(seqs, true); }

    // Both-strand search (zoe_cuda.h): the better of seqs[i] and its reverse complement for every pair, with the strand;
    // a reverse-strand result's coordinates and CIGAR refer to the reverse complement.
    std::vector<std::pair<MaybeAligned<uint32_t>, Strand>> sw_score_both_strands(const std::vector<std::string> &seqs) {
        std::vector<uint8_t> strand;
        return with_strand(scores(seqs, &strand), strand);
    }
    std::vector<std::pair<MaybeAligned<ScoreAndRanges>, Strand>> sw_score_ranges_both_strands(const std::vector<std::string> &seqs) {
        std::vector<uint8_t> strand;
        return with_strand(ranges(seqs, &strand), strand);
    }
    std::vector<std::pair<MaybeAligned<Alignment>, Strand>> sw_align_both_strands(const std::vector<std::string> &seqs) {
        std::vector<uint8_t> strand;
        return with_strand(align(seqs, false, &strand), strand);
    }
    std::vector<std::pair<MaybeAligned<Alignment>, Strand>> sw_align_3pass_both_strands(const std::vector<std::string> &seqs) {
        std::vector<uint8_t> strand;
        return with_strand(align(seqs, true, &strand), strand);
    }

    // Best-hit search (zoe_cuda.h): per streamed sequence, its best profiled sequence and strand (both_strands), the
    // alignment of that pair and the runner-up score (SAM XS).
    struct BestHit {
        uint32_t index = 0;
        Strand strand = Strand::Forward;
        MaybeAligned<Alignment> result;
        uint32_t runner_up = 0;
    };
    std::vector<BestHit> sw_align_best_hit(const std::vector<std::string> &seqs, bool both_strands = false,
                                           bool three_pass = false) {
        std::vector<uint8_t> buf;
        std::vector<uint64_t> off;
        pack(seqs, buf, off);
        const size_t n = seqs.size();
        std::vector<uint32_t> hit(n + 1), score(n + 1), ru(n + 1), rs(n + 1), re(n + 1), qs(n + 1), qe(n + 1);
        std::vector<uint8_t> strand(n + 1), status(n + 1), tier(n + 1);
        std::vector<uint64_t> coff(n + 2);
        std::vector<uint32_t> cig(16 * n + 1024);
        auto call = [&]() {
            return zoe_cuda_sw_align_best_hit_batch(ctx_, buf.data(), off.data(), n, both_strands ? 1 : 0, three_pass ? 1 : 0,
                                                    hit.data(), strand.data(), score.data(), status.data(), tier.data(),
                                                    ru.data(), rs.data(), re.data(), qs.data(), qe.data(), cig.data(),
                                                    coff.data(), cig.size(), nullptr);
        };
        int rc = call();
        if (rc == ZOE_CUDA_E_CIGAR_CAP) {
            cig.resize(coff[0] + 16);
            rc = call();
        }
        check(rc);
        std::vector<BestHit> out(n);
        for (size_t i = 0; i < n; ++i)
            out[i] = best_hit_at(i, hit[i], seqs[i], strand, score, status, ru, rs, re, qs, qe, coff, cig);
        return out;
    }

    // Paired-end best-hit search (zoe_cuda.h), an FR library: per read pair (mates1[i], mates2[i]), the profiled sequence
    // and orientation both mates support best, each mate's alignment, proper-pair flag and mate 1's TLEN.
    struct PairedHit {
        uint32_t index = 0;
        bool proper = false;
        int32_t tlen = 0;
        BestHit mate1, mate2;
    };
    std::vector<PairedHit> sw_align_paired_best_hit(const std::vector<std::string> &mates1,
                                                    const std::vector<std::string> &mates2, uint32_t min_insert,
                                                    uint32_t max_insert, bool three_pass = false) {
        if (mates1.size() != mates2.size()) throw std::invalid_argument("mate lists differ in length");
        std::vector<uint8_t> buf1, buf2;
        std::vector<uint64_t> off1, off2;
        pack(mates1, buf1, off1);
        pack(mates2, buf2, off2);
        const size_t n = mates1.size(), m = 2 * n + 1;
        std::vector<uint32_t> hit(n + 1), score(m), ru(m), rs(m), re(m), qs(m), qe(m);
        std::vector<int> tlen(n + 1);
        std::vector<uint8_t> proper(n + 1), strand(m), status(m), tier(m);
        std::vector<uint64_t> coff(m + 1);
        std::vector<uint32_t> cig(16 * m + 1024);
        auto call = [&]() {
            return zoe_cuda_sw_align_paired_best_hit_batch(
                ctx_, buf1.data(), off1.data(), buf2.data(), off2.data(), n, three_pass ? 1 : 0, min_insert, max_insert,
                hit.data(), proper.data(), tlen.data(), strand.data(), score.data(), status.data(), tier.data(), ru.data(),
                rs.data(), re.data(), qs.data(), qe.data(), cig.data(), coff.data(), cig.size(), nullptr);
        };
        int rc = call();
        if (rc == ZOE_CUDA_E_CIGAR_CAP) {
            cig.resize(coff[0] + 16);
            rc = call();
        }
        check(rc);
        std::vector<PairedHit> out(n);
        for (size_t i = 0; i < n; ++i) {
            out[i].index = hit[i];
            out[i].proper = proper[i] != 0;
            out[i].tlen = tlen[i];
            out[i].mate1 = best_hit_at(2 * i, hit[i], mates1[i], strand, score, status, ru, rs, re, qs, qe, coff, cig);
            out[i].mate2 = best_hit_at(2 * i + 1, hit[i], mates2[i], strand, score, status, ru, rs, re, qs, qe, coff, cig);
        }
        return out;
    }

  private:
    // Entry k of a best-hit or paired call's per-sequence outputs, for streamed sequence seq placed on profiled j.
    BestHit best_hit_at(size_t k, uint32_t j, const std::string &seq, const std::vector<uint8_t> &strand,
                        const std::vector<uint32_t> &score, const std::vector<uint8_t> &status,
                        const std::vector<uint32_t> &ru, const std::vector<uint32_t> &rs, const std::vector<uint32_t> &re,
                        const std::vector<uint32_t> &qs, const std::vector<uint32_t> &qe,
                        const std::vector<uint64_t> &coff, const std::vector<uint32_t> &cig) const {
        static const char ops[] = {'M', 'I', 'D', '?', 'S'};
        BestHit b;
        b.index = j;
        b.strand = static_cast<Strand>(strand[k]);
        b.runner_up = ru[k];
        b.result.status = static_cast<Status>(status[k]);
        if (!b.result.is_some()) return b;
        Alignment &a = b.result.value;
        a.score = score[k];
        a.ref_range = {rs[k], re[k]};
        a.query_range = {qs[k], qe[k]};
        for (uint64_t w = coff[k]; w < coff[k + 1]; ++w) a.states.push_back({cig[w] >> 4, ops[cig[w] & 7]});
        const bool streamed_is_query = streamed_are_ == SeqSrc::Query;
        a.ref_len = (uint32_t)(streamed_is_query ? targets_[j].size() : seq.size());
        a.query_len = (uint32_t)(streamed_is_query ? seq.size() : targets_[j].size());
        return b;
    }

    template <class T>
    static std::vector<std::pair<T, Strand>> with_strand(std::vector<T> v, const std::vector<uint8_t> &strand) {
        std::vector<std::pair<T, Strand>> out;
        out.reserve(v.size());
        for (size_t k = 0; k < v.size(); ++k) out.emplace_back(std::move(v[k]), static_cast<Strand>(strand[k]));
        return out;
    }

    // strand != nullptr: the both-strand entry point, the strand of every pair into *strand
    std::vector<MaybeAligned<uint32_t>> scores(const std::vector<std::string> &seqs, std::vector<uint8_t> *strand) {
        std::vector<uint8_t> buf;
        std::vector<uint64_t> off;
        pack(seqs, buf, off);
        size_t pairs = seqs.size() * targets_.size();
        std::vector<uint32_t> score(pairs + 1);
        std::vector<uint8_t> status(pairs + 1), tier(pairs + 1);
        if (strand) {
            strand->assign(pairs + 1, 0);
            check(zoe_cuda_sw_score_both_strands_batch(ctx_, buf.data(), off.data(), seqs.size(), score.data(), status.data(),
                                                       tier.data(), strand->data()));
        } else {
            check(zoe_cuda_sw_score_batch(ctx_, buf.data(), off.data(), seqs.size(), score.data(), status.data(), tier.data()));
        }
        std::vector<MaybeAligned<uint32_t>> out(pairs);
        for (size_t k = 0; k < pairs; ++k) out[k] = {static_cast<Status>(status[k]), score[k]};
        return out;
    }

    std::vector<MaybeAligned<ScoreAndRanges>> ranges(const std::vector<std::string> &seqs, std::vector<uint8_t> *strand) {
        std::vector<uint8_t> buf;
        std::vector<uint64_t> off;
        pack(seqs, buf, off);
        size_t pairs = seqs.size() * targets_.size();
        std::vector<uint32_t> score(pairs + 1), rs(pairs + 1), re(pairs + 1), qs(pairs + 1), qe(pairs + 1);
        std::vector<uint8_t> status(pairs + 1), tier(pairs + 1);
        if (strand) {
            strand->assign(pairs + 1, 0);
            check(zoe_cuda_sw_score_ranges_both_strands_batch(ctx_, buf.data(), off.data(), seqs.size(), score.data(),
                                                              status.data(), tier.data(), rs.data(), re.data(), qs.data(),
                                                              qe.data(), strand->data()));
        } else {
            check(zoe_cuda_sw_score_ranges_batch(ctx_, buf.data(), off.data(), seqs.size(), score.data(), status.data(),
                                                 tier.data(), rs.data(), re.data(), qs.data(), qe.data()));
        }
        std::vector<MaybeAligned<ScoreAndRanges>> out(pairs);
        for (size_t k = 0; k < pairs; ++k) {
            out[k].status = static_cast<Status>(status[k]);
            if (out[k].is_some()) out[k].value = ScoreAndRanges{score[k], {rs[k], re[k]}, {qs[k], qe[k]}};
        }
        return out;
    }

    std::vector<MaybeAligned<Alignment>> align(const std::vector<std::string> &seqs, bool three_pass,
                                               std::vector<uint8_t> *strand = nullptr) {
        std::vector<uint8_t> buf;
        std::vector<uint64_t> off;
        pack(seqs, buf, off);
        size_t pairs = seqs.size() * targets_.size();
        std::vector<uint32_t> score(pairs + 1), rs(pairs + 1), re(pairs + 1), qs(pairs + 1), qe(pairs + 1);
        std::vector<uint8_t> status(pairs + 1), tier(pairs + 1);
        std::vector<uint64_t> coff(pairs + 2);
        std::vector<uint32_t> cig(16 * pairs + 1024);
        if (strand) strand->assign(pairs + 1, 0);
        auto call = [&]() {
            if (strand)
                return three_pass
                           ? zoe_cuda_sw_align_3pass_both_strands_batch(ctx_, buf.data(), off.data(), seqs.size(), score.data(),
                                                                        status.data(), tier.data(), rs.data(), re.data(),
                                                                        qs.data(), qe.data(), cig.data(), coff.data(),
                                                                        cig.size(), strand->data())
                           : zoe_cuda_sw_align_both_strands_batch(ctx_, buf.data(), off.data(), seqs.size(), score.data(),
                                                                  status.data(), tier.data(), rs.data(), re.data(), qs.data(),
                                                                  qe.data(), cig.data(), coff.data(), cig.size(), nullptr,
                                                                  strand->data());
            return three_pass
                       ? zoe_cuda_sw_align_3pass_batch(ctx_, buf.data(), off.data(), seqs.size(), score.data(), status.data(),
                                                       tier.data(), rs.data(), re.data(), qs.data(), qe.data(), cig.data(),
                                                       coff.data(), cig.size())
                       : zoe_cuda_sw_align_batch(ctx_, buf.data(), off.data(), seqs.size(), score.data(), status.data(),
                                                 tier.data(), rs.data(), re.data(), qs.data(), qe.data(), cig.data(),
                                                 coff.data(), cig.size(), nullptr);
        };
        int rc = call();
        if (rc == ZOE_CUDA_E_CIGAR_CAP) {
            cig.resize(coff[0] + 16);
            rc = call();
        }
        check(rc);
        static const char ops[] = {'M', 'I', 'D', '?', 'S'};
        std::vector<MaybeAligned<Alignment>> out(pairs);
        for (size_t i = 0; i < seqs.size(); ++i)
            for (size_t j = 0; j < targets_.size(); ++j) {
                size_t k = i * targets_.size() + j;
                out[k].status = static_cast<Status>(status[k]);
                if (!out[k].is_some()) continue;
                Alignment &a = out[k].value;
                a.score = score[k];
                a.ref_range = {rs[k], re[k]};
                a.query_range = {qs[k], qe[k]};
                for (uint64_t w = coff[k]; w < coff[k + 1]; ++w) a.states.push_back({cig[w] >> 4, ops[cig[w] & 7]});
                bool streamed_is_query = streamed_are_ == SeqSrc::Query;  // (a sequence and its reverse complement: same length)
                a.ref_len = (uint32_t)(streamed_is_query ? targets_[j].size() : seqs[i].size());
                a.query_len = (uint32_t)(streamed_is_query ? seqs[i].size() : targets_[j].size());
            }
        return out;
    }

    CudaProfiles(const std::vector<std::string> &targets, const WeightMatrix &m, int8_t go, int8_t ge, int l8, int l16,
                 int l32, SeqSrc streamed_are, int n_devices)
        : targets_(targets), streamed_are_(streamed_are) {
        // validate_profile_args (profile.rs:32-44) -- before touching the device, like zoe
        if (targets.empty()) throw ProfileError(ProfileError::EmptySequence, "no profiled sequence");
        for (const std::string &t : targets)
            if (t.empty()) throw ProfileError(ProfileError::EmptySequence, "empty profiled sequence");
        if (go < -127 || go > 0) throw ProfileError(ProfileError::GapOpenOutOfRange, "gap_open out of -127..=0");
        if (ge < -127 || ge > 0) throw ProfileError(ProfileError::GapExtendOutOfRange, "gap_extend out of -127..=0");
        if (ge < go) throw ProfileError(ProfileError::BadGapWeights, "gap_extend < gap_open");
        int rc = zoe_cuda_create(&ctx_, nullptr, n_devices);
        if (rc) throw CudaError(rc, "zoe_cuda_create failed (no usable CUDA device; there is no CPU fallback)");
        check(zoe_cuda_set_scoring(ctx_, m.weights.data(), m.S, m.byte_to_index, go, ge, streamed_are == SeqSrc::Reference));
        check(zoe_cuda_set_lanes(ctx_, l8, l16, l32));
        std::vector<uint8_t> buf;
        std::vector<uint64_t> off;
        pack(targets, buf, off);
        check(zoe_cuda_set_profiled(ctx_, buf.data(), off.data(), (uint32_t)targets.size()));
    }
    static void pack(const std::vector<std::string> &seqs, std::vector<uint8_t> &buf, std::vector<uint64_t> &off) {
        off.assign(1, 0);
        for (const std::string &s : seqs) {
            buf.insert(buf.end(), s.begin(), s.end());
            off.push_back(buf.size());
        }
        if (buf.empty()) buf.push_back(0);
    }
    void check(int rc) {
        if (rc == 0) return;
        std::string msg = zoe_cuda_last_error(ctx_);
        switch (rc) {
            case ZOE_CUDA_E_EMPTY_SEQUENCE: throw ProfileError(ProfileError::EmptySequence, msg);
            case ZOE_CUDA_E_GAP_OPEN_RANGE: throw ProfileError(ProfileError::GapOpenOutOfRange, msg);
            case ZOE_CUDA_E_GAP_EXTEND_RANGE: throw ProfileError(ProfileError::GapExtendOutOfRange, msg);
            case ZOE_CUDA_E_BAD_GAP_WEIGHTS: throw ProfileError(ProfileError::BadGapWeights, msg);
            default: throw CudaError(rc, msg);
        }
    }
    zoe_cuda_ctx *ctx_ = nullptr;
    std::vector<std::string> targets_;
    SeqSrc streamed_are_;
};

// sneaky_snake(reference, query, threshold) -> Option<bool> (src/alignment/sneaky_snake.rs:78-131) for pair i =
// (references[i], queries[i]); std::nullopt = zoe's None.
inline std::vector<std::optional<bool>> sneaky_snake_batch(const std::vector<std::string> &references,
                                                           const std::vector<std::string> &queries, float threshold,
                                                           int n_devices = 1) {
    if (references.size() != queries.size()) throw std::invalid_argument("references and queries must pair up");
    zoe_cuda_ctx *ctx = nullptr;
    int rc = zoe_cuda_create(&ctx, nullptr, n_devices);
    if (rc) throw CudaError(rc, "zoe_cuda_create failed (no usable CUDA device; there is no CPU fallback)");
    auto pack = [](const std::vector<std::string> &v, std::vector<uint8_t> &buf, std::vector<uint64_t> &off) {
        off.assign(1, 0);
        for (const std::string &x : v) {
            buf.insert(buf.end(), x.begin(), x.end());
            off.push_back(buf.size());
        }
        if (buf.empty()) buf.push_back(0);
    };
    std::vector<uint8_t> rb, qb, out(references.size() + 1);
    std::vector<uint64_t> ro, qo;
    pack(references, rb, ro);
    pack(queries, qb, qo);
    rc = zoe_cuda_sneaky_snake_batch(ctx, rb.data(), ro.data(), qb.data(), qo.data(), references.size(), threshold, out.data());
    std::string msg = rc ? zoe_cuda_last_error(ctx) : "";
    zoe_cuda_destroy(ctx);
    if (rc) throw CudaError(rc, msg);
    std::vector<std::optional<bool>> res(references.size());
    for (size_t i = 0; i < res.size(); ++i)
        if (out[i] != ZOE_CUDA_SNAKE_NONE) res[i] = out[i] == ZOE_CUDA_SNAKE_TRUE;
    return res;
}

}  // namespace cuda
}  // namespace zoe
