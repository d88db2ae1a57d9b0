/*
 * zoe_cuda.h -- C ABI of the B200 (sm_100a) backend for zoe's striped Smith-Waterman path.
 *
 * zoe (CDCgov/zoe, pure Rust) has no FFI seam of its own; the drop-in boundary is its Rust
 * API for this path.  Each entry point below names the zoe interface it stands behind
 * (paths relative to the zoe repository root).  A Rust `-sys` crate binds exactly these symbols
 * (see INTEGRATION.md); the C++ mirror (include/zoe_cuda.hpp) and the Python mirror
 * (zoe_b200/) bind the same ones.
 *
 * Vocabulary (SURVEY.md 8(a)): the *profiled* sequences P are the ones a zoe caller builds a
 * `StripedProfile` / `SharedProfiles` from (DP columns c); the *streamed* sequences R are the ones
 * passed to `sw_score(seq)` / `sw_align(SeqSrc)` (DP rows r).  A batch call computes every
 * (streamed i, profiled j) pair; result index = i * n_profiled + j, independent of GPU count.
 *
 * Error model: every call returns 0 on success or a negative ZOE_CUDA_E_* code; the message is
 * available from zoe_cuda_last_error().  No C++ exception crosses this boundary.  A context is
 * NOT thread-safe (one per host thread, like zoe's `LocalProfiles`).  There is no CPU fallback:
 * if no CUDA device is usable, zoe_cuda_create() fails.
 */
#ifndef ZOE_CUDA_H
#define ZOE_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct zoe_cuda_ctx zoe_cuda_ctx;

/* MaybeAligned<T> discriminant: src/alignment/types/output.rs:18-25 */
#define ZOE_CUDA_SOME 0
#define ZOE_CUDA_OVERFLOWED 1
#define ZOE_CUDA_UNMAPPED 2

/* Error codes.  -1..-4 mirror ProfileError (src/alignment/errors.rs:6-15) as raised by
 * validate_profile_args (src/alignment/profile.rs:32-44). */
#define ZOE_CUDA_OK 0
#define ZOE_CUDA_E_EMPTY_SEQUENCE (-1)
#define ZOE_CUDA_E_GAP_OPEN_RANGE (-2)
#define ZOE_CUDA_E_GAP_EXTEND_RANGE (-3)
#define ZOE_CUDA_E_BAD_GAP_WEIGHTS (-4)
#define ZOE_CUDA_E_BAD_ARG (-5)
#define ZOE_CUDA_E_CIGAR_CAP (-6)
#define ZOE_CUDA_E_CUDA (-7)
#define ZOE_CUDA_E_STATE (-8)
#define ZOE_CUDA_E_UNSUPPORTED (-9)

/* CIGAR encoding: BAM style (len << 4) | op with M=0, I=1, D=2, S=4 -- the only operations
 * zoe's SW emits (src/alignment/sw/mod.rs:149-154). */
#define ZOE_CUDA_CIGAR_M 0u
#define ZOE_CUDA_CIGAR_I 1u
#define ZOE_CUDA_CIGAR_D 2u
#define ZOE_CUDA_CIGAR_S 4u

/* Create a context on `n_devices` CUDA devices (device_ids == NULL: devices 0..n-1).  Batches
 * are split over the devices by contiguous streamed-index range; there is no collective.
 * Replaces: nothing in zoe (zoe is single-threaded; callers own parallelism,
 * src/alignment/profile_set.rs:552-560). */
int zoe_cuda_create(zoe_cuda_ctx **ctx, const int *device_ids, int n_devices);
void zoe_cuda_destroy(zoe_cuda_ctx *ctx);
const char *zoe_cuda_last_error(const zoe_cuda_ctx *ctx);

/* Scoring = zoe's (WeightMatrix<i8,S>, gap_open, gap_extend) triple.
 *   weights       S*S row-major, exactly zoe's weights[ref_idx][query_idx]
 *                 (src/data/matrices/mod.rs:230-235)
 *   byte_to_index zoe's ByteIndexMap table (src/data/constants/mappings/byte_index.rs:331-333)
 *   gap_open/gap_extend  as zoe takes them: -127..=0, gap_extend >= gap_open
 *                 (src/alignment/profile.rs:32-44); violations return the ProfileError codes.
 *   profiled_is_query  1: the profiled sequences are queries and streamed sequences are
 *                 references (zoe's SeqSrc::Reference(streamed), no inversion);
 *                 0: the profiled sequences are references, streamed are queries
 *                 (SeqSrc::Query(streamed): the Alignment is invert()ed,
 *                 src/alignment/mod.rs:176-190, src/alignment/types/output.rs:396-425). */
int zoe_cuda_set_scoring(zoe_cuda_ctx *ctx, const int8_t *weights, int S, const uint8_t byte_to_index[256],
                         int8_t gap_open, int8_t gap_extend, int profiled_is_query);

/* Lane counts (M, N, O) of zoe's ProfileSets: they fix the CIGAR tie-break layout of each
 * score-width tier (src/alignment/profile_set.rs:434-483: w128 = 16/8/4, w256 = 32/16/8,
 * w512 = 64/32/16).  Default w256, as Nucleotides::into_local_profile uses
 * (src/data/types/nucleotides/mod.rs:262-300). */
int zoe_cuda_set_lanes(zoe_cuda_ctx *ctx, int lanes_i8, int lanes_i16, int lanes_i32);

/* The profiled sequences (raw bytes, concatenated; offsets has n+1 entries).  Replaces
 * SharedProfiles::new / StripedProfile::new (src/alignment/profile_set.rs:382-390,
 * src/alignment/profile.rs:239-306): validates like zoe, uploads once, replicated per device.
 * Requires set_scoring first. */
int zoe_cuda_set_profiled(zoe_cuda_ctx *ctx, const uint8_t *concat, const uint64_t *offsets, uint32_t n);

/* Batched ProfileSets::sw_score_from_i8 (src/alignment/profile_set.rs:71-78 ->
 * sw_simd_score, src/alignment/sw/striped.rs:65-142, with the i8->i16->i32 escalation of
 * output.rs:81-83).  Host buffers in, host buffers out; outputs have n * n_profiled entries.
 *   score   the local alignment score (0 when not Some)
 *   status  ZOE_CUDA_SOME / OVERFLOWED / UNMAPPED
 *   tier    8, 16 or 32: the narrowest signed width whose run would not have overflowed
 *           (src/alignment/sw/striped.rs:608-633). */
int zoe_cuda_sw_score_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets, uint64_t n,
                            uint32_t *score, uint8_t *status, uint8_t *tier);

/* Batched ProfileSets::sw_align_from_i8 (src/alignment/profile_set.rs:136-145 -> sw_simd_align,
 * src/alignment/sw/striped.rs:449-598, traceback src/alignment/types/backtrack.rs:290-342).
 * Ranges are 0-based half-open and follow zoe's Alignment after make_alignment (i.e. already
 * inverted when profiled_is_query == 0): ref_* index the reference-side sequence, query_* the
 * query-side one.  cigar_off has n_pairs + 1 entries into `cigar` (capacity cigar_cap words);
 * if the CIGARs do not fit the call returns ZOE_CUDA_E_CIGAR_CAP and writes the needed
 * capacity to cigar_off[0] (nothing else is valid).
 *   hazard  (may be NULL) 1 where the pair went through the literal striped-emulation kernel
 *           because its traceback met an E/F tie whose resolution depends on the lane layout.
 * Streamed sequences of any length, as zoe's function: those beyond 1024 residues (one pass of the register-resident
 * kernels) are scored by the chunked-row kernels and aligned by the literal striped kernels, pair by pair -- correct
 * but slow, like the O(mn) memory zoe warns about (striped.rs:410-413); the 3-pass entry point below is the one meant
 * for long reads.  A batch that mixes both kinds is split internally and returned in the caller's order. */
int zoe_cuda_sw_align_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets, uint64_t n,
                            uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *ref_start, uint32_t *ref_end,
                            uint32_t *query_start, uint32_t *query_end, uint32_t *cigar, uint64_t *cigar_off,
                            uint64_t cigar_cap, uint8_t *hazard);

/* Batched ProfileSets::sw_score_ranges_from_i8 (src/alignment/profile_set.rs:313-322 -> sw_simd_score_ranges,
 * src/alignment/sw/striped.rs:355-388): score plus the 0-based half-open alignment ranges, without a traceback
 * matrix (a forward pass finds the end cell, a reverse pass over the truncated, reversed sequences finds the start:
 * sw_simd_score_ends / sw_simd_score_ends_reverse, striped.rs:153-336).  ref_end / query_end are what
 * StripedProfile::sw_score_ends reports (profile.rs:456-460).  Ranges follow zoe's output after make_alignment, i.e.
 * swapped when profiled_is_query == 0 (src/alignment/mod.rs:176-190); they are 0 when status != ZOE_CUDA_SOME.
 * Streamed sequences of any length: batches with a sequence beyond 1024 residues take the chunked-row kernels
 * (sw_ends_long_kernel, forward and reverse). */
int zoe_cuda_sw_score_ranges_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets, uint64_t n,
                                   uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *ref_start, uint32_t *ref_end,
                                   uint32_t *query_start, uint32_t *query_end);

/* Batched ProfileSets::sw_align_from_i8_3pass (src/alignment/profile_set.rs:213-231 -> sw_align_3pass,
 * src/alignment/sw/three_pass.rs:21-104): the memory-light alignment.  Passes 1 and 2 are the ranges pipeline above
 * (score, end cell, start cell; no traceback matrix); pass 3 aligns only the bounding box: the no-gaps shortcut when the
 * diagonal's weights add up to the score, else sw_banded_align (src/alignment/sw/banded.rs:40-133) with band width
 * |ref_len - query_len| + 1 doubled until the banded score matches, else sw_scalar_align on the box
 * (src/alignment/sw/scalar.rs:173-271).  Outputs as zoe_cuda_sw_align_batch (the score is the pass-1 score; the CIGAR
 * carries zoe's soft clips; SeqSrc::Query results are invert()ed).  The CIGAR can differ from sw_align's in equal-score
 * ties, exactly as zoe's two functions differ.  Streamed sequences of any length (band-sized scratch: a 5 kb x 5 kb
 * box costs rows x (2 bw + 1) flag bytes, not rows x columns); alphabets up to 32 symbols. */
int zoe_cuda_sw_align_3pass_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets, uint64_t n,
                                  uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *ref_start, uint32_t *ref_end,
                                  uint32_t *query_start, uint32_t *query_end, uint32_t *cigar, uint64_t *cigar_off,
                                  uint64_t cigar_cap);

/* Both-strand search.  Each entry point takes exactly the arguments of its single-strand twin above plus a trailing
 * `strand` (n * n_profiled entries, may be NULL): 0 = the streamed sequence as given, 1 = its reverse complement.
 * For pair (i, j) let F be what the single-strand call returns for (seq_i, j) and R what it returns for
 * (revcomp(seq_i), j), with the same scoring, lanes, width policy, orientation and align options.  The result is R with
 * strand 1 when R ranks strictly above F, else F with strand 0; the rank is Overflowed > Some(score), ordered by score,
 * > Unmapped, so every tie (equal scores, both Overflowed, both Unmapped, a palindromic read) goes to the forward strand.
 * Every output of the winning strand is returned exactly as the single-strand call returns it (score, status, tier,
 * ranges, CIGAR, hazard): coordinates and CIGAR of a reverse-strand result refer to revcomp(seq_i), as SAM reports a
 * FLAG 16 record, for profiled_is_query 0 and 1 alike.  A 0-length sequence is Unmapped on strand 0.
 *   revcomp  reverses the bytes and maps each through one table: A<->T, C<->G, U->A, R<->Y, K<->M, B<->V, D<->H; S, W, N
 *            map to themselves; lowercase letters map the same way and keep their case; every other byte is unchanged.
 *   cigar_cap  the capacity the selected strands' CIGARs need; ZOE_CUDA_E_CIGAR_CAP reports that need in cigar_off[0].
 * The strands are aligned as one doubled batch, so a call takes at most 2^30 - 1 sequences and, for align / ranges /
 * 3-pass, at most (2^31 - 1) / 2 pairs per device; larger batches fail with ZOE_CUDA_E_BAD_ARG.
 * zoe_cuda_last_stats counts the work done: pairs and cells count both strands, and the tier / overflowed / unmapped
 * counters cover all 2 * n * n_profiled strand-pairs. */
int zoe_cuda_sw_score_both_strands_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets,
                                         uint64_t n, uint32_t *score, uint8_t *status, uint8_t *tier, uint8_t *strand);
int zoe_cuda_sw_score_ranges_both_strands_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets,
                                                uint64_t n, uint32_t *score, uint8_t *status, uint8_t *tier,
                                                uint32_t *ref_start, uint32_t *ref_end, uint32_t *query_start,
                                                uint32_t *query_end, uint8_t *strand);
int zoe_cuda_sw_align_both_strands_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets,
                                         uint64_t n, uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *ref_start,
                                         uint32_t *ref_end, uint32_t *query_start, uint32_t *query_end, uint32_t *cigar,
                                         uint64_t *cigar_off, uint64_t cigar_cap, uint8_t *hazard, uint8_t *strand);
int zoe_cuda_sw_align_3pass_both_strands_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets,
                                               uint64_t n, uint32_t *score, uint8_t *status, uint8_t *tier,
                                               uint32_t *ref_start, uint32_t *ref_end, uint32_t *query_start,
                                               uint32_t *query_end, uint32_t *cigar, uint64_t *cigar_off, uint64_t cigar_cap,
                                               uint8_t *strand);

/* Best-hit search: each streamed sequence's best profiled sequence and strand, chosen on the device; the align entry
 * point aligns only that pair.  For streamed sequence i:
 *   candidates  (j, s) for every profiled j, with s = 0 (seq_i as given) and, when both_strands is set, also s = 1
 *               (revcomp(seq_i), the complement table of the both-strand search).  Each candidate's result is what the
 *               single-strand score call returns for that pair.
 *   selection   the both-strand rank -- Overflowed > Some(score), ordered by score, > Unmapped -- and the highest rank
 *               wins; ties go to the smallest j, then to the forward strand.  A sequence whose candidates are all Unmapped
 *               (a 0-length one too) gets hit 0, strand 0, Unmapped.
 *   hit, strand, score, status, tier   the winner and its score-call result.
 *   runner_up   the largest Some score among candidates with j != hit (either strand); 0 when there is none and when
 *               the winner is not Some.  It is the SAM XS value.
 * The align entry point returns, for the selected pair (seq_i, or revcomp(seq_i) when strand is 1, against hit),
 * exactly what zoe_cuda_sw_align_batch returns (three_pass: zoe_cuda_sw_align_3pass_batch, hazard 0): score, status,
 * tier, ranges, CIGAR, hazard.  Coordinates and CIGAR of a reverse winner refer to revcomp(seq_i).  Winners that are not
 * Some are not aligned: zero ranges, empty CIGAR.
 * Every output has n entries (cigar_off n + 1) and may be NULL, except cigar_off, and cigar when cigar_cap > 0.
 * ZOE_CUDA_E_CIGAR_CAP writes the selected pairs' total need to cigar_off[0].  Limits are those of the score call the
 * search runs (with both_strands, those of zoe_cuda_sw_score_both_strands_batch).  zoe_cuda_last_stats: pairs and cells
 * count the score pass over every candidate plus the aligned pairs; the tier / overflowed / unmapped counters count the
 * score pass; hazard, window and tp_* count the alignments.  A call leaves nothing staged and the profiled set as it was,
 * error or not (DESIGN.md 4.9). */
int zoe_cuda_sw_score_best_hit_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets,
                                     uint64_t n, int both_strands, uint32_t *hit, uint8_t *strand, uint32_t *score,
                                     uint8_t *status, uint8_t *tier, uint32_t *runner_up);
int zoe_cuda_sw_align_best_hit_batch(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets,
                                     uint64_t n, int both_strands, int three_pass, uint32_t *hit, uint8_t *strand,
                                     uint32_t *score, uint8_t *status, uint8_t *tier, uint32_t *runner_up,
                                     uint32_t *ref_start, uint32_t *ref_end, uint32_t *query_start, uint32_t *query_end,
                                     uint32_t *cigar, uint64_t *cigar_off, uint64_t cigar_cap, uint8_t *hazard);

/* Paired-end best-hit search: each read pair's profiled sequence and orientation, chosen on the device from both mates;
 * the align entry point aligns both mates there and reports proper pairs and TLEN.
 *   layout      n_pairs pairs: mate 1 of pair i is sequence i of the mate-1 batch, mate 2 sequence i of the mate-2
 *               batch.  hit, proper and tlen have n_pairs entries; every other output is per mate, 2 n_pairs entries
 *               at index 2i + m (m = 0 for mate 1, 1 for mate 2); cigar_off has 2 n_pairs + 1 entries and the CIGAR
 *               stream is in that order.
 *   candidates  the library is FR, as Illumina paired-end is: the mates come from opposite strands.  Pair i has the
 *               candidates (j, o) for every profiled j and o in {0, 1}; under (j, o) mate 1 is on strand o and mate 2 on
 *               strand 1 - o (strand 1: the reverse complement, with the complement table of the both-strand search).
 *               A mate's result under a candidate is what the single-strand score call returns for that sequence
 *               against j.
 *   selection   each candidate's key is first the number of Overflowed mates (0-2), then the sum of its two mates'
 *               Some scores; the highest key wins, ties go to the smallest j, then to o = 0.  A candidate whose mates
 *               are both Unmapped has key (0, 0); a pair whose candidates all have key (0, 0) -- 0-length mates
 *               included -- gets hit 0, o = 0 and two Unmapped mates.
 *   strand, score, status, tier   each mate's result under the winning candidate.
 *   runner_up   per mate: its largest Some score among candidates with j != hit, on either strand; 0 when the mate is
 *               not Some (the best-hit XS definition, per mate).
 * The align entry point gives each mate that is Some under the winner exactly what zoe_cuda_sw_align_batch returns for
 * (the mate, or its reverse complement on strand 1, against hit); three_pass: zoe_cuda_sw_align_3pass_batch, hazard 0.
 * A mate that is not Some gets zero ranges and an empty CIGAR.  Coordinates and CIGAR of a strand-1 mate refer to its
 * reverse complement, as in the both-strand search.  A mate's panel range is [ref_start, ref_end) when
 * profiled_is_query is 0 and [query_start, query_end) when it is 1.
 *   tlen        when both mates are Some, extent = max(ends) - min(starts); tlen is +extent when mate 1's start is
 *               smaller, or the starts are equal and o = 0, else -extent.  It is mate 1's TLEN (a 32-bit int); mate
 *               2's is -tlen.
 *               0 when the mates are not both Some.
 *   proper      1 iff both mates are Some, the forward-strand mate's start is at most the reverse-strand mate's start
 *               (the mates point inward) and min_insert <= extent <= max_insert.
 * min_insert > max_insert fails with ZOE_CUDA_E_BAD_ARG.  Every output may be NULL, except cigar_off, and cigar when
 * cigar_cap > 0; ZOE_CUDA_E_CIGAR_CAP writes the exact need to cigar_off[0].  Limits are those of
 * zoe_cuda_sw_score_both_strands_batch applied to the 2 n_pairs mates.  zoe_cuda_last_stats counts as the best-hit
 * search does: the score pass over every candidate (4 n_pairs x n_profiled strand-pairs) plus the aligned mates.  A
 * call leaves nothing staged and the profiled set as it was, error or not.  Not covered: RF / FF libraries, mate rescue
 * (re-aligning an unmapped mate near its mapped mate), MAPQ, and supplementary or secondary records (DESIGN.md 4.10). */
int zoe_cuda_sw_score_paired_best_hit_batch(zoe_cuda_ctx *ctx, const uint8_t *mate1_concat, const uint64_t *mate1_offsets,
                                            const uint8_t *mate2_concat, const uint64_t *mate2_offsets, uint64_t n_pairs,
                                            uint32_t *hit, uint8_t *strand, uint32_t *score, uint8_t *status, uint8_t *tier,
                                            uint32_t *runner_up);
int zoe_cuda_sw_align_paired_best_hit_batch(zoe_cuda_ctx *ctx, const uint8_t *mate1_concat, const uint64_t *mate1_offsets,
                                            const uint8_t *mate2_concat, const uint64_t *mate2_offsets, uint64_t n_pairs,
                                            int three_pass, uint32_t min_insert, uint32_t max_insert, uint32_t *hit,
                                            uint8_t *proper, int *tlen, uint8_t *strand, uint32_t *score, uint8_t *status,
                                            uint8_t *tier, uint32_t *runner_up, uint32_t *ref_start, uint32_t *ref_end,
                                            uint32_t *query_start, uint32_t *query_end, uint32_t *cigar, uint64_t *cigar_off,
                                            uint64_t cigar_cap, uint8_t *hazard);

/* Batched sneaky_snake(reference, query, threshold) (src/alignment/sneaky_snake.rs:78-131): the SneakySnake
 * pre-alignment filter for pair i = (reference i, query i).  out[i]: 1 = Some(true) (edits within
 * floor(len(query) * threshold)), 0 = Some(false), 2 = None (threshold outside 0..=1, or the length difference exceeds
 * the edit threshold).  Needs no scoring and no profiled set. */
#define ZOE_CUDA_SNAKE_FALSE 0
#define ZOE_CUDA_SNAKE_TRUE 1
#define ZOE_CUDA_SNAKE_NONE 2
int zoe_cuda_sneaky_snake_batch(zoe_cuda_ctx *ctx, const uint8_t *refs, const uint64_t *ref_offsets, const uint8_t *queries,
                                const uint64_t *query_offsets, uint64_t n, float threshold, uint8_t *out);

/* Which of zoe's integer types may report a result (default 8..32 signed = ProfileSets::sw_*_from_i8).
 *   first_bits..last_bits   8/16/32: the escalation chain starts at first_bits and stops at last_bits:
 *                 (8,32) = sw_score_from_i8 / sw_align_from_i8, (16,32) = ..._from_i16, (32,32) = ..._from_i32
 *                 (src/alignment/profile_set.rs:71-179); first == last = a standalone StripedProfile<T,N,S>
 *                 (src/alignment/profile.rs:440-446, 515-519).  A score beyond last_bits is ZOE_CUDA_OVERFLOWED.
 *   is_unsigned   1: the u8/u16/u32 profiles zoe builds from a biased matrix (WeightMatrix::to_biased_matrix,
 *                 src/data/matrices/mod.rs:471-491): a type holds scores <= MAX - bias - 1
 *                 (score_to_maybe_aligned, src/alignment/sw/striped.rs:608-633); the weights passed to
 *                 zoe_cuda_set_scoring stay the signed ones, the bias is derived from them.
 * `tier` outputs report the bit width of the type that produced the result. */
int zoe_cuda_set_width_policy(zoe_cuda_ctx *ctx, int first_bits, int last_bits, int is_unsigned);

/* Tuning of the align pipeline (results never depend on it; DESIGN.md 4.3).
 *   mode            0 = automatic, 1 = direction bits for the full matrix (what zoe's sw_simd_align stores,
 *                   src/alignment/sw/striped.rs:446-598), 2 = checkpointed window: a score-rate scan parks the
 *                   DP column every 2^checkpoint_log2 columns, the direction bits are recomputed only for the
 *                   window the traceback can reach
 *   checkpoint_log2 2..16 (default 6: 64 columns)
 *   slack           columns kept left of the shortest possible walk (default 16); a walk that needs more
 *                   is redone by the literal kernel and counted in zoe_cuda_stats.window_fallback */
int zoe_cuda_set_align_options(zoe_cuda_ctx *ctx, int mode, int checkpoint_log2, int slack);

/* Upper bound on the device scratch one align / ranges / 3-pass call may hold at a time (checkpoints, direction-bit
 * windows, box scratch); batches that need more are processed in chunks of streamed sequences.  0 = automatic (a
 * fraction of the memory that was free when the context was created, at most 48 GB).  Results never depend on it. */
int zoe_cuda_set_memory_budget(zoe_cuda_ctx *ctx, uint64_t scratch_bytes);

/* ---- measurement hooks (not part of the zoe-facing surface) ---- */

/* Device-resident variant of zoe_cuda_sw_score_batch for kernel-only timing: upload once with
 * zoe_cuda_stage_streamed(), then run the kernels any number of times.  Results stay on the
 * device until zoe_cuda_fetch_scores(). */
int zoe_cuda_stage_streamed(zoe_cuda_ctx *ctx, const uint8_t *streamed_concat, const uint64_t *offsets, uint64_t n);
int zoe_cuda_run_score_staged(zoe_cuda_ctx *ctx);
int zoe_cuda_run_align_staged(zoe_cuda_ctx *ctx);
int zoe_cuda_run_ranges_staged(zoe_cuda_ctx *ctx);
int zoe_cuda_run_3pass_staged(zoe_cuda_ctx *ctx);
int zoe_cuda_fetch_scores(zoe_cuda_ctx *ctx, uint32_t *score, uint8_t *status, uint8_t *tier);

/* Timing of the most recent batch/staged call, from CUDA events on the library's own streams
 * (max over devices): total device time and the share spent in the dominant DP kernel. */
int zoe_cuda_last_timing(const zoe_cuda_ctx *ctx, float *total_ms, float *dp_kernel_ms, uint32_t *kernel_launches);

/* Counters of the most recent batch call: pairs per tier (8/16/32), overflowed, unmapped,
 * pairs re-run at 32 bits, hazard pairs sent to the literal kernel. */
typedef struct {
    uint64_t pairs, cells;
    uint64_t tier8, tier16, tier32, overflowed, unmapped;
    uint64_t rerun_wide, hazard;
    uint64_t window_fallback; /* pairs whose walk left its checkpoint window (re-done by the literal kernel) */
    uint64_t window_pinned;   /* pairs whose maximum recurs in the winning lane: best cell found by a pin sweep */
    /* 3-pass alignment: how pass 3 produced the CIGAR (three_pass.rs:39-84) */
    uint64_t tp_nogaps, tp_banded, tp_scalar, tp_band_attempts;
} zoe_cuda_stats;
int zoe_cuda_last_stats(const zoe_cuda_ctx *ctx, zoe_cuda_stats *out);

/* Integer max-plus issue-rate microbenchmark (the roofline denominator, SURVEY.md 8(d)):
 * kind 0 = VIADDMNMX.S16x2 only, 1 = the score kernel's instruction mix without memory.
 * Returns giga warp-lane-instructions per second on device 0 of the context. */
int zoe_cuda_dpx_peak(zoe_cuda_ctx *ctx, int kind, double *giga_lane_instr_per_s, float *ms);

/* Raw stream handle (cudaStream_t) of device `dev_index`, for external event timing. */
void *zoe_cuda_stream(zoe_cuda_ctx *ctx, int dev_index);

#ifdef __cplusplus
}
#endif
#endif /* ZOE_CUDA_H */
