//! `CudaProfiles`: the batched, B200-resident counterpart of zoe's `SharedProfiles`
//! (src/alignment/profile_set.rs:552-560).  Element-wise equal to
//! `SharedProfiles::sw_score_from_i8` / `sw_align_from_i8` (profile_set.rs:71-78, 136-145).
use std::ffi::CStr;

use zoe::{
    alignment::{Alignment, AlignmentStates, MaybeAligned, ProfileError, ScoreAndRanges, SeqSrc},
    data::{cigar::Ciglet, matrices::WeightMatrix},
};
use zoe_cuda_sys as sys;

pub struct CudaProfiles {
    ctx:               *mut sys::zoe_cuda_ctx,
    profiled_lens:     Vec<usize>,
    profiled_is_query: bool,
}

// One context per host thread (like LocalProfiles); it may be moved, not shared.
unsafe impl Send for CudaProfiles {}

/// Which strand of a streamed sequence a both-strand result belongs to.
#[derive(Debug, Clone, Copy, PartialEq, Eq)]
pub enum Strand {
    Forward = 0,
    Reverse = 1,
}

/// One sequence's result of the best-hit search: the chosen profiled sequence `index` and `strand`, that pair's
/// alignment (of the reverse complement for `Strand::Reverse`), and the best `Some` score against any other profiled
/// sequence (0 if none; SAM `XS`).
#[derive(Debug)]
pub struct BestHit {
    pub index:     usize,
    pub strand:    Strand,
    pub result:    MaybeAligned<Alignment<u32>>,
    pub runner_up: u32,
}

/// One read pair's result of the paired-end best-hit search (an FR library): the profiled sequence `index` both mates
/// were placed on, `proper` (the mates point inward within the insert bounds), `tlen` (mate 1's SAM TLEN; mate 2's is
/// `-tlen`) and each mate's `BestHit`, whose `strand` is the mate's strand in the chosen orientation.
#[derive(Debug)]
pub struct PairedHit {
    pub index:  usize,
    pub proper: bool,
    pub tlen:   i32,
    pub mate1:  BestHit,
    pub mate2:  BestHit,
}

#[derive(Debug)]
pub enum CudaError {
    Profile(ProfileError),
    Cuda { code: i32, message: String },
}

impl CudaProfiles {
    /// `targets` are the profiled sequences.  `profiled_is_query = false` means they are references and the
    /// sequences passed later are queries (`SeqSrc::Query`), the usual read-vs-reference shape.
    pub fn new_with_w256<const S: usize>(
        targets: &[&[u8]], matrix: &WeightMatrix<i8, S>, gap_open: i8, gap_extend: i8, profiled_is_query: bool,
        devices: &[i32],
    ) -> Result<Self, CudaError> {
        Self::new(targets, matrix, gap_open, gap_extend, (32, 16, 8), profiled_is_query, devices)
    }

    pub fn new_with_w128<const S: usize>(
        targets: &[&[u8]], matrix: &WeightMatrix<i8, S>, gap_open: i8, gap_extend: i8, profiled_is_query: bool,
        devices: &[i32],
    ) -> Result<Self, CudaError> {
        Self::new(targets, matrix, gap_open, gap_extend, (16, 8, 4), profiled_is_query, devices)
    }

    pub fn new_with_w512<const S: usize>(
        targets: &[&[u8]], matrix: &WeightMatrix<i8, S>, gap_open: i8, gap_extend: i8, profiled_is_query: bool,
        devices: &[i32],
    ) -> Result<Self, CudaError> {
        Self::new(targets, matrix, gap_open, gap_extend, (64, 32, 16), profiled_is_query, devices)
    }

    fn new<const S: usize>(
        targets: &[&[u8]], matrix: &WeightMatrix<i8, S>, gap_open: i8, gap_extend: i8, lanes: (i32, i32, i32),
        profiled_is_query: bool, devices: &[i32],
    ) -> Result<Self, CudaError> {
        let mut ctx = std::ptr::null_mut();
        let rc = unsafe { sys::zoe_cuda_create(&mut ctx, devices.as_ptr(), devices.len() as i32) };
        if rc != 0 {
            return Err(CudaError::Cuda { code: rc, message: "no usable CUDA device".into() });
        }
        let this = CudaProfiles { ctx, profiled_lens: targets.iter().map(|t| t.len()).collect(), profiled_is_query };
        let weights: Vec<i8> = matrix.weights.iter().flatten().copied().collect();
        let mut lut = [0u8; 256];
        for (b, slot) in lut.iter_mut().enumerate() {
            *slot = matrix.mapping.to_index(b as u8) as u8;
        }
        this.check(unsafe {
            sys::zoe_cuda_set_scoring(ctx, weights.as_ptr(), S as i32, lut.as_ptr(), gap_open, gap_extend, profiled_is_query as i32)
        }, gap_open, gap_extend)?;
        this.check(unsafe { sys::zoe_cuda_set_lanes(ctx, lanes.0, lanes.1, lanes.2) }, gap_open, gap_extend)?;
        let (concat, offsets) = pack(targets);
        this.check(unsafe { sys::zoe_cuda_set_profiled(ctx, concat.as_ptr(), offsets.as_ptr(), targets.len() as u32) }, gap_open, gap_extend)?;
        Ok(this)
    }

    /// `out[i * n_profiled + j] == profiles[j].sw_score_from_i8(seqs[i])`
    pub fn sw_score_batch(&self, seqs: &[&[u8]]) -> Result<Vec<MaybeAligned<u32>>, CudaError> {
        let (concat, offsets) = pack(seqs);
        let pairs = seqs.len() * self.profiled_lens.len();
        let (mut score, mut status, mut tier) = (vec![0u32; pairs], vec![0u8; pairs], vec![0u8; pairs]);
        self.check(unsafe {
            sys::zoe_cuda_sw_score_batch(self.ctx, concat.as_ptr(), offsets.as_ptr(), seqs.len() as u64,
                                         score.as_mut_ptr(), status.as_mut_ptr(), tier.as_mut_ptr())
        }, 0, 0)?;
        Ok(score.iter().zip(&status).map(|(&s, &st)| maybe(st, s)).collect())
    }

    /// `out[i * n_profiled + j] == profiles[j].sw_align_from_i8(seq_src(seqs[i]))` where `seq_src` is
    /// `SeqSrc::Query` when the profiled sequences are references, `SeqSrc::Reference` otherwise.
    pub fn sw_align_batch(&self, seqs: &[&[u8]]) -> Result<Vec<MaybeAligned<Alignment<u32>>>, CudaError> {
        self.align(seqs, false, None)
    }

    /// `out[i * n_profiled + j] == profiles[j].sw_align_from_i8_3pass(seq_src(seqs[i]))` (profile_set.rs:213-231):
    /// ranges from two score passes, then a banded alignment of the bounding box (three_pass.rs:21-104).
    pub fn sw_align_3pass_batch(&self, seqs: &[&[u8]]) -> Result<Vec<MaybeAligned<Alignment<u32>>>, CudaError> {
        self.align(seqs, true, None)
    }

    /// Both-strand search: for every pair, the better of `sw_score_batch` on `seqs[i]` and on its reverse complement
    /// (Overflowed > Some by score > Unmapped; ties to `Strand::Forward`), with the strand.
    pub fn sw_score_both_strands_batch(&self, seqs: &[&[u8]]) -> Result<Vec<(MaybeAligned<u32>, Strand)>, CudaError> {
        let (concat, offsets) = pack(seqs);
        let pairs = seqs.len() * self.profiled_lens.len();
        let (mut score, mut status, mut tier, mut sd) = (vec![0u32; pairs], vec![0u8; pairs], vec![0u8; pairs], vec![0u8; pairs]);
        self.check(unsafe {
            sys::zoe_cuda_sw_score_both_strands_batch(self.ctx, concat.as_ptr(), offsets.as_ptr(), seqs.len() as u64,
                                                      score.as_mut_ptr(), status.as_mut_ptr(), tier.as_mut_ptr(), sd.as_mut_ptr())
        }, 0, 0)?;
        Ok(score.iter().zip(&status).zip(&sd).map(|((&s, &st), &d)| (maybe(st, s), strand(d))).collect())
    }

    /// Both-strand `sw_score_ranges_batch`; a reverse-strand result's ranges refer to the reverse complement.
    pub fn sw_score_ranges_both_strands_batch(&self, seqs: &[&[u8]]) -> Result<Vec<(MaybeAligned<ScoreAndRanges<u32>>, Strand)>, CudaError> {
        let mut sd = vec![0u8; seqs.len() * self.profiled_lens.len()];
        let out = self.ranges(seqs, Some(&mut sd))?;
        Ok(out.into_iter().zip(sd).map(|(m, d)| (m, strand(d))).collect())
    }

    /// Both-strand `sw_align_batch`; a reverse-strand result's ranges and CIGAR refer to the reverse complement (SAM FLAG 16).
    pub fn sw_align_both_strands_batch(&self, seqs: &[&[u8]]) -> Result<Vec<(MaybeAligned<Alignment<u32>>, Strand)>, CudaError> {
        let mut sd = vec![0u8; seqs.len() * self.profiled_lens.len()];
        let out = self.align(seqs, false, Some(&mut sd))?;
        Ok(out.into_iter().zip(sd).map(|(m, d)| (m, strand(d))).collect())
    }

    /// Both-strand `sw_align_3pass_batch`.
    pub fn sw_align_3pass_both_strands_batch(&self, seqs: &[&[u8]]) -> Result<Vec<(MaybeAligned<Alignment<u32>>, Strand)>, CudaError> {
        let mut sd = vec![0u8; seqs.len() * self.profiled_lens.len()];
        let out = self.align(seqs, true, Some(&mut sd))?;
        Ok(out.into_iter().zip(sd).map(|(m, d)| (m, strand(d))).collect())
    }

    /// Best-hit search: one `BestHit` per sequence -- its best profiled sequence (and strand, with `both_strands`) by the
    /// both-strand rank, ties to the smallest index and then `Strand::Forward`; the alignment of that pair as
    /// `sw_align_batch` (`three_pass`: `sw_align_3pass_batch`) aligns it; the runner-up score (SAM XS).
    pub fn sw_align_best_hit_batch(&self, seqs: &[&[u8]], both_strands: bool, three_pass: bool) -> Result<Vec<BestHit>, CudaError> {
        let (concat, offsets) = pack(seqs);
        let n = seqs.len();
        let (mut hit, mut score, mut ru) = (vec![0u32; n + 1], vec![0u32; n + 1], vec![0u32; n + 1]);
        let (mut sd, mut status, mut tier) = (vec![0u8; n + 1], vec![0u8; n + 1], vec![0u8; n + 1]);
        let (mut rs, mut re, mut qs, mut qe) = (vec![0u32; n + 1], vec![0u32; n + 1], vec![0u32; n + 1], vec![0u32; n + 1]);
        let mut coff = vec![0u64; n + 2];
        let mut cigar = vec![0u32; 16 * n + 1024];
        loop {
            let rc = unsafe {
                sys::zoe_cuda_sw_align_best_hit_batch(self.ctx, concat.as_ptr(), offsets.as_ptr(), n as u64,
                    both_strands as std::os::raw::c_int, three_pass as std::os::raw::c_int, hit.as_mut_ptr(), sd.as_mut_ptr(),
                    score.as_mut_ptr(), status.as_mut_ptr(), tier.as_mut_ptr(), ru.as_mut_ptr(), rs.as_mut_ptr(),
                    re.as_mut_ptr(), qs.as_mut_ptr(), qe.as_mut_ptr(), cigar.as_mut_ptr(), coff.as_mut_ptr(),
                    cigar.len() as u64, std::ptr::null_mut())
            };
            if rc == sys::ZOE_CUDA_E_CIGAR_CAP {
                cigar.resize(coff[0] as usize + 16, 0);
                continue;
            }
            self.check(rc, 0, 0)?;
            break;
        }
        Ok(seqs.iter().enumerate().map(|(i, seq)| {
            let j = hit[i] as usize;
            let result = self.hit_alignment(seq, j, status[i], score[i], [rs[i], re[i], qs[i], qe[i]],
                                            &cigar[coff[i] as usize..coff[i + 1] as usize]);
            BestHit { index: j, strand: strand(sd[i]), result, runner_up: ru[i] }
        }).collect())
    }

    /// Paired-end best-hit search: one `PairedHit` per read pair `(mates1[i], mates2[i])`.  The pair's profiled
    /// sequence and orientation maximise (Overflowed mates, sum of the mates' Some scores), ties to the smallest index
    /// and then to mate 1 forward; each mate is aligned as `sw_align_batch` (`three_pass`: `sw_align_3pass_batch`)
    /// aligns it, or its reverse complement on `Strand::Reverse`.  `proper` and `tlen` use the insert bounds.
    pub fn sw_align_paired_best_hit_batch(&self, mates1: &[&[u8]], mates2: &[&[u8]], three_pass: bool, min_insert: u32,
                                          max_insert: u32) -> Result<Vec<PairedHit>, CudaError> {
        assert_eq!(mates1.len(), mates2.len(), "mate lists differ in length");
        let ((c1, o1), (c2, o2)) = (pack(mates1), pack(mates2));
        let n = mates1.len();
        let m = 2 * n + 1;
        let (mut hit, mut proper, mut tlen) = (vec![0u32; n + 1], vec![0u8; n + 1], vec![0i32; n + 1]);
        let (mut score, mut ru) = (vec![0u32; m], vec![0u32; m]);
        let (mut sd, mut status, mut tier) = (vec![0u8; m], vec![0u8; m], vec![0u8; m]);
        let (mut rs, mut re, mut qs, mut qe) = (vec![0u32; m], vec![0u32; m], vec![0u32; m], vec![0u32; m]);
        let mut coff = vec![0u64; m + 1];
        let mut cigar = vec![0u32; 16 * m + 1024];
        loop {
            let rc = unsafe {
                sys::zoe_cuda_sw_align_paired_best_hit_batch(self.ctx, c1.as_ptr(), o1.as_ptr(), c2.as_ptr(), o2.as_ptr(),
                    n as u64, three_pass as std::os::raw::c_int, min_insert, max_insert, hit.as_mut_ptr(),
                    proper.as_mut_ptr(), tlen.as_mut_ptr(), sd.as_mut_ptr(), score.as_mut_ptr(), status.as_mut_ptr(),
                    tier.as_mut_ptr(), ru.as_mut_ptr(), rs.as_mut_ptr(), re.as_mut_ptr(), qs.as_mut_ptr(), qe.as_mut_ptr(),
                    cigar.as_mut_ptr(), coff.as_mut_ptr(), cigar.len() as u64, std::ptr::null_mut())
            };
            if rc == sys::ZOE_CUDA_E_CIGAR_CAP {
                cigar.resize(coff[0] as usize + 16, 0);
                continue;
            }
            self.check(rc, 0, 0)?;
            break;
        }
        let mate = |k: usize, seq: &[u8], j: usize| BestHit {
            index: j,
            strand: strand(sd[k]),
            result: self.hit_alignment(seq, j, status[k], score[k], [rs[k], re[k], qs[k], qe[k]],
                                       &cigar[coff[k] as usize..coff[k + 1] as usize]),
            runner_up: ru[k],
        };
        Ok((0..n).map(|i| {
            let j = hit[i] as usize;
            PairedHit { index: j, proper: proper[i] != 0, tlen: tlen[i], mate1: mate(2 * i, mates1[i], j),
                        mate2: mate(2 * i + 1, mates2[i], j) }
        }).collect())
    }

    /// One best-hit or paired result's alignment against profiled sequence `j`; `ranges` = ref_start, ref_end,
    /// query_start, query_end.
    fn hit_alignment(&self, seq: &[u8], j: usize, status: u8, score: u32, ranges: [u32; 4], words: &[u32])
                     -> MaybeAligned<Alignment<u32>> {
        const OPS: [u8; 5] = [b'M', b'I', b'D', b'?', b'S'];
        match status {
            sys::ZOE_CUDA_SOME => {
                let ciglets = words.iter().map(|w| Ciglet { inc: (w >> 4) as usize, op: OPS[(w & 7) as usize] });
                let (ref_len, query_len) =
                    if self.profiled_is_query { (seq.len(), self.profiled_lens[j]) } else { (self.profiled_lens[j], seq.len()) };
                MaybeAligned::Some(Alignment {
                    score,
                    ref_range: ranges[0] as usize..ranges[1] as usize,
                    query_range: ranges[2] as usize..ranges[3] as usize,
                    states: AlignmentStates::from_ciglets_unchecked(ciglets),
                    ref_len,
                    query_len,
                })
            }
            sys::ZOE_CUDA_OVERFLOWED => MaybeAligned::Overflowed,
            _ => MaybeAligned::Unmapped,
        }
    }

    /// `strand`: the both-strand entry points, the strand of every pair written there.
    fn align(&self, seqs: &[&[u8]], three_pass: bool, mut strand: Option<&mut Vec<u8>>) -> Result<Vec<MaybeAligned<Alignment<u32>>>, CudaError> {
        let (concat, offsets) = pack(seqs);
        let np = self.profiled_lens.len();
        let pairs = seqs.len() * np;
        let mut score = vec![0u32; pairs];
        let (mut status, mut tier) = (vec![0u8; pairs], vec![0u8; pairs]);
        let (mut rs, mut re, mut qs, mut qe) = (vec![0u32; pairs], vec![0u32; pairs], vec![0u32; pairs], vec![0u32; pairs]);
        let mut coff = vec![0u64; pairs + 1];
        let mut cigar = vec![0u32; 16 * pairs + 1024];
        loop {
            let rc = unsafe {
                if let Some(sd) = strand.as_deref_mut() {
                    if three_pass {
                        sys::zoe_cuda_sw_align_3pass_both_strands_batch(self.ctx, concat.as_ptr(), offsets.as_ptr(), seqs.len() as u64,
                            score.as_mut_ptr(), status.as_mut_ptr(), tier.as_mut_ptr(), rs.as_mut_ptr(), re.as_mut_ptr(),
                            qs.as_mut_ptr(), qe.as_mut_ptr(), cigar.as_mut_ptr(), coff.as_mut_ptr(), cigar.len() as u64,
                            sd.as_mut_ptr())
                    } else {
                        sys::zoe_cuda_sw_align_both_strands_batch(self.ctx, concat.as_ptr(), offsets.as_ptr(), seqs.len() as u64,
                            score.as_mut_ptr(), status.as_mut_ptr(), tier.as_mut_ptr(), rs.as_mut_ptr(), re.as_mut_ptr(),
                            qs.as_mut_ptr(), qe.as_mut_ptr(), cigar.as_mut_ptr(), coff.as_mut_ptr(), cigar.len() as u64,
                            std::ptr::null_mut(), sd.as_mut_ptr())
                    }
                } else if three_pass {
                    sys::zoe_cuda_sw_align_3pass_batch(self.ctx, concat.as_ptr(), offsets.as_ptr(), seqs.len() as u64,
                        score.as_mut_ptr(), status.as_mut_ptr(), tier.as_mut_ptr(), rs.as_mut_ptr(), re.as_mut_ptr(),
                        qs.as_mut_ptr(), qe.as_mut_ptr(), cigar.as_mut_ptr(), coff.as_mut_ptr(), cigar.len() as u64)
                } else {
                    sys::zoe_cuda_sw_align_batch(self.ctx, concat.as_ptr(), offsets.as_ptr(), seqs.len() as u64,
                        score.as_mut_ptr(), status.as_mut_ptr(), tier.as_mut_ptr(), rs.as_mut_ptr(), re.as_mut_ptr(),
                        qs.as_mut_ptr(), qe.as_mut_ptr(), cigar.as_mut_ptr(), coff.as_mut_ptr(), cigar.len() as u64,
                        std::ptr::null_mut())
                }
            };
            if rc == sys::ZOE_CUDA_E_CIGAR_CAP {
                cigar.resize(coff[0] as usize + 16, 0);
                continue;
            }
            self.check(rc, 0, 0)?;
            break;
        }
        const OPS: [u8; 5] = [b'M', b'I', b'D', b'?', b'S'];
        let mut out = Vec::with_capacity(pairs);
        for (i, seq) in seqs.iter().enumerate() {
            for j in 0..np {
                let k = i * np + j;
                if status[k] != sys::ZOE_CUDA_SOME {
                    out.push(if status[k] == sys::ZOE_CUDA_OVERFLOWED { MaybeAligned::Overflowed } else { MaybeAligned::Unmapped });
                    continue;
                }
                let ciglets = cigar[coff[k] as usize..coff[k + 1] as usize]
                    .iter()
                    .map(|w| Ciglet { inc: (w >> 4) as usize, op: OPS[(w & 7) as usize] });
                let (ref_len, query_len) =
                    if self.profiled_is_query { (seq.len(), self.profiled_lens[j]) } else { (self.profiled_lens[j], seq.len()) };
                out.push(MaybeAligned::Some(Alignment {
                    score: score[k],
                    ref_range: rs[k] as usize..re[k] as usize,
                    query_range: qs[k] as usize..qe[k] as usize,
                    states: AlignmentStates::from_ciglets_unchecked(ciglets),
                    ref_len,
                    query_len,
                }));
            }
        }
        Ok(out)
    }

    /// `out[i * n_profiled + j] == profiles[j].sw_score_ranges_from_i8(seq_src(seqs[i]))`
    /// (profile_set.rs:313-322): score plus 0-based half-open ranges, no traceback matrix.
    pub fn sw_score_ranges_batch(&self, seqs: &[&[u8]]) -> Result<Vec<MaybeAligned<ScoreAndRanges<u32>>>, CudaError> {
        self.ranges(seqs, None)
    }

    /// `strand`: the both-strand entry point, the strand of every pair written there.
    fn ranges(&self, seqs: &[&[u8]], strand: Option<&mut Vec<u8>>) -> Result<Vec<MaybeAligned<ScoreAndRanges<u32>>>, CudaError> {
        let (concat, offsets) = pack(seqs);
        let pairs = seqs.len() * self.profiled_lens.len();
        let mut score = vec![0u32; pairs];
        let (mut status, mut tier) = (vec![0u8; pairs], vec![0u8; pairs]);
        let (mut rs, mut re, mut qs, mut qe) = (vec![0u32; pairs], vec![0u32; pairs], vec![0u32; pairs], vec![0u32; pairs]);
        self.check(unsafe {
            match strand {
                Some(sd) => sys::zoe_cuda_sw_score_ranges_both_strands_batch(self.ctx, concat.as_ptr(), offsets.as_ptr(),
                    seqs.len() as u64, score.as_mut_ptr(), status.as_mut_ptr(), tier.as_mut_ptr(), rs.as_mut_ptr(),
                    re.as_mut_ptr(), qs.as_mut_ptr(), qe.as_mut_ptr(), sd.as_mut_ptr()),
                None => sys::zoe_cuda_sw_score_ranges_batch(self.ctx, concat.as_ptr(), offsets.as_ptr(), seqs.len() as u64,
                    score.as_mut_ptr(), status.as_mut_ptr(), tier.as_mut_ptr(), rs.as_mut_ptr(), re.as_mut_ptr(),
                    qs.as_mut_ptr(), qe.as_mut_ptr()),
            }
        }, 0, 0)?;
        Ok((0..pairs).map(|k| match status[k] {
            sys::ZOE_CUDA_SOME => MaybeAligned::Some(ScoreAndRanges {
                score: score[k],
                ref_range: rs[k] as usize..re[k] as usize,
                query_range: qs[k] as usize..qe[k] as usize,
            }),
            sys::ZOE_CUDA_OVERFLOWED => MaybeAligned::Overflowed,
            _ => MaybeAligned::Unmapped,
        }).collect())
    }

    /// Which integer types may answer: `(8, 32, false)` = `sw_*_from_i8` (default), `(16, 32, false)` =
    /// `..._from_i16`, `(32, 32, false)` = `..._from_i32` (profile_set.rs:71-179); `first == last` = a standalone
    /// `StripedProfile<T, N, S>`; `unsigned` = the u8/u16/u32 profiles over `to_biased_matrix()`.
    pub fn set_width_policy(&self, first_bits: i32, last_bits: i32, unsigned: bool) -> Result<(), CudaError> {
        self.check(unsafe { sys::zoe_cuda_set_width_policy(self.ctx, first_bits, last_bits, unsigned as i32) }, 0, 0)
    }

    /// Tuning of the align pipeline (never changes results): 0 auto, 1 full-matrix flags, 2 checkpointed window.
    pub fn set_align_options(&self, mode: i32, checkpoint_log2: i32, slack: i32) -> Result<(), CudaError> {
        self.check(unsafe { sys::zoe_cuda_set_align_options(self.ctx, mode, checkpoint_log2, slack) }, 0, 0)
    }

    /// Upper bound on the device scratch of one align / ranges / 3-pass call (0 = automatic): larger batches are
    /// processed in chunks of streamed sequences.  Never changes results.
    pub fn set_memory_budget(&self, scratch_bytes: u64) -> Result<(), CudaError> {
        self.check(unsafe { sys::zoe_cuda_set_memory_budget(self.ctx, scratch_bytes) }, 0, 0)
    }

    /// The SeqSrc this context's batches correspond to (alignment/mod.rs:157-162).
    pub fn seq_src<'a>(&self, seq: &'a [u8]) -> SeqSrc<&'a [u8]> {
        if self.profiled_is_query { SeqSrc::Reference(seq) } else { SeqSrc::Query(seq) }
    }

    fn check(&self, rc: i32, gap_open: i8, gap_extend: i8) -> Result<(), CudaError> {
        match rc {
            0 => Ok(()),
            sys::ZOE_CUDA_E_EMPTY_SEQUENCE => Err(CudaError::Profile(ProfileError::EmptySequence)),
            sys::ZOE_CUDA_E_GAP_OPEN_RANGE => Err(CudaError::Profile(ProfileError::GapOpenOutOfRange { gap_open })),
            sys::ZOE_CUDA_E_GAP_EXTEND_RANGE => Err(CudaError::Profile(ProfileError::GapExtendOutOfRange { gap_extend })),
            sys::ZOE_CUDA_E_BAD_GAP_WEIGHTS => Err(CudaError::Profile(ProfileError::BadGapWeights { gap_open, gap_extend })),
            code => {
                let message = unsafe { CStr::from_ptr(sys::zoe_cuda_last_error(self.ctx)) }.to_string_lossy().into_owned();
                Err(CudaError::Cuda { code, message })
            }
        }
    }
}

impl Drop for CudaProfiles {
    fn drop(&mut self) {
        unsafe { sys::zoe_cuda_destroy(self.ctx) }
    }
}

/// `out[i] == zoe::alignment::sneaky_snake(references[i], queries[i], threshold)`
/// (src/alignment/sneaky_snake.rs:78-131) on the given devices.
pub fn sneaky_snake_batch(references: &[&[u8]], queries: &[&[u8]], threshold: f32, devices: &[i32]) -> Result<Vec<Option<bool>>, CudaError> {
    assert_eq!(references.len(), queries.len(), "references and queries must pair up");
    let mut ctx = std::ptr::null_mut();
    let rc = unsafe { sys::zoe_cuda_create(&mut ctx, devices.as_ptr(), devices.len() as i32) };
    if rc != 0 {
        return Err(CudaError::Cuda { code: rc, message: "no usable CUDA device".into() });
    }
    let (rb, ro) = pack(references);
    let (qb, qo) = pack(queries);
    let mut out = vec![0u8; references.len().max(1)];
    let rc = unsafe {
        sys::zoe_cuda_sneaky_snake_batch(ctx, rb.as_ptr(), ro.as_ptr(), qb.as_ptr(), qo.as_ptr(), references.len() as u64,
                                         threshold, out.as_mut_ptr())
    };
    let message = if rc != 0 { unsafe { CStr::from_ptr(sys::zoe_cuda_last_error(ctx)) }.to_string_lossy().into_owned() } else { String::new() };
    unsafe { sys::zoe_cuda_destroy(ctx) };
    if rc != 0 {
        return Err(CudaError::Cuda { code: rc, message });
    }
    Ok(out[..references.len()].iter().map(|&v| match v { 0 => Some(false), 1 => Some(true), _ => None }).collect())
}

fn maybe(status: u8, score: u32) -> MaybeAligned<u32> {
    match status {
        sys::ZOE_CUDA_SOME => MaybeAligned::Some(score),
        sys::ZOE_CUDA_OVERFLOWED => MaybeAligned::Overflowed,
        _ => MaybeAligned::Unmapped,
    }
}

fn strand(v: u8) -> Strand {
    if v == 1 { Strand::Reverse } else { Strand::Forward }
}

fn pack(seqs: &[&[u8]]) -> (Vec<u8>, Vec<u64>) {
    let mut concat = Vec::with_capacity(seqs.iter().map(|s| s.len()).sum::<usize>().max(1));
    let mut offsets = Vec::with_capacity(seqs.len() + 1);
    offsets.push(0u64);
    for s in seqs {
        concat.extend_from_slice(s);
        offsets.push(concat.len() as u64);
    }
    if concat.is_empty() {
        concat.push(0);
    }
    (concat, offsets)
}
