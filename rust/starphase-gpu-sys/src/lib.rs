//! `extern "C"` mirror of include/starphase_gpu.h plus the small safe wrapper the pb-StarPhase call sites use.
//! One `GpuScorer` per process per GPU; calls are blocking, like the `Aligner::map` calls they replace.
#![allow(non_camel_case_types)]
use std::ffi::{c_char, c_int, c_void, CStr};

#[repr(C)]
pub struct sp_seqset {
    pub bases: *const u8,
    pub offsets: *const i64,
    pub n: i64,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct sp_pair_rec {
    pub score: u64,
    pub score2: u64,
    pub i: u32,
    pub j: u32,
    pub c1: u32,
    pub _pad: u32,
}

/// One traceback alignment (include/starphase_gpu.h `sp_align_rec`): the minimap2::Mapping fields
/// HlaProcessedMatch::add_mapping reads (src/hla/processed_match.rs:53-100).
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct sp_align_rec {
    pub dist: i32,
    pub nm: i32,
    pub p_start: i32,
    pub p_end: i32,
    pub t_start: i32,
    pub t_end: i32,
    pub n_cigar: i32,
    pub _pad: i32,
    pub cigar_off: i64,
}

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct sp_affine_costs {
    pub a: i32,
    pub b: i32,
    pub q: i32,
    pub e: i32,
    pub q2: i32,
    pub e2: i32,
}

pub enum sp_ctx {}
pub enum sp_patterns {}
pub enum sp_targets {}
pub enum sp_dmatrix {}
pub enum sp_comm {}
pub enum sp_consensus {}

/// One sp_consensus_run call with its handle (sp_consensus_run_batch).
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct sp_consensus_job {
    pub c: *mut sp_consensus,
    pub n_sides: i32,
    pub src: [i32; 2],
    pub dst: [i32; 2],
    pub ed: *mut i32,
    pub votes: *mut u8,
    pub full: *mut i32,
    pub min_count: i32,
    pub min_af_permille: i32,
    pub cost_limit: i64,
    pub size_limit: i64,
    pub cost_cap: i64,
    pub max_steps: i32,
    pub steps: *mut u8,
    pub n_steps: *mut i32,
}

/// One sp_consensus_extend call with its handle (sp_consensus_extend_batch).
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct sp_consensus_ext {
    pub c: *mut sp_consensus,
    pub n_tasks: i32,
    pub src: *const i32,
    pub symbols: *const u8,
    pub dst: *const i32,
    pub ed: *mut i32,
    pub votes: *mut u8,
    pub full: *mut i32,
}
pub const SP_COMM_ID_BYTES: usize = 128;

pub const SP_INFIX: c_int = 0;
pub const SP_PREFIX: c_int = 1;

extern "C" {
    pub fn sp_ctx_create(device: c_int, stream: *mut c_void, out: *mut *mut sp_ctx) -> c_int;
    pub fn sp_ctx_destroy(ctx: *mut sp_ctx);
    pub fn sp_ctx_synchronize(ctx: *mut sp_ctx) -> c_int;
    pub fn sp_ctx_share_device(ctx: *mut sp_ctx, on: c_int) -> c_int;
    pub fn sp_pinned_alloc(ctx: *mut sp_ctx, bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn sp_pinned_free(ctx: *mut sp_ctx, p: *mut c_void);
    pub fn sp_version() -> *const c_char;
    pub fn sp_launch_count(ctx: *const sp_ctx) -> u64;
    pub fn sp_last_kernel_ms(ctx: *mut sp_ctx, which: c_int) -> f32;
    pub fn sp_int_peak(ctx: *mut sp_ctx, kind: c_int, ops_per_s: *mut f64) -> c_int;
    pub fn sp_host_alloc(ctx: *mut sp_ctx, bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn sp_host_free(ctx: *mut sp_ctx, ptr: *mut c_void);
    pub fn sp_plan_lane_classes(lens: *const i64, n: i64, max_classes: c_int, n_classes: *mut c_int, widths: *mut c_int,
                                n_patterns: *mut i64, n_warps: *mut i64, padded_rows: *mut i64) -> c_int;
    pub fn sp_patterns_count(p: *const sp_patterns) -> i64;
    pub fn sp_patterns_total_len(p: *const sp_patterns) -> i64;
    pub fn sp_patterns_padded_rows(p: *const sp_patterns) -> i64;
    pub fn sp_targets_count(t: *const sp_targets) -> i64;
    pub fn sp_targets_total_len(t: *const sp_targets) -> i64;
    pub fn sp_score_into(ctx: *mut sp_ctx, t: *const sp_targets, p: *const sp_patterns, dst: *mut sp_dmatrix, pattern_row0: i64) -> c_int;
    pub fn sp_dmatrix_to_host_u16(ctx: *mut sp_ctx, d: *const sp_dmatrix, dist: *mut u16) -> c_int;
    pub fn sp_dmatrix_device_ptr(d: *const sp_dmatrix) -> *mut c_void;
    pub fn sp_dmatrix_ld(d: *const sp_dmatrix) -> i64;
    pub fn sp_dmatrix_elem_bits(d: *const sp_dmatrix) -> c_int;
    pub fn sp_dmatrix_wrap(ctx: *mut sp_ctx, dev_ptr: *mut c_void, n_targets: i64, n_patterns: i64, ld: i64, elem_bits: c_int,
                           out: *mut *mut sp_dmatrix) -> c_int;
    pub fn sp_last_error(ctx: *const sp_ctx) -> *const c_char;
    pub fn sp_patterns_create(ctx: *mut sp_ctx, p: *const sp_seqset, mode: c_int, out: *mut *mut sp_patterns) -> c_int;
    pub fn sp_patterns_destroy(p: *mut sp_patterns);
    pub fn sp_targets_create(ctx: *mut sp_ctx, t: *const sp_seqset, out: *mut *mut sp_targets) -> c_int;
    pub fn sp_targets_derive(ctx: *mut sp_ctx, src: *const sp_targets, n_out: i64, src_index: *const i32, iv_off: *const i64, iv_begin: *const i32,
                             iv_end: *const i32, revcomp: *const u8, out: *mut *mut sp_targets) -> c_int;
    pub fn sp_targets_read(t: *const sp_targets, bases: *mut u8, offsets: *mut i64) -> c_int;
    pub fn sp_targets_destroy(t: *mut sp_targets);
    pub fn sp_score_device(ctx: *mut sp_ctx, t: *const sp_targets, p: *const sp_patterns, elem_bits: c_int,
                           want_end_col: c_int, out: *mut *mut sp_dmatrix) -> c_int;
    pub fn sp_dmatrix_to_host(ctx: *mut sp_ctx, d: *const sp_dmatrix, dist: *mut i32, end_col: *mut i32) -> c_int;
    pub fn sp_dmatrix_destroy(d: *mut sp_dmatrix);
    pub fn sp_score_batch(ctx: *mut sp_ctx, targets: *const sp_seqset, patterns: *const sp_seqset, mode: c_int,
                          dist: *mut i32, end_col: *mut i32) -> c_int;
    pub fn sp_score_spans(ctx: *mut sp_ctx, targets: *const sp_seqset, patterns: *const sp_seqset, dist: *mut i32,
                          start_col: *mut i32, end_col: *mut i32) -> c_int;
    pub fn sp_score_spans_filtered(ctx: *mut sp_ctx, targets: *const sp_seqset, patterns: *const sp_seqset, max_dist_permille: c_int,
                                   dist: *mut i32, start_col: *mut i32, end_col: *mut i32) -> c_int;
    pub fn sp_align_pairs(ctx: *mut sp_ctx, targets: *const sp_seqset, patterns: *const sp_seqset, n_pairs: i64,
                          pair_target: *const i32, pair_pattern: *const i32, recs: *mut sp_align_rec, cigar: *mut u32,
                          cigar_cap: i64, cigar_used: *mut i64) -> c_int;
    pub fn sp_align_windows(ctx: *mut sp_ctx, targets: *const sp_seqset, patterns: *const sp_seqset, n_pairs: i64,
                            pair_target: *const i32, pair_pattern: *const i32, win_begin: *const i32, win_end: *const i32,
                            recs: *mut sp_align_rec, cigar: *mut u32, cigar_cap: i64, cigar_used: *mut i64) -> c_int;
    pub fn sp_row_topk(ctx: *mut sp_ctx, d: *const sp_dmatrix, k: c_int, idx: *mut i32, dist: *mut i32) -> c_int;
    pub fn sp_row_topk_biased(ctx: *mut sp_ctx, d: *const sp_dmatrix, pattern_bias: *const i32, k: c_int, idx: *mut i32,
                              dist: *mut i32) -> c_int;
    pub fn sp_row_topk_weighted(ctx: *mut sp_ctx, d: *const sp_dmatrix, dist_weight: c_int, pattern_bias: *const i32, k: c_int, idx: *mut i32,
                                dist: *mut i32) -> c_int;
    pub fn sp_variant_match(ctx: *mut sp_ctx, n_seq: i64, n_hap: i64, n_var: i64, seq_alleles: *const u8, hap_alleles: *const u8,
                            is_vi: *const u8, vi_match: *mut u32, all_match: *mut u32) -> c_int;
    pub fn sp_chain_window_scores(ctx: *mut sp_ctx, n_chains: i64, chain_off: *const i32, chain_items: *const i32, n_reads: i64,
                                  seg_off: *const i32, w: *const u32, n_haps: i64, out: *mut *mut sp_dmatrix) -> c_int;
    pub fn sp_pair_minsum_full(ctx: *mut sp_ctx, d: *const sp_dmatrix, s: *mut u64) -> c_int;
    pub fn sp_pair_minsum_topk(ctx: *mut sp_ctx, d: *const sp_dmatrix, d2: *const sp_dmatrix, i_begin: i64,
                               i_end: i64, k: c_int, out: *mut sp_pair_rec, n_out: *mut c_int) -> c_int;
    pub fn sp_pair_minsum_topk_host(ctx: *mut sp_ctx, d: *const i32, d2: *const i32, r: i64, a: i64, k: c_int,
                                    out: *mut sp_pair_rec, n_out: *mut c_int) -> c_int;
    pub fn sp_pair_minsum_full_host(ctx: *mut sp_ctx, d: *const i32, r: i64, a: i64, s: *mut u64) -> c_int;
    pub fn sp_align_resident(ctx: *mut sp_ctx, texts: *const sp_targets, patterns: *const sp_targets, n_pairs: i64, pair_text: *const i32,
                             pair_pattern: *const i32, win_begin: *const i32, win_end: *const i32, recs: *mut sp_align_rec, cigar: *mut u32,
                             cigar_cap: i64, cigar_used: *mut i64) -> c_int;
    // K9: the reference's affine cost model for selected pairs
    pub fn sp_align_affine_resident(ctx: *mut sp_ctx, texts: *const sp_targets, patterns: *const sp_targets, n_pairs: i64, pair_text: *const i32,
                                    pair_pattern: *const i32, win_begin: *const i32, win_end: *const i32, band_centre: *const i32, band: i32,
                                    pair_band: *const i32, costs: *const sp_affine_costs, recs: *mut sp_align_rec, scores: *mut i32, cigar: *mut u32, cigar_cap: i64,
                                    cigar_used: *mut i64) -> c_int;
    // K7: consensus extension
    pub fn sp_consensus_create(ctx: *mut sp_ctx, reads: *const sp_seqset, offsets: *const i32, offset_window: i32, band: i32, max_tracks: i32,
                               out: *mut *mut sp_consensus) -> c_int;
    pub fn sp_consensus_destroy(c: *mut sp_consensus);
    pub fn sp_consensus_num_reads(c: *const sp_consensus) -> i32;
    pub fn sp_consensus_num_tracks(c: *const sp_consensus) -> i32;
    pub fn sp_consensus_reset(c: *mut sp_consensus, track: i32) -> c_int;
    pub fn sp_consensus_extend(c: *mut sp_consensus, n_tasks: i32, src: *const i32, symbols: *const u8, dst: *const i32, ed: *mut i32,
                               votes: *mut u8, full: *mut i32) -> c_int;
    pub fn sp_consensus_run_supported(c: *const sp_consensus, n_sides: i32) -> i32;
    pub fn sp_consensus_run(c: *mut sp_consensus, n_sides: i32, src: *const i32, dst: *const i32, ed: *mut i32, votes: *mut u8, full: *mut i32,
                            min_count: i32, min_af_permille: i32, cost_limit: i64, size_limit: i64, cost_cap: i64, max_steps: i32, steps: *mut u8,
                            n_steps: *mut i32) -> c_int;
    pub fn sp_consensus_run_batch(ctx: *mut sp_ctx, n_jobs: i32, jobs: *const sp_consensus_job) -> c_int;
    pub fn sp_consensus_extend_batch(ctx: *mut sp_ctx, n_lists: i32, lists: *const sp_consensus_ext) -> c_int;
    // K8: sequence-to-variant-graph alignment
    pub fn sp_graph_align(ctx: *mut sp_ctx, n_problems: i32, gchars: *const u8, gchar_off: *const i64, pred_off: *const i32, preds: *const i32,
                          diag: *const i32, end_off: *const i32, ends: *const i32, seqs: *const u8, seq_off: *const i64, band: i32,
                          score: *mut i32, columns: *mut i32) -> c_int;
    pub fn sp_graph_traverse(ctx: *mut sp_ctx, n_problems: i32, gchars: *const u8, gchar_off: *const i64, pred_off: *const i32, preds: *const i32,
                             diag: *const i32, end_off: *const i32, ends: *const i32, seqs: *const u8, seq_off: *const i64, band: i32,
                             score: *mut i32, on_path: *mut u8) -> c_int;
    // multi-GPU (one sp_comm per context; ranks are processes or threads, every call below is a collective)
    pub fn sp_comm_unique_id(id: *mut u8) -> c_int;
    pub fn sp_comm_create(ctx: *mut sp_ctx, id: *const u8, rank: c_int, world: c_int, out: *mut *mut sp_comm) -> c_int;
    pub fn sp_comm_destroy(c: *mut sp_comm);
    pub fn sp_comm_rank(c: *const sp_comm) -> c_int;
    pub fn sp_comm_world(c: *const sp_comm) -> c_int;
    pub fn sp_comm_barrier(c: *mut sp_comm) -> c_int;
    pub fn sp_shard_plan(lens: *const i64, n: i64, world: c_int, rank: c_int, idx: *mut i64, n_idx: *mut i64) -> c_int;
    pub fn sp_triangle_rows(n: i64, world: c_int, rank: c_int, lo: *mut i64, hi: *mut i64) -> c_int;
    pub fn sp_comm_bcast_targets(c: *mut sp_comm, targets: *const sp_seqset, root: c_int, out: *mut *mut sp_targets) -> c_int;
    pub fn sp_comm_score_allgather(c: *mut sp_comm, t: *const sp_targets, shard: *const sp_patterns, shard_idx: *const i64,
                                   n_total: i64, elem_bits: c_int, out: *mut *mut sp_dmatrix) -> c_int;
    pub fn sp_comm_pair_minsum_topk(c: *mut sp_comm, d: *const sp_dmatrix, d2: *const sp_dmatrix, k: c_int, out: *mut sp_pair_rec,
                                    n_out: *mut c_int) -> c_int;
}

/// Concatenated sequences in the layout of `sp_seqset`.
pub struct SeqSet {
    bases: Vec<u8>,
    offsets: Vec<i64>,
}

impl SeqSet {
    pub fn new<'a>(seqs: impl IntoIterator<Item = &'a [u8]>) -> Self {
        let mut bases = Vec::new();
        let mut offsets = vec![0i64];
        for s in seqs {
            bases.extend_from_slice(s);
            offsets.push(bases.len() as i64);
        }
        SeqSet { bases, offsets }
    }
    pub fn len(&self) -> usize { self.offsets.len() - 1 }
    pub fn is_empty(&self) -> bool { self.len() == 0 }
    pub fn seq_len(&self, i: usize) -> usize { (self.offsets[i + 1] - self.offsets[i]) as usize }
    fn raw(&self) -> sp_seqset {
        sp_seqset { bases: self.bases.as_ptr(), offsets: self.offsets.as_ptr(), n: self.len() as i64 }
    }
}

pub struct GpuScorer { ctx: *mut sp_ctx }

impl GpuScorer {
    pub fn new(device: i32) -> Result<Self, Box<dyn std::error::Error>> {
        let mut ctx = std::ptr::null_mut();
        let st = unsafe { sp_ctx_create(device, std::ptr::null_mut(), &mut ctx) };
        if st != 0 { return Err(Self::err(std::ptr::null()).into()); }
        Ok(GpuScorer { ctx })
    }
    fn err(ctx: *const sp_ctx) -> String {
        unsafe { CStr::from_ptr(sp_last_error(ctx)).to_string_lossy().into_owned() }
    }
    /// `nm + unmapped` of every pattern against every target: `ret[t * patterns.len() + p]`.
    pub fn score_batch(&self, targets: &SeqSet, patterns: &SeqSet) -> Result<Vec<i32>, Box<dyn std::error::Error>> {
        let mut d = vec![0i32; targets.len() * patterns.len()];
        let st = unsafe { sp_score_batch(self.ctx, &targets.raw(), &patterns.raw(), SP_INFIX, d.as_mut_ptr(), std::ptr::null_mut()) };
        if st != 0 { return Err(Self::err(self.ctx).into()); }
        Ok(d)
    }
    /// Same plus the text span `[start, end)` of an optimal placement (CYP2D6 overlap scores).
    pub fn score_spans(&self, targets: &SeqSet, patterns: &SeqSet) -> Result<(Vec<i32>, Vec<i32>, Vec<i32>), Box<dyn std::error::Error>> {
        let n = targets.len() * patterns.len();
        let (mut d, mut s, mut e) = (vec![0i32; n], vec![0i32; n], vec![0i32; n]);
        let st = unsafe { sp_score_spans(self.ctx, &targets.raw(), &patterns.raw(), d.as_mut_ptr(), s.as_mut_ptr(), e.as_mut_ptr()) };
        if st != 0 { return Err(Self::err(self.ctx).into()); }
        Ok((d, s, e))
    }
    /// `score_spans` for the pairs an aligner would report: `start < 0` where the distance exceeds `max_dist_permille` / 1000 of
    /// the pattern length (weight_sequence uses 350; src/cyp2d6/chaining.rs:58-62 then keeps the default weight).
    pub fn score_spans_filtered(&self, targets: &SeqSet, patterns: &SeqSet, max_dist_permille: i32)
        -> Result<(Vec<i32>, Vec<i32>, Vec<i32>), Box<dyn std::error::Error>> {
        let n = targets.len() * patterns.len();
        let (mut d, mut s, mut e) = (vec![0i32; n], vec![0i32; n], vec![0i32; n]);
        let st = unsafe {
            sp_score_spans_filtered(self.ctx, &targets.raw(), &patterns.raw(), max_dist_permille as c_int, d.as_mut_ptr(), s.as_mut_ptr(),
                                    e.as_mut_ptr())
        };
        if st != 0 { return Err(Self::err(self.ctx).into()); }
        Ok((d, s, e))
    }
    /// (vi_match, all_match) of every (observed allele vector, star-allele definition) pair, `[n_seq][n_hap]` row-major: the
    /// haplotype loop of `Cyp2d6Extractor::assign_haplotype` (src/cyp2d6/haplotyper.rs:470-517).
    pub fn variant_match(&self, seq_alleles: &[u8], n_seq: usize, hap_alleles: &[u8], n_hap: usize, is_vi: &[u8])
        -> Result<(Vec<u32>, Vec<u32>), Box<dyn std::error::Error>> {
        let n_var = is_vi.len();
        assert!(seq_alleles.len() == n_seq * n_var && hap_alleles.len() == n_hap * n_var);
        let (mut vi, mut all) = (vec![0u32; n_seq * n_hap], vec![0u32; n_seq * n_hap]);
        let st = unsafe {
            sp_variant_match(self.ctx, n_seq as i64, n_hap as i64, n_var as i64, seq_alleles.as_ptr(), hap_alleles.as_ptr(), is_vi.as_ptr(),
                             vi.as_mut_ptr(), all.as_mut_ptr())
        };
        if st != 0 { return Err(Self::err(self.ctx).into()); }
        Ok((vi, all))
    }
    /// Traceback alignment of the listed (target, pattern) pairs: what `aligner.map(..)` + `select_best_mapping` hand to
    /// `HlaProcessedMatch::add_mapping` (query = pattern = allele, target = text = consensus).  Returns the records and
    /// the shared CIGAR buffer of `(len << 4) | op` entries (ops 1 = I, 2 = D, 7 = '=', 8 = X).
    pub fn align_pairs(&self, targets: &SeqSet, patterns: &SeqSet, pairs: &[(i32, i32)])
        -> Result<(Vec<sp_align_rec>, Vec<u32>), Box<dyn std::error::Error>> {
        let pt: Vec<i32> = pairs.iter().map(|p| p.0).collect();
        let pp: Vec<i32> = pairs.iter().map(|p| p.1).collect();
        let cap: i64 = pairs.iter().map(|&(t, p)| {
            let (n, m) = (targets.seq_len(t as usize) as i64, patterns.seq_len(p as usize) as i64);
            m + n.min(2 * m) + 1
        }).sum();
        let mut recs = vec![sp_align_rec::default(); pairs.len()];
        let mut cigar = vec![0u32; cap.max(1) as usize];
        let mut used: i64 = 0;
        let st = unsafe {
            sp_align_pairs(self.ctx, &targets.raw(), &patterns.raw(), pairs.len() as i64, pt.as_ptr(), pp.as_ptr(),
                           recs.as_mut_ptr(), cigar.as_mut_ptr(), cap, &mut used)
        };
        if st != 0 { return Err(Self::err(self.ctx).into()); }
        cigar.truncate(used as usize);
        Ok((recs, cigar))
    }
    /// k best allele pairs by (sum_r min(D[r,i], D[r,j]), same on D2, i, j); D, D2 are [R][A] row-major.
    pub fn pair_topk(&self, d: &[i32], d2: Option<&[i32]>, r: usize, a: usize, k: usize) -> Result<Vec<sp_pair_rec>, Box<dyn std::error::Error>> {
        let mut out = vec![sp_pair_rec::default(); k];
        let mut n: c_int = 0;
        let st = unsafe {
            sp_pair_minsum_topk_host(self.ctx, d.as_ptr(), d2.map_or(std::ptr::null(), |x| x.as_ptr()), r as i64, a as i64,
                                     k as c_int, out.as_mut_ptr(), &mut n)
        };
        if st != 0 { return Err(Self::err(self.ctx).into()); }
        out.truncate(n as usize);
        Ok(out)
    }
}

impl Drop for GpuScorer {
    fn drop(&mut self) { unsafe { sp_ctx_destroy(self.ctx) } }
}
