/*
 * starphase_gpu.h -- C ABI of libstarphase_gpu.so (B200 / sm_100a scoring path).
 *
 * This is the drop-in boundary for pb-StarPhase's data-parallel hot path.  The
 * reference (Rust, single process, no FFI of its own) reaches all of its
 * alignment arithmetic through `minimap2::Aligner::map` (call sites listed
 * below); a thin `extern "C"` crate (rust/starphase-gpu-sys, INTEGRATION.md)
 * binds exactly the entry points declared here.  Plain pointers and sizes only;
 * every buffer is caller-owned and borrowed for the duration of one call;
 * calls are blocking and not re-entrant per context (the reference host is
 * single-threaded, src/cli/diplotype.rs:185-191).
 *
 * Distance definition (SURVEY.md §8c):
 *     D(P, T) = min over placements of pattern P inside text T of
 *               (edits + unaligned P bases)            [unit costs]
 * = the reference's `nm + unmapped` for a unit-cost-optimal minimap2 mapping:
 *   - HLA allele vs consensus/read, query side penalised
 *       src/hla/caller.rs:1433-1462, src/util/mapping.rs:22-57   (P = allele)
 *   - HLA read vs allele index, allele side penalised
 *       src/hla/realigner.rs:116-146                             (P = allele)
 *   - CYP2D6 read segment vs consensus, segment fully explained
 *       src/cyp2d6/chaining.rs:48-94                             (P = segment)
 *   - CYP2D6 read vs 39 D6/D7/hybrid templates
 *       src/cyp2d6/haplotyper.rs:193-249                         (P = template)
 * Non-ACGT bytes (N, *) match nothing.  Empty pattern => 0; empty text => |P|.
 *
 * There is NO CPU fallback: every entry point fails with SP_ERR_CUDA when no
 * sm_100 device is usable.
 */
#ifndef STARPHASE_GPU_H
#define STARPHASE_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum sp_status {
    SP_OK = 0,
    SP_ERR_INVALID = 1,     /* bad argument (null pointer, bad offsets, k out of range ...)          */
    SP_ERR_CUDA = 2,        /* CUDA runtime failure or no usable device; see sp_last_error            */
    SP_ERR_TOO_LONG = 3,    /* a pattern exceeds SP_MAX_PATTERN_LEN or a text exceeds the tile budget  */
    SP_ERR_NOMEM = 4,       /* host or device allocation failed                                       */
    SP_ERR_RANGE = 5        /* value does not fit the device format (e.g. > 65535 alleles for top-k)  */
} sp_status;

/* Longest pattern one warp can hold: 32 lanes x 24 words x 32 rows (lane widths above 16 words are compiled for sets that hold
 * such a pattern only).  Longer patterns are rejected with SP_ERR_TOO_LONG -- the reference's aligner has no such limit; the
 * HLA-A / HLA-B alleles of IMGT 3.57 reach 4.1 kb, CYP2D6 regions 6.2 kb, the longest class II genomic alleles (DRB1) ~17 kb.
 * The C++ host skips over-long alleles one by one (they score as "no mapping") instead of failing the gene. */
#define SP_MAX_PATTERN_LEN 24576

/* Concatenated ASCII sequences: sequence i = bases[offsets[i] .. offsets[i+1]).
 * Mirrors how the reference hands `&[u8]` sequences to Aligner::with_seq / map. */
typedef struct sp_seqset {
    const uint8_t *bases;
    const int64_t *offsets; /* n + 1 entries, offsets[0] may be > 0, non-decreasing */
    int64_t n;
} sp_seqset;

/* Text boundary mode.  SP_INFIX: both text ends free (every reference call site).
 * SP_PREFIX: the placement must start at text position 0 (used on reversed
 * sequences to recover the start of the aligned span). */
typedef enum sp_mode { SP_INFIX = 0, SP_PREFIX = 1 } sp_mode;

typedef struct sp_ctx sp_ctx;           /* one per process per GPU; owns stream, events, scratch */
typedef struct sp_patterns sp_patterns; /* device-resident packed pattern set (alleles / segments) */
typedef struct sp_targets sp_targets;   /* device-resident packed text set (reads / consensuses)   */
typedef struct sp_dmatrix sp_dmatrix;   /* device-resident distance matrix, u16 or i32             */

/* One ranked pair: allele-pair for HLA (north_star K2), chain-pair for CYP2D6
 * (src/cyp2d6/chaining.rs:409-534).  Ordering key is (score, score2, i, j) ascending,
 * i <= j -- the reference's ChainScore::compare_tuple (chaining.rs:188-197), with the
 * optional secondary sum playing the role of the DNA score behind the cDNA score in
 * HlaMappingScore's lexicographic order (src/hla/mapping.rs:111-117).
 * c1 = #{reads r : (D[r,i], D2[r,i]) <= (D[r,j], D2[r,j])} so the host can apply
 * is_passing_dual (src/hla/caller.rs:1225-1247) unchanged. */
typedef struct sp_pair_rec {
    uint64_t score;  /* sum over reads of min(D[r,i], D[r,j]) on the primary matrix            */
    uint64_t score2; /* same on the secondary matrix (0 when none was given)                   */
    uint32_t i, j;
    uint32_t c1;
    uint32_t _pad;
} sp_pair_rec;

/* ---- context ------------------------------------------------------------------------- */
/* device: CUDA ordinal.  stream: a cudaStream_t to launch on (e.g. the host framework's
 * current stream), or NULL to create a private non-blocking stream.  The legacy default stream (handle 0) cannot
 * be passed; a host that mixes its own work (e.g. NCCL collectives) with these calls must share an explicit stream. */
sp_status sp_ctx_create(int device, void *stream, sp_ctx **out);
void sp_ctx_destroy(sp_ctx *ctx);
/* Message for the last failing call on this context ("" if none).  Maps to the
 * reference's Box<dyn Error> strings.  ctx may be NULL for creation failures. */
const char *sp_last_error(const sp_ctx *ctx);
/* Device time in ms of the most recent launch of kernel `which`
 * (0 = K1 scoring, 1 = K2 pair scoring, 2 = pattern pack, 3 = text pack, 4 = K4 alignment), measured
 * with CUDA events on the context stream; < 0 if it has not run.  Synchronises. */
float sp_last_kernel_ms(sp_ctx *ctx, int which);
/* Number of kernel launches issued by this context since creation. */
uint64_t sp_launch_count(const sp_ctx *ctx);
/* Block until all work queued on the context stream has finished. */
sp_status sp_ctx_synchronize(sp_ctx *ctx);
/* Several contexts on one GPU, each driven by its own host thread (a cohort worker pool: the reference runs one sample per
 * process, src/cli/diplotype.rs; a cohort is many such runs side by side).  With on != 0 the context launches K1 -- the one long
 * kernel of the path -- one CTA per work item instead of as a persistent grid, and launches of several rounds go to a side stream
 * of the lowest priority, so the short kernels of the other contexts (their streams have the highest priority) are dispatched
 * as soon as any K1 CTA retires.  Results are bit-identical either way.  A context alone on its GPU should leave this off. */
sp_status sp_ctx_share_device(sp_ctx *ctx, int on);
/* Page-locked host memory for result buffers (CIGAR pools, matrices): every entry point accepts pageable memory, but device ->
 * host copies into page-locked memory run at PCIe speed and skip the first-touch page faults of a fresh allocation.  The caller
 * owns the block and releases it with sp_pinned_free (NULL is ignored). */
sp_status sp_pinned_alloc(sp_ctx *ctx, size_t bytes, void **out);
void sp_pinned_free(sp_ctx *ctx, void *p);

/* ---- K1: batched infix edit distance ---------------------------------------------------- */
/* Upload + 2-bit/Peq-pack a pattern set (the allele database of one gene, or the read
 * segments of one CYP2D6 sample).  Done once per database, like HlaRealigner::new builds the
 * allele index once (src/hla/realigner.rs:42-91).  mode selects the pad-row encoding. */
sp_status sp_patterns_create(sp_ctx *ctx, const sp_seqset *patterns, sp_mode mode, sp_patterns **out);
void sp_patterns_destroy(sp_patterns *p);
int64_t sp_patterns_count(const sp_patterns *p);
/* sum of |P| over the set (for GCUPS accounting) */
int64_t sp_patterns_total_len(const sp_patterns *p);
/* rows the packed layout really computes per text column (>= total_len; padding included) */
int64_t sp_patterns_padded_rows(const sp_patterns *p);

/* Host-only (no device touched): how sp_patterns_create would split patterns of the given lengths into
 * lane-width classes (each class = one K1 launch; a warp of width U holds 32 lanes x U words x 32 rows).
 * Outputs are arrays of max_classes entries; padded_rows = rows the layout computes per text column. */
sp_status sp_plan_lane_classes(const int64_t *lens, int64_t n, int max_classes, int *n_classes, int *widths,
                               int64_t *n_patterns, int64_t *n_warps, int64_t *padded_rows);

/* Upload + pack a text set (reads / consensus sequences) into tile streams. */
sp_status sp_targets_create(sp_ctx *ctx, const sp_seqset *targets, sp_targets **out);
/* A text set built on the device from pieces of a resident one (row N4 of SURVEY.md 8f): output sequence q = the concatenation
 * of the intervals [iv_begin[k], iv_end[k]), k in [iv_off[q], iv_off[q + 1]), of source sequence src_index[q], reverse-complemented
 * as a whole when revcomp[q] != 0 (A<->T, C<->G in either case; N and any other byte stay; revcomp NULL = none).  This is
 * splice_read's cDNA (src/hla/caller.rs:1518-1576: the exon intervals in read coordinates, which the host gets from the record's
 * CIGAR) and the strand handling of :1337-1368 and src/hla/realigner.rs:511-515 without the bases crossing PCIe again: only the
 * interval tables go up.  The result is an ordinary sp_targets (K1 texts, either side of K4 / K9). */
sp_status sp_targets_derive(sp_ctx *ctx, const sp_targets *src, int64_t n_out, const int32_t *src_index, const int64_t *iv_off,
                            const int32_t *iv_begin, const int32_t *iv_end, const uint8_t *revcomp, sp_targets **out);
/* Copies a text set back: bases[sp_targets_total_len] and offsets[sp_targets_count + 1] (offsets[0] = 0). */
sp_status sp_targets_read(const sp_targets *t, uint8_t *bases, int64_t *offsets);
void sp_targets_destroy(sp_targets *t);
int64_t sp_targets_count(const sp_targets *t);
int64_t sp_targets_total_len(const sp_targets *t);

/* Score every (target, pattern) pair on the device; result stays in HBM.
 * elem_bits: 16 (uint16, for K2) or 32 (int32).  Layout: D[p * ld + t] ("allele-major",
 * reads contiguous) with ld = targets rounded up to a multiple of 64.
 * want_end_col != 0 also records the smallest end column of a best placement. */
sp_status sp_score_device(sp_ctx *ctx, const sp_targets *t, const sp_patterns *p,
                          int elem_bits, int want_end_col, sp_dmatrix **out);
/* Same, but writes rows [pattern_row0, pattern_row0 + n_patterns) of a caller-provided matrix
 * (e.g. the slot of this rank's allele shard inside an NCCL all-gather buffer wrapped with
 * sp_dmatrix_wrap).  The destination needs n_targets <= its ld / n_targets. */
sp_status sp_score_into(sp_ctx *ctx, const sp_targets *t, const sp_patterns *p, sp_dmatrix *dst,
                        int64_t pattern_row0);
void sp_dmatrix_destroy(sp_dmatrix *d);
/* Copy to host as int32 D[t * n_patterns + p] (row = target), optionally end columns. */
sp_status sp_dmatrix_to_host(sp_ctx *ctx, const sp_dmatrix *d, int32_t *D, int32_t *end_col);
/* 16-bit read-back of a 16-bit matrix (half the PCIe bytes): D[t * n_patterns + p]. */
sp_status sp_dmatrix_to_host_u16(sp_ctx *ctx, const sp_dmatrix *d, uint16_t *D);
/* Pinned (page-locked) host memory: sequence and result buffers allocated here move over PCIe at full speed.
 * Any host pointer is accepted everywhere; pageable ones are staged by the driver and are several times slower. */
sp_status sp_host_alloc(sp_ctx *ctx, size_t bytes, void **out);
void sp_host_free(sp_ctx *ctx, void *ptr);
/* Raw device pointer / geometry for zero-copy consumers (torch, NCCL all-gather). */
void *sp_dmatrix_device_ptr(const sp_dmatrix *d);
int64_t sp_dmatrix_ld(const sp_dmatrix *d);
int sp_dmatrix_elem_bits(const sp_dmatrix *d);
/* Wrap caller-owned device memory (e.g. an all-gathered matrix) as a dmatrix view. */
sp_status sp_dmatrix_wrap(sp_ctx *ctx, void *dev_ptr, int64_t n_targets, int64_t n_patterns,
                          int64_t ld, int elem_bits, sp_dmatrix **out);

/* One-call form with host buffers on both sides (seams S1/S2/S3 of SURVEY.md §8b):
 * D[t * n_patterns + p], caller-allocated; end_col optional (NULL to skip). */
sp_status sp_score_batch(sp_ctx *ctx, const sp_seqset *targets, const sp_seqset *patterns,
                         sp_mode mode, int32_t *D, int32_t *end_col);

/* K3 (CYP2D6 seams S3 / a10): distance plus the text span [start_col, end_col) of an optimal placement, for every
 * (target, pattern): end_col = smallest end of a best placement, start_col = the rightmost start among best
 * placements ending there (recovered by an anchored pass over the reversed sequences).  Feeds the overlap score of
 * weight_sequence (src/cyp2d6/chaining.rs:69-81: clipped_start = start_col, clipped_end = |T| - end_col) and the
 * read span of find_base_type_in_sequence (src/cyp2d6/haplotyper.rs:203-249).  All three outputs are
 * [n_targets][n_patterns] row-major int32, caller-allocated.  Meant for CYP2D6-sized batches (one warp per pair). */
sp_status sp_score_spans(sp_ctx *ctx, const sp_seqset *targets, const sp_seqset *patterns, int32_t *D,
                         int32_t *start_col, int32_t *end_col);
/* Same; pairs whose distance exceeds max_dist_permille / 1000 of the pattern length get start_col = -1 and cost no
 * second pass (D and end_col are still written).  weight_sequence uses 350: sequences that far apart (unrelated DNA sits
 * near 500) are pairs for which the reference's aligner returns no mapping at all (src/cyp2d6/chaining.rs:58-62 then
 * leaves the default (|S|, 0.0)).  A negative value disables the filter. */
sp_status sp_score_spans_filtered(sp_ctx *ctx, const sp_seqset *targets, const sp_seqset *patterns, int max_dist_permille,
                                  int32_t *D, int32_t *start_col, int32_t *end_col);

/* K3 (seam S4, src/cyp2d6/chaining.rs:683-731): the window scan of containment_score hoisted out of the pair loop.
 * Chains are CSR lists of haplotype (consensus) indices; read r owns segments seg_off[r] .. seg_off[r+1]) and
 * W[segment][hap] is the edit distance of weight_sequence.  Result: device matrix B (int32, chains x reads in the K2
 * layout) with B[c][r] = best window sum of chain c for read r, or 2 * (sum of per-segment maxima) when the chain is
 * shorter than the read's segment count.  sp_pair_minsum_full / _topk on B then give, for every chain pair,
 * sum_r min(B[i][r], B[j][r]) = the reference's summed best_score (its ED is that minus sum_r optimum_r). */
sp_status sp_chain_window_scores(sp_ctx *ctx, int64_t n_chains, const int32_t *chain_off, const int32_t *chain_items,
                                 int64_t n_reads, const int32_t *seg_off, const uint32_t *W, int64_t n_haps,
                                 sp_dmatrix **out);

/* ---- K4: traceback alignment of selected pairs ------------------------------------------ */
/* What the host reads from a minimap2::Mapping at the HLA call sites (src/hla/processed_match.rs:53-100:
 * query_start / query_end / target_start / target_end / alignment.nm / alignment.cigar with the EQX flag
 * of src/hla/caller.rs:1395), for the pattern (minimap2's query: the allele) placed inside the text
 * (minimap2's target: the consensus / read):
 *   dist = nm + (|P| - (p_end - p_start)) = D(P, T); nm = edits inside the aligned span;
 *   [p_start, p_end) aligned part of the pattern (clipped ends are the "unmapped" bases of MappingStats,
 *   src/data_types/mapping.rs:7-22); [t_start, t_end) aligned part of the text, t_end = the smallest end of
 *   a best placement (the end column of K1 / K3);
 *   cigar[cigar_off .. cigar_off + n_cigar) = run-length entries (len << 4) | op, BAM op codes
 *   1 = I (pattern base without a text base), 2 = D (text base without a pattern base), 7 = '=', 8 = X,
 *   no clip entries -- exactly what process_mm_cigar (processed_match.rs:210-263) iterates over.
 * The path is the canonical unit-cost optimum: walking back from (|P|, t_end) the diagonal is taken whenever it
 * explains the cell, then I, then D (gaps end up left-aligned, as in ksw2). */
typedef struct sp_align_rec {
    int32_t dist, nm;
    int32_t p_start, p_end;
    int32_t t_start, t_end;
    int32_t n_cigar, _pad;
    int64_t cigar_off;
} sp_align_rec;
/* Align pair q = (targets[pair_target[q]], patterns[pair_pattern[q]]) for q in [0, n_pairs); recs has n_pairs
 * entries; cigar has room for cigar_cap entries.  *cigar_used (optional) receives the entries needed; when that
 * exceeds cigar_cap the call fails with SP_ERR_RANGE and nothing else is written
 * (sum over pairs of |P| + min(|T|, 2|P|) + 1 always suffices). */
sp_status sp_align_pairs(sp_ctx *ctx, const sp_seqset *targets, const sp_seqset *patterns, int64_t n_pairs,
                         const int32_t *pair_target, const int32_t *pair_pattern, sp_align_rec *recs,
                         uint32_t *cigar, int64_t cigar_cap, int64_t *cigar_used);

/* Same for windows of the texts: pair q is aligned inside targets[pair_target[q]][win_begin[q], win_end[q]) only, and
 * t_start / t_end of its record are relative to win_begin[q].  The template search of find_base_type_in_sequence
 * (src/cyp2d6/haplotyper.rs:193-249) aligns 39 templates per read on the placement windows K1 reported: thousands of
 * overlapping windows of ~100 reads, which this call takes as (read, begin, end) instead of as copied sub-strings.
 * win_begin == win_end == NULL is sp_align_pairs. */
sp_status sp_align_windows(sp_ctx *ctx, const sp_seqset *targets, const sp_seqset *patterns, int64_t n_pairs,
                           const int32_t *pair_target, const int32_t *pair_pattern, const int32_t *win_begin,
                           const int32_t *win_end, sp_align_rec *recs, uint32_t *cigar, int64_t cigar_cap,
                           int64_t *cigar_used);

/* Resident form: both sequence sets are already on the device.  sp_targets_create uploads any sequence set as ASCII, texts and
 * patterns alike (the allele database of a gene is kept this way next to its packed sp_patterns form; the reads of a sample are
 * uploaded once for K1 and K4).  A call then moves only the pair list in and the records + run-length CIGARs out.  Pairs are
 * packed several to a warp by pattern length (lane width 4 / 8 / 12 / 16 words), each pair streaming its own text.
 * cigar[recs[q].cigar_off ..) holds pair q's entries; the order of the pairs inside `cigar` is unspecified. */
sp_status sp_align_resident(sp_ctx *ctx, const sp_targets *texts, const sp_targets *patterns, int64_t n_pairs,
                            const int32_t *pair_text, const int32_t *pair_pattern, const int32_t *win_begin,
                            const int32_t *win_end, sp_align_rec *recs, uint32_t *cigar, int64_t cigar_cap,
                            int64_t *cigar_used);

/* ---- K9: the reference's cost model for selected pairs ------------------------------------------ */
/* minimap2's two-piece affine costs as the reference configures them: match +a, mismatch -b, ambiguous base -1, a gap of k bases
 * -min(q + k e, q2 + k e2).  map-hifi: {1, 4, 6, 2, 26, 1} (src/util/mapping.rs:8-14); allele scoring sets a = 5
 * (src/hla/caller.rs:1370-1381). */
typedef struct sp_affine_costs { int32_t a, b, q, e, q2, e2; } sp_affine_costs;
/* Best-scoring LOCAL alignment of pattern q inside its text window under `costs`, restricted to the diagonal band
 * |(j - i) - band_centre[q]| <= band (i = pattern base, j = window column, both 1-based; band <= 255; band_centre NULL = 0): what
 * minimap2 reports for one co-linear chain.  pair_band (optional) gives every pair its own half width in [1, 255] and `band` is
 * ignored; pairs are grouped by width class (<= 31, 63, 127, 255) and the classes run side by side.  The host centres the band on
 * the diagonal hull of the placement K4 found.  recs as for
 * sp_align_pairs (dist = nm + clipped pattern bases; p_start / p_end = minimap2's query_start / query_end; t_start / t_end relative to
 * the window), scores[q] = the DP score minimap2 compares with -s (0 and an empty record when nothing scores above 0).  Ties: the
 * diagonal, then the short-gap deletion, short-gap insertion, long-gap deletion, long-gap insertion (ksw2's order); the first best
 * end cell in anti-diagonal order; the walk back stops at the first zero.  Inside the band the result equals the unbanded optimum
 * (tests/test_affine_gpu.py). */
sp_status sp_align_affine_resident(sp_ctx *ctx, const sp_targets *texts, const sp_targets *patterns, int64_t n_pairs,
                                   const int32_t *pair_text, const int32_t *pair_pattern, const int32_t *win_begin,
                                   const int32_t *win_end, const int32_t *band_centre, int32_t band, const int32_t *pair_band,
                                   const sp_affine_costs *costs, sp_align_rec *recs, int32_t *scores, uint32_t *cigar,
                                   int64_t cigar_cap, int64_t *cigar_used);

/* ---- K5: candidate lists -------------------------------------------------------------------- */
/* The k best patterns of every target of a device matrix (k <= 16): idx / dist are [n_targets][k] row-major, ordered
 * by (distance, pattern index) ascending; entries beyond n_patterns are -1.  Plays the role of minimap2's best_n hit
 * list in HlaRealigner::realign_record (src/hla/realigner.rs:116-146, best_n = 5 from src/util/mapping.rs:8-14): only
 * these candidates go on to sp_align_pairs, and R x k records cross PCIe instead of the R x A matrix. */
sp_status sp_row_topk(sp_ctx *ctx, const sp_dmatrix *d, int k, int32_t *idx, int32_t *dist);
/* Same, ranked by distance + pattern_bias[p] (bias in [0, 2^30), NULL = none); dist still returns the plain distance.
 * With bias = max |P| - |P_p| the order is "most pattern bases explained first" (|P_p| - distance descending), the stand-in
 * for minimap2 ranking its hits by alignment score: a read that covers only part of a long allele then keeps that allele
 * ahead of short alleles lying wholly inside the read (src/hla/realigner.rs:116-146 picks among the reported hits). */
sp_status sp_row_topk_biased(sp_ctx *ctx, const sp_dmatrix *d, const int32_t *pattern_bias, int k, int32_t *idx, int32_t *dist);
/* Same, ranked by dist_weight * distance + pattern_bias[p] (dist_weight in [1, 64]; distances as K1 writes them, < 2^24).  minimap2's DP score under map-hifi is
 * about (aligned bases) - 5 * (edits): a mismatch costs b = 4 and forfeits the match's a = 1, a gap more.  With dist_weight = 5
 * and bias = max |P| - |P_p| the candidate list follows that score: against the affine cost model the realigner's assignment
 * agrees for 91 of 96 simulated reads on the IMGT 3.57 HLA-A / HLA-B alleles, 83 of 96 with dist_weight = 1 (DESIGN.md 3). */
sp_status sp_row_topk_weighted(sp_ctx *ctx, const sp_dmatrix *d, int dist_weight, const int32_t *pattern_bias, int k, int32_t *idx,
                               int32_t *dist);

/* ---- K6: CYP2D6 allele-vector match (row N3 of SURVEY.md 8f) ------------------------------- */
/* Replaces the haplotype loop of Cyp2d6Extractor::assign_haplotype (src/cyp2d6/haplotyper.rs:470-517): for every
 * (sequence s, haplotype h) the number of variant sites whose observed state agrees with the haplotype definition,
 * over all sites (all_match) and over the VI sites only (vi_match).  seq_alleles[s][v]: 0 = REF, 1 = ALT,
 * 2 = ambiguous (agrees with anything), 3 = unset (agrees with nothing); hap_alleles[h][v]: 0 / 1; is_vi[v]: 0 / 1.
 * Other values fail with SP_ERR_INVALID (the reference panics on them, :489, :496).  Outputs are [n_seq][n_hap]
 * row-major.  The host keeps the reference's (vi_match, all_match) arg-max and its tie handling. */
sp_status sp_variant_match(sp_ctx *ctx, int64_t n_seq, int64_t n_hap, int64_t n_var, const uint8_t *seq_alleles,
                           const uint8_t *hap_alleles, const uint8_t *is_vi, uint32_t *vi_match, uint32_t *all_match);

/* ---- K2: pair scoring -------------------------------------------------------------------- */
/* S[i,j] = sum_r min(D[r,i], D[r,j]) for i in [i_begin, i_end), j in [i, n_patterns);
 * d2 (may be NULL) is a secondary matrix of the same geometry giving S2 the same way;
 * writes the k smallest by (S, S2, i, j) into out (k <= 64), returns the count in *n_out.
 * Restricting i to a row range is how allele-pair blocks are sharded across GPUs; merging the
 * per-shard lists by the same key reproduces the single-GPU answer exactly. */
sp_status sp_pair_minsum_topk(sp_ctx *ctx, const sp_dmatrix *d, const sp_dmatrix *d2, int64_t i_begin,
                              int64_t i_end, int k, sp_pair_rec *out, int *n_out);
/* Full upper-triangular matrix S[i * n + j] (j >= i; other entries 0) to host memory.  Used by the
 * CYP2D6 chain-pair path where float penalties are added on the host (chaining.rs:459-497). */
sp_status sp_pair_minsum_full(sp_ctx *ctx, const sp_dmatrix *d, uint64_t *S);
/* Host-buffer convenience: D (and D2, may be NULL) are [R][A] row-major int32 (R reads, A alleles / chains).
 * Values must lie in [0, 2^27) (SP_ERR_RANGE otherwise): the kernel adds 32 reads in 32 bits before it widens to 64.  The same
 * holds for 32-bit device matrices handed to the calls above; matrices written by sp_score_device hold distances <= the
 * longest pattern and always qualify. */
sp_status sp_pair_minsum_topk_host(sp_ctx *ctx, const int32_t *D, const int32_t *D2, int64_t R, int64_t A, int k,
                                   sp_pair_rec *out, int *n_out);
sp_status sp_pair_minsum_full_host(sp_ctx *ctx, const int32_t *D, int64_t R, int64_t A, uint64_t *S);

/* ---- K7: consensus extension (row N1 of SURVEY.md 8f) ---------------------------------------- */
/* The reference builds consensus sequences with waffle_con's dynamic-WFA search (DualConsensusDWFA / ConsensusDWFA /
 * PriorityConsensusDWFA: src/hla/caller.rs:1097-1219, :727-755, src/cyp2d6/caller.rs:145-280): candidate consensus prefixes
 * grow one symbol at a time, every read keeps its edit distance to the prefix, and the reads vote for the next symbol.  The
 * data-parallel step -- extend candidate X by symbol s for all reads -- is what these calls put on the device; the search
 * policy (queue, vote thresholds, dual split) stays with the host (pb_starphase_b200/host/sp_host_consensus.cpp).
 * A handle owns `max_tracks` tracks; a track = the DP column of every read against one consensus prefix, banded
 * (`band` rows either side of the read's diagonal, widened by offset_window / 2).  offsets[r] >= 0 is where read r is expected to
 * start inside the consensus (waffle_con's add_sequence_offset(.., Some(offset))): the read may start anywhere within
 * offset_window / 2 of it for free and is inactive before; offsets[r] < 0 (or offsets == NULL) anchors the read at the start of
 * the consensus (add_sequence / offset None).  Read bytes: A C G T (either case); '*' is a wildcard that matches every consensus
 * symbol at no cost and votes for none (CdwfaConfig::wildcard as src/cyp2d6/caller.rs:148 sets it); any other byte matches nothing. */
typedef struct sp_consensus sp_consensus;
sp_status sp_consensus_create(sp_ctx *ctx, const sp_seqset *reads, const int32_t *offsets, int32_t offset_window, int32_t band,
                              int32_t max_tracks, sp_consensus **out);
void sp_consensus_destroy(sp_consensus *c);
int32_t sp_consensus_num_reads(const sp_consensus *c);
int32_t sp_consensus_num_tracks(const sp_consensus *c);
/* Track `track` becomes the empty consensus. */
sp_status sp_consensus_reset(sp_consensus *c, int32_t track);
/* n_tasks extensions in one launch: track dst[q] = track src[q] with symbols[q] appended ('A' 'C' 'G' 'T'; any other byte matches
 * nothing; 0 = no extension, just report the state of src[q], copied to dst[q]).  dst entries are distinct; a track written by
 * one task may not be read by another (src[q] == dst[q] is fine).  Outputs, [n_tasks][n_reads]:
 *   ed    = min over read prefixes of the edit distance to the extended consensus (0 while the read is inactive)
 *   votes = bit 0..3: A / C / G / T follows a prefix reaching that minimum, bit 4: another byte follows, bit 5: the whole read
 *           reaches it, bit 6: the read is not active yet
 *   full  = min over the columns so far of the distance with the whole read consumed (0x3FFFFFFF: never reached): the read's
 *           cost once the consensus has grown past its end. */
sp_status sp_consensus_extend(sp_consensus *c, int32_t n_tasks, const int32_t *src, const uint8_t *symbols, const int32_t *dst,
                              int32_t *ed, uint8_t *votes, int32_t *full);
/* The extension step in a loop on the device, for the stretches of a search where the reads agree (most of a consensus): starting
 * from a node -- one consensus (n_sides = 1) or a dual pair (2), tracks src[], with the per-read state ed / votes / full
 * ([n_sides][n_reads]) the step that made it returned -- keep appending while every side has at most one symbol with the votes and
 * at least one side has one, the extended node orders before the best competitor of the caller's search -- cost < cost_limit, or
 * cost == cost_limit and total length > size_limit -- its cost is <= cost_cap, and fewer than max_steps rounds were done.
 * Vote rule: a read votes when it is active and not already consumed at a better column (full >= ed), one vote split evenly over
 * its candidate symbols; in a dual node a read counts towards, and votes for, the side(s) it is closest to (cost = 0 while
 * inactive, else min(ed, full)); a symbol passes with >= min_count votes and >= min_af_permille / 1000 of its side's votes; when
 * none passes the first best-voted symbol does; a side nobody votes on is finished and stays as it is.  Node cost = sum over reads
 * of the cost to the closest side.  On return dst[] hold the tracks of the last node, ed / votes / full its state, steps[q] the
 * symbols of round q (low nibble: code 0..3 = ACGT appended to side 0, high nibble: side 1; 15 = side not extended) and *n_steps
 * the number of rounds (0: the start node does not qualify; dst[] are then copies of src[]).  The read set has to fit on chip:
 * sp_consensus_run_supported() tells (<= 2,048 read-sides, band <= 255 + window, reads <= 60,000 bases); SP_ERR_RANGE otherwise.
 * src / dst as for sp_consensus_extend (dst[s] may equal src[s]). */
int32_t sp_consensus_run_supported(const sp_consensus *c, int32_t n_sides);
sp_status sp_consensus_run(sp_consensus *c, int32_t n_sides, const int32_t *src, const int32_t *dst, int32_t *ed, uint8_t *votes,
                           int32_t *full, int32_t min_count, int32_t min_af_permille, int64_t cost_limit, int64_t size_limit,
                           int64_t cost_cap, int32_t max_steps, uint8_t *steps, int32_t *n_steps);
/* Many independent searches in one device pass.  A job is the argument list of sp_consensus_run with its handle; a list is the
 * argument list of sp_consensus_extend with its handle.  Each job's / list's outputs equal those of the single call.  Every handle
 * belongs to ctx; jobs may share a handle when their tracks are disjoint, lists may share one when the tracks of all their tasks
 * obey the rules of a single sp_consensus_extend call.  Everything is checked before anything is launched: on a refusal
 * (SP_ERR_INVALID for a bad argument, a track out of range, overlapping tracks or a foreign handle; SP_ERR_RANGE for a job that
 * does not fit on chip) no output is written.  sp_consensus_run_batch runs one thread-block cluster per job, one launch per
 * on-chip size class; sp_consensus_extend_batch runs every (task, read) of every list in one launch. */
typedef struct sp_consensus_job {
    sp_consensus *c;
    int32_t n_sides;
    int32_t src[2], dst[2];
    int32_t *ed;
    uint8_t *votes;
    int32_t *full;
    int32_t min_count, min_af_permille;
    int64_t cost_limit, size_limit, cost_cap;
    int32_t max_steps;
    uint8_t *steps;
    int32_t *n_steps;
} sp_consensus_job;
typedef struct sp_consensus_ext {
    sp_consensus *c;
    int32_t n_tasks;
    const int32_t *src;
    const uint8_t *symbols;
    const int32_t *dst;
    int32_t *ed;
    uint8_t *votes;
    int32_t *full;
} sp_consensus_ext;
sp_status sp_consensus_run_batch(sp_ctx *ctx, int32_t n_jobs, const sp_consensus_job *jobs);
sp_status sp_consensus_extend_batch(sp_ctx *ctx, int32_t n_lists, const sp_consensus_ext *lists);

/* ---- K8: sequence-to-variant-graph alignment (row N3 of SURVEY.md 8f) ------------------------- */
/* The forward half of what Cyp2d6Extractor::assign_haplotype gets from hiphase's WFAGraph::edit_distance_with_pruning
 * (src/cyp2d6/haplotyper.rs:430-450): the unit-cost end-to-end alignment of a sequence to a graph of the CYP2D6 backbone with one
 * bubble per database variant, for a batch of (graph, sequence) problems.  Graphs arrive linearised (host/sp_host_graph.cpp
 * builds them): position = one character; preds[pred_off[q] .. pred_off[q+1]) = the problem-local positions a path can come
 * from (-1 = before the first character), all smaller than q; diag[q] = the sequence row the position is expected to align to
 * (band centre); ends = positions at which a path may end.  Offsets are global over the concatenated problems and start at 0.
 * score[p] = the edit distance (0x3FFFFFFF when the band excludes every path); columns (optional, host memory,
 * [total positions][2 * band + 1] int32) = the DP matrix, row i of position q at index i - diag[q] + band.  sp_graph_traverse
 * below returns the positions on optimal alignments (`traversed_nodes`, :454-468) instead. */
sp_status sp_graph_align(sp_ctx *ctx, int32_t n_problems, const uint8_t *gchars, const int64_t *gchar_off, const int32_t *pred_off,
                         const int32_t *preds, const int32_t *diag, const int32_t *end_off, const int32_t *ends, const uint8_t *seqs,
                         const int64_t *seq_off, int32_t band, int32_t *score, int32_t *columns);
/* The whole of that call on the device: the forward pass of sp_graph_align, then a backward pass over the DP matrix, which stays
 * in device memory.  Inputs, band limits and checks are those of sp_graph_align; score as there.  on_path[q] (required when there
 * are positions, [total positions]) = 1 when position q has a cell on an optimal alignment, else 0.  The cells on an optimal
 * alignment are the end cells (e, m) with D[e][m] == score (e >= 0; m = sequence length) and, from each such cell (q, i), the
 * cells (q, i-1) when D[q][i-1] + 1 == D[q][i]; (pr, i) when D[pr][i] + 1 == D[q][i]; (pr, i-1) when D[pr][i-1] + sub == D[q][i],
 * for every predecessor pr >= 0 of q, where sub = 0 when the graph character is A/C/G/T and equals the sequence character
 * (either case), else 1.  Cells outside the band or outside rows 0..m take part in nothing, and the start column is never marked.
 * These are the cells with forward + backward == score inside the band.  A problem whose score is 0x3FFFFFFF gets all zeros.
 * The traversed nodes are { node of q : on_path[q] == 1 }. */
sp_status sp_graph_traverse(sp_ctx *ctx, int32_t n_problems, const uint8_t *gchars, const int64_t *gchar_off, const int32_t *pred_off,
                            const int32_t *preds, const int32_t *diag, const int32_t *end_off, const int32_t *ends, const uint8_t *seqs,
                            const int64_t *seq_off, int32_t band, int32_t *score, uint8_t *on_path);

/* ---- multi-GPU: the path over the GPUs of one box (SURVEY.md 8b / 8e) ------------------------ */
/* The reference is one process on one thread (src/cli/diplotype.rs:185-191) and has no distributed code; the north_star
 * partitions this path as: allele set sharded for K1, read set broadcast, allele-pair row blocks sharded for K2, per-shard
 * top-k merged with NCCL.  One sp_comm per (sp_ctx, GPU).  The ranks of a communicator are processes (one per GPU) or
 * threads of one process, each driving its own context; every sp_comm_* call below is a collective: all ranks make it, in
 * the same order.  NCCL is loaded with dlopen on first use ($SP_NCCL_LIB, else libnccl.so.2): hosts that use one GPU
 * never need it.  world == 1 communicators work without NCCL. */
typedef struct sp_comm sp_comm;
#define SP_COMM_ID_BYTES 128
/* Rank 0 draws the id (ncclGetUniqueId) and the host program carries the bytes to the other ranks. */
sp_status sp_comm_unique_id(uint8_t *id /* SP_COMM_ID_BYTES */);
sp_status sp_comm_create(sp_ctx *ctx, const uint8_t *id, int rank, int world, sp_comm **out);
void sp_comm_destroy(sp_comm *c);
int sp_comm_rank(const sp_comm *c);
int sp_comm_world(const sp_comm *c);
/* Returns when every rank has made the call and this rank's stream has drained. */
sp_status sp_comm_barrier(sp_comm *c);

/* Host-only.  Which patterns of a set (lengths lens[0..n)) rank `rank` of `world` owns: dealt in length order so that every
 * shard packs into the same lane-width classes as the whole set (equal K1 cost per rank).  idx has room for n entries and
 * receives the owned indices in ascending order. */
sp_status sp_shard_plan(const int64_t *lens, int64_t n, int world, int rank, int64_t *idx, int64_t *n_idx);
/* Host-only.  Row range [lo, hi) of the pair triangle i <= j < n that `rank` scores in sp_comm_pair_minsum_topk
 * (equal pair counts per rank). */
sp_status sp_triangle_rows(int64_t n, int world, int rank, int64_t *lo, int64_t *hi);

/* Read-set broadcast: `targets` is read on `root` only (may be NULL elsewhere); every rank gets device-resident targets. */
sp_status sp_comm_bcast_targets(sp_comm *c, const sp_seqset *targets, int root, sp_targets **out);
/* K1 over the sharded database: `shard` holds this rank's patterns (created with sp_patterns_create from the sequences
 * sp_shard_plan selected, in that order), shard_idx[i] = database index of its i-th pattern, n_total = size of the database.
 * Every rank scores its shard, the shards are all-gathered and the rows put into database order: *out is the full
 * [n_total patterns x targets] matrix (same layout as sp_score_device) on every rank, bit-identical for any world size. */
sp_status sp_comm_score_allgather(sp_comm *c, const sp_targets *t, const sp_patterns *shard, const int64_t *shard_idx,
                                  int64_t n_total, int elem_bits, sp_dmatrix **out);
/* K2 over the pair triangle, rows split by sp_triangle_rows, per-rank lists all-gathered and merged by
 * (score, score2, i, j): every rank returns the list sp_pair_minsum_topk(0, n) would give on one GPU. */
sp_status sp_comm_pair_minsum_topk(sp_comm *c, const sp_dmatrix *d, const sp_dmatrix *d2, int k, sp_pair_rec *out, int *n_out);

/* ---- misc -------------------------------------------------------------------------------- */
/* Integer-ALU microbenchmark used for the roofline denominator (SURVEY.md §8d): runs a
 * dependent-free loop on every SM and returns achieved 32-bit lane-ops per second.
 * kind: 0 = LOP3 (ALU pipe), 1 = IMAD (FMA pipe), 2 = LOP3 + IMAD alternating, 3 = IADD,
 *       4 = IMAD.HI (FMA pipe), 5 = LOP3 + IMAD.HI alternating. */
sp_status sp_int_peak(sp_ctx *ctx, int kind, double *ops_per_s);
const char *sp_version(void);

#ifdef __cplusplus
}
#endif
#endif /* STARPHASE_GPU_H */
