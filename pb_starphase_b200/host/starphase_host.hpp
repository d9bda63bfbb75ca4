// starphase_host.hpp -- C++ host side above the C ABI (include/starphase_gpu.h).
//
// pb-StarPhase's own host is Rust and stays the reference's code (north_star); neither cargo nor rustc
// exists in this image, so this is the compiled-language mirror of the reference's operator interface for
// the hot path: same names, argument meaning and error behaviour as the Rust functions cited at each
// declaration (paths relative to the pb-StarPhase v2.0.1 tree), with every alignment number coming from
// libstarphase_gpu.so.  Nothing here computes an alignment on the CPU.
//
//   src/data_types/mapping.rs, src/hla/mapping.rs   MappingStats, HlaMappingStats, scores
//   src/util/mapping.rs:22-57                       select_best_mapping
//   src/hla/processed_match.rs                      process_mm_cigar, HlaProcessedMatch
//   src/hla/caller.rs:1332-1511                     score_read            (K1 + K4)
//   src/hla/realigner.rs:98-211                     HlaRealigner::realign_records   (K1 + K4)
//   north_star (2) + src/hla/caller.rs:889-901, :1225-1247   diplotype_hla_gene (K1 + K2)
//   src/cyp2d6/chaining.rs:28-103                   weight_sequences      (K3 spans)
//   src/cyp2d6/caller.rs:430-537                    build_chains
//   src/cyp2d6/chaining.rs:223-592                  find_best_chain_pair  (K3 chain windows + K2)
//   src/cyp2d6/caller.rs:907-957                    convert_chain_to_hap
//   src/data_types/starphase_json.rs, src/util/file_io.rs:37-52   result JSON (serde pretty)
//   src/hla/debug.rs                                HlaDebug / ReadMappingStats / DualPassingStats (hla_debug.json)
//   src/hla/caller.rs:1259-1319, :1337-1368, :1518-1576   score_consensus target preparation, splice_read
//   src/hla/caller.rs:1583-1653                     is_hemizygous_better
#pragma once
#include <cstdint>
#include <functional>
#include <map>
#include <memory>
#include <optional>
#include <set>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../../include/starphase_gpu.h"

namespace starphase {

// Box<dyn Error> of the reference: one exception type carrying the message
struct HostError : std::runtime_error {
    using std::runtime_error::runtime_error;
};

// ------------------------------------------------------------------------------------------
// JSON value with serde_json's pretty printer (2-space indent, insertion-ordered objects)
// ------------------------------------------------------------------------------------------
class Json {
  public:
    enum Kind { Null, Bool, Int, Float, Str, Arr, Obj };
    Json() : kind_(Null) {}
    Json(std::nullptr_t) : kind_(Null) {}
    Json(bool b) : kind_(Bool), i_(b) {}
    Json(int v) : kind_(Int), i_(v) {}
    Json(long v) : kind_(Int), i_(v) {}
    Json(long long v) : kind_(Int), i_(v) {}
    Json(unsigned long v) : kind_(Int), i_(static_cast<long long>(v)) {}
    Json(const char *s) : kind_(Str), s_(s) {}
    Json(std::string s) : kind_(Str), s_(std::move(s)) {}
    // f64 as serde_json writes it: ryu's shortest round-trip digits and notation, non-finite -> null
    static Json number(double v) { Json j; j.kind_ = Float; j.f_ = v; return j; }
    static Json array() { Json j; j.kind_ = Arr; return j; }
    static Json object() { Json j; j.kind_ = Obj; return j; }
    Json &push(Json v) { a_.push_back(std::move(v)); return *this; }
    Json &set(const std::string &k, Json v) { o_.emplace_back(k, std::move(v)); return *this; }
    std::string pretty(int indent = 0) const;

  private:
    Kind kind_;
    long long i_ = 0;
    double f_ = 0.0;
    std::string s_;
    std::vector<Json> a_;
    std::vector<std::pair<std::string, Json>> o_;
};

// ------------------------------------------------------------------------------------------
// scores -- src/data_types/mapping.rs, src/hla/mapping.rs
// ------------------------------------------------------------------------------------------
struct MappingStats {  // src/data_types/mapping.rs:7-22
    size_t seq_len = 0, nm = 0, unmapped = 0;
    std::optional<size_t> clipped_start, clipped_end;
    MappingStats() = default;
    MappingStats(size_t l, size_t n, size_t u) : seq_len(l), nm(n), unmapped(u) {}
    double custom_score(bool penalize_unmapped) const;  // :69-85
    double mapping_score() const { return custom_score(true); }
    Json to_json() const;
    bool operator==(const MappingStats &o) const {
        return seq_len == o.seq_len && nm == o.nm && unmapped == o.unmapped && clipped_start == o.clipped_start &&
               clipped_end == o.clipped_end;
    }
};

// MappingScore::harmonic_mean, src/data_types/mapping.rs:172-183; throws on a score <= 0 ("dna_score must be > 0.0")
double harmonic_mean(const std::vector<double> &scores);

struct HlaMappingStats {  // src/hla/mapping.rs:9-14
    std::optional<MappingStats> cdna_stats, dna_stats;
    std::pair<double, double> mapping_score() const;  // (cDNA, DNA), missing side = 1.0 (:66-83, :111-117)
    Json to_json() const;
};

// the fields of minimap2::Mapping the reference reads (SURVEY.md §8b); produced from sp_align_rec
struct Mapping {
    size_t query_start = 0, query_end = 0, query_len = 0;
    size_t target_start = 0, target_end = 0, target_len = 0;
    size_t nm = 0;
    bool forward = true;
    std::vector<std::pair<uint32_t, uint8_t>> cigar;  // (length, op), minimap2 op codes
};

// src/util/mapping.rs:22-57: index of the best mapping (or nullopt) and its stats
std::pair<std::optional<size_t>, MappingStats> select_best_mapping(const std::vector<Mapping> &mappings,
                                                                   bool unmapped_from_target, bool penalize_unmapped,
                                                                   std::optional<size_t> base_length_override);

// src/hla/processed_match.rs:210-263; throws HostError("Unexpected cigar type: ..") like the reference bails
std::vector<size_t> process_mm_cigar(const std::vector<std::pair<uint32_t, uint8_t>> &cigar, size_t target_offset,
                                     size_t target_len, size_t clip_start, size_t clip_end);

class HlaProcessedMatch {  // src/hla/processed_match.rs:10-184
  public:
    explicit HlaProcessedMatch(std::string haplotype) : haplotype_(std::move(haplotype)) {}
    static HlaProcessedMatch worst_match(size_t num_sequences);
    void add_mapping(const std::optional<Mapping> &m);
    bool is_better_match(const HlaProcessedMatch &rhs) const;
    const std::string &haplotype() const { return haplotype_; }
    const std::vector<std::optional<MappingStats>> &full_mapping_stats() const { return full_mapping_stats_; }
    const std::vector<std::optional<std::vector<size_t>>> &processed_cigars() const { return processed_cigars_; }
    const std::vector<std::pair<size_t, size_t>> &processed_ranges() const { return processed_ranges_; }

  private:
    std::string haplotype_;
    std::vector<std::optional<MappingStats>> full_mapping_stats_;
    std::vector<std::optional<std::vector<size_t>>> processed_cigars_;
    std::vector<std::pair<size_t, size_t>> processed_ranges_;
};

// ------------------------------------------------------------------------------------------
// statistics -- src/util/stats.rs, statrs 0.16 pieces it calls
// ------------------------------------------------------------------------------------------
double ln_gamma(double x);
double ln_factorial(uint64_t x);
double multinomial_ln_pmf(const std::vector<double> &probs, const std::vector<uint64_t> &obs);  // src/util/stats.rs:11-36
double binomial_cdf(uint64_t n, double p, uint64_t k);
double beta_reg(double a, double b, double x);  // statrs 0.16 function::beta::beta_reg (continued fraction)
double binomial_ln_pmf(uint64_t n, double p, uint64_t x);          // statrs 0.16 Binomial::ln_pmf
double normal_ln_pdf(double mean, double std_dev, double x);       // statrs 0.16 Normal::ln_pdf
// src/hla/caller.rs:1225-1247 (defaults of src/cli/diplotype.rs)
bool is_passing_dual(size_t counts1, size_t counts2, double min_consensus_fraction = 0.10, double min_cdf = 0.001,
                     double expected_maf = 0.45);

struct DualPassingStats {  // src/hla/debug.rs:186-226
    bool is_passing = false, is_dual = false;
    std::optional<size_t> counts1, counts2;
    std::optional<double> maf, cdf;
    static DualPassingStats new_dual(bool is_passing, size_t c1, size_t c2, double maf, double cdf);
    static DualPassingStats new_non_dual() { return DualPassingStats(); }
    Json to_json() const;
};
// is_passing_dual with everything it reports (src/hla/caller.rs:1225-1247); is_dual = false gives new_non_dual()
DualPassingStats dual_passing_stats(bool is_dual, size_t counts1, size_t counts2, double min_consensus_fraction = 0.10,
                                    double min_cdf = 0.001, double expected_maf = 0.45);

// src/hla/caller.rs:1583-1653.  scores1 / scores2: per read, the edit distance to consensus 1 / 2 (nullopt = not
// scored: the other score + dual_max_ed_delta is assumed, :1597-1599); is_consensus1: the read's assignment.  In the
// north_star form the scores are the K1 columns D[r, allele1], D[r, allele2] of the called pair.
bool is_hemizygous_better(const std::vector<std::optional<size_t>> &scores1, const std::vector<std::optional<size_t>> &scores2,
                          const std::vector<bool> &is_consensus1, bool is_dual, size_t dual_max_ed_delta,
                          std::optional<double> normalized_coverage);

// ------------------------------------------------------------------------------------------
// GPU: RAII view of the C ABI; every failure becomes HostError(sp_last_error)
// ------------------------------------------------------------------------------------------
using SeqList = std::vector<std::string>;

struct Alignment {  // sp_align_rec + its CIGAR
    int32_t dist = 0, nm = 0, p_start = 0, p_end = 0, t_start = 0, t_end = 0;
    std::vector<std::pair<uint32_t, uint8_t>> cigar;
    long score = 0;       // DP score under the reference's costs (what minimap2 compares with -s); set by align_pairs(.., match_score > 0)
    int64_t t_base = 0;   // text coordinate t_start / t_end are relative to (the window begin; moves when K9 widened the window)
    bool refined = false; // the record is K9's (affine cost model) rather than K4's (unit-cost placement)
};

class GpuAligner;

// sequences uploaded once as ASCII (sp_targets): the texts of K1 and either side of K4 (sp_align_resident) without another
// host -> device copy -- the reads of a sample, the 39 CYP2D6 templates, the allele database next to its packed form
class ResidentSeqs {
  public:
    ~ResidentSeqs();
    ResidentSeqs(const ResidentSeqs &) = delete;
    ResidentSeqs &operator=(const ResidentSeqs &) = delete;
    size_t size() const { return seqs_.size(); }
    const SeqList &sequences() const { return seqs_; }

  private:
    friend class GpuAligner;
    ResidentSeqs() = default;
    sp_targets *t_ = nullptr;
    SeqList seqs_;
};

// device-resident packed pattern set (sp_patterns): the allele database of a gene, built once like HlaRealigner::new builds
// its index once (src/hla/realigner.rs:42-91); its ASCII form stays on the device too, for the K4 tracebacks
class PatternSet {
  public:
    ~PatternSet();
    PatternSet(const PatternSet &) = delete;
    PatternSet &operator=(const PatternSet &) = delete;
    size_t size() const { return ascii_->size(); }
    const SeqList &sequences() const { return ascii_->sequences(); }
    const ResidentSeqs &resident() const { return *ascii_; }

  private:
    friend class GpuAligner;
    PatternSet() = default;
    sp_patterns *p_ = nullptr;
    std::shared_ptr<ResidentSeqs> ascii_;
};

// device-resident distance matrix (sp_dmatrix, u16): stays in HBM between K1, K2 and K5
class DeviceMatrix {
  public:
    ~DeviceMatrix();
    DeviceMatrix(const DeviceMatrix &) = delete;
    DeviceMatrix &operator=(const DeviceMatrix &) = delete;
    int64_t n_targets() const { return nt_; }
    int64_t n_patterns() const { return np_; }

  private:
    friend class GpuAligner;
    DeviceMatrix() = default;
    sp_dmatrix *d_ = nullptr;
    int64_t nt_ = 0, np_ = 0;
};

class GpuAligner {
  public:
    explicit GpuAligner(int device = 0);
    ~GpuAligner();
    GpuAligner(const GpuAligner &) = delete;
    GpuAligner &operator=(const GpuAligner &) = delete;
    // D[t * patterns.size() + p]; end_col (optional) = smallest end column of a best placement
    std::vector<int32_t> score_batch(const SeqList &targets, const SeqList &patterns, std::vector<int32_t> *end_col = nullptr);
    // start = -1 where D * 1000 > |pattern| * max_dist_permille (no span computed); negative = every pair
    void score_spans(const SeqList &targets, const SeqList &patterns, std::vector<int32_t> &D, std::vector<int32_t> &start,
                     std::vector<int32_t> &end, int max_dist_permille = -1);
    // windows (optional, one [begin, end) per pair): align inside that part of the text only; t_start / t_end are relative to begin
    std::vector<Alignment> align_pairs(const SeqList &targets, const SeqList &patterns,
                                       const std::vector<std::pair<int32_t, int32_t>> &pairs,
                                       const std::vector<std::pair<int32_t, int32_t>> *windows = nullptr, int match_score = 0);
    std::vector<sp_pair_rec> pair_minsum_topk(const std::vector<int32_t> &D, const std::vector<int32_t> *D2, int64_t R, int64_t A,
                                              int k);
    // resident path: nothing of size reads x alleles crosses PCIe, no sequence is uploaded twice
    std::shared_ptr<ResidentSeqs> upload(const SeqList &seqs);
    // a resident set built on the device from pieces of another (sp_targets_derive): output q = the concatenation of the
    // intervals pieces[q].second of source sequence pieces[q].first, reverse-complemented as a whole where revcomp[q]; only the
    // interval tables cross PCIe (the host copy of the result is cut from the host copy of the source)
    std::shared_ptr<ResidentSeqs> derive(const ResidentSeqs &src, const std::vector<std::pair<size_t, std::vector<std::pair<size_t, size_t>>>> &pieces,
                                         const std::vector<bool> &revcomp);
    std::shared_ptr<PatternSet> prepare_patterns(const SeqList &patterns);
    std::unique_ptr<DeviceMatrix> score_device(const SeqList &targets, const PatternSet &patterns);          // K1
    std::unique_ptr<DeviceMatrix> score_device(const ResidentSeqs &targets, const PatternSet &patterns, bool want_end_col = false);
    // D[t * n_patterns + p] (and end columns) of a device matrix scored with 32-bit elements / end columns
    void matrix_to_host(const DeviceMatrix &d, std::vector<int32_t> &D, std::vector<int32_t> *end_col);
    // K4; with match_score > 0 (the `a` of the call site: 5 for allele scoring, 1 elsewhere) followed by K9: every placement whose
    // diagonal band fits (half width = half the diagonal hull of the unit-cost path + 24 <= 255) is re-aligned under the
    // reference's two-piece affine costs inside that band, within `bounds` (optional, per pair [lo, hi) of the text; default the
    // whole text), and `score` is filled for every pair; pairs scoring below report_floor come back without their CIGAR (callers
    // that treat them as "no mapping" anyway save the decode of long junk CIGARs)
    std::vector<Alignment> align_pairs(const ResidentSeqs &texts, const ResidentSeqs &patterns,
                                       const std::vector<std::pair<int32_t, int32_t>> &pairs,
                                       const std::vector<std::pair<int32_t, int32_t>> *windows = nullptr, int match_score = 0,
                                       const std::vector<std::pair<int32_t, int32_t>> *bounds = nullptr, long report_floor = -(1l << 62));
    std::vector<sp_pair_rec> pair_minsum_topk(const DeviceMatrix &d, const DeviceMatrix *d2, int k);           // K2
    // K5; ranking key = dist_weight * distance + pattern_bias[p] (bias optional, one entry per pattern); dist returns the plain distance
    void row_topk(const DeviceMatrix &d, int k, std::vector<int32_t> &idx, std::vector<int32_t> &dist,
                  const std::vector<int32_t> *pattern_bias = nullptr, int dist_weight = 1);
    // S[i * n_chains + j], j >= i: sum over reads of min(B[i][r], B[j][r]) for the chain-window matrix B
    std::vector<uint64_t> chain_pair_sums(const std::vector<std::vector<int32_t>> &chains,
                                          const std::vector<std::vector<std::vector<uint32_t>>> &read_weights, int64_t n_haps);
    // K6: (vi_match, all_match)[s * n_hap + h] for site-state rows (0 REF, 1 ALT, 2 ambiguous, 3 unset) against 0/1 haplotype rows
    void variant_match(const std::vector<std::vector<uint8_t>> &seq_alleles, const std::vector<std::vector<uint8_t>> &hap_alleles,
                       const std::vector<uint8_t> &is_vi, std::vector<uint32_t> &vi_match, std::vector<uint32_t> &all_match);
    uint64_t launch_count() const;
    // several aligners on one GPU, one host thread each (a cohort worker pool): sp_ctx_share_device
    void share_device(bool on);
    sp_ctx *raw() { return ctx_; }

  private:
    // K4 alone: records + the run-length CIGAR pool (page-locked buffer `slot`, valid until that slot is used again)
    struct UnitResult {
        std::vector<sp_align_rec> recs;
        const uint32_t *cigar = nullptr;
    };
    UnitResult align_pairs_unit(const ResidentSeqs &texts, const ResidentSeqs &patterns,
                                const std::vector<std::pair<int32_t, int32_t>> &pairs,
                                const std::vector<std::pair<int32_t, int32_t>> *windows);
    uint32_t *cigar_buffer(int slot, int64_t entries);  // grow-only, page-locked (sp_pinned_alloc)
    void check(sp_status st, const char *what);
    sp_ctx *ctx_ = nullptr;
    uint32_t *cig_buf_[2] = {nullptr, nullptr};
    int64_t cig_cap_[2] = {0, 0};
    int64_t cigar_entries_per_pair_ = 256;  // first guess of the CIGAR pool size; grows with what the calls really needed
    int64_t affine_entries_per_pair_ = 64;  // the same for K9's pool
};

// ------------------------------------------------------------------------------------------
// Stand-ins for decisions minimap2 makes inside the reference and an exhaustive aligner cannot copy: whether a mapping is
// reported at all, and which five hits of an index come back.  They have no counterpart in the reference's own code; each is
// measured against the affine cost model in DESIGN.md 3 and listed as a known deviation in INTEGRATION.md.  One process-wide
// set, adjustable by the embedding host.
// ------------------------------------------------------------------------------------------
struct AlignerStandIns {
    long min_dp_score = 200;        // minimap2 -s of map-hifi: a K4 path scoring less (a=1|5 b=4 q=6 e=2 q2=26 e2=1) counts as "no mapping"
    int no_mapping_permille = 350;  // weight_sequence: (segment, consensus) pairs further apart than this share of the segment have no hit
    int candidate_edit_weight = 5;  // realigner candidates: smallest weight * (nm + unmapped) - |allele| (map-hifi: one edit ~ b + a = 5)
    bool template_half_prefilter = true;  // template search: pairs with more than half the template unexplained skip the traceback
    bool affine_refine = true;      // K9 after K4: mapping fields (nm, clips, spans, CIGAR, DP score) from the affine cost model where the band fits
};
AlignerStandIns &aligner_stand_ins();

// ------------------------------------------------------------------------------------------
// HLA
// ------------------------------------------------------------------------------------------
struct HlaAlleleDefinition {  // the members of src/hla/alleles.rs the path reads
    std::string hla_id, gene_name;
    std::vector<std::string> star_allele;
    std::optional<std::string> dna_sequence;
    std::string cdna_sequence;
};
using HlaDatabase = std::map<std::string, HlaAlleleDefinition>;  // BTreeMap<hla_id, def>: iteration order is semantics

struct DiplotypeSettings;
// src/hla/caller.rs:1090-1095: the allele belongs to the gene and has a DNA sequence (unless hla_require_dna is off)
bool is_allowed_allele_def(const HlaAlleleDefinition &def, const std::string &gene_name, const DiplotypeSettings &cli_settings);

struct DiplotypeSettings {  // the members of src/cli/diplotype.rs the path reads
    bool disable_cdna_scoring = false;
    bool hla_require_dna = true;
    double min_consensus_fraction = 0.10, min_cdf = 0.001, expected_maf = 0.45;
    size_t min_consensus_count = 3, dual_max_ed_delta = 100;  // src/cli/diplotype.rs:172-183
    // minimap2's "-s" (min_dp_max, 200 for map-hifi) decides whether a mapping exists at all; the exhaustive aligner
    // always places the allele somewhere, so the same DP score (a=5 b=4 q=6 e=2 q2=26 e2=1, src/hla/caller.rs:1381)
    // of the reported CIGAR is held against that threshold
    int min_dp_score = 200;
};

// minimap2's DP score of a CIGAR: match_score 5 is the scoring of src/hla/caller.rs:1370-1381, 1 the map-hifi default
// of standard_hifi_aligner (src/util/mapping.rs:8-14); b=4 q=6 e=2 q2=26 e2=1 in both
long dp_score(const std::vector<std::pair<uint32_t, uint8_t>> &cigar, long match_score = 5);

// ---- hla_debug.json (src/hla/debug.rs): the artefact to diff against a reference run with --debug-folder ----
struct DetailedMappingStats {  // src/hla/debug.rs:135-183 (DetailedMappingStats::from_mapping)
    size_t query_len = 0, target_len = 0, match_len = 0, nm = 0, query_unmapped = 0, target_unmapped = 0;
    std::string cigar, md;
    Json to_json() const;
};
// minimap2's cigar_str ("12=1X3I..") and MD string (format.c write_MD_core: match runs, mismatched / deleted target
// bases) of an alignment of `query` (the pattern) inside `target` (the text)
std::string cigar_string(const std::vector<std::pair<uint32_t, uint8_t>> &cigar);
std::string md_string(const std::vector<std::pair<uint32_t, uint8_t>> &cigar, const std::string &target, size_t target_start,
                      const std::string &query, size_t query_start);
DetailedMappingStats detailed_mapping_stats(const Mapping &m, const std::string &target, const std::string &query);

struct PairedMappingStats {  // src/hla/debug.rs:126-132
    std::optional<DetailedMappingStats> cdna_mapping, dna_mapping;
    Json to_json() const;
};
class ReadMappingStats {  // src/hla/debug.rs:64-123
  public:
    void set_best_match(std::string id, std::string star) { best_match_id_ = std::move(id); best_match_star_ = std::move(star); }
    const std::optional<std::string> &best_match_id() const { return best_match_id_; }
    const std::optional<std::string> &best_match_star() const { return best_match_star_; }
    const std::map<std::string, PairedMappingStats> &mapping_stats() const { return mapping_stats_; }
    // throws HostError("Entry {hla_id} is already occupied!") like the reference bails
    void add_mapping(const std::string &hla_id, std::optional<DetailedMappingStats> cdna, std::optional<DetailedMappingStats> dna);
    Json to_json() const;

  private:
    std::optional<std::string> best_match_id_, best_match_star_;
    std::map<std::string, PairedMappingStats> mapping_stats_;
};
class HlaDebug {  // src/hla/debug.rs:6-62
  public:
    void add_read(const std::string &gene, const std::string &qname, ReadMappingStats stats);
    void add_dual_passing_stats(const std::string &gene, DualPassingStats stats);
    Json to_json() const;
    std::string pretty() const { return to_json().pretty(); }  // save_json, src/util/file_io.rs:37-52

  private:
    std::map<std::string, std::map<std::string, ReadMappingStats>> read_mapping_stats_;
    std::optional<std::map<std::string, DualPassingStats>> dual_passing_stats_;
};

struct ScoreReadResult {  // score_read's (HashMap<String, HlaMappingStats>, ReadMappingStats)
    std::map<std::string, HlaMappingStats> stats;
    std::string best_hla_id, best_star_allele;
    ReadMappingStats read_mapping_stats;  // keyed by star allele (all_hla_targets = true, src/hla/caller.rs:1397, :1473-1477)
};

// ---- what score_consensus / score_read do to a consensus before the allele loop ----
// src/hla/caller.rs:1518-1576 on plain values: `sequence` aligned at reference position `pos` (0-based) with `cigar`
// (BAM op codes: 0 M, 1 I, 2 D, 3 N, 4 S, 5 H, 7 =, 8 X); exons = half-open reference ranges in the gene
// definition's order.  Returns (spliced bases, offset of the first covered exon base).
// the read intervals splice_read concatenates (:1541-1562) and its offset into the first exon: what sp_targets_derive needs to
// build the cDNA on the device
std::pair<std::vector<std::pair<size_t, size_t>>, size_t> splice_segments(size_t sequence_len, int64_t pos,
                                                                          const std::vector<std::pair<uint32_t, uint8_t>> &cigar,
                                                                          const std::vector<std::pair<uint64_t, uint64_t>> &exons);
std::pair<std::string, size_t> splice_read(const std::string &sequence, int64_t pos, const std::vector<std::pair<uint32_t, uint8_t>> &cigar,
                                           const std::vector<std::pair<uint64_t, uint64_t>> &exons);
std::string reverse_complement(const std::string &s);  // src/util/sequence.rs; throws on a non-ACGTN byte like the reference
struct ScoreReadTargets {
    std::string dna_target, cdna_target;
};
// src/hla/caller.rs:1337-1368: gene-strand DNA target and spliced cDNA target ("N" when nothing splices or cDNA scoring is off)
ScoreReadTargets prepare_score_read_targets(const std::string &read_sequence, int64_t pos, const std::vector<std::pair<uint32_t, uint8_t>> &cigar,
                                            const std::vector<std::pair<uint64_t, uint64_t>> &exons, bool is_forward_strand,
                                            const DiplotypeSettings &settings);
// src/hla/caller.rs:1332-1511.  dna_target / cdna_target: the consensus on the gene's strand and its spliced cDNA
// ("N" when empty), prepared by the host exactly as lines 1337-1368.
ScoreReadResult score_read(GpuAligner &gpu, const std::string &dna_target, const std::string &cdna_target, const HlaDatabase &database,
                           const std::string &gene_name, const DiplotypeSettings &settings);

// src/hla/caller.rs:1259-1319: the consensus (hg38 forward strand) is aligned to the gene's reference region (K4 in place of
// ref_aligner.map), the mapping becomes the CIGAR of an artificial record at ref_start + target_start with the unaligned consensus
// ends soft-clipped (convert_mapping_to_cigar, src/visualization/debug_bam_writer.rs:310-344), and that record goes through
// splice_read / the strand handling into score_read.  exons: absolute reference coordinates.  An empty consensus or one that does
// not align gives the empty result of :1264-1268 / :1283-1288.
ScoreReadResult score_consensus(GpuAligner &gpu, const std::string &reference_sequence, int64_t ref_start, const std::string &consensus,
                                const HlaDatabase &database, const std::string &gene_name,
                                const std::vector<std::pair<uint64_t, uint64_t>> &exons, bool is_forward_strand,
                                const DiplotypeSettings &settings);

struct PgxMappingDetails {  // src/data_types/starphase_json.rs:271-283
    std::string read_qname, best_hla_id, best_star_allele;
    HlaMappingStats best_mapping_stats;
    bool is_ignored = false;
    Json to_json() const;
};

// src/util/homopolymers.rs:18-42
std::string hpc(const std::string &sequence);
size_t hpc_pos(const std::string &sequence, size_t position);

struct HlaGeneDefinition {  // the members of src/hla/alleles.rs' gene definition the realigner reads
    bool is_forward_strand = true;
    // hg38 forward-strand sequence of the gene region +- 100 bp (src/hla/realigner.rs:72-77, `gene_ref_sequence`)
    std::string reference_sequence;
};
struct RealignedHlaRecord {  // src/hla/realigner.rs:417-478 (without the cloned bam::Record)
    size_t segment_start = 0, segment_end = 0;  // the part of the read handed to the consensus step
    std::string dna_sequence, hpc_sequence;
    size_t dna_offset = 0, hpc_offset = 0;
};
struct RealignmentResult {  // src/hla/realigner.rs:358-414
    std::string gene_name;
    ReadMappingStats read_mapping_stats;
    PgxMappingDetails mapping_details;
    std::optional<RealignedHlaRecord> realigned_record;
    bool is_realigned() const { return realigned_record.has_value(); }
};

class HlaRealigner {  // src/hla/realigner.rs:22-350
  public:
    // builds the resident allele index once: every allele of the listed genes that has a DNA sequence (create_hla_fasta, :497-526);
    // sequences are taken as stored (database side only: realign_records)
    HlaRealigner(GpuAligner &gpu, const std::vector<std::string> &gene_list, const HlaDatabase &database);
    // HlaRealigner::new (:42-91): alleles of reverse-strand genes are reverse-complemented into hg38 orientation
    // (create_hla_fasta :511-515) and every gene keeps its buffered hg38 sequence for the offset step (realign_records_full)
    HlaRealigner(GpuAligner &gpu, const std::vector<std::string> &gene_list, const HlaDatabase &database,
                 const std::map<std::string, HlaGeneDefinition> &gene_definitions);
    // one PgxMappingDetails per read, in input order; n_candidates plays the role of minimap2's best_n = 5.
    // K1 over the index (matrix stays on the device), K5 candidate lists, K4 traceback of the candidates.
    std::vector<PgxMappingDetails> realign_records(const std::vector<std::pair<std::string, std::string>> &qname_and_sequence,
                                                   int n_candidates = 5);
    // same, on a distance matrix K1 already produced for these reads against this index
    std::vector<PgxMappingDetails> realign_records_scored(const std::vector<std::pair<std::string, std::string>> &qname_and_sequence,
                                                          const DeviceMatrix &D, int n_candidates = 5,
                                                          const ResidentSeqs *resident_reads = nullptr);
    // realign_record in full (:98-350) for a batch of reads (hg38 forward strand): best database allele as above, then the
    // buffered read segment against the gene's hg38 sequence and, when that starts later than the allele mapping, the allele
    // against hg38 (two more K4 batches) for the segment range and the DNA / HPC offsets the consensus step consumes
    std::vector<RealignmentResult> realign_records_full(const std::vector<std::pair<std::string, std::string>> &qname_and_sequence,
                                                        int n_candidates = 5);
    size_t n_alleles() const { return alleles_.size(); }
    const PatternSet &index() const { return *index_; }
    const std::vector<std::string> &skipped_alleles() const { return skipped_; }  // longer than SP_MAX_PATTERN_LEN: not in the index

  private:
    std::vector<std::string> skipped_;
    struct BestHit { int allele = -1; MappingStats stats; Alignment aln; };
    // resident_reads: the reads as already uploaded for K1 (nullptr: uploaded here)
    std::vector<BestHit> best_hits(const std::vector<std::pair<std::string, std::string>> &reads, const DeviceMatrix &D, int n_candidates,
                                   const ResidentSeqs *resident_reads = nullptr);
    GpuAligner &gpu_;
    std::vector<const HlaAlleleDefinition *> alleles_;
    std::shared_ptr<PatternSet> index_;
    std::map<std::string, HlaGeneDefinition> gene_definitions_;
};

struct HlaRead {
    std::string qname, dna_target, cdna_target;
};
struct Diplotype {  // src/data_types/pgx_diplotype.rs:9-66
    std::string hap1, hap2;
    std::string diplotype() const { return hap1 + "/" + hap2; }
    std::string pharmcat_diplotype() const;  // :51-65: a haplotype holding a '+' goes into brackets ("[*4 + *68]/*1")
    Json to_json() const;
};
struct HlaGeneCall {
    Diplotype diplotype;
    std::string hla_id1, hla_id2;
    uint64_t pair_score_cdna = 0, pair_score_dna = 0;
    size_t counts1 = 0, counts2 = 0;
    std::vector<PgxMappingDetails> mapping_details;
    Json gene_details() const;  // PgxGeneDetails::new_from_mappings, src/data_types/starphase_json.rs:147-161
};
// One gene's resident database: the allowed alleles in BTreeMap order with their DNA / cDNA pattern sets on the device
// and the realigner over the same DNA index.  Built once per database, reused for every sample of a cohort.
struct HlaRecord;
class HlaGeneIndex {
  public:
    HlaGeneIndex(GpuAligner &gpu, const HlaDatabase &database, const std::string &gene_name, const DiplotypeSettings &settings);
    const std::string &gene_name() const { return gene_name_; }
    size_t n_alleles() const { return allowed_.size(); }
    // alleles longer than SP_MAX_PATTERN_LEN: left out of the index (cannot be called), listed here for the caller's warning
    const std::vector<std::string> &skipped_alleles() const { return skipped_; }

  private:
    std::vector<std::string> skipped_;
    friend HlaGeneCall diplotype_hla_gene(GpuAligner &, HlaGeneIndex &, const std::vector<HlaRead> &, const DiplotypeSettings &);
    friend HlaGeneCall diplotype_hla_gene_records(GpuAligner &, HlaGeneIndex &, const std::vector<HlaRecord> &,
                                                  const std::vector<std::pair<uint64_t, uint64_t>> &, bool, const DiplotypeSettings &);
    friend HlaGeneCall diplotype_from_targets(GpuAligner &, HlaGeneIndex &, const std::vector<std::string> &, const std::shared_ptr<ResidentSeqs> &,
                                              const std::shared_ptr<ResidentSeqs> &, const DiplotypeSettings &);
    std::string gene_name_;
    HlaDatabase gene_db_;  // owns the allele definitions the realigner points to
    std::vector<const HlaAlleleDefinition *> allowed_;
    std::shared_ptr<PatternSet> cdna_;
    std::unique_ptr<HlaRealigner> realigner_;  // holds the DNA pattern set
};
// north_star (2): exhaustive read x allele scoring, allele-pair min-sum ranking with the (cDNA, DNA) key, then the
// reference's het/hom decision (src/hla/caller.rs:889-901) and diplotype strings (:1046-1065)
HlaGeneCall diplotype_hla_gene(GpuAligner &gpu, HlaGeneIndex &index, const std::vector<HlaRead> &reads, const DiplotypeSettings &settings);
// the same call from aligned records (what the reference holds when it reaches score_read, src/hla/caller.rs:1337-1368): the
// read sequences are uploaded once; the DNA targets (reverse-complemented for a reverse-strand gene) and the cDNA targets
// (splice_read's exon intervals, "N" when nothing is left or cDNA scoring is off) are built on the device from them
struct HlaRecord {
    std::string qname, sequence;
    int64_t pos = 0;
    std::vector<std::pair<uint32_t, uint8_t>> cigar;
};
HlaGeneCall diplotype_hla_gene_records(GpuAligner &gpu, HlaGeneIndex &index, const std::vector<HlaRecord> &records,
                                       const std::vector<std::pair<uint64_t, uint64_t>> &exons, bool is_forward_strand,
                                       const DiplotypeSettings &settings);
// convenience: builds the index for this one call
HlaGeneCall diplotype_hla_gene(GpuAligner &gpu, const HlaDatabase &database, const std::string &gene_name,
                               const std::vector<HlaRead> &reads, const DiplotypeSettings &settings);

// ------------------------------------------------------------------------------------------
// CYP2D6
// ------------------------------------------------------------------------------------------
enum class Cyp2d6RegionType { Unknown, Rep6, Cyp2d6, LinkRegion, Rep7, Spacer, Cyp2d7, Cyp2d6Deletion, Hybrid, FalseAllele };

struct Cyp2d6RegionLabel {  // src/cyp2d6/region_label.rs:72-266
    Cyp2d6RegionType region_type = Cyp2d6RegionType::Unknown;
    std::optional<std::string> subtype_label;
    bool is_cyp2d() const;
    bool is_rep() const;
    bool is_reported_allele() const;
    std::string full_allele() const;
    std::string simplify_allele(bool detailed, const std::map<std::string, std::string> &cyp_translate) const;
    bool is_allowed_label() const;
    bool is_allowed_label_pair(const Cyp2d6RegionLabel &next) const;
    bool is_normalizing_allele(bool normalize_all) const;
    bool is_candidate_chain_head(bool normalize_all) const;
    void mark_false_allele() { region_type = Cyp2d6RegionType::FalseAllele; }
};
const char *region_type_name(Cyp2d6RegionType t);
Cyp2d6RegionType region_type_from_name(const std::string &s);

// ---- allele-vector typing: the in-tree half of Cyp2d6Extractor::assign_haplotype (src/cyp2d6/haplotyper.rs:452-601) ----
enum class VariantAlleleRelationship {  // src/data_types/region_variants.rs:5-23
    Unknown, Match, Unexpected, Missing, AmbiguousUnexpected, AmbiguousMissing, UnknownUnexpected, UnknownMissing
};
const char *variant_state_name(VariantAlleleRelationship s);
struct RegionVariant {  // src/data_types/region_variants.rs:26-34
    std::string label;
    bool is_vi = false;
    VariantAlleleRelationship variant_state = VariantAlleleRelationship::Unknown;
    std::string to_string() const;  // "=label" / "+label" / "-label" / "?label"
    Json to_json() const;
};
struct VariantMetadata {  // the members of LoadedVariants the typing reads (src/cyp2d6/haplotyper.rs:617-640, :812)
    std::string label;
    bool is_vi = false;
};
struct Cyp2d6Region {  // src/cyp2d6/region.rs:17-25
    Cyp2d6RegionLabel label;
    std::optional<size_t> unique_id;
    std::optional<std::vector<RegionVariant>> variants;  // set by the allele-vector typing (assign_haplotypes_from_alleles)
    std::string index_label() const;  // :50-56
    std::string deep_label() const;   // :60-95: index label + "+rs.." (unexpected) / "-rs.." (missing) / "?rs.." (ambiguous) deltas
};

struct AlleleMapping {  // src/cyp2d6/haplotyper.rs:836-869
    Cyp2d6RegionLabel allele_label;
    size_t region_start = 0, region_end = 0;  // coordinates inside the searched sequence
    MappingStats mapping_stats;               // relative to the template, with clippings
};

// src/cyp2d6/haplotyper.rs:877-893: shared length over the shorter of the two ranges [s1, e1), [s2, e2)
double overlap_score(size_t s1, size_t e1, size_t s2, size_t e2);

// The search half of Cyp2d6Extractor (src/cyp2d6/haplotyper.rs:142-315): which of the D6 / D7 / hybrid / REP / spacer /
// link / *5 templates (generate_cyp_hybrids, src/cyp2d6/definitions.rs:346-464) occur where in a sequence.
struct Cyp2d6TypingDb;
class Cyp2d6Extractor {
  public:
    // hybrid_sequences: (label, template sequence); iterated in full_allele() string order like :175-183
    Cyp2d6Extractor(GpuAligner &gpu, std::vector<std::pair<Cyp2d6RegionLabel, std::string>> hybrid_sequences);
    // find_base_type_in_sequence for a batch of sequences (reads or consensuses).  One K1 launch scores every
    // (sequence, template) pair; promising pairs get a K4 traceback on the placement window; every accepted hit
    // re-opens the search in the unexplained remainders left and right of it for the same template (minimap2 reports
    // up to best_n = 5 mappings per query, e.g. both copies of a duplication), then the reference's overlap collapse
    // and missing-fraction filter run unchanged.
    std::vector<std::vector<AlleleMapping>> find_base_type_in_sequences(const SeqList &search_sequences, bool penalize_unmapped,
                                                                        double max_missing_frac);
    const std::vector<std::pair<Cyp2d6RegionLabel, std::string>> &hybrid_sequences() const { return templates_; }
    // find_full_type_in_sequence (:326-361) for a batch of consensuses: template search with unmapped bases penalised, the
    // lowest-scoring match (first on ties); a match listed in db.mapped_hybrids goes through assign_haplotype (:371-601):
    // the consensus is mapped onto the backbone (K4 + K9, a = 1), the variant graph of the aligned backbone stretch is built
    // and the aligned part of the consensus aligned to it end to end (K8), the traversed nodes give the allele vector, K6
    // scores it against every haplotype definition.  nullopt = "no matches found" (the reference's error).
    std::vector<std::optional<Cyp2d6Region>> find_full_type_in_sequences(const SeqList &search_sequences, double max_missing_frac,
                                                                         bool force_assignment, const Cyp2d6TypingDb &db,
                                                                         size_t graph_band = 128);

  private:
    GpuAligner &gpu_;
    std::vector<std::pair<Cyp2d6RegionLabel, std::string>> templates_;
    std::shared_ptr<PatternSet> tmpl_patterns_;  // built at the first search
};

// :454-468: per-site state from the nodes a WFA-graph traversal visited (3 = unset, conflicting assignments -> 2)
std::vector<uint8_t> alleles_from_traversal(size_t num_variants, const std::vector<size_t> &traversed_nodes,
                                            const std::map<size_t, std::vector<std::pair<size_t, uint8_t>>> &node_to_alleles);
struct HaplotypeAssignment {
    Cyp2d6RegionLabel label;                              // Unknown when ambiguous and not forced
    std::optional<std::vector<RegionVariant>> variants;   // None for Unknown
    size_t vi_match = 0, all_match = 0;                   // best_score
};
// :470-601 for a batch of observed vectors: K6 scores every (vector, haplotype) pair on the GPU, the host keeps the
// reference's arg-max over (vi_match, all_match) in BTreeMap order, its tie handling (sorted by full_allele, first one
// if force_assignment else Unknown) and the RegionVariant list.  haplotype_lookup: star allele -> 0/1 vector.
std::vector<HaplotypeAssignment> assign_haplotypes_from_alleles(GpuAligner &gpu, const std::vector<std::vector<uint8_t>> &alleles,
                                                                const std::map<std::string, std::vector<uint8_t>> &haplotype_lookup,
                                                                const std::vector<VariantMetadata> &variants, bool force_assignment);

struct Cyp2d6Config {  // the members of src/cyp2d6/definitions.rs:128-336 the chaining code reads
    std::map<std::string, std::string> cyp_translate;
    std::set<std::pair<std::string, std::string>> inferred_connections;
    std::set<std::string> unexpected_singletons;
    static Cyp2d6Config default_config();
};

enum class Cyp2d6DetailLevel { CoreAlleles, SubAlleles, DeepAlleles };
// src/cyp2d6/caller.rs:907-957
std::string convert_chain_to_hap(const std::vector<size_t> &chain, const std::vector<Cyp2d6Region> &hap_regions,
                                 Cyp2d6DetailLevel level, const std::map<std::string, std::string> &cyp_translate);

using SequenceWeights = std::vector<std::pair<size_t, double>>;  // src/cyp2d6/chaining.rs:18
// weight_sequence (src/cyp2d6/chaining.rs:28-103) for a batch of read segments against all consensuses: one K3 span
// launch instead of one aligner per segment.  Result[s] is empty when the best hit misses more than 5 % (:96-102).
std::vector<SequenceWeights> weight_sequences(GpuAligner &gpu, const SeqList &segments, const SeqList &consensuses,
                                              const std::vector<Cyp2d6Region> &con_regions);

struct ChainBuild {  // src/cyp2d6/caller.rs:430-537
    std::map<std::string, std::vector<std::vector<size_t>>> qname_chains;
    std::map<std::string, std::vector<SequenceWeights>> qname_chain_scores;
    std::vector<size_t> best_allele_mapping_counts;
};
// read_weights[qname] = weight_sequence result per region of the read, read order (empty = region skipped)
ChainBuild build_chains(const std::map<std::string, std::vector<SequenceWeights>> &read_weights, size_t n_haps);

struct ChainPenalties {  // src/cyp2d6/chaining.rs:107-139
    double lasso_penalty = 4.0, ln_ed_penalty = 2.0, unexpected_chain_penalty = 10.0, inferred_edge_penalty = 2.0;
};
struct ChainPairResult {
    std::vector<std::vector<size_t>> best_chains;  // two chains, sorted
    std::vector<std::string> dangling_alleles;      // CallerWarning::DanglingAllele names
    double score = 0.0;
    size_t index1 = 0, index2 = 0, n_possible_chains = 0, n_full_evaluations = 0;
    uint64_t edit_distance = 0;
};
struct NoChainingHead : HostError { NoChainingHead() : HostError("NoChainingHead") {} };
struct NoChainsFound : HostError { NoChainsFound() : HostError("NoChainsFound") {} };
struct NoScorePairs : HostError { NoScorePairs() : HostError("NoScorePairs") {} };
// src/cyp2d6/chaining.rs:223-592.  The integer ED term of every chain pair comes from the GPU (chain windows + K2);
// pairs are then visited in increasing lower bound (all other terms are >= 0) and the float terms (hap weights ->
// multinomial) are evaluated only until the bound passes the best score: the same arg-min (score, i, j) as the
// reference's exhaustive loop with its 10-entry heap.
ChainPairResult find_best_chain_pair(GpuAligner &gpu, const Cyp2d6Config &cfg,
                                     const std::map<std::string, std::vector<std::vector<size_t>>> &obs_chains,
                                     const std::map<std::string, std::vector<SequenceWeights>> &chain_scores,
                                     const std::vector<Cyp2d6Region> &hap_regions, bool infer_connections, bool normalize_all_alleles,
                                     const ChainPenalties &penalties, bool ignore_chain_label_limits);

struct Cyp2d6ReadRegion {
    size_t start = 0, end = 0;  // coordinates in the read of the extracted sequence
    std::string sequence;
};
struct Cyp2d6Call {
    ChainPairResult chain_pair;
    Diplotype diplotype, simple_diplotype, deep_diplotype;
    std::vector<Cyp2d6Region> hap_regions;  // after FalseAllele marking
    Json multi_mapping_details = Json::array();
    Json gene_details() const;  // PgxGeneDetails::new_from_multi_mappings, src/data_types/starphase_json.rs:169-188
};
// the chaining half of diplotype_cyp2d6 (src/cyp2d6/caller.rs:430-739): weights, chains, false alleles, best pair, strings
Cyp2d6Call call_cyp2d6_chains(GpuAligner &gpu, const Cyp2d6Config &cfg, const SeqList &consensuses,
                              std::vector<Cyp2d6Region> hap_regions,
                              const std::map<std::string, std::vector<Cyp2d6ReadRegion>> &regions_of_interest,
                              bool infer_connections, bool normalize_all_alleles);

// cyp2d6_alleles.json (DeeplotypeDebug, src/cyp2d6/debug.rs:8-71): the three forms of both haplotypes + the variants of every typed allele
std::string cyp2d6_alleles_json(const std::vector<std::vector<size_t>> &best_diplotype_indices, const std::vector<Cyp2d6Region> &hap_regions,
                                const std::map<std::string, std::string> &cyp_translate);

// ------------------------------------------------------------------------------------------
// variant graph typing (row N3 of SURVEY.md 8f) -- what assign_haplotype gets from hiphase's WFAGraph
// (src/cyp2d6/haplotyper.rs:430-468): graph of the backbone with one bubble per variant, end-to-end edit distance of a consensus
// (forward DP on the device, K8), the nodes on optimal alignments, and from them the 0 / 1 / 2 / 3 allele vector K6 scores.
// ------------------------------------------------------------------------------------------
struct GraphVariant {  // position in reference coordinates, VCF-style alleles; the order of the list defines the variant indices
    size_t position = 0;
    std::string ref_allele, alt_allele;
};
struct VariantGraph {
    std::vector<std::string> seqs;            // node sequences (only the unlabelled source / sink may be empty)
    std::vector<std::vector<size_t>> preds;   // predecessor nodes
    std::vector<size_t> coord;                // backbone offset at which the node starts
    std::map<size_t, std::vector<std::pair<size_t, uint8_t>>> node_to_alleles;  // NodeAlleleMap of the reference (:431)
    size_t sink = 0;
    // WFAGraph::from_reference_variants(chrom_seq, variants, start, end) (:432-441): backbone = reference[region_start, +len)
    static VariantGraph from_reference_variants(const std::string &backbone, size_t region_start, const std::vector<GraphVariant> &variants);
    size_t get_num_nodes() const { return seqs.size(); }
    size_t add(std::string seq, std::vector<size_t> preds, size_t coord);
};
struct GraphAlignment {  // WFAResult: score() and traversed_nodes()
    bool found = false;   // false: the band excluded every path
    size_t score = 0;
    std::vector<size_t> traversed_nodes;
};
// what assign_haplotype reads from the config, the reference genome and the database (src/cyp2d6/haplotyper.rs:40-130, :371-452)
struct Cyp2d6TypingDb {
    std::string backbone;                 // reference[backbone_start, backbone_start + |backbone|): cyp_coordinates["CYP2D6_wfa_backbone"]
    size_t backbone_start = 0;
    std::vector<GraphVariant> variants;   // loaded_variants.ordered_variants(), reference coordinates
    std::vector<VariantMetadata> metadata;                            // same order
    std::map<std::string, std::vector<uint8_t>> haplotype_lookup;     // star allele -> 0/1 vector (:40-70)
    std::vector<Cyp2d6RegionLabel> mapped_hybrids;                    // labels that go through deep genotyping (:117-124)
};
// edit_distance_with_pruning for a batch: one (graph, sequence) problem per entry, one device call
std::vector<GraphAlignment> graph_edit_distance(GpuAligner &gpu, const std::vector<const VariantGraph *> &graphs, const SeqList &sequences,
                                                size_t band = 128);
// :452-468: the allele of every variant from the traversed nodes (3 unset, 2 both alleles on optimal alignments)
std::vector<uint8_t> graph_alleles(const VariantGraph &g, const GraphAlignment &aln, size_t num_variants);

// ------------------------------------------------------------------------------------------
// consensus (row N1 of SURVEY.md 8f) -- the interface of waffle_con's ConsensusDWFA / DualConsensusDWFA as the reference uses it
// (src/hla/caller.rs:1097-1219, :727-755), the per-read extension step on the device (K7, sp_consensus_extend), the search policy
// here.  The policy restates the published outline of waffle_con's search, not its code (DESIGN.md 3: parity unpinned).
// ------------------------------------------------------------------------------------------
struct CdwfaConfig {  // the members the reference sets at src/hla/caller.rs:1103-1116
    size_t min_count = 3;
    double min_af = 0.10;
    bool allow_early_termination = false;
    size_t max_queue_size = 20;
    size_t max_capacity_per_size = 10;
    size_t offset_window = 0;
    size_t band = 32;  // rows either side of a read's diagonal kept on the device (HiFi drift); widened by offset_window / 2
    // accepted for interface compatibility, not modelled: dual_max_ed_delta, weighted_by_ed (the reference sets false),
    // consensus_cost (the reference sets L1Distance, which is what is implemented), offset_compare_length
    size_t dual_max_ed_delta = 20;
};
struct Consensus {  // waffle_con::consensus::Consensus
    std::string sequence;
    std::vector<size_t> scores;  // per read, in insertion order
};
struct DualConsensus {  // waffle_con::dual_consensus::DualConsensus
    std::string consensus1;
    std::optional<std::string> consensus2;
    std::vector<bool> is_consensus1;
    std::vector<std::optional<size_t>> scores1, scores2;
    bool is_dual() const { return consensus2.has_value(); }
};
// the outcome of one search of a batch: its solutions, or the message of the HostError its consensus() would throw
template <typename T>
struct SearchResult {
    std::vector<T> list;
    std::optional<std::string> error;
};
class ConsensusDWFA {
  public:
    ConsensusDWFA(GpuAligner &gpu, CdwfaConfig config) : gpu_(gpu), config_(config) {}
    void add_sequence(const std::string &sequence) { add_sequence_offset(sequence, std::nullopt); }
    void add_sequence_offset(const std::string &sequence, std::optional<size_t> offset);
    std::vector<Consensus> consensus();  // every best solution, first = the one the reference takes
    // independent searches on one GpuAligner, their device calls gathered: each round of the batch is at most one
    // sp_consensus_extend_batch and one sp_consensus_run_batch for all searches still running.  result[i] is what
    // searches[i]->consensus() returns or throws; a failed device call throws for the whole batch.
    static std::vector<SearchResult<Consensus>> consensus_batch(const std::vector<ConsensusDWFA *> &searches);
    size_t n_extension_calls() const { return n_calls_; }

  protected:
    friend class DualConsensusDWFA;
    GpuAligner &gpu_;
    CdwfaConfig config_;
    SeqList reads_;
    std::vector<int32_t> offsets_;
    size_t n_calls_ = 0;
};
class DualConsensusDWFA {
  public:
    DualConsensusDWFA(GpuAligner &gpu, CdwfaConfig config) : inner_(gpu, config) {}
    void add_sequence(const std::string &sequence) { inner_.add_sequence(sequence); }
    void add_sequence_offset(const std::string &sequence, std::optional<size_t> offset) { inner_.add_sequence_offset(sequence, offset); }
    std::vector<DualConsensus> consensus();
    static std::vector<SearchResult<DualConsensus>> consensus_batch(const std::vector<DualConsensusDWFA *> &searches);  // as ConsensusDWFA's
    size_t n_extension_calls() const { return inner_.n_calls_; }

  private:
    ConsensusDWFA inner_;
};

// waffle_con's PriorityConsensusDWFA as the CYP2D6 caller drives it (src/cyp2d6/caller.rs:145-280): every input is a chain of
// representations of one read segment (there: homopolymer-compressed first, then the raw bases), an offset per level and an
// optional seed; the result groups the inputs and gives every group one consensus per level.  Restated outline (parity unpinned,
// DESIGN.md 4.7): inputs with different seeds never share a group; a group is examined level by level with DualConsensusDWFA -- a
// dual answer splits it in two (both halves are examined again at the same level), a single answer moves it to the next level,
// after the last level it is final; groups come out ordered by their smallest input index.
struct PriorityConsensus {
    std::vector<std::vector<Consensus>> consensuses;  // [group][level]; scores in the order of the group's members
    std::vector<size_t> sequence_indices;             // group of every input, in insertion order
};
class PriorityConsensusDWFA {
  public:
    PriorityConsensusDWFA(GpuAligner &gpu, CdwfaConfig config) : gpu_(gpu), config_(config) {}
    void add_seeded_sequence_chain(const std::vector<std::string> &sequence_chain, const std::vector<std::optional<size_t>> &offset_chain,
                                   std::optional<uint64_t> seed);
    size_t n_sequences() const { return chains_.size(); }
    PriorityConsensus consensus();

  private:
    GpuAligner &gpu_;
    CdwfaConfig config_;
    std::vector<std::vector<std::string>> chains_;
    std::vector<std::vector<std::optional<size_t>>> offsets_;
    std::vector<std::optional<uint64_t>> seeds_;
};

// ---- the consensus step of the HLA caller (src/hla/caller.rs:1097-1247) ----
// dwfa_config_from_cli (:1097-1116): min_count / min_af / dual_max_ed_delta from the CLI, queue 20, capacity 10, offset_window 400
CdwfaConfig dwfa_config_from_cli(const DiplotypeSettings &cli_settings, bool allow_early_termination);
// is_passing_dual on a DualConsensus (:1225-1247): counts from is_consensus1
DualPassingStats is_passing_dual(const DualConsensus &dual_consensus, const DiplotypeSettings &cli_settings);
// run_dual_consensus (:1126-1139): segments in key order, first solution
DualConsensus run_dual_consensus(GpuAligner &gpu, const std::map<std::string, std::string> &segments, const DiplotypeSettings &cli_settings);
// run_dual_consensus_with_offsets (:1151-1219): on the homopolymer-compressed sequences first (offsets relative to the smallest,
// + half the window; the smallest itself anchored); when that result does not pass is_passing_dual, on the full-length DNA
DualConsensus run_dual_consensus_with_offsets(GpuAligner &gpu, const std::map<std::string, RealignmentResult> &segments,
                                              const DiplotypeSettings &cli_settings);
// the re-consensus of the two read groups on full-length DNA (:706-760): (consensus 1, consensus 2 or nullopt); a group whose
// consensus fails comes back as the empty string (tagged unknown downstream)
std::pair<std::string, std::optional<std::string>> consensus_per_group(GpuAligner &gpu, const std::map<std::string, RealignmentResult> &segments,
                                                                       const std::vector<bool> &is_consensus1, bool is_dual,
                                                                       const DiplotypeSettings &cli_settings);

// ---- the consensus stage of the CYP2D6 caller (src/cyp2d6/caller.rs:145-310, :750-893) ----
// hpc_with_guide (src/util/homopolymers.rs:53-64): (homopolymer-compressed sequence, position of guide_offset in the compressed guide)
std::pair<std::string, size_t> hpc_with_guide(const std::string &sequence, const std::string &guide_sequence, size_t guide_offset);
// the CdwfaConfig of :149-162 ('*' wildcard, early termination, queue 20, capacity 10, offset_window 2 x 50)
CdwfaConfig cyp2d6_consensus_config(const DiplotypeSettings &cli_settings);
// what the loop at :168-212 collects from the regions of interest, in BTreeMap order of the read ids
struct Cyp2d6ConsensusInputs {
    SeqList raw_sequences;            // the part of the read matching the region
    SeqList hpc_sequences;            // its homopolymer-compressed form
    std::vector<size_t> base_offsets, hpc_offsets;  // 0 = anchored at the start; else clipped template start (+ offset_window)
    std::vector<std::string> sequence_ids;          // "{read_id}_{start}_{end}_{allele_label}"
    std::vector<std::pair<std::string, AlleleMapping>> flattened_regions_of_interest;
    std::vector<std::optional<uint64_t>> seeds;     // :224-231: *5, REP6, REP7, spacer and link regions never share a group
};
Cyp2d6ConsensusInputs cyp2d6_consensus_inputs(const std::map<std::string, std::string> &read_sequences,
                                              const std::map<std::string, std::vector<AlleleMapping>> &regions_of_interest,
                                              const Cyp2d6Extractor &d6_typer, double max_missing_consensus_frac, size_t offset_window = 50);
// :163-262 + :283: the priority chain (HPC first, then the raw bases) over those inputs
PriorityConsensus cyp2d6_priority_consensus(GpuAligner &gpu, const Cyp2d6ConsensusInputs &inputs, const CdwfaConfig &config);
struct MultiConsensus {  // waffle_con::multi_consensus::MultiConsensus
    std::vector<Consensus> consensuses;
    std::vector<size_t> sequence_indices;
};
// merge_consensus_results (:750-893): consensuses with the same HPC form and the same (sub-allele) type become one -- typed with
// find_full_type_in_sequences (K4 / K9 / K8 / K6), merged groups re-solved with ConsensusDWFA on the raw sequences (K7); groups
// that cannot be typed join the single typed group with their HPC form, or stay an UNKNOWN pile (none), or are emptied (several)
MultiConsensus merge_consensus_results(GpuAligner &gpu, const SeqList &sequences, const std::vector<size_t> &offsets,
                                       const CdwfaConfig &cdwfa_config, const PriorityConsensus &raw_consensus_result,
                                       Cyp2d6Extractor &d6_typer, const Cyp2d6TypingDb &db, const Cyp2d6Config &cyp2d6_config,
                                       double max_missing_consensus_frac);

// StarphaseJson, src/data_types/starphase_json.rs:13-21; metadata order of src/database/pgx_database.rs:359-371
std::string starphase_json(const std::string &pbstarphase_version, const std::map<std::string, std::string> &database_metadata,
                           const std::map<std::string, Json> &gene_details);

}  // namespace starphase
