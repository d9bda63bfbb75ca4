// sp_host_py.cpp -- pybind11 view of the C++ host (module pb_starphase_b200._starphase_host) so that the parity
// tests can drive the same functions a C++ host would call.  No logic here.
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include "starphase_host.hpp"

namespace py = pybind11;
using namespace starphase;

static HlaDatabase make_db(const std::vector<std::tuple<std::string, std::string, std::vector<std::string>, std::optional<std::string>, std::string>> &rows) {
    HlaDatabase db;
    for (const auto &r : rows) {
        HlaAlleleDefinition d;
        d.hla_id = std::get<0>(r); d.gene_name = std::get<1>(r); d.star_allele = std::get<2>(r);
        d.dna_sequence = std::get<3>(r); d.cdna_sequence = std::get<4>(r);
        db.emplace(d.hla_id, std::move(d));
    }
    return db;
}

static std::vector<Cyp2d6Region> make_regions(const std::vector<std::tuple<std::string, std::optional<std::string>, std::optional<size_t>>> &rows) {
    std::vector<Cyp2d6Region> out;
    for (const auto &r : rows) {
        Cyp2d6Region g;
        g.label.region_type = region_type_from_name(std::get<0>(r));
        g.label.subtype_label = std::get<1>(r);
        g.unique_id = std::get<2>(r);
        out.push_back(std::move(g));
    }
    return out;
}

PYBIND11_MODULE(_starphase_host, m) {
    m.doc() = "C++ host mirror of pb-StarPhase's hot-path interface above libstarphase_gpu.so";
    py::register_exception<HostError>(m, "HostError");
    py::register_exception<NoChainingHead>(m, "NoChainingHead", m.attr("HostError").ptr());
    py::register_exception<NoChainsFound>(m, "NoChainsFound", m.attr("HostError").ptr());
    py::register_exception<NoScorePairs>(m, "NoScorePairs", m.attr("HostError").ptr());

    py::class_<Json>(m, "Json").def("pretty", [](const Json &j) { return j.pretty(); });

    // variant graph typing (K8 forward + marking pass): (backbone, region_start, [(pos, ref, alt)], sequences, band)
    m.def("graph_typing", [](GpuAligner &g, const std::string &backbone, size_t region_start,
                             const std::vector<std::tuple<size_t, std::string, std::string>> &variants, const SeqList &sequences, size_t band) {
        std::vector<GraphVariant> vs;
        for (const auto &v : variants) vs.push_back({std::get<0>(v), std::get<1>(v), std::get<2>(v)});
        const VariantGraph graph = VariantGraph::from_reference_variants(backbone, region_start, vs);
        std::vector<const VariantGraph *> gs(sequences.size(), &graph);
        py::list out;
        for (const GraphAlignment &a : graph_edit_distance(g, gs, sequences, band))
            out.append(py::make_tuple(a.found, a.score, a.traversed_nodes, graph_alleles(graph, a, vs.size())));
        py::list nodes;
        for (size_t k = 0; k < graph.seqs.size(); ++k) nodes.append(py::make_tuple(py::bytes(graph.seqs[k]), graph.preds[k], graph.coord[k]));
        return py::make_tuple(out, nodes, graph.node_to_alleles, graph.sink);
    });

    // consensus (K7 + host search): (sequences, offsets or None, config dict) -> solutions
    auto cfg_from = [](const py::dict &d) {
        CdwfaConfig c;
        if (d.contains("min_count")) c.min_count = d["min_count"].cast<size_t>();
        if (d.contains("min_af")) c.min_af = d["min_af"].cast<double>();
        if (d.contains("allow_early_termination")) c.allow_early_termination = d["allow_early_termination"].cast<bool>();
        if (d.contains("max_queue_size")) c.max_queue_size = d["max_queue_size"].cast<size_t>();
        if (d.contains("max_capacity_per_size")) c.max_capacity_per_size = d["max_capacity_per_size"].cast<size_t>();
        if (d.contains("offset_window")) c.offset_window = d["offset_window"].cast<size_t>();
        if (d.contains("band")) c.band = d["band"].cast<size_t>();
        return c;
    };
    m.def("consensus", [cfg_from](GpuAligner &g, const SeqList &reads, const std::vector<std::optional<size_t>> &offsets, const py::dict &cfg) {
        ConsensusDWFA c(g, cfg_from(cfg));
        for (size_t r = 0; r < reads.size(); ++r) c.add_sequence_offset(reads[r], r < offsets.size() ? offsets[r] : std::nullopt);
        py::list out;
        for (const Consensus &s : c.consensus()) out.append(py::make_tuple(py::bytes(s.sequence), s.scores));
        return py::make_tuple(out, c.n_extension_calls());
    });
    // priority consensus: chains[i] = the representations of input i (e.g. HPC, raw), offsets[i] one per level (None = anchored),
    // seeds[i] or None -> (consensuses[group][level] = (sequence, scores), group of every input)
    m.def("priority_consensus", [cfg_from](GpuAligner &g, const std::vector<std::vector<std::string>> &chains,
                                           const std::vector<std::vector<std::optional<size_t>>> &offsets,
                                           const std::vector<std::optional<uint64_t>> &seeds, const py::dict &cfg) {
        PriorityConsensusDWFA p(g, cfg_from(cfg));
        for (size_t i = 0; i < chains.size(); ++i) p.add_seeded_sequence_chain(chains[i], offsets[i], seeds[i]);
        const PriorityConsensus r = p.consensus();
        py::list groups;
        for (const auto &levels : r.consensuses) {
            py::list one;
            for (const Consensus &c : levels) one.append(py::make_tuple(py::bytes(c.sequence), c.scores));
            groups.append(one);
        }
        return py::make_tuple(groups, r.sequence_indices);
    });
    m.def("dual_consensus", [cfg_from](GpuAligner &g, const SeqList &reads, const std::vector<std::optional<size_t>> &offsets, const py::dict &cfg) {
        DualConsensusDWFA c(g, cfg_from(cfg));
        for (size_t r = 0; r < reads.size(); ++r) c.add_sequence_offset(reads[r], r < offsets.size() ? offsets[r] : std::nullopt);
        py::list out;
        for (const DualConsensus &s : c.consensus()) {
            py::dict d;
            d["consensus1"] = py::bytes(s.consensus1);
            d["consensus2"] = s.consensus2 ? py::object(py::bytes(*s.consensus2)) : py::object(py::none());
            d["is_consensus1"] = s.is_consensus1;
            d["scores1"] = s.scores1;
            d["scores2"] = s.scores2;
            out.append(d);
        }
        return py::make_tuple(out, c.n_extension_calls());
    });
    // many independent searches in one batch: groups = [(sequences, offsets)] -> per group (solutions, device calls, error or None)
    // as consensus / dual_consensus return them, with the message of a failed search instead of an exception
    using Groups = std::vector<std::pair<SeqList, std::vector<std::optional<size_t>>>>;
    m.def("consensus_batch", [cfg_from](GpuAligner &g, const Groups &groups, const py::dict &cfg) {
        std::vector<std::unique_ptr<ConsensusDWFA>> own;
        std::vector<ConsensusDWFA *> batch;
        for (const auto &grp : groups) {
            own.push_back(std::make_unique<ConsensusDWFA>(g, cfg_from(cfg)));
            for (size_t r = 0; r < grp.first.size(); ++r) own.back()->add_sequence_offset(grp.first[r], r < grp.second.size() ? grp.second[r] : std::nullopt);
            batch.push_back(own.back().get());
        }
        const auto results = ConsensusDWFA::consensus_batch(batch);
        py::list out;
        for (size_t k = 0; k < results.size(); ++k) {
            py::list sols;
            for (const Consensus &s : results[k].list) sols.append(py::make_tuple(py::bytes(s.sequence), s.scores));
            out.append(py::make_tuple(sols, batch[k]->n_extension_calls(), results[k].error ? py::object(py::str(*results[k].error)) : py::object(py::none())));
        }
        return out;
    });
    m.def("dual_consensus_batch", [cfg_from](GpuAligner &g, const Groups &groups, const py::dict &cfg) {
        std::vector<std::unique_ptr<DualConsensusDWFA>> own;
        std::vector<DualConsensusDWFA *> batch;
        for (const auto &grp : groups) {
            own.push_back(std::make_unique<DualConsensusDWFA>(g, cfg_from(cfg)));
            for (size_t r = 0; r < grp.first.size(); ++r) own.back()->add_sequence_offset(grp.first[r], r < grp.second.size() ? grp.second[r] : std::nullopt);
            batch.push_back(own.back().get());
        }
        const auto results = DualConsensusDWFA::consensus_batch(batch);
        py::list out;
        for (size_t k = 0; k < results.size(); ++k) {
            py::list sols;
            for (const DualConsensus &s : results[k].list) {
                py::dict d;
                d["consensus1"] = py::bytes(s.consensus1);
                d["consensus2"] = s.consensus2 ? py::object(py::bytes(*s.consensus2)) : py::object(py::none());
                d["is_consensus1"] = s.is_consensus1;
                d["scores1"] = s.scores1;
                d["scores2"] = s.scores2;
                sols.append(d);
            }
            out.append(py::make_tuple(sols, batch[k]->n_extension_calls(), results[k].error ? py::object(py::str(*results[k].error)) : py::object(py::none())));
        }
        return out;
    });

    py::class_<MappingStats>(m, "MappingStats")
        .def(py::init<size_t, size_t, size_t>())
        .def_readwrite("seq_len", &MappingStats::seq_len)
        .def_readwrite("nm", &MappingStats::nm)
        .def_readwrite("unmapped", &MappingStats::unmapped)
        .def("custom_score", &MappingStats::custom_score)
        .def("mapping_score", &MappingStats::mapping_score)
        .def("as_tuple", [](const MappingStats &s) { return std::make_tuple(s.seq_len, s.nm, s.unmapped); });

    py::class_<HlaMappingStats>(m, "HlaMappingStats")
        .def(py::init<>())
        .def_readwrite("cdna_stats", &HlaMappingStats::cdna_stats)
        .def_readwrite("dna_stats", &HlaMappingStats::dna_stats)
        .def("mapping_score", &HlaMappingStats::mapping_score)
        .def("to_json", &HlaMappingStats::to_json);

    py::class_<Mapping>(m, "Mapping")
        .def(py::init([](size_t qs, size_t qe, size_t ql, size_t ts, size_t te, size_t tl, size_t nm, bool fwd,
                         std::vector<std::pair<uint32_t, uint8_t>> cigar) {
                 Mapping x;
                 x.query_start = qs; x.query_end = qe; x.query_len = ql; x.target_start = ts; x.target_end = te; x.target_len = tl;
                 x.nm = nm; x.forward = fwd; x.cigar = std::move(cigar);
                 return x;
             }),
             py::arg("query_start"), py::arg("query_end"), py::arg("query_len"), py::arg("target_start"), py::arg("target_end"),
             py::arg("target_len"), py::arg("nm"), py::arg("forward") = true, py::arg("cigar") = std::vector<std::pair<uint32_t, uint8_t>>());

    m.def("select_best_mapping", [](const std::vector<Mapping> &ms, bool from_target, bool pen, std::optional<size_t> ov) {
        auto r = select_best_mapping(ms, from_target, pen, ov);
        return std::make_pair(r.first, std::make_tuple(r.second.seq_len, r.second.nm, r.second.unmapped));
    }, py::arg("mappings"), py::arg("unmapped_from_target"), py::arg("penalize_unmapped"), py::arg("base_length_override") = std::nullopt);
    m.def("process_mm_cigar", &process_mm_cigar);
    m.def("dp_score", &dp_score, py::arg("cigar"), py::arg("match_score") = 5);

    py::class_<HlaProcessedMatch>(m, "HlaProcessedMatch")
        .def(py::init<std::string>())
        .def_static("worst_match", &HlaProcessedMatch::worst_match)
        .def("add_mapping", &HlaProcessedMatch::add_mapping)
        .def("is_better_match", &HlaProcessedMatch::is_better_match)
        .def("haplotype", &HlaProcessedMatch::haplotype)
        .def("processed_cigars", &HlaProcessedMatch::processed_cigars)
        .def("processed_ranges", &HlaProcessedMatch::processed_ranges);

    m.def("ln_gamma", &ln_gamma);
    m.def("ln_factorial", &ln_factorial);
    m.def("multinomial_ln_pmf", &multinomial_ln_pmf);
    m.def("binomial_cdf", &binomial_cdf);
    m.def("is_passing_dual", static_cast<bool (*)(size_t, size_t, double, double, double)>(&is_passing_dual), py::arg("counts1"), py::arg("counts2"), py::arg("min_consensus_fraction") = 0.10,
          py::arg("min_cdf") = 0.001, py::arg("expected_maf") = 0.45);

    m.def("beta_reg", &beta_reg);
    m.def("binomial_ln_pmf", &binomial_ln_pmf);
    m.def("normal_ln_pdf", &normal_ln_pdf);
    m.def("json_f64", [](double v) { return Json::number(v).pretty(); });
    m.def("dual_passing_stats_json", [](bool is_dual, size_t c1, size_t c2, double min_fraction, double min_cdf, double expected_maf) {
        return dual_passing_stats(is_dual, c1, c2, min_fraction, min_cdf, expected_maf).to_json().pretty();
    }, py::arg("is_dual"), py::arg("counts1"), py::arg("counts2"), py::arg("min_consensus_fraction") = 0.10, py::arg("min_cdf") = 0.001,
          py::arg("expected_maf") = 0.45);
    m.def("is_hemizygous_better", &is_hemizygous_better, py::arg("scores1"), py::arg("scores2"), py::arg("is_consensus1"), py::arg("is_dual"),
          py::arg("dual_max_ed_delta"), py::arg("normalized_coverage"));
    m.def("cigar_string", &cigar_string);
    m.def("md_string", &md_string, py::arg("cigar"), py::arg("target"), py::arg("target_start"), py::arg("query"), py::arg("query_start"));
    m.def("reverse_complement", &reverse_complement);
    m.def("is_allowed_allele_def", [](const std::string &def_gene, bool has_dna, const std::string &gene_name, bool hla_require_dna) {
        HlaAlleleDefinition d;
        d.hla_id = "HLA1"; d.gene_name = def_gene; d.cdna_sequence = "AG";
        if (has_dna) d.dna_sequence = "ACGT";
        DiplotypeSettings s;
        s.hla_require_dna = hla_require_dna;
        return is_allowed_allele_def(d, gene_name, s);
    });
    m.def("splice_read", &splice_read, py::arg("sequence"), py::arg("pos"), py::arg("cigar"), py::arg("exons"));
    m.def("prepare_score_read_targets", [](const std::string &seq, int64_t pos, const std::vector<std::pair<uint32_t, uint8_t>> &cigar,
                                           const std::vector<std::pair<uint64_t, uint64_t>> &exons, bool fwd, const DiplotypeSettings &s) {
        const ScoreReadTargets t = prepare_score_read_targets(seq, pos, cigar, exons, fwd, s);
        return py::make_tuple(t.dna_target, t.cdna_target);
    });

    py::class_<DiplotypeSettings>(m, "DiplotypeSettings")
        .def(py::init<>())
        .def_readwrite("disable_cdna_scoring", &DiplotypeSettings::disable_cdna_scoring)
        .def_readwrite("hla_require_dna", &DiplotypeSettings::hla_require_dna)
        .def_readwrite("min_consensus_fraction", &DiplotypeSettings::min_consensus_fraction)
        .def_readwrite("min_cdf", &DiplotypeSettings::min_cdf)
        .def_readwrite("expected_maf", &DiplotypeSettings::expected_maf)
        .def_readwrite("min_dp_score", &DiplotypeSettings::min_dp_score)
        .def_readwrite("min_consensus_count", &DiplotypeSettings::min_consensus_count)
        .def_readwrite("dual_max_ed_delta", &DiplotypeSettings::dual_max_ed_delta);

    // the consensus step of the HLA caller: records = (qname, dna_sequence, hpc_sequence, dna_offset, hpc_offset), taken in qname order
    // -> (dual consensus of run_dual_consensus_with_offsets, is_passing, (consensus 1, consensus 2 or None) of the per-group re-consensus)
    m.def("hla_consensus_step", [](GpuAligner &g, const std::vector<std::tuple<std::string, std::string, std::string, size_t, size_t>> &records,
                                   const DiplotypeSettings &s) {
        std::map<std::string, RealignmentResult> segs;
        for (const auto &r : records) {
            RealignmentResult rr;
            RealignedHlaRecord rec;
            rec.dna_sequence = std::get<1>(r); rec.hpc_sequence = std::get<2>(r); rec.dna_offset = std::get<3>(r); rec.hpc_offset = std::get<4>(r);
            rr.realigned_record = rec;
            segs[std::get<0>(r)] = rr;
        }
        const DualConsensus d = run_dual_consensus_with_offsets(g, segs, s);
        py::dict out;
        out["consensus1"] = py::bytes(d.consensus1);
        out["consensus2"] = d.consensus2 ? py::object(py::bytes(*d.consensus2)) : py::object(py::none());
        out["is_consensus1"] = d.is_consensus1;
        out["scores1"] = d.scores1;
        out["scores2"] = d.scores2;
        const auto groups = consensus_per_group(g, segs, d.is_consensus1, d.is_dual(), s);
        py::object g2 = groups.second ? py::object(py::bytes(*groups.second)) : py::object(py::none());
        return py::make_tuple(out, is_passing_dual(d, s).is_passing, py::make_tuple(py::bytes(groups.first), g2));
    });

    // the process-wide aligner stand-ins (starphase_host.hpp): stand_ins() reads them, set_stand_ins(name=value, ...) changes them
    m.def("stand_ins", []() {
        const AlignerStandIns &s = aligner_stand_ins();
        py::dict d;
        d["min_dp_score"] = s.min_dp_score; d["no_mapping_permille"] = s.no_mapping_permille;
        d["candidate_edit_weight"] = s.candidate_edit_weight; d["template_half_prefilter"] = s.template_half_prefilter;
        d["affine_refine"] = s.affine_refine;
        return d;
    });
    m.def("set_stand_ins", [](const py::kwargs &kw) {
        AlignerStandIns &s = aligner_stand_ins();
        for (auto item : kw) {
            const std::string k = py::cast<std::string>(item.first);
            if (k == "min_dp_score") s.min_dp_score = py::cast<long>(item.second);
            else if (k == "no_mapping_permille") s.no_mapping_permille = py::cast<int>(item.second);
            else if (k == "candidate_edit_weight") s.candidate_edit_weight = py::cast<int>(item.second);
            else if (k == "template_half_prefilter") s.template_half_prefilter = py::cast<bool>(item.second);
            else if (k == "affine_refine") s.affine_refine = py::cast<bool>(item.second);
            else throw std::invalid_argument("set_stand_ins: unknown setting " + k);
        }
    });

    py::class_<GpuAligner>(m, "GpuAligner")
        .def(py::init<int>(), py::arg("device") = 0)
        .def("score_batch", [](GpuAligner &g, const SeqList &t, const SeqList &p) { return g.score_batch(t, p); })
        .def("launch_count", &GpuAligner::launch_count)
        .def("share_device", &GpuAligner::share_device, py::arg("on") = true)
        .def("align_pairs", [](GpuAligner &g, const SeqList &t, const SeqList &p, const std::vector<std::pair<int32_t, int32_t>> &pairs, int match_score) {
            py::list out;
            for (const Alignment &a : g.align_pairs(t, p, pairs, nullptr, match_score)) {
                py::dict d;
                d["dist"] = a.dist; d["nm"] = a.nm; d["p_start"] = a.p_start; d["p_end"] = a.p_end; d["t_start"] = a.t_start; d["t_end"] = a.t_end;
                d["score"] = a.score; d["refined"] = a.refined;
                py::list c;
                for (const auto &e : a.cigar) c.append(py::make_tuple(e.first, static_cast<int>(e.second)));
                d["cigar"] = c;
                out.append(d);
            }
            return out;
        }, py::arg("texts"), py::arg("patterns"), py::arg("pairs"), py::arg("match_score") = 0);

    // ---- HLA ----
    using DbRows = std::vector<std::tuple<std::string, std::string, std::vector<std::string>, std::optional<std::string>, std::string>>;
    m.def("score_read", [](GpuAligner &g, const std::string &dna_target, const std::string &cdna_target, const DbRows &rows,
                           const std::string &gene, const DiplotypeSettings &s) {
        const HlaDatabase db = make_db(rows);
        ScoreReadResult r = score_read(g, dna_target, cdna_target, db, gene, s);
        py::dict stats;
        for (const auto &kv : r.stats) {
            auto tup = [](const std::optional<MappingStats> &x) -> py::object {
                if (!x) return py::none();
                return py::make_tuple(x->seq_len, x->nm, x->unmapped);
            };
            stats[py::str(kv.first)] = py::make_tuple(tup(kv.second.cdna_stats), tup(kv.second.dna_stats));
        }
        return py::make_tuple(stats, r.best_hla_id, r.best_star_allele);
    });
    m.def("score_consensus", [](GpuAligner &g, const std::string &reference_sequence, int64_t ref_start, const std::string &consensus,
                                const DbRows &rows, const std::string &gene, const std::vector<std::pair<uint64_t, uint64_t>> &exons,
                                bool is_forward_strand, const DiplotypeSettings &s) {
        const HlaDatabase db = make_db(rows);
        ScoreReadResult r = score_consensus(g, reference_sequence, ref_start, consensus, db, gene, exons, is_forward_strand, s);
        py::dict stats;
        for (const auto &kv : r.stats) {
            auto tup = [](const std::optional<MappingStats> &x) -> py::object {
                if (!x) return py::none();
                return py::make_tuple(x->seq_len, x->nm, x->unmapped);
            };
            stats[py::str(kv.first)] = py::make_tuple(tup(kv.second.cdna_stats), tup(kv.second.dna_stats));
        }
        return py::make_tuple(stats, r.best_hla_id, r.best_star_allele, r.read_mapping_stats.to_json().pretty());
    });
    // hla_debug.json of one gene scored like diplotype_hla_batch does it (src/hla/caller.rs:805, :877, :914): one score_read per
    // consensus under the names consensus1 / consensus2 + the gene's DualPassingStats
    m.def("hla_debug_json", [](GpuAligner &g, const DbRows &rows, const std::string &gene,
                               const std::vector<std::tuple<std::string, std::string, std::string>> &consensuses /* qname, dna target, cdna target */,
                               bool is_dual, size_t counts1, size_t counts2, const DiplotypeSettings &s) {
        const HlaDatabase db = make_db(rows);
        HlaDebug dbg;
        for (const auto &c : consensuses)
            dbg.add_read(gene, std::get<0>(c), score_read(g, std::get<1>(c), std::get<2>(c), db, gene, s).read_mapping_stats);
        dbg.add_dual_passing_stats(gene, dual_passing_stats(is_dual, counts1, counts2, s.min_consensus_fraction, s.min_cdf, s.expected_maf));
        return dbg.pretty();
    });
    m.def("realign_records", [](GpuAligner &g, const std::vector<std::string> &genes, const DbRows &rows,
                                const std::vector<std::pair<std::string, std::string>> &reads, int n_candidates) {
        const HlaDatabase db = make_db(rows);
        HlaRealigner r(g, genes, db);
        Json arr = Json::array();
        for (const auto &d : r.realign_records(reads, n_candidates)) arr.push(d.to_json());
        return arr;
    }, py::arg("gpu"), py::arg("gene_list"), py::arg("database"), py::arg("reads"), py::arg("n_candidates") = 5);
    m.def("diplotype_strings", [](const std::string &h1, const std::string &h2) {
        const Diplotype d{h1, h2};
        return py::make_tuple(d.diplotype(), d.pharmcat_diplotype(), d.to_json().pretty());
    });
    m.def("harmonic_mean", &harmonic_mean);
    m.def("hpc", &hpc);
    m.def("hpc_pos", &hpc_pos);
    m.def("realign_records_full", [](GpuAligner &g, const std::vector<std::string> &genes, const DbRows &rows,
                                     const std::map<std::string, std::pair<bool, std::string>> &gene_defs,
                                     const std::vector<std::pair<std::string, std::string>> &reads, int n_candidates) {
        const HlaDatabase db = make_db(rows);
        std::map<std::string, HlaGeneDefinition> defs;
        for (const auto &kv : gene_defs) defs[kv.first] = HlaGeneDefinition{kv.second.first, kv.second.second};
        HlaRealigner r(g, genes, db, defs);
        py::list out;
        for (const RealignmentResult &res : r.realign_records_full(reads, n_candidates)) {
            py::dict d;
            d["gene_name"] = res.gene_name;
            d["read_mapping_stats"] = res.read_mapping_stats.to_json().pretty();
            d["mapping_details"] = res.mapping_details.to_json().pretty();
            if (res.realigned_record) {
                const RealignedHlaRecord &x = *res.realigned_record;
                d["realigned_record"] = py::make_tuple(x.segment_start, x.segment_end, x.dna_offset, x.hpc_offset, x.dna_sequence, x.hpc_sequence);
            } else {
                d["realigned_record"] = py::none();
            }
            out.append(d);
        }
        return out;
    }, py::arg("gpu"), py::arg("gene_list"), py::arg("database"), py::arg("gene_definitions"), py::arg("reads"), py::arg("n_candidates") = 5);
    m.def("diplotype_hla_gene", [](GpuAligner &g, const DbRows &rows, const std::string &gene,
                                   const std::vector<std::tuple<std::string, std::string, std::string>> &reads, const DiplotypeSettings &s) {
        const HlaDatabase db = make_db(rows);
        std::vector<HlaRead> rs;
        for (const auto &r : reads) rs.push_back({std::get<0>(r), std::get<1>(r), std::get<2>(r)});
        const HlaGeneCall c = diplotype_hla_gene(g, db, gene, rs, s);
        py::dict d;
        d["hla_id1"] = c.hla_id1; d["hla_id2"] = c.hla_id2; d["counts1"] = c.counts1; d["counts2"] = c.counts2;
        d["pair_score_cdna"] = c.pair_score_cdna; d["pair_score_dna"] = c.pair_score_dna;
        d["gene_details"] = c.gene_details();
        return d;
    });

    py::class_<HlaGeneIndex>(m, "HlaGeneIndex")
        .def(py::init([](GpuAligner &g, const DbRows &rows, const std::string &gene, const DiplotypeSettings &s) {
                 return new HlaGeneIndex(g, make_db(rows), gene, s);
             }), py::keep_alive<1, 2>())
        .def("n_alleles", &HlaGeneIndex::n_alleles)
        .def("gene_name", &HlaGeneIndex::gene_name);
    m.def("diplotype_hla_gene_indexed", [](GpuAligner &g, HlaGeneIndex &index,
                                           const std::vector<std::tuple<std::string, std::string, std::string>> &reads, const DiplotypeSettings &s) {
        std::vector<HlaRead> rs;
        for (const auto &r : reads) rs.push_back({std::get<0>(r), std::get<1>(r), std::get<2>(r)});
        // the interpreter lock is dropped for the C++ call: a cohort driver runs one sample per thread (one GpuAligner each)
        const HlaGeneCall c = [&] { py::gil_scoped_release nogil; return diplotype_hla_gene(g, index, rs, s); }();
        py::dict d;
        d["hla_id1"] = c.hla_id1; d["hla_id2"] = c.hla_id2; d["counts1"] = c.counts1; d["counts2"] = c.counts2;
        d["pair_score_cdna"] = c.pair_score_cdna; d["pair_score_dna"] = c.pair_score_dna;
        d["gene_details"] = c.gene_details();
        return d;
    });

    // records: (qname, read sequence, pos, cigar [(len, op)]); the DNA / cDNA targets are derived on the device (sp_targets_derive)
    m.def("diplotype_hla_gene_records", [](GpuAligner &g, HlaGeneIndex &index,
                                           const std::vector<std::tuple<std::string, std::string, int64_t, std::vector<std::pair<uint32_t, uint8_t>>>> &records,
                                           const std::vector<std::pair<uint64_t, uint64_t>> &exons, bool is_forward_strand, const DiplotypeSettings &s) {
        std::vector<HlaRecord> rs;
        for (const auto &r : records) rs.push_back({std::get<0>(r), std::get<1>(r), std::get<2>(r), std::get<3>(r)});
        const HlaGeneCall c = diplotype_hla_gene_records(g, index, rs, exons, is_forward_strand, s);
        py::dict d;
        d["hla_id1"] = c.hla_id1; d["hla_id2"] = c.hla_id2; d["counts1"] = c.counts1; d["counts2"] = c.counts2;
        d["pair_score_cdna"] = c.pair_score_cdna; d["pair_score_dna"] = c.pair_score_dna;
        d["gene_details"] = c.gene_details();
        return d;
    });

    // ---- CYP2D6 ----
    using RegionRows = std::vector<std::tuple<std::string, std::optional<std::string>, std::optional<size_t>>>;
    m.def("label_ops", [](const std::string &type, const std::optional<std::string> &sub, const std::string &type2,
                          const std::optional<std::string> &sub2, bool normalize_all) {
        const Cyp2d6Config cfg = Cyp2d6Config::default_config();
        Cyp2d6RegionLabel a{region_type_from_name(type), sub}, b{region_type_from_name(type2), sub2};
        py::dict d;
        d["full_allele"] = a.full_allele();
        d["simple"] = a.simplify_allele(false, cfg.cyp_translate);
        d["detailed"] = a.simplify_allele(true, cfg.cyp_translate);
        d["allowed"] = a.is_allowed_label();
        d["allowed_pair"] = a.is_allowed_label_pair(b);
        d["head"] = a.is_candidate_chain_head(normalize_all);
        d["normalizing"] = a.is_normalizing_allele(normalize_all);
        return d;
    });
    m.def("find_base_type_in_sequences", [](GpuAligner &g, const std::vector<std::tuple<std::string, std::optional<std::string>, std::string>> &templates,
                                            const SeqList &seqs, bool penalize_unmapped, double max_missing_frac) {
        std::vector<std::pair<Cyp2d6RegionLabel, std::string>> ts;
        for (const auto &t : templates) ts.push_back({Cyp2d6RegionLabel{region_type_from_name(std::get<0>(t)), std::get<1>(t)}, std::get<2>(t)});
        std::vector<std::vector<AlleleMapping>> all_hits;
        {
            py::gil_scoped_release nogil;
            Cyp2d6Extractor ex(g, std::move(ts));
            all_hits = ex.find_base_type_in_sequences(seqs, penalize_unmapped, max_missing_frac);
        }
        py::list out;
        for (const auto &hits : all_hits) {
            py::list one;
            for (const AlleleMapping &h : hits)
                one.append(py::make_tuple(h.allele_label.full_allele(), h.region_start, h.region_end,
                                          py::make_tuple(h.mapping_stats.seq_len, h.mapping_stats.nm, h.mapping_stats.unmapped,
                                                         h.mapping_stats.clipped_start, h.mapping_stats.clipped_end)));
            out.append(one);
        }
        return out;
    });
    // find_full_type_in_sequences: db = (backbone, backbone_start, variants [(pos, ref, alt)], metadata [(label, is_vi)],
    // haplotype lookup {star: 0/1 vector}, mapped hybrids [(type, subtype)]); per sequence None or (type, subtype, variants JSON or None)
    m.def("find_full_type_in_sequences", [](GpuAligner &g, const std::vector<std::tuple<std::string, std::optional<std::string>, std::string>> &templates,
                                            const SeqList &seqs, double max_missing_frac, bool force_assignment, const std::string &backbone,
                                            size_t backbone_start, const std::vector<std::tuple<size_t, std::string, std::string>> &variants,
                                            const std::vector<std::pair<std::string, bool>> &metadata,
                                            const std::map<std::string, std::vector<uint8_t>> &lookup,
                                            const std::vector<std::pair<std::string, std::optional<std::string>>> &mapped_hybrids, size_t graph_band) {
        std::vector<std::pair<Cyp2d6RegionLabel, std::string>> ts;
        for (const auto &t : templates) ts.push_back({Cyp2d6RegionLabel{region_type_from_name(std::get<0>(t)), std::get<1>(t)}, std::get<2>(t)});
        Cyp2d6Extractor ex(g, std::move(ts));
        Cyp2d6TypingDb db;
        db.backbone = backbone; db.backbone_start = backbone_start; db.haplotype_lookup = lookup;
        for (const auto &v : variants) db.variants.push_back({std::get<0>(v), std::get<1>(v), std::get<2>(v)});
        for (const auto &v : metadata) db.metadata.push_back({v.first, v.second});
        for (const auto &h : mapped_hybrids) db.mapped_hybrids.push_back(Cyp2d6RegionLabel{region_type_from_name(h.first), h.second});
        py::list out;
        for (const std::optional<Cyp2d6Region> &r : ex.find_full_type_in_sequences(seqs, max_missing_frac, force_assignment, db, graph_band)) {
            if (!r) { out.append(py::none()); continue; }
            py::object rv = py::none();
            if (r->variants) {
                Json arr = Json::array();
                for (const RegionVariant &v : *r->variants) arr.push(v.to_json());
                rv = py::str(arr.pretty());
            }
            py::object sub = r->label.subtype_label ? py::object(py::str(*r->label.subtype_label)) : py::object(py::none());
            out.append(py::make_tuple(region_type_name(r->label.region_type), sub, rv));
        }
        return out;
    }, py::arg("gpu"), py::arg("templates"), py::arg("sequences"), py::arg("max_missing_frac"), py::arg("force_assignment"), py::arg("backbone"),
       py::arg("backbone_start"), py::arg("variants"), py::arg("metadata"), py::arg("haplotype_lookup"), py::arg("mapped_hybrids"),
       py::arg("graph_band") = 128);
    // ---- the consensus stage of the CYP2D6 caller (src/cyp2d6/caller.rs:145-310, :750-893) ----
    m.def("hpc_with_guide", [](const std::string &seq, const std::string &guide, size_t off) {
        const auto r = hpc_with_guide(seq, guide, off);
        return py::make_tuple(py::bytes(r.first), r.second);
    });
    // roi: {read id: [(region type, subtype, start, end, (seq_len, nm, unmapped, clipped_start, clipped_end))]} as find_base_type_in_sequences returns them
    m.def("cyp2d6_consensus_inputs", [](GpuAligner &g, const std::map<std::string, std::string> &read_sequences,
                                        const std::map<std::string, std::vector<std::tuple<std::string, std::optional<std::string>, size_t, size_t,
                                                                                             std::tuple<size_t, size_t, size_t, std::optional<size_t>, std::optional<size_t>>>>> &roi,
                                        const std::vector<std::tuple<std::string, std::optional<std::string>, std::string>> &templates,
                                        double max_missing_consensus_frac) {
        std::vector<std::pair<Cyp2d6RegionLabel, std::string>> ts;
        for (const auto &t : templates) ts.push_back({Cyp2d6RegionLabel{region_type_from_name(std::get<0>(t)), std::get<1>(t)}, std::get<2>(t)});
        Cyp2d6Extractor ex(g, std::move(ts));
        std::map<std::string, std::vector<AlleleMapping>> regions;
        for (const auto &kv : roi)
            for (const auto &r : kv.second) {
                AlleleMapping a;
                a.allele_label = Cyp2d6RegionLabel{region_type_from_name(std::get<0>(r)), std::get<1>(r)};
                a.region_start = std::get<2>(r); a.region_end = std::get<3>(r);
                const auto &st = std::get<4>(r);
                a.mapping_stats = MappingStats(std::get<0>(st), std::get<1>(st), std::get<2>(st));
                a.mapping_stats.clipped_start = std::get<3>(st); a.mapping_stats.clipped_end = std::get<4>(st);
                regions[kv.first].push_back(a);
            }
        const Cyp2d6ConsensusInputs in = cyp2d6_consensus_inputs(read_sequences, regions, ex, max_missing_consensus_frac);
        py::dict d;
        py::list raw, hp;
        for (const auto &x : in.raw_sequences) raw.append(py::bytes(x));
        for (const auto &x : in.hpc_sequences) hp.append(py::bytes(x));
        d["raw_sequences"] = raw; d["hpc_sequences"] = hp; d["base_offsets"] = in.base_offsets; d["hpc_offsets"] = in.hpc_offsets;
        d["sequence_ids"] = in.sequence_ids; d["seeds"] = in.seeds;
        return d;
    });
    // raw: (consensuses[group] = [(hpc sequence, scores), (full sequence, scores)], group of every sequence) as priority_consensus returns it
    m.def("merge_consensus_results", [cfg_from](GpuAligner &g, const SeqList &sequences, const std::vector<size_t> &offsets, const py::dict &cfg,
                                                const std::vector<std::vector<std::pair<std::string, std::vector<size_t>>>> &raw_consensuses,
                                                const std::vector<size_t> &raw_indices,
                                                const std::vector<std::tuple<std::string, std::optional<std::string>, std::string>> &templates,
                                                const std::string &backbone, size_t backbone_start,
                                                const std::vector<std::tuple<size_t, std::string, std::string>> &variants,
                                                const std::vector<std::pair<std::string, bool>> &metadata,
                                                const std::map<std::string, std::vector<uint8_t>> &lookup,
                                                const std::vector<std::pair<std::string, std::optional<std::string>>> &mapped_hybrids,
                                                double max_missing_consensus_frac) {
        std::vector<std::pair<Cyp2d6RegionLabel, std::string>> ts;
        for (const auto &t : templates) ts.push_back({Cyp2d6RegionLabel{region_type_from_name(std::get<0>(t)), std::get<1>(t)}, std::get<2>(t)});
        Cyp2d6Extractor ex(g, std::move(ts));
        Cyp2d6TypingDb db;
        db.backbone = backbone; db.backbone_start = backbone_start; db.haplotype_lookup = lookup;
        for (const auto &v : variants) db.variants.push_back({std::get<0>(v), std::get<1>(v), std::get<2>(v)});
        for (const auto &v : metadata) db.metadata.push_back({v.first, v.second});
        for (const auto &h : mapped_hybrids) db.mapped_hybrids.push_back(Cyp2d6RegionLabel{region_type_from_name(h.first), h.second});
        PriorityConsensus raw;
        raw.sequence_indices = raw_indices;
        for (const auto &levels : raw_consensuses) {
            std::vector<Consensus> one;
            for (const auto &c : levels) one.push_back(Consensus{c.first, c.second});
            raw.consensuses.push_back(std::move(one));
        }
        const MultiConsensus mc = merge_consensus_results(g, sequences, offsets, cfg_from(cfg), raw, ex, db, Cyp2d6Config::default_config(),
                                                          max_missing_consensus_frac);
        py::list cons;
        for (const Consensus &c : mc.consensuses) cons.append(py::make_tuple(py::bytes(c.sequence), c.scores));
        return py::make_tuple(cons, mc.sequence_indices);
    });
    m.def("overlap_score", &overlap_score);
    m.def("region_variant_string", [](const std::string &label, bool is_vi, int state) {
        return RegionVariant{label, is_vi, static_cast<VariantAlleleRelationship>(state)}.to_string();
    });
    // rows: (region type, subtype label, unique id, variants or None); variants: (label, is_vi, state index)
    m.def("cyp2d6_alleles_json", [](const std::vector<std::vector<size_t>> &best,
                                    const std::vector<std::tuple<std::string, std::optional<std::string>, std::optional<size_t>,
                                                                 std::optional<std::vector<std::tuple<std::string, bool, int>>>>> &rows) {
        std::vector<Cyp2d6Region> regions;
        for (const auto &r : rows) {
            Cyp2d6Region g;
            g.label.region_type = region_type_from_name(std::get<0>(r));
            g.label.subtype_label = std::get<1>(r);
            g.unique_id = std::get<2>(r);
            if (std::get<3>(r)) {
                g.variants.emplace();
                for (const auto &v : *std::get<3>(r))
                    g.variants->push_back({std::get<0>(v), std::get<1>(v), static_cast<VariantAlleleRelationship>(std::get<2>(v))});
            }
            regions.push_back(std::move(g));
        }
        return cyp2d6_alleles_json(best, regions, Cyp2d6Config::default_config().cyp_translate);
    });
    m.def("alleles_from_traversal", &alleles_from_traversal);
    m.def("assign_haplotypes_from_alleles", [](GpuAligner &g, const std::vector<std::vector<uint8_t>> &alleles,
                                               const std::map<std::string, std::vector<uint8_t>> &lookup,
                                               const std::vector<std::pair<std::string, bool>> &variants, bool force) {
        std::vector<VariantMetadata> meta;
        for (const auto &v : variants) meta.push_back({v.first, v.second});
        py::list out;
        for (const HaplotypeAssignment &a : assign_haplotypes_from_alleles(g, alleles, lookup, meta, force)) {
            py::object star = a.label.region_type == Cyp2d6RegionType::Unknown ? py::object(py::none()) : py::object(py::str(*a.label.subtype_label));
            py::object rv = py::none();
            if (a.variants) {
                Json arr = Json::array();
                for (const RegionVariant &v : *a.variants) arr.push(v.to_json());
                rv = py::str(arr.pretty());
            }
            out.append(py::make_tuple(star, rv, py::make_tuple(a.vi_match, a.all_match), a.label.full_allele()));
        }
        return out;
    });
    m.def("convert_chain_to_hap", [](const std::vector<size_t> &chain, const RegionRows &rows, const std::string &level) {
        const Cyp2d6Config cfg = Cyp2d6Config::default_config();
        const Cyp2d6DetailLevel lvl = level == "CoreAlleles" ? Cyp2d6DetailLevel::CoreAlleles
                                      : level == "SubAlleles" ? Cyp2d6DetailLevel::SubAlleles : Cyp2d6DetailLevel::DeepAlleles;
        return convert_chain_to_hap(chain, make_regions(rows), lvl, cfg.cyp_translate);
    });
    m.def("weight_sequences", [](GpuAligner &g, const SeqList &segments, const SeqList &consensuses, const RegionRows &rows) {
        return weight_sequences(g, segments, consensuses, make_regions(rows));
    });
    m.def("build_chains", [](const std::map<std::string, std::vector<SequenceWeights>> &rw, size_t n_haps) {
        ChainBuild b = build_chains(rw, n_haps);
        return py::make_tuple(b.qname_chains, b.qname_chain_scores, b.best_allele_mapping_counts);
    });
    m.def("find_best_chain_pair", [](GpuAligner &g, const std::map<std::string, std::vector<std::vector<size_t>>> &obs,
                                     const std::map<std::string, std::vector<SequenceWeights>> &scores, const RegionRows &rows, bool infer,
                                     bool normalize_all, bool ignore_limits, double lasso, double ln_ed, double unexpected,
                                     double inferred_edge) {
        ChainPenalties pen;
        pen.lasso_penalty = lasso; pen.ln_ed_penalty = ln_ed; pen.unexpected_chain_penalty = unexpected; pen.inferred_edge_penalty = inferred_edge;
        const ChainPairResult r = find_best_chain_pair(g, Cyp2d6Config::default_config(), obs, scores, make_regions(rows), infer, normalize_all,
                                                       pen, ignore_limits);
        py::dict d;
        d["best_chains"] = r.best_chains; d["dangling"] = r.dangling_alleles; d["score"] = r.score; d["i"] = r.index1; d["j"] = r.index2;
        d["edit_distance"] = r.edit_distance; d["n_possible_chains"] = r.n_possible_chains; d["n_full_evaluations"] = r.n_full_evaluations;
        return d;
    }, py::arg("gpu"), py::arg("obs_chains"), py::arg("chain_scores"), py::arg("regions"), py::arg("infer"), py::arg("normalize_all"),
          py::arg("ignore_limits") = false, py::arg("lasso_penalty") = 4.0, py::arg("ln_ed_penalty") = 2.0,
          py::arg("unexpected_chain_penalty") = 10.0, py::arg("inferred_edge_penalty") = 2.0);
    m.def("call_cyp2d6_chains", [](GpuAligner &g, const SeqList &consensuses, const RegionRows &rows,
                                   const std::map<std::string, std::vector<std::tuple<size_t, size_t, std::string>>> &roi, bool infer,
                                   bool normalize_all) {
        std::map<std::string, std::vector<Cyp2d6ReadRegion>> regions;
        for (const auto &kv : roi)
            for (const auto &r : kv.second) regions[kv.first].push_back({std::get<0>(r), std::get<1>(r), std::get<2>(r)});
        const Cyp2d6Call c = [&] {
            py::gil_scoped_release nogil;
            return call_cyp2d6_chains(g, Cyp2d6Config::default_config(), consensuses, make_regions(rows), regions, infer, normalize_all);
        }();
        py::dict d;
        d["best_chains"] = c.chain_pair.best_chains; d["score"] = c.chain_pair.score; d["dangling"] = c.chain_pair.dangling_alleles;
        d["n_possible_chains"] = c.chain_pair.n_possible_chains; d["n_full_evaluations"] = c.chain_pair.n_full_evaluations;
        d["gene_details"] = c.gene_details();
        return d;
    });

    m.def("starphase_json", &starphase_json);
}
