// sp_host_graph.cpp -- variant graph + traversal above K8 (sp_graph_traverse): row N3 of SURVEY.md 8f.
//
// Cyp2d6Extractor::assign_haplotype (src/cyp2d6/haplotyper.rs:371-468) builds a graph of the CYP2D6 backbone with one bubble per
// database variant (hiphase::WFAGraph::from_reference_variants, :430-441), aligns the consensus to it end to end
// (edit_distance_with_pruning, :445) and reads every variant's allele off the traversed nodes (:454-468).  Here: VariantGraph
// (the graph and its node -> (variant, allele) labels), its linearisation, and K8 on the device (sp_graph_traverse), which
// returns the positions, and with them the nodes, some optimal alignment passes through.  The graph construction restates the
// published behaviour, not hiphase's code (unvendored): overlapping variants form one site with a REF branch and one ALT branch
// per variant.
#include <algorithm>
#include <set>

#include "starphase_host.hpp"

namespace starphase {

size_t VariantGraph::add(std::string seq, std::vector<size_t> preds, size_t coord) {
    seqs.push_back(std::move(seq)); this->preds.push_back(std::move(preds)); this->coord.push_back(coord);
    return seqs.size() - 1;
}

VariantGraph VariantGraph::from_reference_variants(const std::string &backbone, size_t region_start, const std::vector<GraphVariant> &variants) {
    VariantGraph g;
    const size_t n = backbone.size();
    struct V { size_t pos; const std::string *ref, *alt; size_t index; };
    std::vector<V> inside;
    for (size_t k = 0; k < variants.size(); ++k) {
        const GraphVariant &v = variants[k];
        if (v.position < region_start) continue;
        const size_t p = v.position - region_start;
        if (p + v.ref_allele.size() > n || backbone.compare(p, v.ref_allele.size(), v.ref_allele) != 0) continue;  // not wholly inside / not this reference
        inside.push_back({p, &v.ref_allele, &v.alt_allele, k});
    }
    std::stable_sort(inside.begin(), inside.end(), [](const V &a, const V &b) { return a.pos != b.pos ? a.pos < b.pos : a.index < b.index; });
    std::vector<std::vector<V>> sites;
    size_t cur_end = 0;
    for (const V &v : inside) {
        if (!sites.empty() && (v.pos < cur_end || v.pos == sites.back()[0].pos)) {
            sites.back().push_back(v);
            cur_end = std::max(cur_end, v.pos + v.ref->size());
        } else {
            sites.push_back({v});
            cur_end = v.pos + v.ref->size();
        }
    }
    std::vector<size_t> last = {g.add("", {}, 0)};  // node 0: empty source
    size_t pos = 0;
    for (const auto &site : sites) {
        size_t s0 = site[0].pos, s1 = 0;
        for (const V &v : site) s1 = std::max(s1, v.pos + v.ref->size());
        auto branch = [&](const V &v) { return backbone.substr(s0, v.pos - s0) + *v.alt + backbone.substr(v.pos + v.ref->size(), s1 - (v.pos + v.ref->size())); };
        bool empty_branch = false;
        for (const V &v : site) empty_branch = empty_branch || branch(v).empty();
        if (empty_branch) {  // every branch keeps at least one character (a bare deletion takes a neighbouring backbone base along)
            if (s0 > pos) --s0;
            else if (s1 < n) ++s1;
        }
        if (s0 > pos) last = {g.add(backbone.substr(pos, s0 - pos), last, pos)};
        std::vector<size_t> branches;
        const size_t ref = g.add(backbone.substr(s0, s1 - s0), last, s0);
        for (const V &v : site) g.node_to_alleles[ref].emplace_back(v.index, uint8_t(0));
        branches.push_back(ref);
        for (const V &v : site) {
            const size_t alt = g.add(branch(v), last, s0);
            g.node_to_alleles[alt].emplace_back(v.index, uint8_t(1));
            for (const V &u : site)
                if (u.index != v.index) g.node_to_alleles[alt].emplace_back(u.index, uint8_t(0));
            branches.push_back(alt);
        }
        last = branches;
        pos = s1;
    }
    g.sink = g.add(backbone.substr(pos), last, pos);
    return g;
}

namespace {
struct Linear {
    std::string chars;
    std::vector<int32_t> pred_off, preds, diag, node_of, ends;
};
Linear linearise(const VariantGraph &g) {
    Linear L;
    L.pred_off.push_back(0);
    std::vector<int32_t> lastpos(g.seqs.size(), -1);
    // positions at which a path can stand after `node` (through empty nodes; -1 = before the first character)
    std::function<std::vector<int32_t>(size_t)> tails = [&](size_t node) -> std::vector<int32_t> {
        if (!g.seqs[node].empty()) return {lastpos[node]};
        if (g.preds[node].empty()) return {-1};
        std::set<int32_t> out;
        for (size_t p : g.preds[node])
            for (int32_t t : tails(p)) out.insert(t);
        return std::vector<int32_t>(out.begin(), out.end());
    };
    for (size_t node = 0; node < g.seqs.size(); ++node) {
        const std::string &s = g.seqs[node];
        for (size_t c = 0; c < s.size(); ++c) {
            const int32_t pid = static_cast<int32_t>(L.chars.size());
            if (c == 0) {
                std::set<int32_t> pr;
                for (size_t p : g.preds[node])
                    for (int32_t t : tails(p)) pr.insert(t);
                if (g.preds[node].empty()) pr.insert(-1);
                L.preds.insert(L.preds.end(), pr.begin(), pr.end());
            } else {
                L.preds.push_back(pid - 1);
            }
            L.pred_off.push_back(static_cast<int32_t>(L.preds.size()));
            L.chars.push_back(s[c]);
            L.diag.push_back(static_cast<int32_t>(g.coord[node] + c + 1));
            L.node_of.push_back(static_cast<int32_t>(node));
        }
        if (!s.empty()) lastpos[node] = static_cast<int32_t>(L.chars.size()) - 1;
    }
    L.ends = tails(g.sink);
    return L;
}
}  // namespace

std::vector<GraphAlignment> graph_edit_distance(GpuAligner &gpu, const std::vector<const VariantGraph *> &graphs, const SeqList &sequences, size_t band) {
    if (graphs.size() != sequences.size()) throw HostError("graph_edit_distance: one sequence per graph expected");
    const size_t n = graphs.size();
    std::vector<Linear> lin;
    std::string gchars, seqs;
    std::vector<int64_t> goff(1, 0), soff(1, 0);
    std::vector<int32_t> pred_off(1, 0), preds, diag, end_off(1, 0), ends;
    for (size_t p = 0; p < n; ++p) {
        lin.push_back(linearise(*graphs[p]));
        const Linear &L = lin.back();
        gchars += L.chars;
        for (size_t q = 1; q < L.pred_off.size(); ++q) pred_off.push_back(static_cast<int32_t>(preds.size()) + L.pred_off[q]);
        preds.insert(preds.end(), L.preds.begin(), L.preds.end());
        diag.insert(diag.end(), L.diag.begin(), L.diag.end());
        ends.insert(ends.end(), L.ends.begin(), L.ends.end());
        end_off.push_back(static_cast<int32_t>(ends.size()));
        goff.push_back(static_cast<int64_t>(gchars.size()));
        seqs += sequences[p];
        soff.push_back(static_cast<int64_t>(seqs.size()));
    }
    std::vector<int32_t> score(std::max<size_t>(n, 1));
    std::vector<uint8_t> on_path(std::max<size_t>(gchars.size(), 1));
    if (gchars.empty()) gchars.push_back('N');
    if (seqs.empty()) seqs.push_back('N');
    if (preds.empty()) preds.push_back(-1);
    if (diag.empty()) diag.push_back(0);
    if (n) {
        const sp_status st = sp_graph_traverse(gpu.raw(), static_cast<int32_t>(n), reinterpret_cast<const uint8_t *>(gchars.data()), goff.data(),
                                               pred_off.data(), preds.data(), diag.data(), end_off.data(), ends.data(),
                                               reinterpret_cast<const uint8_t *>(seqs.data()), soff.data(), static_cast<int32_t>(band), score.data(),
                                               on_path.data());
        if (st != SP_OK) throw HostError(std::string("sp_graph_traverse: ") + sp_last_error(gpu.raw()));
    }
    constexpr int32_t kInf = 0x3FFFFFFF;
    std::vector<GraphAlignment> out(n);
    for (size_t p = 0; p < n; ++p) {
        const Linear &L = lin[p];
        out[p].score = static_cast<size_t>(score[p]);
        out[p].found = score[p] < kInf;
        std::set<size_t> nodes;
        for (size_t q = 0; q < L.node_of.size(); ++q)
            if (on_path[static_cast<size_t>(goff[p]) + q]) nodes.insert(static_cast<size_t>(L.node_of[q]));
        out[p].traversed_nodes.assign(nodes.begin(), nodes.end());
    }
    return out;
}

std::vector<uint8_t> graph_alleles(const VariantGraph &g, const GraphAlignment &aln, size_t num_variants) {
    return alleles_from_traversal(num_variants, aln.traversed_nodes, g.node_to_alleles);  // src/cyp2d6/haplotyper.rs:452-468
}

}  // namespace starphase
