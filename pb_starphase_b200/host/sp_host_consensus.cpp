// sp_host_consensus.cpp -- consensus search above K7 (sp_consensus_extend): row N1 of SURVEY.md 8f.
//
// Interface: waffle_con's ConsensusDWFA / DualConsensusDWFA as the reference drives them (src/hla/caller.rs:1124-1219:
// with_config, add_sequence, add_sequence_offset, consensus() -> list of equally good solutions, first one taken).
// Policy: a best-first search over consensus prefixes.  A node is one consensus (or two: a dual node) with, for every read,
// its edit distance to the prefix (end-free in the read) -- kept on the device, one track per consensus; reads vote for the
// next symbol with the bases that follow their best prefixes, one vote per read split evenly; a symbol is extended when it
// has min_count votes and a min_af share (the best-voted symbol when none qualifies); when two symbols qualify on a single
// node, a dual node with one consensus per symbol is opened as well; in a dual node a read counts towards, and votes for,
// the consensus it is closer to; at most max_capacity_per_size nodes are expanded per total length and the queue keeps the
// max_queue_size best nodes; a node nobody votes on is complete, and the cheapest complete nodes are the answer (a dual
// answer needs min_count reads and a min_af share on its minor side).  Every expansion is ONE device call covering all
// (consensus, symbol) extensions of the node -- and a node with a single way forward (one symbol with the votes per side, which is
// most of a consensus) is handed to the device together with the cost of the best competitor: sp_consensus_run keeps extending it
// on chip for as long as this loop would have popped its child next, and returns the last child (identical search, ~1 us instead
// of ~25 us per symbol).  This restates the published outline of waffle_con's search, not its code.
#include <algorithm>
#include <array>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <limits>
#include <map>
#include <memory>
#include <set>

#include "starphase_host.hpp"

namespace starphase {

namespace {
constexpr int32_t kInf = 0x3FFFFFFF;
constexpr uint8_t kFinished = 1u << 5, kInactive = 1u << 6;
constexpr long kVoteUnit = 12;  // one read's vote, split evenly over its 1..4 candidate symbols

struct TrackPool {
    std::vector<int> free_list;
    explicit TrackPool(int n) { for (int t = n - 1; t >= 0; --t) free_list.push_back(t); }
    int take() {
        if (free_list.empty()) throw HostError("consensus: out of device tracks");
        const int t = free_list.back();
        free_list.pop_back();
        return t;
    }
};
struct Side {  // one consensus of a node: its device track and the per-read outputs of the step that made it
    int track = -1;
    TrackPool *pool = nullptr;
    std::vector<int32_t> ed, full;
    std::vector<uint8_t> votes;
    ~Side() { if (pool && track >= 0) pool->free_list.push_back(track); }
    std::vector<long> costs() const {
        std::vector<long> c(ed.size());
        for (size_t r = 0; r < ed.size(); ++r) c[r] = (votes[r] & kInactive) ? 0 : std::min(ed[r], full[r]);
        return c;
    }
};
using SidePtr = std::shared_ptr<Side>;
struct Node {
    long cost = 0;
    std::string c1, c2;
    bool dual = false;
    SidePtr s1, s2;
    size_t size() const { return c1.size() + (dual ? c2.size() : 0); }
};
struct NodeLess {  // (cost, longer first, consensus1, consensus2)
    bool operator()(const std::shared_ptr<Node> &a, const std::shared_ptr<Node> &b) const {
        if (a->cost != b->cost) return a->cost < b->cost;
        if (a->size() != b->size()) return a->size() > b->size();
        if (a->c1 != b->c1) return a->c1 < b->c1;
        return a->c2 < b->c2;
    }
};

std::array<long, 4> tally(const Side &s, const std::vector<char> *voters) {
    std::array<long, 4> t{0, 0, 0, 0};
    for (size_t r = 0; r < s.ed.size(); ++r) {
        if (voters && !(*voters)[r]) continue;
        if ((s.votes[r] & kInactive) || s.full[r] < s.ed[r]) continue;  // inactive, or already consumed at a better column
        const int n = __builtin_popcount(s.votes[r] & 15u);
        for (int k = 0; k < 4 && n; ++k)
            if (s.votes[r] >> k & 1u) t[static_cast<size_t>(k)] += kVoteUnit / n;
    }
    return t;
}
std::vector<int> strictly_passing(const std::array<long, 4> &t, const CdwfaConfig &cfg) {
    const long total = t[0] + t[1] + t[2] + t[3], permille = std::lround(cfg.min_af * 1000.0);
    std::vector<int> ok;
    for (int k = 0; k < 4; ++k)
        if (t[static_cast<size_t>(k)] >= kVoteUnit * static_cast<long>(cfg.min_count) && t[static_cast<size_t>(k)] * 1000 >= total * permille && total > 0)
            ok.push_back(k);
    return ok;
}
std::vector<int> passing(const std::array<long, 4> &t, const CdwfaConfig &cfg) {
    const long total = t[0] + t[1] + t[2] + t[3];
    if (total == 0) return {};
    std::vector<int> ok = strictly_passing(t, cfg);
    if (!ok.empty()) return ok;
    int best = 0;
    for (int k = 1; k < 4; ++k)
        if (t[static_cast<size_t>(k)] > t[static_cast<size_t>(best)]) best = k;
    return {best};
}

// a failed sp_* call inside a search: it fails the whole batch, where a HostError of the search's own fails only that search
struct DeviceError : HostError {
    using HostError::HostError;
};

// One best-first search, resumable: advance() runs the policy on the host until it needs the device and leaves one request --
// an extension list or a run job -- in `need`; the driver below fulfils the requests of many searches together and calls resume().
struct Search {
    GpuAligner &gpu;
    const CdwfaConfig &cfg;
    const SeqList &reads;
    const bool allow_dual;
    sp_consensus *h = nullptr;
    TrackPool pool;
    size_t n_calls = 0, n_run_steps = 0;
    double run_seconds = 0.0;  // inside the sp_consensus_run_batch calls that carried this search's jobs (diagnostic)
    bool can_run[3] = {false, false, false};  // sp_consensus_run fits for 1 / 2 sides
    // the search
    std::multiset<std::shared_ptr<Node>, NodeLess> queue;
    std::vector<std::shared_ptr<Node>> best;
    bool have_best = false;
    long best_cost = 0;
    std::map<size_t, size_t> expanded;
    // the pending request and what its answer is for
    enum class Need { None, Extend, Run } need = Need::None;
    enum class Then { Root, Expand, Run } then = Then::Root;
    std::shared_ptr<Node> cur;  // the node being expanded
    std::vector<int> p1, p2, strict;
    std::vector<int32_t> x_src, x_dst, x_ed, x_full;  // extension list
    std::vector<uint8_t> x_sym, x_votes;
    std::vector<SidePtr> x_out;
    sp_consensus_job job{};  // run job, its buffers
    std::vector<int32_t> r_ed, r_full;
    std::vector<uint8_t> r_votes, r_log;
    int32_t r_n = 0;
    SidePtr r_out[2];
    long r_limit_cost = 0, r_limit_size = 0, r_cap = 0;

    Search(GpuAligner &g, const CdwfaConfig &c, const SeqList &r, const std::vector<int32_t> &offsets, bool dual)
        : gpu(g), cfg(c), reads(r), allow_dual(dual), pool(256) {
        if (reads.empty()) throw HostError("consensus: no sequences were added");
        std::string bases;
        std::vector<int64_t> offs(1, 0);
        for (const auto &s : reads) { bases += s; offs.push_back(static_cast<int64_t>(bases.size())); }
        if (bases.empty()) bases.push_back('N');
        sp_seqset set{reinterpret_cast<const uint8_t *>(bases.data()), offs.data(), static_cast<int64_t>(reads.size())};
        const sp_status st = sp_consensus_create(gpu.raw(), &set, offsets.data(), static_cast<int32_t>(cfg.offset_window), static_cast<int32_t>(cfg.band),
                                                 256, &h);
        if (st != SP_OK) throw HostError(std::string("sp_consensus_create: ") + sp_last_error(gpu.raw()));
        const bool on = getenv("SP_CONSENSUS_NO_RUN") == nullptr;  // A/B switch for measurements: step every symbol from the host
        can_run[1] = on && sp_consensus_run_supported(h, 1) != 0;
        can_run[2] = on && sp_consensus_run_supported(h, 2) != 0;
    }
    ~Search() {
        if (getenv("SP_TIMING"))
            fprintf(stderr, "[sp_timing] consensus search: %zu device calls, %zu symbols appended on the device in %.1f ms\n", n_calls, n_run_steps,
                    1e3 * run_seconds);
        sp_consensus_destroy(h);
    }
    Search(const Search &) = delete;
    Search &operator=(const Search &) = delete;

    // the node has one way forward: ask the device to follow it (see the header of this file)
    void request_run(const Node &node, long cost_limit, long size_limit, long cost_cap) {
        const int ns = node.dual ? 2 : 1;
        const size_t R = reads.size(), s0 = node.size();
        // every node expanded on the way must be below the per-size capacity: stop before the first size that is full
        size_t first_full = static_cast<size_t>(-1);
        for (auto it = expanded.upper_bound(s0); it != expanded.end(); ++it)
            if (it->second >= cfg.max_capacity_per_size) { first_full = it->first; break; }
        size_t max_steps = 1 << 16;
        if (first_full != static_cast<size_t>(-1)) max_steps = std::min<size_t>(max_steps, node.dual ? (first_full - s0 - 1) / 2 + 1 : first_full - s0);
        r_ed.assign(R * static_cast<size_t>(ns), 0); r_full.assign(R * static_cast<size_t>(ns), 0);
        r_votes.assign(R * static_cast<size_t>(ns), 0); r_log.assign(max_steps, 0);
        job = sp_consensus_job{};
        job.c = h; job.n_sides = ns;
        for (int s = 0; s < ns; ++s) {
            const Side &from = s == 0 ? *node.s1 : *node.s2;
            r_out[s] = std::make_shared<Side>();
            r_out[s]->pool = &pool;
            r_out[s]->track = pool.take();
            job.src[s] = from.track; job.dst[s] = r_out[s]->track;
            std::copy(from.ed.begin(), from.ed.end(), r_ed.begin() + static_cast<std::ptrdiff_t>(static_cast<size_t>(s) * R));
            std::copy(from.full.begin(), from.full.end(), r_full.begin() + static_cast<std::ptrdiff_t>(static_cast<size_t>(s) * R));
            std::copy(from.votes.begin(), from.votes.end(), r_votes.begin() + static_cast<std::ptrdiff_t>(static_cast<size_t>(s) * R));
        }
        if (ns == 1) r_out[1] = nullptr;
        job.ed = r_ed.data(); job.votes = r_votes.data(); job.full = r_full.data();
        job.min_count = static_cast<int32_t>(cfg.min_count); job.min_af_permille = static_cast<int32_t>(std::lround(cfg.min_af * 1000.0));
        job.cost_limit = static_cast<int64_t>(cost_limit); job.size_limit = static_cast<int64_t>(size_limit); job.cost_cap = static_cast<int64_t>(cost_cap);
        job.max_steps = static_cast<int32_t>(max_steps); job.steps = r_log.data(); job.n_steps = &r_n;
        r_n = 0; r_limit_cost = cost_limit; r_limit_size = size_limit; r_cap = cost_cap;
        need = Need::Run; then = Then::Run;
    }

    // the run's answer: the last child, or nullptr when the device took no step; `expanded` gets the nodes expanded on the way
    std::shared_ptr<Node> run_result() {
        static const char kSym[4] = {'A', 'C', 'G', 'T'};
        const Node &node = *cur;
        const int ns = node.dual ? 2 : 1;
        const size_t R = reads.size(), s0 = node.size();
        ++n_calls;
        const int32_t n = r_n;
        if (getenv("SP_CONSENSUS_DEBUG"))
            fprintf(stderr, "[consensus] run: dual %d size %zu cost %ld limit (%ld, %ld) cap %ld max_steps %d -> %d steps\n", node.dual ? 1 : 0, s0,
                    node.cost, r_limit_cost, r_limit_size, r_cap, job.max_steps, n);
        SidePtr out[2] = {std::move(r_out[0]), std::move(r_out[1])};
        if (n == 0) return nullptr;
        n_run_steps += static_cast<size_t>(n);
        std::string c1 = node.c1, c2 = node.c2;
        for (int32_t q = 0; q < n; ++q) {
            if (q > 0) ++expanded[c1.size() + (node.dual ? c2.size() : 0)];  // the node this round expanded (round 0: counted by the caller)
            const int a = r_log[static_cast<size_t>(q)] & 15, b = r_log[static_cast<size_t>(q)] >> 4;
            if (a < 4) c1.push_back(kSym[a]);
            if (node.dual && b < 4) c2.push_back(kSym[b]);
        }
        for (int s = 0; s < ns; ++s) {
            out[s]->ed.assign(r_ed.begin() + static_cast<std::ptrdiff_t>(static_cast<size_t>(s) * R), r_ed.begin() + static_cast<std::ptrdiff_t>(static_cast<size_t>(s + 1) * R));
            out[s]->full.assign(r_full.begin() + static_cast<std::ptrdiff_t>(static_cast<size_t>(s) * R), r_full.begin() + static_cast<std::ptrdiff_t>(static_cast<size_t>(s + 1) * R));
            out[s]->votes.assign(r_votes.begin() + static_cast<std::ptrdiff_t>(static_cast<size_t>(s) * R), r_votes.begin() + static_cast<std::ptrdiff_t>(static_cast<size_t>(s + 1) * R));
        }
        return make(std::move(c1), out[0], node.dual, std::move(c2), node.dual ? out[1] : nullptr);
    }

    // one extension list: every (parent side, symbol); symbol 0 = report the fresh track
    void request_extend(const std::vector<std::pair<const Side *, char>> &tasks, Then next) {
        const size_t n = tasks.size(), R = reads.size();
        x_src.assign(n, 0); x_dst.assign(n, 0); x_sym.assign(n, 0);
        x_ed.assign(n * R, 0); x_full.assign(n * R, 0); x_votes.assign(n * R, 0);
        x_out.assign(n, nullptr);
        for (size_t q = 0; q < n; ++q) {
            x_out[q] = std::make_shared<Side>();
            x_out[q]->pool = &pool;
            x_out[q]->track = pool.take();
            if (tasks[q].first) {
                x_src[q] = tasks[q].first->track;
            } else {  // root: a fresh track, reported
                x_src[q] = x_out[q]->track;
                if (sp_consensus_reset(h, x_out[q]->track) != SP_OK) throw DeviceError(std::string("sp_consensus_reset: ") + sp_last_error(gpu.raw()));
            }
            x_dst[q] = x_out[q]->track;
            x_sym[q] = static_cast<uint8_t>(tasks[q].second);
        }
        need = Need::Extend; then = next;
    }
    sp_consensus_ext ext_list() {
        return sp_consensus_ext{h, static_cast<int32_t>(x_src.size()), x_src.data(), x_sym.data(), x_dst.data(), x_ed.data(), x_votes.data(), x_full.data()};
    }
    std::vector<SidePtr> extend_result() {
        const size_t n = x_out.size(), R = reads.size();
        if (n && R) ++n_calls;
        for (size_t q = 0; q < n; ++q) {
            x_out[q]->ed.assign(x_ed.begin() + static_cast<std::ptrdiff_t>(q * R), x_ed.begin() + static_cast<std::ptrdiff_t>((q + 1) * R));
            x_out[q]->full.assign(x_full.begin() + static_cast<std::ptrdiff_t>(q * R), x_full.begin() + static_cast<std::ptrdiff_t>((q + 1) * R));
            x_out[q]->votes.assign(x_votes.begin() + static_cast<std::ptrdiff_t>(q * R), x_votes.begin() + static_cast<std::ptrdiff_t>((q + 1) * R));
        }
        return std::move(x_out);
    }

    std::shared_ptr<Node> make(std::string c1, SidePtr s1, bool dual, std::string c2, SidePtr s2) {
        auto n = std::make_shared<Node>();
        n->c1 = std::move(c1); n->s1 = std::move(s1); n->dual = dual; n->c2 = std::move(c2); n->s2 = std::move(s2);
        const std::vector<long> a = n->s1->costs();
        if (!dual) {
            for (long x : a) n->cost += x;
        } else {
            const std::vector<long> b = n->s2->costs();
            for (size_t r = 0; r < a.size(); ++r) n->cost += std::min(a[r], b[r]);
        }
        return n;
    }

    void start() { request_extend({{nullptr, 0}}, Then::Root); }

    // the device has answered the pending request: take its results and go on to the next request (need == None: done)
    void resume() {
        static const char kSym[4] = {'A', 'C', 'G', 'T'};
        need = Need::None;
        if (then == Then::Root) {
            queue.insert(make("", extend_result()[0], false, "", nullptr));
        } else if (then == Then::Run) {
            if (const std::shared_ptr<Node> child = run_result()) {
                queue.insert(child);
            } else {
                request_expand();
                return;
            }
        } else {
            const std::vector<SidePtr> ext = extend_result();
            const Node &node = *cur;
            if (!node.dual) {
                for (size_t a = 0; a < p1.size(); ++a) queue.insert(make(node.c1 + kSym[p1[a]], ext[a], false, "", nullptr));
                if (allow_dual && strict.size() >= 2)
                    for (size_t ia = 0; ia < strict.size(); ++ia)
                        for (size_t ib = ia + 1; ib < strict.size(); ++ib) {
                            const size_t a = static_cast<size_t>(std::find(p1.begin(), p1.end(), strict[ia]) - p1.begin());
                            const size_t b = static_cast<size_t>(std::find(p1.begin(), p1.end(), strict[ib]) - p1.begin());
                            queue.insert(make(node.c1 + kSym[strict[ia]], ext[a], true, node.c1 + kSym[strict[ib]], ext[b]));
                        }
            } else {
                // a finished side stays as it is
                const size_t n1 = std::max<size_t>(p1.size(), 1), n2 = std::max<size_t>(p2.size(), 1);
                for (size_t a = 0; a < n1; ++a)
                    for (size_t b = 0; b < n2; ++b) {
                        const bool e1 = !p1.empty(), e2 = !p2.empty();
                        queue.insert(make(e1 ? node.c1 + kSym[p1[a]] : node.c1, e1 ? ext[a] : node.s1, true,
                                          e2 ? node.c2 + kSym[p2[b]] : node.c2, e2 ? ext[p1.size() + b] : node.s2));
                    }
            }
            while (queue.size() > cfg.max_queue_size) queue.erase(std::prev(queue.end()));
        }
        advance();
    }

    // the current node's expansion on the host: one extension per (side, passing symbol)
    void request_expand() {
        static const char kSym[4] = {'A', 'C', 'G', 'T'};
        if (getenv("SP_CONSENSUS_DEBUG"))
            fprintf(stderr, "[consensus] host: dual %d size %zu cost %ld p1 %zu p2 %zu queue %zu\n", cur->dual ? 1 : 0, cur->size(), cur->cost, p1.size(),
                    p2.size(), queue.size());
        std::vector<std::pair<const Side *, char>> tasks;
        for (int k : p1) tasks.emplace_back(cur->s1.get(), kSym[k]);
        for (int k : p2) tasks.emplace_back(cur->s2.get(), kSym[k]);
        request_extend(tasks, Then::Expand);
    }

    // pops nodes until one needs the device
    void advance() {
        const long permille = std::lround(cfg.min_af * 1000.0);
        while (!queue.empty()) {
            const std::shared_ptr<Node> node = *queue.begin();
            queue.erase(queue.begin());
            if (have_best && node->cost > best_cost) break;
            p1.clear(); p2.clear(); strict.clear();
            std::vector<long> c1, c2;
            if (!node->dual) {
                const auto t1 = tally(*node->s1, nullptr);
                p1 = passing(t1, cfg);
                strict = strictly_passing(t1, cfg);
            } else {
                c1 = node->s1->costs(); c2 = node->s2->costs();
                std::vector<char> v1(c1.size()), v2(c1.size());
                for (size_t r = 0; r < c1.size(); ++r) { v1[r] = c1[r] <= c2[r]; v2[r] = c2[r] <= c1[r]; }
                p1 = passing(tally(*node->s1, &v1), cfg);
                p2 = passing(tally(*node->s2, &v2), cfg);
            }
            if (p1.empty() && p2.empty()) {  // nobody wants to go on: complete
                if (node->dual) {
                    size_t n1 = 0;
                    for (size_t r = 0; r < c1.size(); ++r) n1 += c1[r] <= c2[r];
                    const size_t n2 = c1.size() - n1, mn = std::min(n1, n2);
                    if (mn < cfg.min_count || static_cast<long>(mn) * 1000 < static_cast<long>(n1 + n2) * permille) continue;
                }
                if (!have_best || node->cost < best_cost) { best.assign(1, node); best_cost = node->cost; have_best = true; }
                else if (node->cost == best_cost) best.push_back(node);
                continue;
            }
            size_t &cnt = expanded[node->size()];
            if (cnt >= cfg.max_capacity_per_size) continue;
            ++cnt;
            cur = node;
            const bool one_way = node->dual ? (p1.size() <= 1 && p2.size() <= 1) : p1.size() == 1;
            if (one_way && can_run[node->dual ? 2 : 1]) {
                // the child is popped next for as long as it orders before every other node (cheaper, or as cheap and longer; equal
                // on both: the strings decide, here) and is not dearer than the best answer
                const long kMax = std::numeric_limits<long>::max();
                const long limit_cost = queue.empty() ? kMax : (*queue.begin())->cost;
                const long limit_size = queue.empty() ? 0 : static_cast<long>((*queue.begin())->size());
                request_run(*node, limit_cost, limit_size, have_best ? best_cost : kMax);
                return;
            }
            request_expand();
            return;
        }
        cur = nullptr;
    }
};

// Runs the searches to their end together.  Each round gathers the pending requests of every search still running into at most
// one sp_consensus_extend_batch and one sp_consensus_run_batch, then resumes each search with its own results.  A HostError of a
// search ends that search alone (errors[i]); a failed device call throws.
void drive(sp_ctx *ctx, const std::vector<Search *> &ss, std::vector<std::optional<std::string>> &errors) {
    auto step = [&](size_t i, auto &&fn) {
        try {
            fn();
        } catch (const DeviceError &) {
            throw;
        } catch (const HostError &e) {
            errors[i] = e.what();
            ss[i]->need = Search::Need::None;
        }
    };
    for (size_t i = 0; i < ss.size(); ++i)
        if (ss[i] && !errors[i]) step(i, [&] { ss[i]->start(); });
    for (;;) {
        std::vector<sp_consensus_ext> lists;
        std::vector<sp_consensus_job> jobs;
        std::vector<size_t> live;
        for (size_t i = 0; i < ss.size(); ++i) {
            if (!ss[i] || errors[i] || ss[i]->need == Search::Need::None) continue;
            live.push_back(i);
            if (ss[i]->need == Search::Need::Extend) lists.push_back(ss[i]->ext_list());
            else jobs.push_back(ss[i]->job);
        }
        if (live.empty()) break;
        if (!lists.empty() && sp_consensus_extend_batch(ctx, static_cast<int32_t>(lists.size()), lists.data()) != SP_OK)
            throw DeviceError(std::string("sp_consensus_extend_batch: ") + sp_last_error(ctx));
        if (!jobs.empty()) {
            const auto t0 = std::chrono::steady_clock::now();
            if (sp_consensus_run_batch(ctx, static_cast<int32_t>(jobs.size()), jobs.data()) != SP_OK)
                throw DeviceError(std::string("sp_consensus_run_batch: ") + sp_last_error(ctx));
            const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            for (size_t i : live)
                if (ss[i]->need == Search::Need::Run) ss[i]->run_seconds += dt;
        }
        for (size_t i : live) step(i, [&] { ss[i]->resume(); });
    }
}

struct SearchSpec {  // what a ConsensusDWFA holds
    GpuAligner *gpu;
    const CdwfaConfig *cfg;
    const SeqList *reads;
    const std::vector<int32_t> *offsets;
};

// builds one search per spec (a HostError there is that search's failure: no search, or errors[i]) and drives them all.  The
// searches are handed back because their answers (`best`) hold tracks of their pools.
std::vector<std::unique_ptr<Search>> run_searches(const std::vector<SearchSpec> &objs, bool allow_dual, std::vector<std::optional<std::string>> &errors) {
    const size_t n = objs.size();
    errors.assign(n, std::nullopt);
    std::vector<std::unique_ptr<Search>> own(n);
    if (n == 0) return own;
    sp_ctx *ctx = objs[0].gpu->raw();
    std::vector<Search *> ss(n, nullptr);
    for (size_t i = 0; i < n; ++i) {
        if (objs[i].gpu->raw() != ctx) throw HostError("consensus_batch: every search of a batch runs on the same GpuAligner");
        try {
            own[i] = std::make_unique<Search>(*objs[i].gpu, *objs[i].cfg, *objs[i].reads, *objs[i].offsets, allow_dual);
            ss[i] = own[i].get();
        } catch (const HostError &e) {
            errors[i] = e.what();
        }
    }
    drive(ctx, ss, errors);
    return own;
}
}  // namespace

void ConsensusDWFA::add_sequence_offset(const std::string &sequence, std::optional<size_t> offset) {
    reads_.push_back(sequence);
    offsets_.push_back(offset ? static_cast<int32_t>(*offset) : -1);  // -1: anchored at the consensus start
}

std::vector<SearchResult<Consensus>> ConsensusDWFA::consensus_batch(const std::vector<ConsensusDWFA *> &searches) {
    std::vector<std::optional<std::string>> errors;
    std::vector<SearchSpec> specs;
    for (ConsensusDWFA *c : searches) specs.push_back({&c->gpu_, &c->config_, &c->reads_, &c->offsets_});
    const std::vector<std::unique_ptr<Search>> ss = run_searches(specs, false, errors);
    std::vector<SearchResult<Consensus>> out(searches.size());
    for (size_t i = 0; i < searches.size(); ++i) {
        searches[i]->n_calls_ = ss[i] ? ss[i]->n_calls : 0;
        out[i].error = errors[i];
        if (errors[i]) continue;
        for (const auto &n : ss[i]->best) {
            Consensus c;
            c.sequence = n->c1;
            for (long x : n->s1->costs()) c.scores.push_back(static_cast<size_t>(x));
            out[i].list.push_back(std::move(c));
        }
    }
    return out;
}

std::vector<Consensus> ConsensusDWFA::consensus() {
    std::vector<SearchResult<Consensus>> r = consensus_batch({this});
    if (r[0].error) throw HostError(*r[0].error);
    return std::move(r[0].list);
}

std::vector<SearchResult<DualConsensus>> DualConsensusDWFA::consensus_batch(const std::vector<DualConsensusDWFA *> &searches) {
    std::vector<ConsensusDWFA *> inner;
    for (DualConsensusDWFA *d : searches) inner.push_back(&d->inner_);
    std::vector<std::optional<std::string>> errors;
    std::vector<SearchSpec> specs;
    for (ConsensusDWFA *c : inner) specs.push_back({&c->gpu_, &c->config_, &c->reads_, &c->offsets_});
    const std::vector<std::unique_ptr<Search>> ss = run_searches(specs, true, errors);
    std::vector<SearchResult<DualConsensus>> out(searches.size());
    for (size_t i = 0; i < searches.size(); ++i) {
        inner[i]->n_calls_ = ss[i] ? ss[i]->n_calls : 0;
        out[i].error = errors[i];
        if (errors[i]) continue;
        for (const auto &n : ss[i]->best) {
            DualConsensus d;
            d.consensus1 = n->c1;
            const std::vector<long> a = n->s1->costs();
            if (!n->dual) {
                d.is_consensus1.assign(a.size(), true);
                for (long x : a) d.scores1.emplace_back(static_cast<size_t>(x));
                d.scores2.assign(a.size(), std::nullopt);
            } else {
                d.consensus2 = n->c2;
                const std::vector<long> b = n->s2->costs();
                for (size_t r = 0; r < a.size(); ++r) {
                    d.is_consensus1.push_back(a[r] <= b[r]);
                    d.scores1.emplace_back(static_cast<size_t>(a[r]));
                    d.scores2.emplace_back(static_cast<size_t>(b[r]));
                }
            }
            out[i].list.push_back(std::move(d));
        }
    }
    return out;
}

std::vector<DualConsensus> DualConsensusDWFA::consensus() {
    std::vector<SearchResult<DualConsensus>> r = consensus_batch({this});
    if (r[0].error) throw HostError(*r[0].error);
    return std::move(r[0].list);
}

// ------------------------------------------------------------------------------------------
// PriorityConsensusDWFA (see starphase_host.hpp for the outline restated here)
// ------------------------------------------------------------------------------------------
void PriorityConsensusDWFA::add_seeded_sequence_chain(const std::vector<std::string> &sequence_chain,
                                                      const std::vector<std::optional<size_t>> &offset_chain, std::optional<uint64_t> seed) {
    if (sequence_chain.empty() || sequence_chain.size() != offset_chain.size()) throw HostError("priority consensus: one offset per chain level expected");
    if (!chains_.empty() && chains_[0].size() != sequence_chain.size()) throw HostError("priority consensus: every chain needs the same number of levels");
    chains_.push_back(sequence_chain); offsets_.push_back(offset_chain); seeds_.push_back(seed);
}

PriorityConsensus PriorityConsensusDWFA::consensus() {
    if (chains_.empty()) throw HostError("priority consensus: no sequences were added");
    const size_t levels = chains_[0].size();
    struct Group {
        std::vector<size_t> members;
        size_t level = 0;
        std::vector<std::optional<Consensus>> known;  // single consensus of exactly these members, per level, where a run gave it
    };
    // seeds first: unseeded inputs together, then one group per seed value (ascending)
    std::map<std::pair<bool, uint64_t>, std::vector<size_t>> by_seed;
    for (size_t i = 0; i < chains_.size(); ++i) by_seed[{seeds_[i].has_value(), seeds_[i].value_or(0)}].push_back(i);
    std::vector<Group> work, done;
    for (auto it = by_seed.rbegin(); it != by_seed.rend(); ++it) work.push_back({it->second, 0, std::vector<std::optional<Consensus>>(levels)});
    // every group in `work` is independent of the others: each round examines all of them in one batch
    while (!work.empty()) {
        std::vector<Group> round;
        for (Group &g : work) (g.level == levels ? done : round).push_back(std::move(g));
        work.clear();
        std::vector<std::unique_ptr<DualConsensusDWFA>> dwfas;
        std::vector<DualConsensusDWFA *> batch;
        for (const Group &g : round) {
            dwfas.push_back(std::make_unique<DualConsensusDWFA>(gpu_, config_));
            for (size_t i : g.members) dwfas.back()->add_sequence_offset(chains_[i][g.level], offsets_[i][g.level]);
            batch.push_back(dwfas.back().get());
        }
        const std::vector<SearchResult<DualConsensus>> results = DualConsensusDWFA::consensus_batch(batch);
        for (size_t k = 0; k < round.size(); ++k) {
            Group &g = round[k];
            if (results[k].error) throw HostError(*results[k].error);
            if (results[k].list.empty()) throw HostError("priority consensus: no consensus found");
            const DualConsensus &d = results[k].list[0];
            if (d.is_dual()) {  // two groups, each examined again at this level
                Group a{{}, g.level, std::vector<std::optional<Consensus>>(levels)}, b = a;
                for (size_t m = 0; m < g.members.size(); ++m) (d.is_consensus1[m] ? a : b).members.push_back(g.members[m]);
                work.push_back(std::move(b)); work.push_back(std::move(a));
            } else {
                Consensus c;
                c.sequence = d.consensus1;
                for (const auto &x : d.scores1) c.scores.push_back(x.value_or(0));
                g.known[g.level] = std::move(c);
                ++g.level;
                work.push_back(std::move(g));
            }
        }
    }
    std::sort(done.begin(), done.end(), [](const Group &a, const Group &b) { return a.members.front() < b.members.front(); });
    // the split happened at a later level: the levels only seen for the larger group, every (group, level) in one batch
    std::vector<std::unique_ptr<ConsensusDWFA>> singles;
    std::vector<ConsensusDWFA *> batch;
    std::vector<std::pair<size_t, size_t>> slot;  // (group, level) of every single
    for (size_t gi = 0; gi < done.size(); ++gi)
        for (size_t l = 0; l < levels; ++l)
            if (!done[gi].known[l]) {
                singles.push_back(std::make_unique<ConsensusDWFA>(gpu_, config_));
                for (size_t i : done[gi].members) singles.back()->add_sequence_offset(chains_[i][l], offsets_[i][l]);
                batch.push_back(singles.back().get());
                slot.emplace_back(gi, l);
            }
    const std::vector<SearchResult<Consensus>> results = ConsensusDWFA::consensus_batch(batch);
    for (size_t k = 0; k < slot.size(); ++k) {
        if (results[k].error) throw HostError(*results[k].error);
        if (results[k].list.empty()) throw HostError("priority consensus: no consensus found");
        done[slot[k].first].known[slot[k].second] = results[k].list[0];
    }
    PriorityConsensus out;
    out.sequence_indices.assign(chains_.size(), 0);
    for (size_t gi = 0; gi < done.size(); ++gi) {
        Group &g = done[gi];
        std::vector<Consensus> per_level;
        for (size_t l = 0; l < levels; ++l) per_level.push_back(*g.known[l]);
        out.consensuses.push_back(std::move(per_level));
        for (size_t i : g.members) out.sequence_indices[i] = gi;
    }
    return out;
}

// ------------------------------------------------------------------------------------------
// the consensus step of the HLA caller
// ------------------------------------------------------------------------------------------
CdwfaConfig dwfa_config_from_cli(const DiplotypeSettings &cli, bool allow_early_termination) {  // src/hla/caller.rs:1097-1116
    CdwfaConfig c;
    c.min_count = cli.min_consensus_count;
    c.min_af = cli.min_consensus_fraction;
    c.dual_max_ed_delta = cli.dual_max_ed_delta;
    c.allow_early_termination = allow_early_termination;
    c.max_queue_size = 20;
    c.max_capacity_per_size = 10;
    c.offset_window = 400;
    return c;
}

DualPassingStats is_passing_dual(const DualConsensus &d, const DiplotypeSettings &cli) {  // :1225-1247
    size_t counts1 = 0;
    for (bool b : d.is_consensus1) counts1 += b;
    return dual_passing_stats(d.is_dual(), counts1, d.is_consensus1.size() - counts1, cli.min_consensus_fraction, cli.min_cdf, cli.expected_maf);
}

DualConsensus run_dual_consensus(GpuAligner &gpu, const std::map<std::string, std::string> &segments, const DiplotypeSettings &cli) {  // :1126-1139
    DualConsensusDWFA dwfa(gpu, dwfa_config_from_cli(cli, false));
    for (const auto &kv : segments) dwfa.add_sequence(kv.second);
    std::vector<DualConsensus> list = dwfa.consensus();
    if (list.empty()) throw HostError("run_dual_consensus: no consensus found");
    return list[0];  // "Found multiple solutions, selecting first."
}

namespace {
// one pass of :1163-1177 / :1196-1211: every record's sequence with its offset relative to the smallest (+ half the window; the
// smallest anchored); which = the HPC or the full-length members of RealignedHlaRecord
DualConsensus dual_pass(GpuAligner &gpu, const std::map<std::string, RealignmentResult> &segments, const CdwfaConfig &config, bool hpc) {
    const size_t half_window = config.offset_window / 2;
    size_t min_offset = static_cast<size_t>(-1);
    for (const auto &kv : segments) {
        if (!kv.second.realigned_record) throw HostError("run_dual_consensus_with_offsets: a record was not realigned");
        min_offset = std::min(min_offset, hpc ? kv.second.realigned_record->hpc_offset : kv.second.realigned_record->dna_offset);
    }
    DualConsensusDWFA dwfa(gpu, config);
    for (const auto &kv : segments) {
        const RealignedHlaRecord &rec = *kv.second.realigned_record;
        const size_t o = hpc ? rec.hpc_offset : rec.dna_offset;
        dwfa.add_sequence_offset(hpc ? rec.hpc_sequence : rec.dna_sequence, o == min_offset ? std::nullopt : std::optional<size_t>(o - min_offset + half_window));
    }
    std::vector<DualConsensus> list = dwfa.consensus();
    if (list.empty()) throw HostError("run_dual_consensus_with_offsets: no consensus found");
    return list[0];
}
}  // namespace

DualConsensus run_dual_consensus_with_offsets(GpuAligner &gpu, const std::map<std::string, RealignmentResult> &segments,
                                              const DiplotypeSettings &cli) {  // :1151-1219
    if (segments.empty()) throw HostError("run_dual_consensus_with_offsets: no records");
    const CdwfaConfig config = dwfa_config_from_cli(cli, true);
    const DualConsensus hpc = dual_pass(gpu, segments, config, true);
    if (is_passing_dual(hpc, cli).is_passing) return hpc;  // :1180-1190
    return dual_pass(gpu, segments, config, false);         // HPC did not find a difference: full-length DNA
}

std::pair<std::string, std::optional<std::string>> consensus_per_group(GpuAligner &gpu, const std::map<std::string, RealignmentResult> &segments,
                                                                       const std::vector<bool> &is_consensus1, bool is_dual,
                                                                       const DiplotypeSettings &cli) {  // :706-760, :817-836
    if (is_consensus1.size() != segments.size()) throw HostError("consensus_per_group: one assignment per record expected");
    const CdwfaConfig config = dwfa_config_from_cli(cli, true);
    const size_t half_window = config.offset_window / 2;
    size_t min1 = static_cast<size_t>(-1), min2 = static_cast<size_t>(-1), r = 0;
    for (const auto &kv : segments) {
        if (!kv.second.realigned_record) throw HostError("consensus_per_group: a record was not realigned");
        size_t &m = is_consensus1[r++] ? min1 : min2;
        m = std::min(m, kv.second.realigned_record->dna_offset);
    }
    ConsensusDWFA d1(gpu, config), d2(gpu, config);
    size_t n1 = 0, n2 = 0;
    r = 0;
    for (const auto &kv : segments) {
        const RealignedHlaRecord &rec = *kv.second.realigned_record;
        const bool first = is_consensus1[r++];
        const size_t mn = first ? min1 : min2;
        (first ? d1 : d2).add_sequence_offset(rec.dna_sequence, rec.dna_offset == mn ? std::nullopt : std::optional<size_t>(rec.dna_offset - mn + half_window));
        ++(first ? n1 : n2);
    }
    // both groups in one batch; a failed consensus is the empty string (:735-749), and does not stop the other group
    std::vector<ConsensusDWFA *> batch;
    if (n1) batch.push_back(&d1);
    if (is_dual && n2) batch.push_back(&d2);
    const std::vector<SearchResult<Consensus>> results = ConsensusDWFA::consensus_batch(batch);
    auto first_or_empty = [&](const ConsensusDWFA &d) -> std::string {
        for (size_t k = 0; k < batch.size(); ++k)
            if (batch[k] == &d) return results[k].error || results[k].list.empty() ? std::string() : results[k].list[0].sequence;
        return std::string();  // no reads
    };
    std::pair<std::string, std::optional<std::string>> out;
    out.first = first_or_empty(d1);
    if (is_dual) out.second = first_or_empty(d2);
    return out;
}

// ------------------------------------------------------------------------------------------
// the consensus stage of the CYP2D6 caller (src/cyp2d6/caller.rs:145-310, :750-893)
// ------------------------------------------------------------------------------------------
std::pair<std::string, size_t> hpc_with_guide(const std::string &sequence, const std::string &guide_sequence, size_t guide_offset) {
    return {hpc(sequence), hpc_pos(guide_sequence, guide_offset)};  // src/util/homopolymers.rs:53-64
}

CdwfaConfig cyp2d6_consensus_config(const DiplotypeSettings &cli) {  // :145-162
    CdwfaConfig c;
    c.min_count = cli.min_consensus_count;
    c.min_af = cli.min_consensus_fraction;
    c.dual_max_ed_delta = cli.dual_max_ed_delta;
    c.allow_early_termination = true;
    c.max_queue_size = 20;
    c.max_capacity_per_size = 10;
    c.offset_window = 2 * 50;  // "+-50 bp, but the config only lets us look before" (:147-148)
    return c;
}

Cyp2d6ConsensusInputs cyp2d6_consensus_inputs(const std::map<std::string, std::string> &read_sequences,
                                              const std::map<std::string, std::vector<AlleleMapping>> &regions_of_interest,
                                              const Cyp2d6Extractor &d6_typer, double max_missing_consensus_frac, size_t offset_window) {
    Cyp2d6ConsensusInputs in;
    auto get_allele = [&](const Cyp2d6RegionLabel &label) -> const std::string & {  // Cyp2d6Extractor::get_allele
        for (const auto &t : d6_typer.hybrid_sequences())
            if (t.first.region_type == label.region_type && t.first.subtype_label == label.subtype_label) return t.second;
        throw HostError("cyp2d6_consensus_inputs: no template for " + label.full_allele());
    };
    for (const auto &kv : regions_of_interest) {  // BTreeMap order (:178)
        const auto rs = read_sequences.find(kv.first);
        if (rs == read_sequences.end()) throw HostError("cyp2d6_consensus_inputs: no sequence for read " + kv.first);
        for (const AlleleMapping &region : kv.second) {
            if (region.mapping_stats.custom_score(true) > max_missing_consensus_frac) continue;  // :181-184
            if (region.region_end > rs->second.size() || region.region_start > region.region_end)
                throw HostError("cyp2d6_consensus_inputs: region outside read " + kv.first);
            const size_t prefix_len = region.mapping_stats.clipped_start.value_or(0);
            const std::string seq = rs->second.substr(region.region_start, region.region_end - region.region_start);
            const auto hp = hpc_with_guide(seq, get_allele(region.allele_label), prefix_len);  // :200-202
            in.raw_sequences.push_back(seq);
            in.base_offsets.push_back(prefix_len == 0 ? 0 : prefix_len + offset_window);      // :195-199
            in.hpc_sequences.push_back(hp.first);
            in.hpc_offsets.push_back(hp.second == 0 ? 0 : hp.second + offset_window);         // :204-208
            in.sequence_ids.push_back(kv.first + "_" + std::to_string(region.region_start) + "_" + std::to_string(region.region_end) + "_" +
                                      region.allele_label.full_allele());
            in.flattened_regions_of_interest.emplace_back(kv.first, region);
            std::optional<uint64_t> seed;  // :224-231
            switch (region.allele_label.region_type) {
                case Cyp2d6RegionType::Cyp2d6Deletion: seed = 0; break;
                case Cyp2d6RegionType::Rep6: seed = 1; break;
                case Cyp2d6RegionType::Rep7: seed = 2; break;
                case Cyp2d6RegionType::Spacer: seed = 3; break;
                case Cyp2d6RegionType::LinkRegion: seed = 4; break;
                default: break;
            }
            in.seeds.push_back(seed);
        }
    }
    return in;
}

PriorityConsensus cyp2d6_priority_consensus(GpuAligner &gpu, const Cyp2d6ConsensusInputs &in, const CdwfaConfig &config) {
    PriorityConsensusDWFA dwfa(gpu, config);
    auto opt = [](size_t v) { return v == 0 ? std::nullopt : std::optional<size_t>(v); };  // offset 0 = auto-start (:243-254)
    for (size_t i = 0; i < in.raw_sequences.size(); ++i)
        dwfa.add_seeded_sequence_chain({in.hpc_sequences[i], in.raw_sequences[i]}, {opt(in.hpc_offsets[i]), opt(in.base_offsets[i])}, in.seeds[i]);
    return dwfa.consensus();
}

MultiConsensus merge_consensus_results(GpuAligner &gpu, const SeqList &sequences, const std::vector<size_t> &offsets,
                                       const CdwfaConfig &cdwfa_config, const PriorityConsensus &raw, Cyp2d6Extractor &d6_typer,
                                       const Cyp2d6TypingDb &db, const Cyp2d6Config &cyp2d6_config, double max_missing_consensus_frac) {
    if (sequences.size() != offsets.size() || sequences.size() != raw.sequence_indices.size())
        throw HostError("merge_consensus_results: one offset and one consensus index per sequence expected");
    const std::string unknown = Cyp2d6RegionLabel{}.full_allele();
    // every consensus is typed in one batch (:760-782); "no matches found" is the reference's error branch -> unknown
    SeqList to_type;
    for (const auto &levels : raw.consensuses) {
        if (levels.size() < 2) throw HostError("merge_consensus_results: (HPC, full) consensus pairs expected");
        const std::string &full = levels[1].sequence;
        const size_t b = full.find_first_not_of('*'), e = full.find_last_not_of('*');
        to_type.push_back(b == std::string::npos ? std::string() : full.substr(b, e - b + 1));  // trim_matches('*')
    }
    const bool force_assignment = false;
    const std::vector<std::optional<Cyp2d6Region>> typed = d6_typer.find_full_type_in_sequences(to_type, max_missing_consensus_frac, force_assignment, db);
    std::map<std::pair<std::string, std::string>, std::vector<size_t>> consensus_set;
    std::map<std::string, std::vector<size_t>> unknown_set;
    for (size_t i = 0; i < raw.consensuses.size(); ++i) {
        const Cyp2d6RegionLabel label = typed[i] ? typed[i]->label : Cyp2d6RegionLabel{};
        const std::string reduced = label.simplify_allele(true, cyp2d6_config.cyp_translate);  // keeps sub-alleles such as "*4.001"
        if (!label.is_allowed_label()) unknown_set[raw.consensuses[i][0].sequence].push_back(i);
        else consensus_set[{raw.consensuses[i][0].sequence, reduced}].push_back(i);
    }
    std::set<std::pair<std::string, std::string>> intentional_ignore;  // :797-835
    for (auto &kv : unknown_set) {
        std::vector<std::pair<std::string, std::string>> other_keys;
        for (const auto &ck : consensus_set)
            if (ck.first.first == kv.first) other_keys.push_back(ck.first);
        if (other_keys.size() == 1) {
            std::vector<size_t> &entry = consensus_set[other_keys[0]];
            entry.insert(entry.end(), kv.second.begin(), kv.second.end());
        } else {
            const std::pair<std::string, std::string> key{kv.first, unknown};
            if (other_keys.size() > 1) intentional_ignore.insert(key);
            if (!consensus_set.emplace(key, kv.second).second) throw HostError("merge_consensus_results: duplicate unknown key");
        }
    }
    MultiConsensus out;
    out.sequence_indices.assign(raw.sequence_indices.size(), std::numeric_limits<size_t>::max());
    std::vector<std::unique_ptr<ConsensusDWFA>> merges;  // the merged groups, re-solved together below
    std::vector<size_t> merge_slot;                      // their place in out.consensuses
    for (const auto &kv : consensus_set) {
        const std::vector<size_t> &con_indices = kv.second;
        const size_t con_index = out.consensuses.size();
        auto contains = [&](size_t v) { return std::find(con_indices.begin(), con_indices.end(), v) != con_indices.end(); };
        Consensus consensus;
        if (intentional_ignore.count(kv.first)) {  // a group with several possible parents: kept empty (:842-854)
            size_t num_scored = 0;
            for (size_t i = 0; i < raw.sequence_indices.size(); ++i)
                if (contains(raw.sequence_indices[i])) { out.sequence_indices[i] = con_index; ++num_scored; }
            consensus.scores.assign(num_scored, 0);
        } else if (con_indices.size() == 1) {  // the full-length consensus as it is (:855-864)
            for (size_t i = 0; i < raw.sequence_indices.size(); ++i)
                if (raw.sequence_indices[i] == con_indices[0]) out.sequence_indices[i] = con_index;
            consensus = raw.consensuses[con_indices[0]][1];
        } else {  // a merge: one consensus of all their raw sequences (:865-886)
            merges.push_back(std::make_unique<ConsensusDWFA>(gpu, cdwfa_config));
            merge_slot.push_back(con_index);
            for (size_t si = 0; si < sequences.size(); ++si)
                if (contains(raw.sequence_indices[si])) {
                    merges.back()->add_sequence_offset(sequences[si], offsets[si] == 0 ? std::nullopt : std::optional<size_t>(offsets[si]));
                    out.sequence_indices[si] = con_index;
                }
        }
        out.consensuses.push_back(std::move(consensus));
    }
    std::vector<ConsensusDWFA *> batch;
    for (const auto &m : merges) batch.push_back(m.get());
    const std::vector<SearchResult<Consensus>> results = ConsensusDWFA::consensus_batch(batch);
    for (size_t k = 0; k < merges.size(); ++k) {
        if (results[k].error) throw HostError(*results[k].error);
        if (results[k].list.empty()) throw HostError("merge_consensus_results: no consensus for a merged group");
        out.consensuses[merge_slot[k]] = results[k].list[0];  // "Multiple consensuses found during collapse, picking first."
    }
    for (size_t v : out.sequence_indices)
        if (v >= out.consensuses.size()) throw HostError("merge_consensus_results: a sequence lost its consensus");
    return out;
}

}  // namespace starphase
