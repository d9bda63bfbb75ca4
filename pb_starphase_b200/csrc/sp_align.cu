// sp_align.cu -- K4 host side: sp_align_resident / sp_align_pairs / sp_align_windows (include/starphase_gpu.h), and the
// pair-call steps K4 and K9 (sp_affine.cu) share: argument checks, pair resolution, buffers and the readback.
//
// Plan (host, O(pairs log pairs)): every pair gets the lane width its pattern needs (U = 4 / 8 / 12 / 16 / 20 / 24); the pairs
// of one width are packed best-fit-decreasing into 32-lane bins -- several pairs per warp, each with its own text -- and every
// width is one launch of k4_align<U> over a work list of bins, two passes per pair (sp_align.cuh).  The sequences are
// device-resident (sp_targets handles): a call moves only the pair list and the plan tables in, the records and the dense
// CIGAR pool out.
#include "sp_internal.cuh"

#define SP_NO_GLOBAL_KERNELS  // the non-template kernels of sp_kernels.cuh are instantiated in starphase_gpu.cu
#include "sp_kernels.cuh"
#include "sp_align.cuh"

using namespace sp;

static_assert(sizeof(sp_align_rec) == sizeof(AlignRecDev), "sp_align_rec layout");

sp_status pair_call_check(sp_ctx *ctx, const char *fn, const void *texts, const void *patterns, int64_t n_pairs, const int32_t *pair_text,
                          const int32_t *pair_pattern, const int32_t *win_begin, const int32_t *win_end, const sp_align_rec *recs,
                          const uint32_t *cigar, int64_t cigar_cap, int64_t *cigar_used) {
    const std::string f(fn);
    if (!texts || !patterns) return fail(ctx, SP_ERR_INVALID, f + ": NULL sequence set");
    if ((win_begin == nullptr) != (win_end == nullptr)) return fail(ctx, SP_ERR_INVALID, f + ": win_begin and win_end go together");
    if (n_pairs < 0 || (n_pairs > 0 && (!pair_text || !pair_pattern || !recs)) || cigar_cap < 0 || (cigar_cap > 0 && !cigar))
        return fail(ctx, SP_ERR_INVALID, f + ": bad argument");
    if (cigar_used) *cigar_used = 0;
    if (n_pairs > 0x7FFFFFF0ll) return fail(ctx, SP_ERR_RANGE, f + ": too many pairs");
    return SP_OK;
}

sp_status pair_resolve(sp_ctx *ctx, const char *fn, const sp_targets *texts, const sp_targets *patterns, int64_t q, const int32_t *pair_text,
                       const int32_t *pair_pattern, const int32_t *win_begin, const int32_t *win_end, int64_t &t_off, int64_t &n, int64_t &m) {
    const int64_t t = pair_text[q], pi = pair_pattern[q];
    if (t < 0 || t >= texts->n || pi < 0 || pi >= patterns->n)
        return fail(ctx, SP_ERR_INVALID, std::string(fn) + ": pair index outside the sequence sets");
    m = patterns->h_offs[static_cast<size_t>(pi) + 1] - patterns->h_offs[static_cast<size_t>(pi)];
    n = texts->h_offs[static_cast<size_t>(t) + 1] - texts->h_offs[static_cast<size_t>(t)];
    t_off = texts->h_offs[static_cast<size_t>(t)];
    if (win_begin) {
        if (win_begin[q] < 0 || win_end[q] < win_begin[q] || win_end[q] > n)
            return fail(ctx, SP_ERR_INVALID, std::string(fn) + ": window outside its text");
        t_off += win_begin[q];
        n = win_end[q] - win_begin[q];
    }
    return SP_OK;
}

PairCall::~PairCall() {
    dev_free(ctx, recs); dev_free(ctx, scores); dev_free(ctx, used);
}

sp_status PairCall::alloc(int64_t n_pairs, int64_t cig_total, int64_t cigar_cap, bool with_scores, int n_used) {
    sp_status st = cuda_status(ctx, fn, ctx_pool(ctx, 1, static_cast<size_t>(cig_total) * 4, reinterpret_cast<void **>(&cigar)), "cigar pool");
    if (st == SP_OK)
        st = cuda_status(ctx, fn, ctx_pool(ctx, 3, static_cast<size_t>(std::max<int64_t>(cigar_cap, 4)) * 4, reinterpret_cast<void **>(&dense)),
                         "dense cigar pool");
    const size_t rec_bytes = static_cast<size_t>(n_pairs) * sizeof(AlignRecDev);
    if (st == SP_OK) st = cuda_status(ctx, fn, dev_malloc(ctx, &recs, rec_bytes), "cudaMalloc recs");
    if (st == SP_OK) st = cuda_status(ctx, fn, cudaMemsetAsync(recs, 0, rec_bytes, ctx->stream), "memset");
    if (st == SP_OK && with_scores) st = cuda_status(ctx, fn, dev_malloc(ctx, &scores, static_cast<size_t>(n_pairs) * 4), "cudaMalloc scores");
    if (st == SP_OK) st = cuda_status(ctx, fn, dev_malloc(ctx, &used, n_used * sizeof(unsigned long long)), "cudaMalloc");
    if (st == SP_OK) st = cuda_status(ctx, fn, cudaMemsetAsync(used, 0, n_used * sizeof(unsigned long long), ctx->stream), "memset");
    return st;
}

sp_status PairCall::finish(int64_t n_pairs, sp_align_rec *out_recs, int32_t *out_scores, uint32_t *out_cigar, int64_t cigar_cap,
                           int64_t *cigar_used, PhaseTimer &tm) {
    std::vector<sp_align_rec> hrec(static_cast<size_t>(n_pairs));  // AlignRecDev has sp_align_rec's layout
    std::vector<int32_t> hscores(scores ? static_cast<size_t>(n_pairs) : 0);
    unsigned long long fill = 0;
    sp_status st = cuda_status(ctx, fn, cudaMemcpyAsync(hrec.data(), recs, hrec.size() * sizeof(sp_align_rec), cudaMemcpyDeviceToHost, ctx->stream), "D2H recs");
    if (st == SP_OK && scores)
        st = cuda_status(ctx, fn, cudaMemcpyAsync(hscores.data(), scores, hscores.size() * 4, cudaMemcpyDeviceToHost, ctx->stream), "D2H scores");
    if (st == SP_OK) st = cuda_status(ctx, fn, cudaMemcpyAsync(&fill, used, sizeof(fill), cudaMemcpyDeviceToHost, ctx->stream), "D2H");
    if (st == SP_OK) st = cuda_status(ctx, fn, cudaStreamSynchronize(ctx->stream), "kernels");
    if (st != SP_OK) return st;
    tm.mark("kernels + recs D2H");
    if (cigar_used) *cigar_used = static_cast<int64_t>(fill);
    if (fill > static_cast<unsigned long long>(cigar_cap))
        return fail(ctx, SP_ERR_RANGE, std::string(fn) + ": cigar buffer too small: " + std::to_string(fill) + " entries needed");
    if (fill > 0) {
        st = cuda_status(ctx, fn, cudaMemcpyAsync(out_cigar, dense, static_cast<size_t>(fill) * 4, cudaMemcpyDeviceToHost, ctx->stream), "D2H cigar");
        if (st == SP_OK) st = cuda_status(ctx, fn, cudaStreamSynchronize(ctx->stream), "D2H cigar");
        if (st != SP_OK) return st;
    }
    std::copy(hrec.begin(), hrec.end(), out_recs);
    std::copy(hscores.begin(), hscores.end(), out_scores);
    tm.mark("cigar D2H");
    return SP_OK;
}

namespace {

struct PairPlan {
    int64_t q;       // index in the caller's pair list
    int32_t p;       // pattern index
    int32_t m, n;    // pattern length, text (window) length
    int32_t nl;      // lanes
    int64_t t_off;   // first text byte in the device buffer
};

struct ClassPlan {
    int U = 0;
    std::vector<PairPlan> pairs;
    // filled by pack_bins
    int n_bins = 0;
    std::vector<int32_t> lane_pair, lane_first;
    LaneTables lanes;
    std::vector<AlignPairDev> dev_pairs;
    int64_t slot_words = 4;
};

int lane_width_for(int64_t m) { return m <= 4096 ? 4 : m <= 8192 ? 8 : m <= 12288 ? 12 : m <= 16384 ? 16 : m <= 20480 ? 20 : 24; }

// pairs of equal lane count stay in order of decreasing text length, so the pairs sharing a warp have similar pass lengths
void pack_bins(ClassPlan &c, int64_t &cig_total) {
    const int U = c.U;
    const int64_t rows = 32ll * U;
    std::stable_sort(c.pairs.begin(), c.pairs.end(), [](const PairPlan &a, const PairPlan &b) {
        if (a.nl != b.nl) return a.nl > b.nl;
        return a.n > b.n;
    });
    std::vector<int> nl(c.pairs.size());
    for (size_t k = 0; k < c.pairs.size(); ++k) nl[k] = c.pairs[k].nl;
    std::vector<LaneSlot> at;
    c.n_bins = sp_internal_pack_lanes(nl, &at);
    c.lanes.resize(c.n_bins);
    c.lane_pair.assign(static_cast<size_t>(c.n_bins) * 32, -1);
    c.lane_first.assign(static_cast<size_t>(c.n_bins) * 32, 0);
    std::vector<int64_t> bin_words(static_cast<size_t>(c.n_bins), 0);
    c.dev_pairs.resize(c.pairs.size());
    for (size_t k = 0; k < c.pairs.size(); ++k) {
        const PairPlan &pp = c.pairs[k];
        const int bin = at[k].bin, start = at[k].lane0;
        c.lanes.place(bin, start, pp.nl, pp.p, pp.m, U);
        for (int li = 0; li < pp.nl; ++li) {
            const size_t o = static_cast<size_t>(bin) * 32 + start + li;
            c.lane_pair[o] = static_cast<int32_t>(k);
            c.lane_first[o] = start;
        }
        const int64_t pad = static_cast<int64_t>(pp.nl) * rows - pp.m;
        const int64_t ncols = std::min<int64_t>(pp.n, 2ll * pp.m);  // pass 2's window = m + d columns, d <= m
        const int64_t Wp = static_cast<int64_t>(pp.nl) * U - ((pad >> 5) & ~3ll);
        AlignPairDev &d = c.dev_pairs[k];
        d.t_off = pp.t_off;
        d.scr_off = bin_words[static_cast<size_t>(bin)];
        d.cig_off = cig_total;
        d.n = pp.n; d.m = pp.m;
        d.cig_len = static_cast<int32_t>(pp.m + ncols + 1);
        d.out = static_cast<int32_t>(pp.q);
        bin_words[static_cast<size_t>(bin)] += (ncols * 2 * Wp + 7) / 8 * 8;  // 32-byte aligned pair regions (STG.256)
        cig_total += d.cig_len;
    }
    for (int64_t w : bin_words) c.slot_words = std::max(c.slot_words, w);
    c.slot_words = (c.slot_words + 7) / 8 * 8;
}

template <int U>
sp_status launch_class(sp_ctx *ctx, const AlignParams &prm, int grid) {
    const size_t smem = static_cast<size_t>(K4_WARPS) * blob_words(U) * 4;
    SP_CUDA(ctx, cudaFuncSetAttribute(k4_align<U>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    k4_align<U><<<grid, 32 * K4_WARPS, smem, ctx->stream>>>(prm);
    ++ctx->launches;
    SP_CUDA(ctx, cudaGetLastError());
    return SP_OK;
}

template <int U>
int class_occupancy() {
    int occ = 0;
    const size_t smem = static_cast<size_t>(K4_WARPS) * blob_words(U) * 4;
    cudaFuncSetAttribute(k4_align<U>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k4_align<U>, 32 * K4_WARPS, smem) != cudaSuccess) occ = 1;
    return std::max(occ, 1);
}

}  // namespace

extern "C" sp_status sp_align_resident(sp_ctx *ctx, const sp_targets *texts, const sp_targets *patterns, int64_t n_pairs,
                                       const int32_t *pair_text, const int32_t *pair_pattern, const int32_t *win_begin,
                                       const int32_t *win_end, sp_align_rec *recs, uint32_t *cigar, int64_t cigar_cap,
                                       int64_t *cigar_used) {
    if (!ctx) return SP_ERR_INVALID;
    const char *fn = "sp_align_resident";
    sp_status st = pair_call_check(ctx, fn, texts, patterns, n_pairs, pair_text, pair_pattern, win_begin, win_end, recs, cigar, cigar_cap, cigar_used);
    if (st != SP_OK || n_pairs == 0) return st;
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    PhaseTimer tm;

    // ---- plan ----
    std::map<int, ClassPlan> classes;  // key = U
    for (int64_t q = 0; q < n_pairs; ++q) {
        int64_t t_off, n, m;
        st = pair_resolve(ctx, fn, texts, patterns, q, pair_text, pair_pattern, win_begin, win_end, t_off, n, m);
        if (st != SP_OK) return st;
        if (m > SP_MAX_PATTERN_LEN) return fail(ctx, SP_ERR_TOO_LONG, "sp_align_resident: pattern exceeds SP_MAX_PATTERN_LEN");
        if (n > 0x7FFFFF00ll) return fail(ctx, SP_ERR_TOO_LONG, "sp_align_resident: text too long");
        if (m == 0) continue;  // empty pattern: distance 0, empty placement at column 0 = the zeroed record
        const int U = lane_width_for(m);
        ClassPlan &c = classes[U];
        c.U = U;
        PairPlan pp;
        pp.q = q; pp.p = pair_pattern[q];
        pp.m = static_cast<int32_t>(m); pp.n = static_cast<int32_t>(n);
        pp.nl = static_cast<int32_t>((m + 32ll * U - 1) / (32ll * U));
        pp.t_off = t_off;
        c.pairs.push_back(pp);
    }
    if (classes.empty()) {  // only empty patterns: nothing to launch
        std::fill(recs, recs + n_pairs, sp_align_rec{});
        return SP_OK;
    }
    int64_t cig_total = 0, max_slot_words = 4, max_bins = 0, blob_words_max = 0;
    for (auto &kv : classes) {
        pack_bins(kv.second, cig_total);
        max_slot_words = std::max(max_slot_words, kv.second.slot_words);
        max_bins = std::max<int64_t>(max_bins, kv.second.n_bins);
        blob_words_max = std::max<int64_t>(blob_words_max, static_cast<int64_t>(kv.second.n_bins) * blob_words(kv.second.U));
    }
    tm.mark("plan");
    if (max_slot_words > (24ll << 30) / 4) return fail(ctx, SP_ERR_NOMEM, "sp_align_resident: traceback scratch of one warp exceeds 24 GB");

    // ---- device buffers: scratch / CIGAR regions / blobs / dense pool live in the context's grow-only pools ----
    static int occ_cache[6] = {0, 0, 0, 0, 0, 0};  // resident CTAs per SM of k4_align<4 / 8 / 12 / 16 / 20 / 24>
    auto occupancy = [&](int U) -> int {
        int &o = occ_cache[U / 4 - 1];
        if (!o)
            o = U == 4 ? class_occupancy<4>() : U == 8 ? class_occupancy<8>() : U == 12 ? class_occupancy<12>() : U == 16 ? class_occupancy<16>()
                : U == 20 ? class_occupancy<20>() : class_occupancy<24>();
        return o;
    };
    // scratch budget: a quarter of the memory that was free when the pool last had to grow, within [4, 16] GB.  cudaMemGetInfo
    // costs milliseconds next to multi-GB allocations, so it is asked again only when this call would grow the pool.
    auto budget_of = [&]() { return std::max<int64_t>(4ll << 30, std::min<int64_t>(16ll << 30, static_cast<int64_t>(ctx->free_mem_cached / 4))) / 4; };
    auto need_words = [&](int64_t budget_words) {
        int64_t need = 0;
        for (auto &kv : classes) {
            ClassPlan &c = kv.second;
            int64_t n_slots = std::min<int64_t>(c.n_bins, static_cast<int64_t>(ctx->num_sms) * occupancy(c.U) * K4_WARPS);
            n_slots = std::max<int64_t>(1, std::min(n_slots, budget_words / c.slot_words));
            need = std::max(need, n_slots * c.slot_words);
        }
        return need;
    };
    if (!ctx->free_mem_cached || static_cast<size_t>(need_words(budget_of())) * 4 > 2 * ctx->pool_bytes[0]) {
        size_t free_b = 0, total_b = 0;
        SP_CUDA(ctx, cudaMemGetInfo(&free_b, &total_b));
        ctx->free_mem_cached = free_b + ctx->pool_bytes[0];
    }
    const int64_t budget_words = budget_of();
    uint32_t *d_blobs = nullptr, *d_scratch = nullptr;
    char *d_tables = nullptr;
    PairCall call(ctx, fn);
    auto cleanup = [&]() { dev_free(ctx, d_tables); };
    auto cu = [&](cudaError_t e, const char *what) { return cuda_status(ctx, fn, e, what); };
#define SP_TRY(x)                                   \
    do {                                            \
        sp_status s__ = (x);                        \
        if (s__ != SP_OK) { cleanup(); return s__; } \
    } while (0)
    SP_TRY(cu(ctx_pool(ctx, 2, static_cast<size_t>(blob_words_max) * 4, reinterpret_cast<void **>(&d_blobs)), "blob pool"));
    SP_TRY(call.alloc(n_pairs, cig_total, cigar_cap, false, 1));
    // the plan tables of all classes: one page-locked block, one H2D copy
    auto up16 = [](size_t x) { return (x + 15) / 16 * 16; };
    size_t tables_bytes = 0;
    std::vector<size_t> class_base;
    for (auto &kv : classes) {
        class_base.push_back(tables_bytes);
        tables_bytes += 5 * up16(static_cast<size_t>(kv.second.n_bins) * 32 * 4) + up16(kv.second.dev_pairs.size() * sizeof(AlignPairDev));
    }
    char *h_tables = nullptr;
    SP_TRY(cu(ctx_stage(ctx, tables_bytes, reinterpret_cast<void **>(&h_tables)), "cudaHostAlloc"));
    SP_TRY(cu(dev_malloc(ctx, &d_tables, tables_bytes), "cudaMalloc tables"));
    {
        size_t ci = 0;
        for (auto &kv : classes) {
            ClassPlan &c = kv.second;
            const size_t tab = up16(static_cast<size_t>(c.n_bins) * 32 * 4), raw = static_cast<size_t>(c.n_bins) * 32 * 4;
            char *dst = h_tables + class_base[ci++];
            memcpy(dst, c.lane_pair.data(), raw);
            memcpy(dst + tab, c.lane_first.data(), raw);
            memcpy(dst + 2 * tab, c.lanes.pat.data(), raw);
            memcpy(dst + 3 * tab, c.lanes.row0.data(), raw);
            memcpy(dst + 4 * tab, c.lanes.info1.data(), raw);
            memcpy(dst + 5 * tab, c.dev_pairs.data(), c.dev_pairs.size() * sizeof(AlignPairDev));
        }
    }
    SP_TRY(cu(cudaMemcpyAsync(d_tables, h_tables, tables_bytes, cudaMemcpyHostToDevice, ctx->stream), "H2D tables"));

    bool first_launch = true;
    size_t ci = 0;
    for (auto &kv : classes) {
        ClassPlan &c = kv.second;
        // one scratch slot per warp in flight, capped by the memory budget
        int64_t n_slots = std::min<int64_t>(c.n_bins, static_cast<int64_t>(ctx->num_sms) * occupancy(c.U) * K4_WARPS);
        n_slots = std::max<int64_t>(1, std::min(n_slots, budget_words / c.slot_words));
        {   // hysteresis: re-growing a multi-GB scratch costs ~100 ms; a pool holding at least half of the wanted slots is used as is
            const int64_t have = static_cast<int64_t>(ctx->pool_bytes[0] / 4) / c.slot_words;
            if (have < n_slots && have * 2 >= n_slots) n_slots = have;
        }
        const int grid = static_cast<int>((n_slots + K4_WARPS - 1) / K4_WARPS);
        SP_TRY(cu(ctx_scratch(ctx, static_cast<size_t>(grid) * K4_WARPS * c.slot_words * 4, reinterpret_cast<void **>(&d_scratch)), "traceback scratch"));
        const size_t tab = up16(static_cast<size_t>(c.n_bins) * 32 * 4);
        char *base = d_tables + class_base[ci++];
        const int32_t *d_lane_pair = reinterpret_cast<const int32_t *>(base), *d_lane_first = reinterpret_cast<const int32_t *>(base + tab);
        const int32_t *d_lane_pat = reinterpret_cast<const int32_t *>(base + 2 * tab), *d_lane_row0 = reinterpret_cast<const int32_t *>(base + 3 * tab);
        const uint32_t *d_lane_info1 = reinterpret_cast<const uint32_t *>(base + 4 * tab);
        const AlignPairDev *d_pairs = reinterpret_cast<const AlignPairDev *>(base + 5 * tab);
        if (first_launch) ev_begin(ctx, 4);  // the K4 timer spans the pack and align launches of all classes of one call
        first_launch = false;
        SP_TRY(sp_internal_pack_blobs(ctx, patterns->d_bases, patterns->d_offs, d_lane_pat, d_lane_row0, d_lane_info1, d_blobs, c.n_bins, c.U, 0, 0));
        SP_TRY(cu(cudaMemsetAsync(ctx->d_counter, 0, sizeof(int), ctx->stream), "memset"));
        AlignParams prm;
        prm.blobs = d_blobs; prm.tbases = texts->d_bases; prm.lane_pair = d_lane_pair; prm.lane_first = d_lane_first; prm.pairs = d_pairs;
        prm.cigar = call.cigar; prm.dense = call.dense; prm.dense_used = call.used; prm.dense_cap = static_cast<unsigned long long>(cigar_cap);
        prm.scratch = d_scratch; prm.slot_words = c.slot_words; prm.recs = call.recs; prm.n_bins = c.n_bins;
        prm.next_bin = ctx->d_counter; prm.one = 1u; prm.m1 = 0xFFFFFFFFu;
        switch (c.U) {
            case 4: SP_TRY(launch_class<4>(ctx, prm, grid)); break;
            case 8: SP_TRY(launch_class<8>(ctx, prm, grid)); break;
            case 12: SP_TRY(launch_class<12>(ctx, prm, grid)); break;
            case 16: SP_TRY(launch_class<16>(ctx, prm, grid)); break;
            case 20: SP_TRY(launch_class<20>(ctx, prm, grid)); break;
            default: SP_TRY(launch_class<24>(ctx, prm, grid)); break;
        }
    }
    ev_end(ctx, 4);
    tm.mark("upload + launches");
    SP_TRY(call.finish(n_pairs, recs, nullptr, cigar, cigar_cap, cigar_used, tm));
#undef SP_TRY
    cleanup();
    return SP_OK;
}

extern "C" sp_status sp_align_pairs(sp_ctx *ctx, const sp_seqset *targets, const sp_seqset *patterns, int64_t n_pairs,
                                    const int32_t *pair_target, const int32_t *pair_pattern, sp_align_rec *recs,
                                    uint32_t *cigar, int64_t cigar_cap, int64_t *cigar_used) {
    return sp_align_windows(ctx, targets, patterns, n_pairs, pair_target, pair_pattern, nullptr, nullptr, recs, cigar, cigar_cap, cigar_used);
}

// Host-buffer form: only the sequences some pair names travel to the device, then the resident path.
extern "C" sp_status sp_align_windows(sp_ctx *ctx, const sp_seqset *targets, const sp_seqset *patterns, int64_t n_pairs,
                                      const int32_t *pair_target, const int32_t *pair_pattern, const int32_t *win_begin,
                                      const int32_t *win_end, sp_align_rec *recs, uint32_t *cigar, int64_t cigar_cap,
                                      int64_t *cigar_used) {
    if (!ctx) return SP_ERR_INVALID;
    sp_status st = pair_call_check(ctx, "sp_align_windows", targets, patterns, n_pairs, pair_target, pair_pattern, win_begin, win_end, recs,
                                   cigar, cigar_cap, cigar_used);
    if (st == SP_OK) st = check_seqset(ctx, targets, "targets");
    if (st == SP_OK) st = check_seqset(ctx, patterns, "patterns");
    if (st != SP_OK) return st;
    if (n_pairs == 0) return SP_OK;
    std::vector<int32_t> t_local(static_cast<size_t>(targets->n), -1), p_local(static_cast<size_t>(patterns->n), -1);
    std::vector<int64_t> t_ids, p_ids;
    std::vector<int32_t> pt(static_cast<size_t>(n_pairs)), pp(static_cast<size_t>(n_pairs));
    for (int64_t q = 0; q < n_pairs; ++q) {
        const int64_t t = pair_target[q], pi = pair_pattern[q];
        if (t < 0 || t >= targets->n || pi < 0 || pi >= patterns->n)
            return fail(ctx, SP_ERR_INVALID, "sp_align_windows: pair index outside the sequence sets");
        if (t_local[static_cast<size_t>(t)] < 0) { t_local[static_cast<size_t>(t)] = static_cast<int32_t>(t_ids.size()); t_ids.push_back(t); }
        if (p_local[static_cast<size_t>(pi)] < 0) { p_local[static_cast<size_t>(pi)] = static_cast<int32_t>(p_ids.size()); p_ids.push_back(pi); }
        pt[static_cast<size_t>(q)] = t_local[static_cast<size_t>(t)];
        pp[static_cast<size_t>(q)] = p_local[static_cast<size_t>(pi)];
    }
    auto gather = [](const sp_seqset *s, const std::vector<int64_t> &ids, std::vector<uint8_t> &bases, std::vector<int64_t> &offs) {
        offs.assign(1, 0);
        for (int64_t id : ids) {
            bases.insert(bases.end(), s->bases + s->offsets[id], s->bases + s->offsets[id + 1]);
            offs.push_back(static_cast<int64_t>(bases.size()));
        }
        if (bases.empty()) bases.push_back(0);
    };
    std::vector<uint8_t> tb, pbs;
    std::vector<int64_t> to, po;
    gather(targets, t_ids, tb, to);
    gather(patterns, p_ids, pbs, po);
    sp_seqset tset = {tb.data(), to.data(), static_cast<int64_t>(t_ids.size())};
    sp_seqset pset = {pbs.data(), po.data(), static_cast<int64_t>(p_ids.size())};
    sp_targets *T = nullptr, *P = nullptr;
    st = sp_targets_create(ctx, &tset, &T);
    if (st == SP_OK) st = sp_targets_create(ctx, &pset, &P);
    if (st == SP_OK)
        st = sp_align_resident(ctx, T, P, n_pairs, pt.data(), pp.data(), win_begin, win_end, recs, cigar, cigar_cap, cigar_used);
    sp_targets_destroy(T); sp_targets_destroy(P);
    return st;
}
