// sp_affine.cu -- K9 host side: sp_align_affine_resident (include/starphase_gpu.h).
#include "sp_internal.cuh"

#define SP_NO_GLOBAL_KERNELS
#include "sp_kernels.cuh"
#include "sp_affine.cuh"

using namespace sp;

namespace {
template <int CELLS>
int k9_occupancy() {
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k9_affine_local<CELLS>, 128, 0) != cudaSuccess) occ = 1;
    return std::max(occ, 1);
}
}  // namespace

extern "C" sp_status sp_align_affine_resident(sp_ctx *ctx, const sp_targets *texts, const sp_targets *patterns, int64_t n_pairs,
                                              const int32_t *pair_text, const int32_t *pair_pattern, const int32_t *win_begin,
                                              const int32_t *win_end, const int32_t *band_centre, int32_t band, const int32_t *pair_band,
                                              const sp_affine_costs *costs, sp_align_rec *recs, int32_t *scores, uint32_t *cigar,
                                              int64_t cigar_cap, int64_t *cigar_used) {
    if (!ctx) return SP_ERR_INVALID;
    const char *fn = "sp_align_affine_resident";
    if (!costs) return fail(ctx, SP_ERR_INVALID, "sp_align_affine_resident: NULL argument");
    if (n_pairs > 0 && !scores) return fail(ctx, SP_ERR_INVALID, "sp_align_affine_resident: bad argument");
    if (!pair_band && (band < 1 || band > 255)) return fail(ctx, SP_ERR_INVALID, "sp_align_affine_resident: band must be in [1, 255]");
    if (costs->a < 1 || costs->b < 0 || costs->q < 0 || costs->e < 1 || costs->q2 < 0 || costs->e2 < 1 || costs->a > 100 || costs->b > 1000 ||
        costs->q > 10000 || costs->q2 > 10000 || costs->e > 1000 || costs->e2 > 1000)
        return fail(ctx, SP_ERR_INVALID, "sp_align_affine_resident: costs out of range");
    if (sp_status s = pair_call_check(ctx, fn, texts, patterns, n_pairs, pair_text, pair_pattern, win_begin, win_end, recs, cigar, cigar_cap,
                                      cigar_used); s != SP_OK || n_pairs == 0)
        return s;
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    PhaseTimer tm;
    // width classes: band cells per lane (the last cell of lane 31 is never a band cell: 2 W + 1 <= 32 cells - 1)
    static const int kCells[4] = {2, 4, 8, 16};
    auto class_of = [](int w) { return w <= 31 ? 0 : w <= 63 ? 1 : w <= 127 ? 2 : 3; };
    int64_t cnt[4] = {0, 0, 0, 0}, first[4], fill[4], max_trace[4] = {16, 16, 16, 16};
    for (int64_t q = 0; q < n_pairs; ++q) {
        const int w = pair_band ? pair_band[q] : band;
        if (w < 1 || w > 255) return fail(ctx, SP_ERR_INVALID, "sp_align_affine_resident: pair_band must be in [1, 255]");
        ++cnt[class_of(w)];
    }
    first[0] = 0;
    for (int c = 1; c < 4; ++c) first[c] = first[c - 1] + cnt[c - 1];
    for (int c = 0; c < 4; ++c) fill[c] = first[c];
    std::vector<AffinePairDev> pairs(static_cast<size_t>(n_pairs));  // class by class
    int64_t cig_total = 0;
    for (int64_t q = 0; q < n_pairs; ++q) {
        int64_t t_off, n, m;
        if (sp_status s = pair_resolve(ctx, fn, texts, patterns, q, pair_text, pair_pattern, win_begin, win_end, t_off, n, m); s != SP_OK) return s;
        if (m > 0x3FFFFFFF || n > 0x3FFFFFFF) return fail(ctx, SP_ERR_TOO_LONG, "sp_align_affine_resident: sequence too long");
        const int w = pair_band ? pair_band[q] : band, c = class_of(w);
        AffinePairDev &d = pairs[static_cast<size_t>(fill[c]++)];
        d.t_off = t_off; d.p_off = patterns->h_offs[static_cast<size_t>(pair_pattern[q])];
        d.n = static_cast<int32_t>(n); d.m = static_cast<int32_t>(m);
        d.centre = band_centre ? band_centre[q] : 0;
        d.trace_off = 0;
        d.cig_off = cig_total;
        d.cig_len = static_cast<int32_t>(std::min<int64_t>(m + std::min<int64_t>(n, m + 2ll * w) + 2, 0x7FFFFFF0ll));
        d.out = static_cast<int32_t>(q); d.band = w;
        cig_total += d.cig_len;
        max_trace[c] = std::max<int64_t>(max_trace[c], m * 32 * kCells[c]);  // one row = 32 * cells trace bytes
    }
    tm.mark("k9 plan");
    // one trace slot per resident warp, every class inside its share of the scratch budget
    const int occ[4] = {k9_occupancy<2>(), k9_occupancy<4>(), k9_occupancy<8>(), k9_occupancy<16>()};
    int grid[4] = {0, 0, 0, 0};
    int64_t trace_off[4] = {0, 0, 0, 0}, trace_total = 0;
    int n_classes = 0;
    for (int c = 0; c < 4; ++c) n_classes += cnt[c] > 0;
    const int64_t budget = (8ll << 30) / std::max(n_classes, 1);
    for (int c = 0; c < 4; ++c) {
        if (!cnt[c]) continue;
        int64_t n_slots = std::min<int64_t>(cnt[c], static_cast<int64_t>(ctx->num_sms) * occ[c] * 4);
        n_slots = std::max<int64_t>(1, std::min(n_slots, budget / max_trace[c]));
        grid[c] = static_cast<int>((n_slots + 3) / 4);
        trace_off[c] = trace_total;
        trace_total += static_cast<int64_t>(grid[c]) * 4 * max_trace[c];
    }
    if (tm.on) fprintf(stderr, "[sp_timing] k9 pairs %lld (classes %lld %lld %lld %lld) trace %lld MB cig_total %lld\n", static_cast<long long>(n_pairs),
                       static_cast<long long>(cnt[0]), static_cast<long long>(cnt[1]), static_cast<long long>(cnt[2]), static_cast<long long>(cnt[3]),
                       static_cast<long long>(trace_total >> 20), static_cast<long long>(cig_total));
    uint8_t *d_trace = nullptr;
    AffinePairDev *d_pairs = nullptr;
    PairCall call(ctx, fn);  // used: [0] = dense pool fill, then the four work counters
    auto cleanup = [&]() { dev_free(ctx, d_pairs); };
    auto cu = [&](cudaError_t e, const char *what) { return cuda_status(ctx, fn, e, what); };
#define SP_TRY(x)                                   \
    do {                                            \
        sp_status s__ = (x);                        \
        if (s__ != SP_OK) { cleanup(); return s__; } \
    } while (0)
    SP_TRY(cu(ctx_aux(ctx), "side streams"));
    SP_TRY(cu(ctx_scratch(ctx, static_cast<size_t>(trace_total), reinterpret_cast<void **>(&d_trace)), "trace scratch"));
    SP_TRY(call.alloc(n_pairs, cig_total, cigar_cap, true, 4));
    SP_TRY(cu(dev_malloc(ctx, &d_pairs, pairs.size() * sizeof(AffinePairDev)), "cudaMalloc"));
    SP_TRY(cu(cudaMemcpyAsync(d_pairs, pairs.data(), pairs.size() * sizeof(AffinePairDev), cudaMemcpyHostToDevice, ctx->stream), "H2D"));
    tm.mark("k9 buffers + H2D");
    ev_begin(ctx, 4);
    SP_TRY(cu(cudaEventRecord(ctx->aux_fork, ctx->stream), "fork"));
    int lane_stream = 0;  // the first class runs on the context stream, the others beside it
    bool joined[3] = {false, false, false};
    for (int c = 3; c >= 0; --c) {  // widest (slowest per pair) first
        if (!cnt[c]) continue;
        cudaStream_t st = ctx->stream;
        if (lane_stream > 0) {
            st = ctx->aux[lane_stream - 1];
            SP_TRY(cu(cudaStreamWaitEvent(st, ctx->aux_fork, 0), "fork"));
        }
        AffineParams prm;
        prm.tbases = texts->d_bases; prm.pbases = patterns->d_bases; prm.pairs = d_pairs + first[c]; prm.trace = d_trace + trace_off[c];
        prm.slot_bytes = max_trace[c];
        prm.cigar = call.cigar; prm.dense = call.dense; prm.dense_used = call.used; prm.dense_cap = static_cast<unsigned long long>(cigar_cap);
        prm.recs = call.recs; prm.scores = call.scores; prm.n_pairs = static_cast<int>(cnt[c]);
        prm.a = costs->a; prm.b = costs->b; prm.q = costs->q; prm.e = costs->e; prm.q2 = costs->q2; prm.e2 = costs->e2;
        prm.next_pair = reinterpret_cast<int *>(call.used + 1) + c;
        if (c == 0) k9_affine_local<2><<<grid[c], 128, 0, st>>>(prm);
        else if (c == 1) k9_affine_local<4><<<grid[c], 128, 0, st>>>(prm);
        else if (c == 2) k9_affine_local<8><<<grid[c], 128, 0, st>>>(prm);
        else k9_affine_local<16><<<grid[c], 128, 0, st>>>(prm);
        ++ctx->launches;
        SP_TRY(cu(cudaGetLastError(), "k9_affine_local launch"));
        if (lane_stream > 0) {
            SP_TRY(cu(cudaEventRecord(ctx->aux_join[lane_stream - 1], st), "join"));
            joined[lane_stream - 1] = true;
        }
        ++lane_stream;
    }
    for (int i = 0; i < 3; ++i)
        if (joined[i]) SP_TRY(cu(cudaStreamWaitEvent(ctx->stream, ctx->aux_join[i], 0), "join"));
    ev_end(ctx, 4);
    SP_TRY(call.finish(n_pairs, recs, scores, cigar, cigar_cap, cigar_used, tm));
#undef SP_TRY
    cleanup();
    return SP_OK;
}
