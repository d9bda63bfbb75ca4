// sp_graph.cu -- K8 host side: sp_graph_align and sp_graph_traverse (include/starphase_gpu.h), row N3 of SURVEY.md 8f.
#include "sp_internal.cuh"

#include "sp_graph.cuh"

using namespace sp;

static uint8_t graph_code_of(uint8_t c) {
    switch (c) {
        case 'A': case 'a': return 0;
        case 'C': case 'c': return 1;
        case 'G': case 'g': return 2;
        case 'T': case 't': return 3;
        default: return 4;
    }
}

// The one path behind both entry points: argument checks, uploads, the forward pass, then either the column matrix out
// (sp_graph_align, `columns` optional) or the marking pass and on_path out (sp_graph_traverse, `traverse`).
static sp_status graph_run(sp_ctx *ctx, const char *who, bool traverse, int32_t n_problems, const uint8_t *gchars, const int64_t *gchar_off,
                           const int32_t *pred_off, const int32_t *preds, const int32_t *diag, const int32_t *end_off, const int32_t *ends,
                           const uint8_t *seqs, const int64_t *seq_off, int32_t band, int32_t *score, int32_t *columns, uint8_t *on_path) {
    const std::string name(who);
    if (!ctx) return SP_ERR_INVALID;
    if (n_problems < 0 || band < 1 || band > 271) return fail(ctx, SP_ERR_INVALID, name + ": band must be in [1, 271]");
    if (n_problems == 0) return SP_OK;
    if (!gchar_off || !pred_off || !end_off || !seq_off || !score) return fail(ctx, SP_ERR_INVALID, name + ": NULL argument");
    const int64_t npos = gchar_off[n_problems] - gchar_off[0], nseq = seq_off[n_problems] - seq_off[0];
    if (gchar_off[0] != 0 || seq_off[0] != 0 || end_off[0] != 0) return fail(ctx, SP_ERR_INVALID, name + ": offsets must start at 0");
    if ((npos > 0 && (!gchars || !preds || !diag || (traverse && !on_path))) || (nseq > 0 && !seqs)) return fail(ctx, SP_ERR_INVALID, name + ": NULL argument");
    if (npos > 0x7FFFFFF0ll / (2 * band + 1)) return fail(ctx, SP_ERR_RANGE, name + ": graphs too large for one call");
    const int64_t n_pred = pred_off[npos], n_end = end_off[n_problems];
    for (int32_t pr = 0; pr < n_problems; ++pr) {
        const int64_t np = gchar_off[pr + 1] - gchar_off[pr];
        if (np < 0 || seq_off[pr + 1] < seq_off[pr] || end_off[pr + 1] <= end_off[pr]) return fail(ctx, SP_ERR_INVALID, name + ": bad offsets");
        for (int64_t q = gchar_off[pr]; q < gchar_off[pr + 1]; ++q) {
            if (pred_off[q + 1] <= pred_off[q]) return fail(ctx, SP_ERR_INVALID, name + ": a position without predecessor");
            for (int32_t k = pred_off[q]; k < pred_off[q + 1]; ++k)
                if (preds[k] < -1 || preds[k] >= q - gchar_off[pr]) return fail(ctx, SP_ERR_INVALID, name + ": predecessors must come earlier");
        }
        for (int32_t k = end_off[pr]; k < end_off[pr + 1]; ++k)
            if (ends[k] < -1 || ends[k] >= np) return fail(ctx, SP_ERR_INVALID, name + ": end position out of range");
    }
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    std::vector<uint8_t> gc(static_cast<size_t>(std::max<int64_t>(npos, 1))), sc(static_cast<size_t>(std::max<int64_t>(nseq, 1)));
    for (int64_t i = 0; i < npos; ++i) gc[static_cast<size_t>(i)] = graph_code_of(gchars[i]);
    for (int64_t i = 0; i < nseq; ++i) sc[static_cast<size_t>(i)] = graph_code_of(seqs[i]);
    std::vector<long long> goff(gchar_off, gchar_off + n_problems + 1), soff(seq_off, seq_off + n_problems + 1);
    const int nb = 2 * band + 1;
    uint8_t *d_gc = nullptr, *d_sc = nullptr, *d_marks = nullptr, *d_on = nullptr;
    long long *d_goff = nullptr, *d_soff = nullptr;
    int32_t *d_pred_off = nullptr, *d_preds = nullptr, *d_diag = nullptr, *d_end_off = nullptr, *d_ends = nullptr, *d_cols = nullptr, *d_score = nullptr;
    auto cleanup = [&]() {
        dev_free(ctx, d_gc); dev_free(ctx, d_sc); dev_free(ctx, d_goff); dev_free(ctx, d_soff); dev_free(ctx, d_pred_off); dev_free(ctx, d_preds);
        dev_free(ctx, d_diag); dev_free(ctx, d_end_off); dev_free(ctx, d_ends); dev_free(ctx, d_cols); dev_free(ctx, d_score);
        dev_free(ctx, d_marks); dev_free(ctx, d_on);
    };
    cudaError_t e = cudaSuccess;
    auto up = [&](auto **dst, const void *src, size_t bytes) {
        if (e != cudaSuccess) return;
        e = dev_malloc(ctx, dst, std::max<size_t>(bytes, 16));
        if (e == cudaSuccess && bytes) e = cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream);
    };
    up(&d_gc, gc.data(), static_cast<size_t>(npos));
    up(&d_sc, sc.data(), static_cast<size_t>(nseq));
    up(&d_goff, goff.data(), goff.size() * sizeof(long long));
    up(&d_soff, soff.data(), soff.size() * sizeof(long long));
    up(&d_pred_off, pred_off, static_cast<size_t>(npos + 1) * 4);
    up(&d_preds, preds, static_cast<size_t>(n_pred) * 4);
    up(&d_diag, diag, static_cast<size_t>(npos) * 4);
    up(&d_end_off, end_off, static_cast<size_t>(n_problems + 1) * 4);
    up(&d_ends, ends, static_cast<size_t>(n_end) * 4);
    if (e == cudaSuccess) e = dev_malloc(ctx, &d_cols, std::max<size_t>(static_cast<size_t>(npos) * nb * 4, 16));
    if (e == cudaSuccess) e = dev_malloc(ctx, &d_score, static_cast<size_t>(n_problems) * 4);
    // marking pass: the pushed marks ([npos][nb]) and the hit flags ([npos]) in one zeroed block, on_path beside it
    const size_t mark_bytes = static_cast<size_t>(npos) * (nb + 1);
    if (traverse && e == cudaSuccess) e = dev_malloc(ctx, &d_marks, std::max<size_t>(mark_bytes, 16));
    if (traverse && e == cudaSuccess) e = dev_malloc(ctx, &d_on, std::max<size_t>(static_cast<size_t>(npos), 16));
    if (traverse && e == cudaSuccess) e = cudaMemsetAsync(d_marks, 0, mark_bytes, ctx->stream);
    if (e == cudaSuccess) {
        GraphParams prm;
        prm.gcodes = d_gc; prm.goff = d_goff; prm.pred_off = d_pred_off; prm.preds = d_preds; prm.diag = d_diag; prm.end_off = d_end_off;
        prm.ends = d_ends; prm.scodes = d_sc; prm.soff = d_soff; prm.columns = d_cols; prm.score = d_score; prm.n_problems = n_problems; prm.W = band;
        prm.marks = d_marks; prm.hit = d_marks ? d_marks + static_cast<size_t>(npos) * nb : nullptr; prm.on_path = d_on;
        const unsigned grid = static_cast<unsigned>((static_cast<long long>(n_problems) * 32 + 127) / 128);
        const int cells = (nb + 31) / 32;
        if (cells <= 3) k8_graph_forward<3><<<grid, 128, 0, ctx->stream>>>(prm);
        else if (cells <= 5) k8_graph_forward<5><<<grid, 128, 0, ctx->stream>>>(prm);
        else if (cells <= 9) k8_graph_forward<9><<<grid, 128, 0, ctx->stream>>>(prm);
        else k8_graph_forward<17><<<grid, 128, 0, ctx->stream>>>(prm);
        ++ctx->launches;
        if (traverse) {
            if (cells <= 3) k8_graph_mark<3><<<grid, 128, 0, ctx->stream>>>(prm);
            else if (cells <= 5) k8_graph_mark<5><<<grid, 128, 0, ctx->stream>>>(prm);
            else if (cells <= 9) k8_graph_mark<9><<<grid, 128, 0, ctx->stream>>>(prm);
            else k8_graph_mark<17><<<grid, 128, 0, ctx->stream>>>(prm);
            ++ctx->launches;
        }
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(score, d_score, static_cast<size_t>(n_problems) * 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && columns && npos) e = cudaMemcpyAsync(columns, d_cols, static_cast<size_t>(npos) * nb * 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && traverse && npos) e = cudaMemcpyAsync(on_path, d_on, static_cast<size_t>(npos), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cleanup();
    if (e != cudaSuccess) return fail(ctx, e == cudaErrorMemoryAllocation ? SP_ERR_NOMEM : SP_ERR_CUDA, name + ": " + cudaGetErrorString(e));
    return SP_OK;
}

extern "C" sp_status sp_graph_align(sp_ctx *ctx, int32_t n_problems, const uint8_t *gchars, const int64_t *gchar_off, const int32_t *pred_off,
                                    const int32_t *preds, const int32_t *diag, const int32_t *end_off, const int32_t *ends,
                                    const uint8_t *seqs, const int64_t *seq_off, int32_t band, int32_t *score, int32_t *columns) {
    return graph_run(ctx, "sp_graph_align", false, n_problems, gchars, gchar_off, pred_off, preds, diag, end_off, ends, seqs, seq_off, band, score,
                     columns, nullptr);
}

extern "C" sp_status sp_graph_traverse(sp_ctx *ctx, int32_t n_problems, const uint8_t *gchars, const int64_t *gchar_off, const int32_t *pred_off,
                                       const int32_t *preds, const int32_t *diag, const int32_t *end_off, const int32_t *ends,
                                       const uint8_t *seqs, const int64_t *seq_off, int32_t band, int32_t *score, uint8_t *on_path) {
    return graph_run(ctx, "sp_graph_traverse", true, n_problems, gchars, gchar_off, pred_off, preds, diag, end_off, ends, seqs, seq_off, band, score,
                     nullptr, on_path);
}
