// sp_consensus.cu -- K7 host side: sp_consensus_* (include/starphase_gpu.h), row N1 of SURVEY.md 8f.
#include "sp_internal.cuh"

#include <cstring>

#include "sp_consensus.cuh"

using namespace sp;

struct sp_consensus {
    sp_ctx *ctx = nullptr;
    int n_reads = 0, n_tracks = 0, W = 0, half_window = 0, cells = 0;
    uint8_t *d_codes = nullptr;
    long long *d_roffs = nullptr;
    int32_t *d_offset = nullptr, *d_band = nullptr, *d_best_full = nullptr, *d_track_len = nullptr;
    int max_read_len = 0;
};

static uint8_t code_of(uint8_t c) {
    switch (c) {
        case 'A': case 'a': return 0;
        case 'C': case 'c': return 1;
        case 'G': case 'g': return 2;
        case 'T': case 't': return 3;
        case '*': return 5;  // wildcard (waffle_con's CdwfaConfig::wildcard as the CYP2D6 caller sets it, src/cyp2d6/caller.rs:148)
        default: return 4;
    }
}

extern "C" sp_status sp_consensus_create(sp_ctx *ctx, const sp_seqset *reads, const int32_t *offsets, int32_t offset_window, int32_t band,
                                         int32_t max_tracks, sp_consensus **out) {
    if (!ctx) return SP_ERR_INVALID;
    if (!out) return fail(ctx, SP_ERR_INVALID, "sp_consensus_create: out is NULL");
    *out = nullptr;
    sp_status st = check_seqset(ctx, reads, "reads");
    if (st != SP_OK) return st;
    if (offset_window < 0 || band < 1 || max_tracks < 1) return fail(ctx, SP_ERR_INVALID, "sp_consensus_create: bad window / band / track count");
    const int W = band + offset_window / 2;  // the band has to hold the drift of the read and the uncertainty of where it starts
    if (2 * W + 1 > 32 * 32) return fail(ctx, SP_ERR_RANGE, "sp_consensus_create: band + offset_window / 2 must stay below 512");
    if (reads->n > 0x7FFFFF) return fail(ctx, SP_ERR_RANGE, "sp_consensus_create: too many reads");
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    sp_consensus *c = new (std::nothrow) sp_consensus();
    if (!c) return fail(ctx, SP_ERR_NOMEM, "out of host memory");
    c->ctx = ctx; c->n_reads = static_cast<int>(reads->n); c->n_tracks = max_tracks; c->W = W; c->half_window = offset_window / 2;
    c->cells = (2 * W + 1 + 31) / 32;
    for (int64_t i = 0; i < reads->n; ++i) c->max_read_len = std::max<int>(c->max_read_len, static_cast<int>(std::min<int64_t>(reads->offsets[i + 1] - reads->offsets[i], 0x7FFFFFFF)));
    const int64_t base0 = reads->n ? reads->offsets[0] : 0, nbytes = reads->n ? reads->offsets[reads->n] - base0 : 0;
    std::vector<uint8_t> codes(static_cast<size_t>(std::max<int64_t>(nbytes, 1)));
    for (int64_t i = 0; i < nbytes; ++i) codes[static_cast<size_t>(i)] = code_of(reads->bases[base0 + i]);
    std::vector<long long> roffs(static_cast<size_t>(reads->n) + 1, 0);
    std::vector<int32_t> offs(static_cast<size_t>(std::max<int64_t>(reads->n, 1)), -1);
    for (int64_t i = 0; i <= reads->n; ++i) roffs[static_cast<size_t>(i)] = reads->n ? reads->offsets[i] - base0 : 0;
    for (int64_t i = 0; i < reads->n; ++i) {
        offs[static_cast<size_t>(i)] = offsets ? std::max(offsets[i], -1) : -1;
    }
    const size_t nr = static_cast<size_t>(std::max(c->n_reads, 1)), nb = static_cast<size_t>(2 * W + 1);
    cudaError_t e = dev_malloc(ctx, &c->d_codes, codes.size());
    if (e == cudaSuccess) e = dev_malloc(ctx, &c->d_roffs, roffs.size() * sizeof(long long));
    if (e == cudaSuccess) e = dev_malloc(ctx, &c->d_offset, offs.size() * 4);
    if (e == cudaSuccess) e = dev_malloc(ctx, &c->d_band, static_cast<size_t>(max_tracks) * nr * nb * 4);
    if (e == cudaSuccess) e = dev_malloc(ctx, &c->d_best_full, static_cast<size_t>(max_tracks) * nr * 4);
    if (e == cudaSuccess) e = dev_malloc(ctx, &c->d_track_len, static_cast<size_t>(max_tracks) * 4);
    if (e == cudaSuccess) e = cudaMemcpyAsync(c->d_codes, codes.data(), codes.size(), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(c->d_roffs, roffs.data(), roffs.size() * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(c->d_offset, offs.data(), offs.size() * 4, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->d_track_len, 0, static_cast<size_t>(max_tracks) * 4, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        sp_consensus_destroy(c);
        return fail(ctx, e == cudaErrorMemoryAllocation ? SP_ERR_NOMEM : SP_ERR_CUDA, std::string("sp_consensus_create: ") + cudaGetErrorString(e));
    }
    for (int t = 0; t < max_tracks; ++t) {
        k7_reset<<<(c->n_reads + 127) / 128 + 1, 128, 0, ctx->stream>>>(c->d_best_full, c->d_track_len, t, c->n_reads);
        ++ctx->launches;
    }
    SP_CUDA(ctx, cudaGetLastError());
    *out = c;
    return SP_OK;
}

extern "C" void sp_consensus_destroy(sp_consensus *c) {
    if (!c) return;
    sp_ctx *ctx = c->ctx;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    dev_free(ctx, c->d_codes); dev_free(ctx, c->d_roffs); dev_free(ctx, c->d_offset); dev_free(ctx, c->d_band);
    dev_free(ctx, c->d_best_full); dev_free(ctx, c->d_track_len);
    delete c;
}

extern "C" int32_t sp_consensus_num_reads(const sp_consensus *c) { return c ? c->n_reads : 0; }
extern "C" int32_t sp_consensus_num_tracks(const sp_consensus *c) { return c ? c->n_tracks : 0; }

extern "C" sp_status sp_consensus_reset(sp_consensus *c, int32_t track) {
    if (!c) return SP_ERR_INVALID;
    sp_ctx *ctx = c->ctx;
    if (track < 0 || track >= c->n_tracks) return fail(ctx, SP_ERR_INVALID, "sp_consensus_reset: track out of range");
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    k7_reset<<<(c->n_reads + 127) / 128 + 1, 128, 0, ctx->stream>>>(c->d_best_full, c->d_track_len, track, c->n_reads);
    ++ctx->launches;
    SP_CUDA(ctx, cudaGetLastError());
    return SP_OK;
}

// ---- sp_consensus_extend(_batch): K7, one warp per (task, read) of every list, in one launch ----
namespace {
size_t up16(size_t x) { return (x + 15) / 16 * 16; }

template <int CELLS>
void launch_extend(const ConsParams &prm, cudaStream_t stream) {
    const unsigned grid = static_cast<unsigned>((prm.n_warps * 32 + 127) / 128);
    k7_extend<CELLS><<<grid, 128, 0, stream>>>(prm);
}

// fn: the entry point named in error messages
sp_status extend_lists(sp_ctx *ctx, const char *fn, int32_t n_lists, const sp_consensus_ext *lists) {
    const std::string f(fn);
    if (n_lists < 0 || (n_lists > 0 && !lists)) return fail(ctx, SP_ERR_INVALID, f + ": bad argument");
    std::map<const sp_consensus *, std::vector<char>> is_dst;  // per handle, over all its lists: the tracks a task writes
    for (int l = 0; l < n_lists; ++l) {
        const sp_consensus_ext &x = lists[l];
        if (!x.c || x.c->ctx != ctx) return fail(ctx, SP_ERR_INVALID, f + ": a handle is NULL or belongs to another context");
        if (x.n_tasks < 0 || (x.n_tasks > 0 && (!x.src || !x.dst || !x.ed || !x.votes || !x.full))) return fail(ctx, SP_ERR_INVALID, f + ": bad argument");
        std::vector<char> &w = is_dst[x.c];
        w.resize(static_cast<size_t>(x.c->n_tracks), 0);
        for (int q = 0; q < x.n_tasks; ++q) {
            if (x.src[q] < 0 || x.src[q] >= x.c->n_tracks || x.dst[q] < 0 || x.dst[q] >= x.c->n_tracks)
                return fail(ctx, SP_ERR_INVALID, f + ": track out of range");
            if (w[static_cast<size_t>(x.dst[q])]) return fail(ctx, SP_ERR_INVALID, f + ": two tasks write the same track");
            w[static_cast<size_t>(x.dst[q])] = 1;
        }
    }
    for (int l = 0; l < n_lists; ++l) {
        const sp_consensus_ext &x = lists[l];
        const std::vector<char> &w = is_dst[x.c];
        for (int q = 0; q < x.n_tasks; ++q)
            if (x.src[q] != x.dst[q] && w[static_cast<size_t>(x.src[q])])
                return fail(ctx, SP_ERR_INVALID, f + ": a track is read by one task and written by another");
    }
    // a list without tasks or reads does nothing at all (no length is bumped)
    std::vector<K7Task> tasks;
    int cells = 0;
    long long n_warps = 0;
    for (int l = 0; l < n_lists; ++l) {
        const sp_consensus_ext &x = lists[l];
        if (x.n_tasks == 0 || x.c->n_reads == 0) continue;
        const sp_consensus *c = x.c;
        cells = std::max(cells, c->cells);
        for (int q = 0; q < x.n_tasks; ++q) {
            K7Task t;
            t.codes = c->d_codes; t.roffs = c->d_roffs; t.offset = c->d_offset; t.band = c->d_band; t.best_full = c->d_best_full;
            t.track_len = c->d_track_len; t.warp0 = n_warps; t.n_reads = c->n_reads; t.W = c->W; t.half_window = c->half_window;
            t.src = x.src[q]; t.dst = x.dst[q];
            t.sym = x.symbols ? (x.symbols[q] == 0 ? 255u : std::min<uint32_t>(code_of(x.symbols[q]), 4u)) : 255u;  // symbol 0: report the track's state only
            tasks.push_back(t);
            n_warps += c->n_reads;
        }
    }
    if (tasks.empty()) return SP_OK;
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    // one block, device and page-locked: [tasks | ed | full | votes]; the tasks go up, the rest comes back, in one copy each
    const size_t o_ed = up16(tasks.size() * sizeof(K7Task)), o_full = o_ed + up16(static_cast<size_t>(n_warps) * 4),
                 o_votes = o_full + up16(static_cast<size_t>(n_warps) * 4), bytes = o_votes + up16(static_cast<size_t>(n_warps));
    uint8_t *h = nullptr, *d = nullptr;
    SP_CUDA(ctx, ctx_stage(ctx, bytes, reinterpret_cast<void **>(&h)));
    SP_CUDA(ctx, ctx_scratch(ctx, bytes, reinterpret_cast<void **>(&d)));
    std::memcpy(h, tasks.data(), tasks.size() * sizeof(K7Task));
    SP_CUDA(ctx, cudaMemcpyAsync(d, h, o_ed, cudaMemcpyHostToDevice, ctx->stream));
    ConsParams prm;
    prm.tasks = reinterpret_cast<const K7Task *>(d); prm.n_tasks = static_cast<int>(tasks.size()); prm.n_warps = n_warps;
    prm.out_ed = reinterpret_cast<int32_t *>(d + o_ed); prm.out_full = reinterpret_cast<int32_t *>(d + o_full); prm.out_votes = d + o_votes;
    switch (cells) {
#define SP_CASE(n) case n: launch_extend<n>(prm, ctx->stream); break
        SP_CASE(1); SP_CASE(2); SP_CASE(3); SP_CASE(4); SP_CASE(5); SP_CASE(6); SP_CASE(7); SP_CASE(8); SP_CASE(9); SP_CASE(10); SP_CASE(11);
        SP_CASE(12); SP_CASE(13); SP_CASE(14); SP_CASE(15); SP_CASE(16); SP_CASE(17); SP_CASE(18); SP_CASE(19); SP_CASE(20); SP_CASE(21);
        SP_CASE(22); SP_CASE(23); SP_CASE(24); SP_CASE(25); SP_CASE(26); SP_CASE(27); SP_CASE(28); SP_CASE(29); SP_CASE(30); SP_CASE(31);
        SP_CASE(32);
#undef SP_CASE
        default: return fail(ctx, SP_ERR_RANGE, f + ": band too wide");
    }
    k7_bump_lengths<<<(prm.n_tasks + 127) / 128, 128, 0, ctx->stream>>>(prm);
    ctx->launches += 2;
    SP_CUDA(ctx, cudaGetLastError());
    SP_CUDA(ctx, cudaMemcpyAsync(h + o_ed, d + o_ed, bytes - o_ed, cudaMemcpyDeviceToHost, ctx->stream));
    SP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    size_t q0 = 0;
    for (int l = 0; l < n_lists; ++l) {
        const sp_consensus_ext &x = lists[l];
        if (x.n_tasks == 0 || x.c->n_reads == 0) continue;
        const size_t row = static_cast<size_t>(tasks[q0].warp0), n = static_cast<size_t>(x.n_tasks) * x.c->n_reads;
        std::memcpy(x.ed, h + o_ed + row * 4, n * 4);
        std::memcpy(x.full, h + o_full + row * 4, n * 4);
        std::memcpy(x.votes, h + o_votes + row, n);
        q0 += static_cast<size_t>(x.n_tasks);
    }
    return SP_OK;
}
}  // namespace

extern "C" sp_status sp_consensus_extend(sp_consensus *c, int32_t n_tasks, const int32_t *src, const uint8_t *symbols, const int32_t *dst,
                                         int32_t *ed, uint8_t *votes, int32_t *full) {
    if (!c) return SP_ERR_INVALID;
    const sp_consensus_ext list{c, n_tasks, src, symbols, dst, ed, votes, full};
    return extend_lists(c->ctx, "sp_consensus_extend", 1, &list);
}

extern "C" sp_status sp_consensus_extend_batch(sp_ctx *ctx, int32_t n_lists, const sp_consensus_ext *lists) {
    if (!ctx) return SP_ERR_INVALID;
    return extend_lists(ctx, "sp_consensus_extend_batch", n_lists, lists);
}

// ---- sp_consensus_run(_batch): K7 in a loop on the device (k7_run), one cluster per job ----
namespace {
struct RunPlan {
    int cells = 0, n_cta = 0;
    size_t smem = 0, smem_max = 0;  // of this job's cluster shape; the most any launch may ask for (the attribute is set once)
};
// cells per lane rounded up to {2, 4, 8, 16}; cluster size and shared memory of one CTA; n_cta = 0: does not fit
RunPlan plan_run(const sp_consensus *c, int n_sides) {
    RunPlan pl;
    const int nb = 2 * c->W + 1, items = c->n_reads * n_sides;
    if (nb > 511 || items < 1 || items > 2048 || c->max_read_len > 60000) return pl;  // columns are kept as u16
    pl.cells = nb < 64 ? 2 : nb < 128 ? 4 : nb < 256 ? 8 : 16;
    const int nwarps = K7_RUN_THREADS / 32;
    int n_cta = 1;
    while (n_cta < 8 && n_cta * nwarps < items) n_cta *= 2;
    if (const char *force = getenv("SP_K7_RUN_CTAS")) n_cta = std::max(1, std::min(8, atoi(force)));  // measurement hook
    const int per_warp = (items + n_cta * nwarps - 1) / (n_cta * nwarps);
    // K7Item + column (u16) + code ring (2 bytes per cell) per slot; ed / full / votes double-buffered per item
    pl.smem = static_cast<size_t>(nwarps) * per_warp * (sizeof(K7Item) + static_cast<size_t>(pl.cells) * 32 * 4) + static_cast<size_t>(items) * 18 + 16;
    const size_t room = static_cast<size_t>(std::max(c->ctx->smem_optin - 1024, 0));  // the kernel's few static bytes come out of the same budget
    if (pl.smem > room) return pl;
    pl.smem_max = room;
    pl.n_cta = n_cta;
    return pl;
}
// n jobs of one CELLS class: n clusters of n_cta CTAs each
template <int CELLS>
cudaError_t launch_run(sp_ctx *ctx, bool &attr_set, const ConsRunParams *d_jobs, int n, int n_cta, size_t smem, size_t smem_max, cudaStream_t stream) {
    if (!attr_set) {
        const cudaError_t e = cudaFuncSetAttribute(k7_run<CELLS>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem_max));
        if (e != cudaSuccess) return e;
        attr_set = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(n * n_cta)); cfg.blockDim = dim3(K7_RUN_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = static_cast<unsigned>(n_cta); attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    ++ctx->launches;
    return cudaLaunchKernelEx(&cfg, k7_run<CELLS>, d_jobs);
}

constexpr int kLogHead = 256;  // log bytes fetched with the state; longer runs take one more copy

sp_status run_jobs(sp_ctx *ctx, const char *fn, int32_t n_jobs, const sp_consensus_job *jobs) {
    const std::string f(fn);
    if (n_jobs < 0 || (n_jobs > 0 && !jobs)) return fail(ctx, SP_ERR_INVALID, f + ": bad argument");
    std::map<const sp_consensus *, std::vector<int>> owner;  // per handle: the job using each track (-1: none)
    for (int j = 0; j < n_jobs; ++j) {
        const sp_consensus_job &x = jobs[j];
        if (!x.c || x.c->ctx != ctx) return fail(ctx, SP_ERR_INVALID, f + ": a handle is NULL or belongs to another context");
        const int ns = x.n_sides;
        if (ns < 1 || ns > 2 || !x.ed || !x.votes || !x.full || !x.steps || !x.n_steps || x.max_steps < 1 || x.min_count < 0 || x.min_af_permille < 0 ||
            x.min_af_permille > 1000)
            return fail(ctx, SP_ERR_INVALID, f + ": bad argument");
        for (int s = 0; s < ns; ++s)
            if (x.src[s] < 0 || x.src[s] >= x.c->n_tracks || x.dst[s] < 0 || x.dst[s] >= x.c->n_tracks) return fail(ctx, SP_ERR_INVALID, f + ": track out of range");
        if (ns == 2 && (x.dst[0] == x.dst[1] || x.dst[0] == x.src[1] || x.dst[1] == x.src[0]))
            return fail(ctx, SP_ERR_INVALID, f + ": the two sides need separate destination tracks");
        std::vector<int> &own = owner[x.c];
        own.resize(static_cast<size_t>(x.c->n_tracks), -1);
        for (int s = 0; s < ns; ++s)
            for (const int t : {x.src[s], x.dst[s]}) {
                int &o = own[static_cast<size_t>(t)];
                if (o >= 0 && o != j) return fail(ctx, SP_ERR_INVALID, f + ": two jobs use the same track");
                o = j;
            }
    }
    // the jobs that launch, by CELLS class (a job of an empty read set takes no step)
    std::vector<RunPlan> plans(static_cast<size_t>(n_jobs));
    std::vector<int> by_class[4];
    for (int j = 0; j < n_jobs; ++j) {
        if (jobs[j].c->n_reads == 0) continue;
        plans[static_cast<size_t>(j)] = plan_run(jobs[j].c, jobs[j].n_sides);
        const RunPlan &pl = plans[static_cast<size_t>(j)];
        if (pl.n_cta == 0) return fail(ctx, SP_ERR_RANGE, f + ": the read set does not fit on chip (sp_consensus_run_supported)");
        by_class[pl.cells == 2 ? 0 : pl.cells == 4 ? 1 : pl.cells == 8 ? 2 : 3].push_back(j);
    }
    std::vector<int> order;  // launch order = slot of the job's parameters
    for (const auto &cl : by_class) order.insert(order.end(), cl.begin(), cl.end());
    if (order.empty()) {
        for (int j = 0; j < n_jobs; ++j) *jobs[j].n_steps = 0;
        return SP_OK;
    }
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    // one block, device and page-locked: [parameters | per job: n_steps, pad | ed | full | votes | log head] up, the per-job part back;
    // then, on the device only, the log beyond its head
    const size_t n_run = order.size(), o_state = up16(n_run * sizeof(ConsRunParams));
    std::vector<size_t> o_job(n_run), o_rest(n_run);
    size_t bytes = o_state;
    for (size_t k = 0; k < n_run; ++k) {
        const sp_consensus_job &x = jobs[order[k]];
        o_job[k] = bytes;
        bytes += 16 + up16(static_cast<size_t>(x.c->n_reads) * x.n_sides * 9) + kLogHead;
    }
    const size_t state_end = bytes;
    for (size_t k = 0; k < n_run; ++k) {
        o_rest[k] = bytes;
        bytes += up16(static_cast<size_t>(std::max(jobs[order[k]].max_steps - kLogHead, 0)));
    }
    uint8_t *h = nullptr, *d = nullptr;
    SP_CUDA(ctx, ctx_stage(ctx, state_end, reinterpret_cast<void **>(&h)));
    SP_CUDA(ctx, ctx_scratch(ctx, bytes, reinterpret_cast<void **>(&d)));
    for (size_t k = 0; k < n_run; ++k) {
        const sp_consensus_job &x = jobs[order[k]];
        const sp_consensus *c = x.c;
        const size_t items = static_cast<size_t>(c->n_reads) * x.n_sides, o_ed = o_job[k] + 16, o_full = o_ed + items * 4, o_votes = o_full + items * 4;
        const size_t o_log = o_job[k] + 16 + up16(items * 9);
        std::memset(h + o_job[k], 0, 16);
        std::memcpy(h + o_ed, x.ed, items * 4);
        std::memcpy(h + o_full, x.full, items * 4);
        std::memcpy(h + o_votes, x.votes, items);
        ConsRunParams prm;
        prm.codes = c->d_codes; prm.roffs = c->d_roffs; prm.offset = c->d_offset; prm.band = c->d_band; prm.best_full = c->d_best_full;
        prm.track_len = c->d_track_len; prm.n_reads = c->n_reads; prm.W = c->W; prm.half_window = c->half_window; prm.n_sides = x.n_sides;
        for (int s = 0; s < 2; ++s) { prm.src[s] = x.src[s < x.n_sides ? s : 0]; prm.dst[s] = x.dst[s < x.n_sides ? s : 0]; }
        prm.ed = reinterpret_cast<int32_t *>(d + o_ed); prm.full = reinterpret_cast<int32_t *>(d + o_full); prm.votes = d + o_votes;
        prm.min_units = 12 * x.min_count; prm.permille = x.min_af_permille; prm.cost_limit = x.cost_limit; prm.size_limit = x.size_limit;
        prm.cost_cap = x.cost_cap; prm.max_steps = x.max_steps;
        prm.log_head = d + o_log; prm.log_rest = d + o_rest[k]; prm.n_steps = reinterpret_cast<int *>(d + o_job[k]);
        std::memcpy(h + k * sizeof(ConsRunParams), &prm, sizeof(prm));
    }
    SP_CUDA(ctx, cudaMemcpyAsync(d, h, state_end, cudaMemcpyHostToDevice, ctx->stream));
    // one launch per class, cluster = the largest any of its jobs asks for; classes side by side on the context's side streams
    SP_CUDA(ctx, ctx_aux(ctx));
    ev_begin(ctx, 4);
    SP_CUDA(ctx, cudaEventRecord(ctx->aux_fork, ctx->stream));
    int lane_stream = 0;
    size_t first = 0;
    for (int ci = 0; ci < 4; ++ci) {
        const std::vector<int> &cl = by_class[ci];
        if (cl.empty()) continue;
        int n_cta = 0;
        size_t smem = 0, smem_max = 0;
        for (int j : cl) {
            n_cta = std::max(n_cta, plans[static_cast<size_t>(j)].n_cta);
            smem = std::max(smem, plans[static_cast<size_t>(j)].smem);
            smem_max = plans[static_cast<size_t>(j)].smem_max;
        }
        cudaStream_t st = ctx->stream;
        if (lane_stream > 0) {
            st = ctx->aux[lane_stream - 1];
            SP_CUDA(ctx, cudaStreamWaitEvent(st, ctx->aux_fork, 0));
        }
        const ConsRunParams *dj = reinterpret_cast<const ConsRunParams *>(d) + first;
        const int n = static_cast<int>(cl.size());
        bool &attr = ctx->k7_run_attr[ci];
        const cudaError_t e = ci == 0 ? launch_run<2>(ctx, attr, dj, n, n_cta, smem, smem_max, st) : ci == 1 ? launch_run<4>(ctx, attr, dj, n, n_cta, smem, smem_max, st)
                              : ci == 2 ? launch_run<8>(ctx, attr, dj, n, n_cta, smem, smem_max, st) : launch_run<16>(ctx, attr, dj, n, n_cta, smem, smem_max, st);
        SP_CUDA(ctx, e);
        if (lane_stream > 0) {
            SP_CUDA(ctx, cudaEventRecord(ctx->aux_join[lane_stream - 1], st));
            SP_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->aux_join[lane_stream - 1], 0));
        }
        ++lane_stream;
        first += cl.size();
    }
    ev_end(ctx, 4);
    SP_CUDA(ctx, cudaMemcpyAsync(h + o_state, d + o_state, state_end - o_state, cudaMemcpyDeviceToHost, ctx->stream));
    SP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    bool more = false;
    for (size_t k = 0; k < n_run; ++k) {
        const sp_consensus_job &x = jobs[order[k]];
        int done = 0;
        std::memcpy(&done, h + o_job[k], sizeof(int));
        if (done > kLogHead) {
            SP_CUDA(ctx, cudaMemcpyAsync(x.steps + kLogHead, d + o_rest[k], static_cast<size_t>(done - kLogHead), cudaMemcpyDeviceToHost, ctx->stream));
            more = true;
        }
    }
    if (more) SP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int j = 0; j < n_jobs; ++j) *jobs[j].n_steps = 0;
    for (size_t k = 0; k < n_run; ++k) {
        const sp_consensus_job &x = jobs[order[k]];
        const size_t items = static_cast<size_t>(x.c->n_reads) * x.n_sides, o_ed = o_job[k] + 16, o_full = o_ed + items * 4, o_votes = o_full + items * 4;
        int done = 0;
        std::memcpy(&done, h + o_job[k], sizeof(int));
        std::memcpy(x.ed, h + o_ed, items * 4);
        std::memcpy(x.full, h + o_full, items * 4);
        std::memcpy(x.votes, h + o_votes, items);
        if (done > 0) std::memcpy(x.steps, h + o_job[k] + 16 + up16(items * 9), static_cast<size_t>(std::min(done, kLogHead)));
        *x.n_steps = done;
    }
    if (getenv("SP_TIMING")) fprintf(stderr, "[sp_timing] k7_run %zu jobs %d classes %.1f us\n", n_run, lane_stream, 1e3 * sp_last_kernel_ms(ctx, 4));
    return SP_OK;
}
}  // namespace

extern "C" int32_t sp_consensus_run_supported(const sp_consensus *c, int32_t n_sides) {
    if (!c || n_sides < 1 || n_sides > 2) return 0;
    return plan_run(c, n_sides).n_cta > 0 ? 1 : 0;
}

extern "C" sp_status sp_consensus_run(sp_consensus *c, int32_t n_sides, const int32_t *src, const int32_t *dst, int32_t *ed, uint8_t *votes,
                                      int32_t *full, int32_t min_count, int32_t min_af_permille, int64_t cost_limit, int64_t size_limit,
                                      int64_t cost_cap, int32_t max_steps, uint8_t *steps, int32_t *n_steps) {
    if (!c) return SP_ERR_INVALID;
    if (n_sides < 1 || n_sides > 2 || !src || !dst || !ed || !votes || !full || !steps || !n_steps || max_steps < 1 || min_count < 0 ||
        min_af_permille < 0 || min_af_permille > 1000)
        return fail(c->ctx, SP_ERR_INVALID, "sp_consensus_run: bad argument");
    *n_steps = 0;  // the single call reports zero rounds on the refusals that follow; a batch writes nothing
    sp_consensus_job job{c, n_sides, {src[0], 0}, {dst[0], 0}, ed, votes, full, min_count, min_af_permille, cost_limit, size_limit, cost_cap,
                         max_steps, steps, n_steps};
    if (n_sides == 2) { job.src[1] = src[1]; job.dst[1] = dst[1]; }
    return run_jobs(c->ctx, "sp_consensus_run", 1, &job);
}

extern "C" sp_status sp_consensus_run_batch(sp_ctx *ctx, int32_t n_jobs, const sp_consensus_job *jobs) {
    if (!ctx) return SP_ERR_INVALID;
    return run_jobs(ctx, "sp_consensus_run_batch", n_jobs, jobs);
}
