// starphase_gpu.cu -- host side of libstarphase_gpu.so: the C ABI of include/starphase_gpu.h.
// No torch types, no CPU fallback: every entry point needs a usable sm_100 device.
// (K4 lives in sp_align.cu, the multi-GPU entry points in sp_comm.cu; shared handles in sp_internal.cuh.)
#include "sp_internal.cuh"

#include "sp_kernels.cuh"
#include "sp_misc.cuh"

using namespace sp;

thread_local std::string g_create_err;

sp_status sp_internal_pack_blobs(sp_ctx *ctx, const uint8_t *d_bases, const long long *d_offs, const int32_t *d_lane_pat,
                                 const int32_t *d_lane_row0, const uint32_t *d_lane_info1, uint32_t *d_blobs, int n_bins, int U,
                                 int prefix_mode, int reverse) {
    const long long total_threads = static_cast<long long>(n_bins) * 32 * U;
    if (total_threads == 0) return SP_OK;
    pack_patterns<<<static_cast<int>((total_threads + 255) / 256), 256, 0, ctx->stream>>>(d_bases, d_offs, d_lane_pat, d_lane_row0, d_lane_info1,
                                                                                             d_blobs, n_bins, U, prefix_mode, reverse);
    ++ctx->launches;
    SP_CUDA(ctx, cudaGetLastError());
    return SP_OK;
}

void LaneTables::resize(int n_bins) {
    const size_t lanes = static_cast<size_t>(n_bins) * 32;
    pat.resize(lanes, -1);
    row0.resize(lanes, 0);
    info1.resize(lanes, INFO_FIRST);
}

void LaneTables::place(int bin, int lane0, int nl, int32_t p, int64_t m, int U) {
    const int64_t rows = 32ll * U, pad = nl * rows - m;
    for (int li = 0; li < nl; ++li) {
        const size_t o = static_cast<size_t>(bin) * 32 + lane0 + li;
        pat[o] = p;
        row0[o] = static_cast<int32_t>(li * rows - pad);
        info1[o] = static_cast<uint32_t>(m) | (li == 0 ? INFO_FIRST : 0u) | (li == nl - 1 ? INFO_LAST : 0u);
    }
}

int sp_internal_pack_lanes(const std::vector<int> &lanes, std::vector<LaneSlot> *slots) {
    std::vector<std::vector<int>> by_rem(33);  // bins by free lanes
    std::vector<int> used;                     // lanes used per bin
    if (slots) slots->resize(lanes.size());
    for (size_t k = 0; k < lanes.size(); ++k) {
        int bin = -1;
        for (int rem = lanes[k]; rem <= 32; ++rem)
            if (!by_rem[rem].empty()) { bin = by_rem[rem].back(); by_rem[rem].pop_back(); break; }
        if (bin < 0) {
            bin = static_cast<int>(used.size());
            used.push_back(0);
        }
        if (slots) (*slots)[k] = {bin, used[bin]};
        used[bin] += lanes[k];
        by_rem[32 - used[bin]].push_back(bin);
    }
    return static_cast<int>(used.size());
}

extern "C" const char *sp_version(void) { return "starphase_gpu 0.1.0 (sm_100a)"; }

extern "C" const char *sp_last_error(const sp_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

extern "C" sp_status sp_ctx_create(int device, void *stream, sp_ctx **out) {
    if (!out) return fail(nullptr, SP_ERR_INVALID, "sp_ctx_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, SP_ERR_CUDA,
                    std::string("no CUDA device available (this library has no CPU fallback): ") +
                        cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(nullptr, SP_ERR_INVALID, "sp_ctx_create: bad device ordinal");
    SP_CUDA(nullptr, cudaSetDevice(device));
    cudaDeviceProp prop;
    SP_CUDA(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(nullptr, SP_ERR_CUDA,
                    "device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                        "; libstarphase_gpu is built for sm_100a only");
    sp_ctx *ctx = new (std::nothrow) sp_ctx();
    if (!ctx) return fail(nullptr, SP_ERR_NOMEM, "out of host memory");
    ctx->device = device;
    ctx->num_sms = prop.multiProcessorCount;
    ctx->smem_optin = static_cast<int>(prop.sharedMemPerBlockOptin);
    if (stream) {
        ctx->stream = static_cast<cudaStream_t>(stream);
    } else {
        // highest priority: when contexts share a GPU (sp_ctx_share_device) their long K1 launches run on a lowest-priority side
        // stream and everything on this one is dispatched ahead of K1's waiting CTAs; alone on a GPU the priority changes nothing
        int prio_lo = 0, prio_hi = 0;
        cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
        if (cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) {
            delete ctx;
            return fail(nullptr, SP_ERR_CUDA, "cudaStreamCreate failed");
        }
        ctx->own_stream = true;
    }
    for (int i = 0; i < 5; ++i)
        for (int j = 0; j < 2; ++j) cudaEventCreate(&ctx->ev[i][j]);
    // a private pool: freed blocks stay here instead of going back to the OS at every synchronisation, and the default pool of
    // the embedding process (torch, NCCL, the Rust host) keeps its own settings
    {
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        if (cudaMemPoolCreate(&ctx->mempool, &props) == cudaSuccess) {
            unsigned long long threshold = ~0ull;
            cudaMemPoolSetAttribute(ctx->mempool, cudaMemPoolAttrReleaseThreshold, &threshold);
        } else {
            ctx->mempool = nullptr;  // falls back to the device's default pool, untouched
        }
    }
    cudaGetLastError();
    if (cudaMalloc(&ctx->d_counter, sizeof(int)) != cudaSuccess) {
        sp_ctx_destroy(ctx);
        return fail(nullptr, SP_ERR_NOMEM, "cudaMalloc failed");
    }
    *out = ctx;
    return SP_OK;
}

extern "C" void sp_ctx_destroy(sp_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (int i = 0; i < 5; ++i)
        for (int j = 0; j < 2; ++j) cudaEventDestroy(ctx->ev[i][j]);
    for (int i = 0; i < 3; ++i) {
        if (ctx->aux[i]) { cudaStreamSynchronize(ctx->aux[i]); cudaStreamDestroy(ctx->aux[i]); }
        if (ctx->aux_join[i]) cudaEventDestroy(ctx->aux_join[i]);
    }
    if (ctx->aux_fork) cudaEventDestroy(ctx->aux_fork);
    if (ctx->bulk) { cudaStreamSynchronize(ctx->bulk); cudaStreamDestroy(ctx->bulk); }
    if (ctx->bulk_fork) cudaEventDestroy(ctx->bulk_fork);
    if (ctx->bulk_join) cudaEventDestroy(ctx->bulk_join);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    for (void *p : ctx->pool) cudaFree(p);
    cudaFree(ctx->d_counter);
    cudaFreeHost(ctx->h_stage);
    if (ctx->mempool) cudaMemPoolDestroy(ctx->mempool);
    delete ctx;
}

extern "C" sp_status sp_ctx_share_device(sp_ctx *ctx, int on) {
    if (!ctx) return SP_ERR_INVALID;
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    if (on) SP_CUDA(ctx, ctx_bulk(ctx));
    ctx->share_device = on != 0;
    return SP_OK;
}

extern "C" sp_status sp_pinned_alloc(sp_ctx *ctx, size_t bytes, void **out) {
    if (!ctx) return SP_ERR_INVALID;
    if (!out) return fail(ctx, SP_ERR_INVALID, "sp_pinned_alloc: NULL argument");
    *out = nullptr;
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    const cudaError_t e = cudaHostAlloc(out, std::max<size_t>(bytes, 1), cudaHostAllocDefault);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *out = nullptr;
        return fail(ctx, SP_ERR_NOMEM, std::string("sp_pinned_alloc: ") + cudaGetErrorString(e));
    }
    return SP_OK;
}

extern "C" void sp_pinned_free(sp_ctx *ctx, void *p) {
    if (!p) return;
    if (ctx) cudaSetDevice(ctx->device);
    cudaFreeHost(p);
}

extern "C" sp_status sp_ctx_synchronize(sp_ctx *ctx) {
    if (!ctx) return SP_ERR_INVALID;
    SP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SP_OK;
}

extern "C" float sp_last_kernel_ms(sp_ctx *ctx, int which) {
    if (!ctx || which < 0 || which > 4 || !ctx->ev_valid[which]) return -1.0f;
    if (cudaEventSynchronize(ctx->ev[which][1]) != cudaSuccess) return -1.0f;
    float ms = -1.0f;
    if (cudaEventElapsedTime(&ms, ctx->ev[which][0], ctx->ev[which][1]) != cudaSuccess) return -1.0f;
    return ms;
}

extern "C" uint64_t sp_launch_count(const sp_ctx *ctx) { return ctx ? ctx->launches : 0; }

// ------------------------------------------------------------------------------------------
// sequence-set validation / upload
// ------------------------------------------------------------------------------------------
sp_status check_seqset(sp_ctx *ctx, const sp_seqset *s, const char *what) {
    if (!s) return fail(ctx, SP_ERR_INVALID, std::string(what) + ": seqset is NULL");
    if (s->n < 0) return fail(ctx, SP_ERR_INVALID, std::string(what) + ": negative count");
    if (s->n > 0 && !s->offsets) return fail(ctx, SP_ERR_INVALID, std::string(what) + ": offsets is NULL");
    for (int64_t i = 0; i < s->n; ++i)
        if (s->offsets[i + 1] < s->offsets[i])
            return fail(ctx, SP_ERR_INVALID, std::string(what) + ": offsets must be non-decreasing");
    if (s->n > 0 && s->offsets[s->n] > s->offsets[0] && !s->bases)
        return fail(ctx, SP_ERR_INVALID, std::string(what) + ": bases is NULL");
    if (s->n > 0x7FFFFFF0ll) return fail(ctx, SP_ERR_RANGE, std::string(what) + ": too many sequences");
    return SP_OK;
}

// copies bases[offsets[0]..offsets[n]) to the device and rebased offsets (offs[0] = 0)
sp_status upload_seqset(sp_ctx *ctx, const sp_seqset *s, uint8_t **d_bases, long long **d_offs) {
    const int64_t base0 = s->n ? s->offsets[0] : 0;
    const int64_t nbytes = s->n ? s->offsets[s->n] - base0 : 0;
    std::vector<long long> offs(static_cast<size_t>(s->n) + 1);
    for (int64_t i = 0; i <= s->n; ++i) offs[static_cast<size_t>(i)] = s->n ? s->offsets[i] - base0 : 0;
    *d_bases = nullptr; *d_offs = nullptr;
    cudaError_t e = dev_malloc(ctx, reinterpret_cast<void **>(d_bases), static_cast<size_t>(std::max<int64_t>(nbytes, 16)));
    if (e == cudaSuccess) e = dev_malloc(ctx, reinterpret_cast<void **>(d_offs), offs.size() * sizeof(long long));
    if (e == cudaSuccess && nbytes)
        e = cudaMemcpyAsync(*d_bases, s->bases + base0, static_cast<size_t>(nbytes), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(*d_offs, offs.data(), offs.size() * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);  // offs is a stack-owned vector
    if (e != cudaSuccess) {  // nothing stays behind on the error path
        dev_free(ctx, *d_bases); dev_free(ctx, *d_offs);
        *d_bases = nullptr; *d_offs = nullptr;
        return fail(ctx, e == cudaErrorMemoryAllocation ? SP_ERR_NOMEM : SP_ERR_CUDA, std::string("sequence upload: ") + cudaGetErrorString(e));
    }
    return SP_OK;
}

// ------------------------------------------------------------------------------------------
// patterns: choose lane width U, bin-pack patterns into 32-lane warps, build Peq blobs on device
// ------------------------------------------------------------------------------------------
// lane widths compiled into the library
static const int kUmin = 4, kUmax = 16;
static const int kULong[2] = {20, 24};  // only for pattern sets holding a pattern of more than 16,384 rows
// modelled ALU-pipe instructions per text column of one warp (DESIGN.md §4.1).  The constants are round 1's count (8 per word + 17 of
// per-column bookkeeping); the kernel is at 7 per word + ~4 now, and the classes chosen for the IMGT-shaped sets are the same for any
// bookkeeping constant between 1 and 17 (lane granularity decides, not the model), so the constants were left alone
static double warp_cost(int U) { return 8.0 * U + 17.0; }

// Packs the non-empty patterns listed in `which` into warps of lane width U, most lanes first (stable); returns the warp
// count and, when `lanes` is given, lays the patterns out in it.  Every pattern fits: choose_classes picked U for it.
static int plan_bins(const std::vector<int64_t> &lens, const std::vector<int32_t> &which, int U, LaneTables *lanes) {
    const int64_t rows = 32ll * U;
    std::vector<std::pair<int, int32_t>> items;  // (lanes, pattern)
    items.reserve(which.size());
    for (int32_t i : which) {
        const int64_t len = lens[static_cast<size_t>(i)];
        if (len > 0) items.emplace_back(static_cast<int>((len + rows - 1) / rows), i);
    }
    std::stable_sort(items.begin(), items.end(),
                     [](const std::pair<int, int32_t> &a, const std::pair<int, int32_t> &b) { return a.first > b.first; });
    std::vector<int> nl(items.size());
    for (size_t k = 0; k < items.size(); ++k) nl[k] = items[k].first;
    std::vector<LaneSlot> at;
    const int n_bins = sp_internal_pack_lanes(nl, lanes ? &at : nullptr);
    if (lanes) {
        lanes->resize(n_bins);
        for (size_t k = 0; k < items.size(); ++k)
            lanes->place(at[k].bin, at[k].lane0, nl[k], items[k].second, lens[static_cast<size_t>(items[k].second)], U);
    }
    return n_bins;
}

// Splits the patterns over up to `max_classes` lane widths.  Every pattern goes to the width in the current set that
// is cheapest for it (cost of a warp of that width / patterns of its lane count a warp holds); widths are added
// greedily while the packed total (warps x modelled cost per column) drops by more than 1 %.
static bool choose_classes(const std::vector<int64_t> &lens, int max_classes, std::vector<int> &Us,
                           std::vector<std::vector<int32_t>> &members) {
    const size_t n = lens.size();
    auto assign = [&](const std::vector<int> &set, std::vector<std::vector<int32_t>> &mem) -> bool {
        mem.assign(set.size(), {});
        for (size_t i = 0; i < n; ++i) {
            if (lens[i] == 0) continue;
            int best = -1;
            double bc = 0;
            for (size_t c = 0; c < set.size(); ++c) {
                const int64_t nl = (lens[i] + 32ll * set[c] - 1) / (32ll * set[c]);
                if (nl > 32) continue;
                const double cost = warp_cost(set[c]) / static_cast<double>(32 / nl);
                if (best < 0 || cost < bc) { best = static_cast<int>(c); bc = cost; }
            }
            if (best < 0) return false;
            mem[static_cast<size_t>(best)].push_back(static_cast<int32_t>(i));
        }
        return true;
    };
    auto total_cost = [&](const std::vector<int> &set, const std::vector<std::vector<int32_t>> &mem) -> double {
        double c = 0;
        for (size_t k = 0; k < set.size(); ++k) {
            const int n_bins = plan_bins(lens, mem[k], set[k], nullptr);
            const int groups = (n_bins + K1_WARPS - 1) / K1_WARPS;
            c += (n_bins + 0.25 * (groups * K1_WARPS - n_bins)) * warp_cost(set[k]);
        }
        return c;
    };
    std::vector<int> cand;
    const char *forceU = getenv("SP_FORCE_U");  // test hook: one fixed lane width
    for (int U = kUmin; U <= kUmax; ++U)
        if (!forceU || atoi(forceU) == U) cand.push_back(U);
    int64_t longest = 0;
    for (int64_t x : lens) longest = std::max(longest, x);
    if (longest > 32ll * 32 * kUmax)
        for (int U : kULong)
            if (!forceU || atoi(forceU) == U) cand.push_back(U);
    if (forceU) max_classes = 1;
    std::vector<int> set;
    std::vector<std::vector<int32_t>> mem;
    double cur = 0;
    while (static_cast<int>(set.size()) < max_classes) {
        int bestU = 0;
        double bestc = 0;
        for (int U : cand) {
            if (std::find(set.begin(), set.end(), U) != set.end()) continue;
            std::vector<int> trial = set;
            trial.push_back(U);
            std::vector<std::vector<int32_t>> tm;
            if (!assign(trial, tm)) continue;
            const double c = total_cost(trial, tm);
            if (!bestU || c < bestc) { bestU = U; bestc = c; }
        }
        if (!bestU) break;
        if (!set.empty() && bestc > 0.99 * cur) break;
        set.push_back(bestU);
        cur = bestc;
    }
    if (set.empty()) return false;
    assign(set, mem);
    Us.clear(); members.clear();
    for (size_t k = 0; k < set.size(); ++k)
        if (!mem[k].empty()) { Us.push_back(set[k]); members.push_back(mem[k]); }
    if (Us.empty()) { Us.push_back(set[0]); members.emplace_back(); }  // only empty patterns
    return true;
}

// Host-only view of the planner (no device needed): which lane widths a pattern set would be split into.
extern "C" sp_status sp_plan_lane_classes(const int64_t *lens, int64_t n, int max_classes, int *n_classes, int *widths,
                                          int64_t *n_patterns, int64_t *n_warps, int64_t *padded_rows) {
    if (!lens || n < 0 || !n_classes || !widths || !n_patterns || !n_warps || !padded_rows || max_classes < 1 ||
        max_classes > 8)
        return SP_ERR_INVALID;
    std::vector<int64_t> v(lens, lens + n);
    for (int64_t x : v)
        if (x < 0) return SP_ERR_INVALID;
        else if (x > SP_MAX_PATTERN_LEN) return SP_ERR_TOO_LONG;
    std::vector<int> Us;
    std::vector<std::vector<int32_t>> members;
    if (!choose_classes(v, max_classes, Us, members)) return SP_ERR_TOO_LONG;
    *n_classes = static_cast<int>(Us.size());
    *padded_rows = 0;
    for (size_t k = 0; k < Us.size(); ++k) {
        const int n_bins = plan_bins(v, members[k], Us[k], nullptr);
        widths[k] = Us[k];
        n_patterns[k] = static_cast<int64_t>(members[k].size());
        n_warps[k] = n_bins;
        *padded_rows += static_cast<int64_t>(n_bins) * 32 * 32 * Us[k];
    }
    return SP_OK;
}

extern "C" sp_status sp_patterns_create(sp_ctx *ctx, const sp_seqset *patterns, sp_mode mode, sp_patterns **out) {
    if (!ctx) return SP_ERR_INVALID;
    if (!out) return fail(ctx, SP_ERR_INVALID, "sp_patterns_create: out is NULL");
    *out = nullptr;
    sp_status st = check_seqset(ctx, patterns, "patterns");
    if (st != SP_OK) return st;
    if (mode != SP_INFIX && mode != SP_PREFIX) return fail(ctx, SP_ERR_INVALID, "bad mode");
    SP_CUDA(ctx, cudaSetDevice(ctx->device));

    std::vector<int64_t> lens(static_cast<size_t>(patterns->n));
    int64_t total = 0, maxlen = 0;
    for (int64_t i = 0; i < patterns->n; ++i) {
        lens[static_cast<size_t>(i)] = patterns->offsets[i + 1] - patterns->offsets[i];
        total += lens[static_cast<size_t>(i)];
        maxlen = std::max(maxlen, lens[static_cast<size_t>(i)]);
    }
    if (maxlen > SP_MAX_PATTERN_LEN)
        return fail(ctx, SP_ERR_TOO_LONG,
                    "pattern of " + std::to_string(maxlen) + " bases exceeds SP_MAX_PATTERN_LEN (" +
                        std::to_string(SP_MAX_PATTERN_LEN) + ")");

    std::vector<int> Us;
    std::vector<std::vector<int32_t>> members;
    const char *maxc = getenv("SP_MAX_CLASSES");
    if (!choose_classes(lens, maxc ? std::max(1, atoi(maxc)) : 4, Us, members))
        return fail(ctx, SP_ERR_TOO_LONG, "no lane width fits the longest pattern");

    sp_patterns *p = new (std::nothrow) sp_patterns();
    if (!p) return fail(ctx, SP_ERR_NOMEM, "out of host memory");
    p->ctx = ctx; p->n = patterns->n; p->total_len = total; p->mode = mode;

    uint8_t *d_bases = nullptr; long long *d_offs = nullptr;
    int32_t *d_lane_pat = nullptr, *d_lane_row0 = nullptr; uint32_t *d_lane_info1 = nullptr;
    auto free_tabs = [&]() {
        dev_free(ctx, d_lane_pat); dev_free(ctx, d_lane_row0); dev_free(ctx, d_lane_info1);
        d_lane_pat = d_lane_row0 = nullptr; d_lane_info1 = nullptr;
    };
    auto cleanup = [&]() { dev_free(ctx, d_bases); dev_free(ctx, d_offs); free_tabs(); };
#define SP_TRY(x)                                   \
    do {                                            \
        sp_status s__ = (x);                        \
        if (s__ != SP_OK) { cleanup(); sp_patterns_destroy(p); return s__; } \
    } while (0)
    auto cu = [&](cudaError_t e, const char *what) -> sp_status {
        if (e != cudaSuccess) return fail(ctx, SP_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
        return SP_OK;
    };
    SP_TRY(upload_seqset(ctx, patterns, &d_bases, &d_offs));
    for (size_t k = 0; k < Us.size(); ++k) {
        const int U = Us[k];
        LaneTables lanes;
        const int n_bins = plan_bins(lens, members[k], U, &lanes);
        PatClass pc;
        pc.U = U;
        pc.n_groups = std::max(1, (n_bins + K1_WARPS - 1) / K1_WARPS);
        pc.n_bins = pc.n_groups * K1_WARPS;
        p->padded_rows += static_cast<int64_t>(n_bins) * 32 * 32 * U;
        const size_t tab = static_cast<size_t>(pc.n_bins) * 32;
        lanes.resize(pc.n_bins);
        SP_TRY(cu(dev_malloc(ctx, reinterpret_cast<void **>(&d_lane_pat), tab * 4), "cudaMalloc lane_pat"));
        SP_TRY(cu(dev_malloc(ctx, reinterpret_cast<void **>(&d_lane_row0), tab * 4), "cudaMalloc lane_row0"));
        SP_TRY(cu(dev_malloc(ctx, reinterpret_cast<void **>(&d_lane_info1), tab * 4), "cudaMalloc lane_info1"));
        SP_TRY(cu(dev_malloc(ctx, reinterpret_cast<void **>(&pc.d_blobs), static_cast<size_t>(pc.n_bins) * blob_words(U) * 4),
                  "cudaMalloc blobs"));
        p->classes.push_back(pc);  // owned by p from here on
        SP_TRY(cu(cudaMemcpyAsync(d_lane_pat, lanes.pat.data(), tab * 4, cudaMemcpyHostToDevice, ctx->stream), "H2D"));
        SP_TRY(cu(cudaMemcpyAsync(d_lane_row0, lanes.row0.data(), tab * 4, cudaMemcpyHostToDevice, ctx->stream), "H2D"));
        SP_TRY(cu(cudaMemcpyAsync(d_lane_info1, lanes.info1.data(), tab * 4, cudaMemcpyHostToDevice, ctx->stream), "H2D"));
        if (k == 0) ev_begin(ctx, 2);
        SP_TRY(sp_internal_pack_blobs(ctx, d_bases, d_offs, d_lane_pat, d_lane_row0, d_lane_info1, pc.d_blobs, pc.n_bins, U,
                                      mode == SP_PREFIX ? 1 : 0, 0));
        SP_TRY(cu(cudaStreamSynchronize(ctx->stream), "pack_patterns"));  // the plan's host vectors die with this iteration
        free_tabs();
    }
    ev_end(ctx, 2);
#undef SP_TRY
    cleanup();
    *out = p;
    return SP_OK;
}

extern "C" void sp_patterns_destroy(sp_patterns *p) {
    if (!p) return;
    cudaSetDevice(p->ctx->device);
    for (auto &c : p->classes) dev_free(p->ctx, c.d_blobs);
    delete p;
}
extern "C" int64_t sp_patterns_count(const sp_patterns *p) { return p ? p->n : 0; }
extern "C" int64_t sp_patterns_total_len(const sp_patterns *p) { return p ? p->total_len : 0; }
extern "C" int64_t sp_patterns_padded_rows(const sp_patterns *p) { return p ? p->padded_rows : 0; }

// ------------------------------------------------------------------------------------------
// targets
// ------------------------------------------------------------------------------------------
// host-side bookkeeping of a text set (chunk counts per text) from its offsets
static sp_status targets_from_offsets(sp_ctx *ctx, const int64_t *offsets, int64_t n, sp_targets **out) {
    sp_targets *t = new (std::nothrow) sp_targets();
    if (!t) return fail(ctx, SP_ERR_NOMEM, "out of host memory");
    t->ctx = ctx; t->n = n;
    t->nch.resize(static_cast<size_t>(n));
    t->h_offs.assign(static_cast<size_t>(n) + 1, 0);
    for (int64_t i = 0; i < n; ++i) {
        const int64_t len = offsets[i + 1] - offsets[i];
        t->h_offs[static_cast<size_t>(i) + 1] = t->h_offs[static_cast<size_t>(i)] + len;
        t->total_len += len;
        const int64_t nc = std::max<int64_t>(1, (len + K1_CHUNK - 1) / K1_CHUNK);
        if (nc > 0x3FFFFFFF) { delete t; return fail(ctx, SP_ERR_TOO_LONG, "text too long"); }
        t->nch[static_cast<size_t>(i)] = static_cast<int32_t>(nc);
        t->max_nch = std::max(t->max_nch, static_cast<int32_t>(nc));
        t->sum_nch += nc;
    }
    *out = t;
    return SP_OK;
}

extern "C" sp_status sp_targets_create(sp_ctx *ctx, const sp_seqset *targets, sp_targets **out) {
    if (!ctx) return SP_ERR_INVALID;
    if (!out) return fail(ctx, SP_ERR_INVALID, "sp_targets_create: out is NULL");
    *out = nullptr;
    sp_status st = check_seqset(ctx, targets, "targets");
    if (st != SP_OK) return st;
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    sp_targets *t = nullptr;
    const int64_t zero[1] = {0};
    st = targets_from_offsets(ctx, targets->n ? targets->offsets : zero, targets->n, &t);
    if (st != SP_OK) return st;
    st = upload_seqset(ctx, targets, &t->d_bases, &t->d_offs);
    if (st != SP_OK) { sp_targets_destroy(t); return st; }
    *out = t;
    return SP_OK;
}

// sp_comm.cu: a text set whose bases / rebased offsets (offs[0] == 0) are already on the device (received by broadcast);
// the handle takes ownership of both buffers (stream-ordered allocations of this context)
sp_status sp_internal_targets_adopt(sp_ctx *ctx, uint8_t *d_bases, long long *d_offs, const int64_t *host_offsets, int64_t n,
                                    sp_targets **out) {
    sp_targets *t = nullptr;
    sp_status st = targets_from_offsets(ctx, host_offsets, n, &t);
    if (st != SP_OK) return st;
    t->d_bases = d_bases; t->d_offs = d_offs;
    *out = t;
    return SP_OK;
}

extern "C" sp_status sp_targets_derive(sp_ctx *ctx, const sp_targets *src, int64_t n_out, const int32_t *src_index, const int64_t *iv_off,
                                       const int32_t *iv_begin, const int32_t *iv_end, const uint8_t *revcomp, sp_targets **out) {
    if (!ctx) return SP_ERR_INVALID;
    if (!out) return fail(ctx, SP_ERR_INVALID, "sp_targets_derive: out is NULL");
    *out = nullptr;
    if (!src || n_out < 0 || (n_out > 0 && (!src_index || !iv_off))) return fail(ctx, SP_ERR_INVALID, "sp_targets_derive: bad argument");
    const int64_t n_iv = n_out ? iv_off[n_out] : 0;
    if (n_out > 0 && (iv_off[0] != 0 || n_iv < 0 || (n_iv > 0 && (!iv_begin || !iv_end)))) return fail(ctx, SP_ERR_INVALID, "sp_targets_derive: bad interval table");
    std::vector<int64_t> out_offs(static_cast<size_t>(n_out) + 1, 0);
    std::vector<long long> iv_prefix(static_cast<size_t>(std::max<int64_t>(n_iv, 1)), 0), iv_off_ll(static_cast<size_t>(n_out) + 1, 0);
    for (int64_t q = 0; q < n_out; ++q) {
        if (src_index[q] < 0 || src_index[q] >= src->n || iv_off[q + 1] < iv_off[q]) return fail(ctx, SP_ERR_INVALID, "sp_targets_derive: bad source index or interval range");
        const int64_t slen = src->h_offs[static_cast<size_t>(src_index[q]) + 1] - src->h_offs[static_cast<size_t>(src_index[q])];
        int64_t len = 0;
        for (int64_t k = iv_off[q]; k < iv_off[q + 1]; ++k) {
            if (iv_begin[k] < 0 || iv_end[k] < iv_begin[k] || iv_end[k] > slen) return fail(ctx, SP_ERR_INVALID, "sp_targets_derive: interval outside its source sequence");
            iv_prefix[static_cast<size_t>(k)] = len;
            len += iv_end[k] - iv_begin[k];
        }
        out_offs[static_cast<size_t>(q) + 1] = out_offs[static_cast<size_t>(q)] + len;
        iv_off_ll[static_cast<size_t>(q) + 1] = iv_off[q + 1];
    }
    // empty intervals would break the "last interval whose prefix <= pos" search: they are dropped from the device tables
    std::vector<int32_t> begin_c;
    std::vector<long long> prefix_c, off_c(static_cast<size_t>(n_out) + 1, 0);
    for (int64_t q = 0; q < n_out; ++q) {
        for (int64_t k = iv_off[q]; k < iv_off[q + 1]; ++k)
            if (iv_end[k] > iv_begin[k]) { begin_c.push_back(iv_begin[k]); prefix_c.push_back(iv_prefix[static_cast<size_t>(k)]); }
        off_c[static_cast<size_t>(q) + 1] = static_cast<long long>(begin_c.size());
    }
    if (begin_c.empty()) { begin_c.push_back(0); prefix_c.push_back(0); }
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t total = out_offs[static_cast<size_t>(n_out)];
    std::vector<long long> out_offs_ll(out_offs.begin(), out_offs.end());
    std::vector<uint8_t> rc(static_cast<size_t>(std::max<int64_t>(n_out, 1)), 0);
    for (int64_t q = 0; q < n_out; ++q) rc[static_cast<size_t>(q)] = revcomp ? revcomp[q] : 0;
    uint8_t *d_bases = nullptr, *d_rc = nullptr;
    long long *d_offs = nullptr, *d_ivoff = nullptr, *d_prefix = nullptr;
    int32_t *d_src = nullptr, *d_begin = nullptr;
    auto cleanup = [&]() { dev_free(ctx, d_rc); dev_free(ctx, d_ivoff); dev_free(ctx, d_prefix); dev_free(ctx, d_src); dev_free(ctx, d_begin); };
    auto bail = [&](cudaError_t e) -> sp_status {
        cleanup(); dev_free(ctx, d_bases); dev_free(ctx, d_offs);
        return fail(ctx, e == cudaErrorMemoryAllocation ? SP_ERR_NOMEM : SP_ERR_CUDA, std::string("sp_targets_derive: ") + cudaGetErrorString(e));
    };
    cudaError_t e = dev_malloc(ctx, &d_bases, static_cast<size_t>(std::max<int64_t>(total, 16)));
    if (e == cudaSuccess) e = dev_malloc(ctx, &d_offs, out_offs_ll.size() * sizeof(long long));
    if (e == cudaSuccess) e = dev_malloc(ctx, &d_rc, rc.size());
    if (e == cudaSuccess) e = dev_malloc(ctx, &d_ivoff, off_c.size() * sizeof(long long));
    if (e == cudaSuccess) e = dev_malloc(ctx, &d_prefix, prefix_c.size() * sizeof(long long));
    if (e == cudaSuccess) e = dev_malloc(ctx, &d_src, static_cast<size_t>(std::max<int64_t>(n_out, 1)) * 4);
    if (e == cudaSuccess) e = dev_malloc(ctx, &d_begin, begin_c.size() * 4);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_offs, out_offs_ll.data(), out_offs_ll.size() * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_rc, rc.data(), rc.size(), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_ivoff, off_c.data(), off_c.size() * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_prefix, prefix_c.data(), prefix_c.size() * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && n_out) e = cudaMemcpyAsync(d_src, src_index, static_cast<size_t>(n_out) * 4, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_begin, begin_c.data(), begin_c.size() * 4, cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) return bail(e);
    if (total > 0) {
        DeriveParams prm;
        prm.src_bases = src->d_bases; prm.src_offs = src->d_offs; prm.src_index = d_src; prm.iv_off = d_ivoff; prm.iv_begin = d_begin;
        prm.iv_prefix = d_prefix; prm.revcomp = d_rc; prm.out_offs = d_offs; prm.out_bases = d_bases; prm.n_out = n_out; prm.total = total;
        derive_texts<<<static_cast<unsigned>((total + 255) / 256), 256, 0, ctx->stream>>>(prm);
        ++ctx->launches;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);  // the host tables above go out of scope
    if (e != cudaSuccess) return bail(e);
    cleanup();
    const sp_status st = sp_internal_targets_adopt(ctx, d_bases, d_offs, out_offs.data(), n_out, out);
    if (st != SP_OK) { dev_free(ctx, d_bases); dev_free(ctx, d_offs); }
    return st;
}

extern "C" sp_status sp_targets_read(const sp_targets *t, uint8_t *bases, int64_t *offsets) {
    if (!t) return SP_ERR_INVALID;
    sp_ctx *ctx = t->ctx;
    if (!offsets || (t->total_len > 0 && !bases)) return fail(ctx, SP_ERR_INVALID, "sp_targets_read: NULL argument");
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    for (int64_t i = 0; i <= t->n; ++i) offsets[i] = t->h_offs[static_cast<size_t>(i)];
    if (t->total_len > 0) {
        SP_CUDA(ctx, cudaMemcpyAsync(bases, t->d_bases, static_cast<size_t>(t->total_len), cudaMemcpyDeviceToHost, ctx->stream));
        SP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return SP_OK;
}

extern "C" void sp_targets_destroy(sp_targets *t) {
    if (!t) return;
    cudaSetDevice(t->ctx->device);
    for (auto &kv : t->packs) {
        dev_free(t->ctx, kv.second.d_text); dev_free(t->ctx, kv.second.d_tile_off); dev_free(t->ctx, kv.second.d_tile_text0);
    }
    dev_free(t->ctx, t->d_bases); dev_free(t->ctx, t->d_offs);
    delete t;
}
extern "C" int64_t sp_targets_count(const sp_targets *t) { return t ? t->n : 0; }
extern "C" int64_t sp_targets_total_len(const sp_targets *t) { return t ? t->total_len : 0; }

// builds (or returns the cached) tile stream for tile capacity tc
static sp_status get_text_pack(sp_ctx *ctx, sp_targets *t, int tc, const TextPack **out) {
    auto it = t->packs.find(tc);
    if (it != t->packs.end()) { *out = &it->second; return SP_OK; }
    std::vector<int32_t> tile_off(1, 0), tile_text0, text_chunk0(static_cast<size_t>(t->n));
    int64_t cur = 0, tile_start = 0;
    bool open = false;
    for (int64_t i = 0; i < t->n; ++i) {
        const int32_t nc = t->nch[static_cast<size_t>(i)];
        if (open && cur - tile_start + nc > tc) {  // close the tile, pad to an even chunk count (16-byte TMA granule)
            cur += (cur - tile_start) & 1;
            tile_off.push_back(static_cast<int32_t>(cur));
            open = false;
        }
        if (!open) { tile_start = cur; tile_text0.push_back(static_cast<int32_t>(i)); open = true; }
        text_chunk0[static_cast<size_t>(i)] = static_cast<int32_t>(cur);
        cur += nc;
        if (cur > 0x7FFFFFF0ll) return fail(ctx, SP_ERR_RANGE, "text set too large for one call");
    }
    if (open) { cur += (cur - tile_start) & 1; tile_off.push_back(static_cast<int32_t>(cur)); }
    TextPack pk;
    pk.tc = tc; pk.n_tiles = static_cast<int>(tile_text0.size()); pk.total_chunks = cur;
    int32_t *d_chunk0 = nullptr, *d_nch = nullptr;
    // on any CUDA error below nothing stays allocated (the pack is not cached either)
#define SP_PACK_CUDA(call)                                                                                       \
    do {                                                                                                         \
        cudaError_t e__ = (call);                                                                                \
        if (e__ != cudaSuccess) {                                                                                \
            dev_free(ctx, pk.d_text); dev_free(ctx, pk.d_tile_off); dev_free(ctx, pk.d_tile_text0);              \
            dev_free(ctx, d_chunk0); dev_free(ctx, d_nch);                                                       \
            return fail(ctx, e__ == cudaErrorMemoryAllocation ? SP_ERR_NOMEM : SP_ERR_CUDA,                      \
                        std::string(#call) + ": " + cudaGetErrorString(e__));                                    \
        }                                                                                                        \
    } while (0)
    SP_PACK_CUDA(dev_malloc(ctx, reinterpret_cast<void **>(&pk.d_text), static_cast<size_t>(std::max<int64_t>(cur, 2)) * 8));
    SP_PACK_CUDA(dev_malloc(ctx, reinterpret_cast<void **>(&pk.d_tile_off), tile_off.size() * 4));
    SP_PACK_CUDA(dev_malloc(ctx, reinterpret_cast<void **>(&pk.d_tile_text0), std::max<size_t>(tile_text0.size(), 1) * 4));
    SP_PACK_CUDA(dev_malloc(ctx, reinterpret_cast<void **>(&d_chunk0), std::max<size_t>(text_chunk0.size(), 1) * 4));
    SP_PACK_CUDA(dev_malloc(ctx, reinterpret_cast<void **>(&d_nch), std::max<size_t>(t->nch.size(), 1) * 4));
    SP_PACK_CUDA(cudaMemsetAsync(pk.d_text, 0x04, static_cast<size_t>(std::max<int64_t>(cur, 2)) * 8, ctx->stream));
    SP_PACK_CUDA(cudaMemcpyAsync(pk.d_tile_off, tile_off.data(), tile_off.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (!tile_text0.empty())
        SP_PACK_CUDA(cudaMemcpyAsync(pk.d_tile_text0, tile_text0.data(), tile_text0.size() * 4, cudaMemcpyHostToDevice,
                                     ctx->stream));
    if (t->n) {
        SP_PACK_CUDA(cudaMemcpyAsync(d_chunk0, text_chunk0.data(), text_chunk0.size() * 4, cudaMemcpyHostToDevice,
                                     ctx->stream));
        SP_PACK_CUDA(cudaMemcpyAsync(d_nch, t->nch.data(), t->nch.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
        const int blocks = static_cast<int>(std::min<int64_t>(t->n, 65535));
        ev_begin(ctx, 3);
        pack_texts<<<blocks, 128, 0, ctx->stream>>>(t->d_bases, t->d_offs, d_chunk0, d_nch, pk.d_text,
                                                    static_cast<int>(t->n));
        ev_end(ctx, 3);
        ++ctx->launches;
        SP_PACK_CUDA(cudaGetLastError());
    }
    SP_PACK_CUDA(cudaStreamSynchronize(ctx->stream));  // host vectors go out of scope
    dev_free(ctx, d_chunk0); dev_free(ctx, d_nch);
    auto ins = t->packs.emplace(tc, pk);
    *out = &ins.first->second;
    return SP_OK;
#undef SP_PACK_CUDA
}

// ------------------------------------------------------------------------------------------
// K1 launch
// ------------------------------------------------------------------------------------------
template <int U, bool TE>
static sp_status launch_k1(sp_ctx *ctx, const K1Params &prm, size_t smem, int n_items, bool first, bool last) {
    SP_CUDA(ctx, cudaFuncSetAttribute(k1_infix<U, TE>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    int occ = 0;
    SP_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k1_infix<U, TE>, K1_THREADS, smem));
    if (occ < 1) return fail(ctx, SP_ERR_CUDA, "K1 does not fit on an SM with the requested shared memory");
    if (first) ev_begin(ctx, 0);  // the K1 timer spans the launches of all lane-width classes of one call
    if (ctx->share_device) {
        // One CTA per item, handed out by the hardware: every retiring CTA is a slot the short kernels of the other contexts
        // on this GPU can take.  A launch of several rounds goes to the lowest-priority side stream, so that those kernels (and
        // this context's own short K1 launches, which stay on the main stream) are dispatched ahead of its waiting CTAs
        K1Params q = prm;
        q.next_item = nullptr;
        const bool bulk = n_items > 2 * ctx->num_sms * occ && !getenv("SP_SHARE_NOBULK");  // experiment hook: everything on the main stream
        if (bulk) {
            SP_CUDA(ctx, cudaEventRecord(ctx->bulk_fork, ctx->stream));
            SP_CUDA(ctx, cudaStreamWaitEvent(ctx->bulk, ctx->bulk_fork, 0));
        }
        k1_infix<U, TE><<<n_items, K1_THREADS, smem, bulk ? ctx->bulk : ctx->stream>>>(q);
        if (bulk) {
            SP_CUDA(ctx, cudaEventRecord(ctx->bulk_join, ctx->bulk));
            SP_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->bulk_join, 0));
        }
    } else {
        // persistent CTAs: a multiple of the SM count, each looping over (pattern-group, text-tile) items
        const int grid = std::min(n_items, ctx->num_sms * occ);
        SP_CUDA(ctx, cudaMemsetAsync(ctx->d_counter, 0, sizeof(int), ctx->stream));
        k1_infix<U, TE><<<grid, K1_THREADS, smem, ctx->stream>>>(prm);
    }
    if (last) ev_end(ctx, 0);
    ++ctx->launches;
    SP_CUDA(ctx, cudaGetLastError());
    return SP_OK;
}

template <bool TE>
static sp_status dispatch_k1(sp_ctx *ctx, int U, const K1Params &prm, size_t smem, int n_items, bool first, bool last) {
    switch (U) {
#define SP_CASE(u) case u: return launch_k1<u, TE>(ctx, prm, smem, n_items, first, last)
        SP_CASE(4); SP_CASE(5); SP_CASE(6); SP_CASE(7); SP_CASE(8); SP_CASE(9); SP_CASE(10); SP_CASE(11);
        SP_CASE(12); SP_CASE(13); SP_CASE(14); SP_CASE(15); SP_CASE(16); SP_CASE(20); SP_CASE(24);
#undef SP_CASE
        default: return fail(ctx, SP_ERR_INVALID, "unsupported lane width");
    }
}

// runs K1 for (t, p) writing D[(row0 + pattern) * ld + text] into caller-provided device memory
static sp_status run_k1(sp_ctx *ctx, sp_targets *t, const sp_patterns *p, void *out, int32_t *out_end, int64_t ld,
                        int elem_bits, int64_t row0) {
    if (t->n == 0 || p->n == 0 || p->total_len == 0) return SP_OK;
    for (size_t k = 0; k < p->classes.size(); ++k) {
        const PatClass &pc = p->classes[k];
        // tile capacity: 32 KB of text by default, grown for long texts, shrunk when the work list would be too short
        const int U = pc.U;
        const size_t blob_bytes = static_cast<size_t>(K1_WARPS) * blob_words(U) * 4;
        const int64_t max_tc = (static_cast<int64_t>(ctx->smem_optin) - static_cast<int64_t>(blob_bytes) - 1024) / 8 / 2 * 2;
        // Tile capacity (chunks).  Tiles hold whole texts; an item costs (chunks in the tile + 31 fill/drain steps) and the
        // persistent grid finishes about half an item late on average, so model  time ~ (tile + 31) * (items / grid + 1/2)
        // and take the best of a few capacities: big tiles when there is plenty of work (bench: 87 k items), small ones when
        // a call brings few reads (cohort: 64 reads per gene -> 1,246 items at 4,096 chunks was 4.2 rounds of 296 CTAs)
        int64_t tc = 4096;
        {
            const double avg = static_cast<double>(t->sum_nch) / static_cast<double>(std::max<int64_t>(t->n, 1));
            const double grid_ctas = 2.0 * ctx->num_sms;
            double best_cost = 0;
            for (int64_t cand : {4096, 3072, 2048, 1536, 1024, 768, 512, 384, 256}) {
                if (cand < t->max_nch && cand != 4096) continue;
                const double per_tile = std::max(1.0, std::floor(static_cast<double>(cand) / std::max(avg, 1.0)));
                const double tiles = std::ceil(static_cast<double>(t->n) / per_tile);
                const double tile_nch = std::min(per_tile, static_cast<double>(t->n)) * avg;
                const double cost = (tile_nch + 31.0) * (tiles * pc.n_groups / grid_ctas + 0.5);
                if (best_cost == 0 || cost < best_cost) { best_cost = cost; tc = cand; }
            }
        }
        if (const char *force_tc = getenv("SP_FORCE_TC")) tc = std::max<int64_t>(64, atoll(force_tc));  // experiment hook: tile capacity in chunks
        tc = std::max<int64_t>(tc, t->max_nch);
        tc = (tc + 1) / 2 * 2;
        if (tc > max_tc)
            return fail(ctx, SP_ERR_TOO_LONG,
                        "text of " + std::to_string(static_cast<long long>(t->max_nch) * K1_CHUNK) +
                            " columns exceeds the shared-memory tile budget (" + std::to_string(max_tc * K1_CHUNK) + ")");
        const TextPack *pk = nullptr;
        sp_status st = get_text_pack(ctx, t, static_cast<int>(tc), &pk);
        if (st != SP_OK) return st;

        K1Params prm;
        prm.blobs = pc.d_blobs; prm.text = pk->d_text; prm.tile_chunk_off = pk->d_tile_off; prm.tile_text0 = pk->d_tile_text0;
        prm.out = static_cast<char *>(out) + static_cast<size_t>(row0 * ld) * (elem_bits / 8);
        prm.out_end = out_end ? out_end + row0 * ld : nullptr;
        prm.ld = ld;
        prm.n_groups = pc.n_groups; prm.n_tiles = pk->n_tiles; prm.out16 = elem_bits == 16;
        prm.prefix_mode = p->mode == SP_PREFIX;
        prm.one = 1u; prm.m1 = 0xFFFFFFFFu; prm.sixteen = 16u;
        prm.next_item = ctx->d_counter;
        const int64_t n_items64 = static_cast<int64_t>(prm.n_groups) * prm.n_tiles;
        if (n_items64 > 0x7FFFFFFFll) return fail(ctx, SP_ERR_RANGE, "work list too large");
        const size_t smem = blob_bytes + static_cast<size_t>(tc + 2) * 8;
        const bool first = k == 0, last = k + 1 == p->classes.size();
        st = out_end ? dispatch_k1<true>(ctx, U, prm, smem, static_cast<int>(n_items64), first, last)
                     : dispatch_k1<false>(ctx, U, prm, smem, static_cast<int>(n_items64), first, last);
        if (st != SP_OK) return st;
    }
    return SP_OK;
}

extern "C" sp_status sp_score_device(sp_ctx *ctx, const sp_targets *t_in, const sp_patterns *p, int elem_bits,
                                     int want_end_col, sp_dmatrix **out) {
    if (!ctx) return SP_ERR_INVALID;
    if (!t_in || !p || !out) return fail(ctx, SP_ERR_INVALID, "sp_score_device: NULL argument");
    if (elem_bits != 16 && elem_bits != 32) return fail(ctx, SP_ERR_INVALID, "elem_bits must be 16 or 32");
    *out = nullptr;
    sp_targets *t = const_cast<sp_targets *>(t_in);  // the tile-stream cache is an implementation detail
    SP_CUDA(ctx, cudaSetDevice(ctx->device));

    sp_dmatrix *d = new (std::nothrow) sp_dmatrix();
    if (!d) return fail(ctx, SP_ERR_NOMEM, "out of host memory");
    d->ctx = ctx; d->nt = t->n; d->np = p->n; d->elem_bits = elem_bits;
    d->ld = (t->n + 63) / 64 * 64;
    const size_t elems = static_cast<size_t>(std::max<int64_t>(d->np * d->ld, 1));
    cudaError_t e = dev_malloc(ctx, &d->d, elems * (elem_bits / 8));
    if (e == cudaSuccess) e = cudaMemsetAsync(d->d, 0, elems * (elem_bits / 8), ctx->stream);
    if (e == cudaSuccess && want_end_col) {
        e = dev_malloc(ctx, reinterpret_cast<void **>(&d->d_end), elems * 4);
        if (e == cudaSuccess) e = cudaMemsetAsync(d->d_end, 0, elems * 4, ctx->stream);
    }
    if (e != cudaSuccess) {
        sp_dmatrix_destroy(d);
        return fail(ctx, e == cudaErrorMemoryAllocation ? SP_ERR_NOMEM : SP_ERR_CUDA,
                    std::string("distance matrix allocation: ") + cudaGetErrorString(e));
    }
    sp_status st = run_k1(ctx, t, p, d->d, d->d_end, d->ld, elem_bits, 0);
    if (st != SP_OK) { sp_dmatrix_destroy(d); return st; }
    *out = d;
    return SP_OK;
}

extern "C" sp_status sp_score_into(sp_ctx *ctx, const sp_targets *t_in, const sp_patterns *p, sp_dmatrix *dst,
                                   int64_t pattern_row0) {
    if (!ctx) return SP_ERR_INVALID;
    if (!t_in || !p || !dst) return fail(ctx, SP_ERR_INVALID, "sp_score_into: NULL argument");
    if (pattern_row0 < 0 || pattern_row0 + p->n > dst->np || t_in->n > dst->nt || t_in->n > dst->ld)
        return fail(ctx, SP_ERR_INVALID, "sp_score_into: destination matrix is too small");
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    // rows of empty patterns are defined as distance 0
    SP_CUDA(ctx, cudaMemsetAsync(static_cast<char *>(dst->d) + static_cast<size_t>(pattern_row0 * dst->ld) * (dst->elem_bits / 8),
                                 0, static_cast<size_t>(p->n * dst->ld) * (dst->elem_bits / 8), ctx->stream));
    return run_k1(ctx, const_cast<sp_targets *>(t_in), p, dst->d, nullptr, dst->ld, dst->elem_bits, pattern_row0);
}

extern "C" void sp_dmatrix_destroy(sp_dmatrix *d) {
    if (!d) return;
    if (d->owned) {
        cudaSetDevice(d->ctx->device);
        cudaStreamSynchronize(d->ctx->stream);
        dev_free(d->ctx, d->d);
        dev_free(d->ctx, d->d_end);
    }
    delete d;
}
extern "C" void *sp_dmatrix_device_ptr(const sp_dmatrix *d) { return d ? d->d : nullptr; }
extern "C" int64_t sp_dmatrix_ld(const sp_dmatrix *d) { return d ? d->ld : 0; }
extern "C" int sp_dmatrix_elem_bits(const sp_dmatrix *d) { return d ? d->elem_bits : 0; }

extern "C" sp_status sp_dmatrix_wrap(sp_ctx *ctx, void *dev_ptr, int64_t n_targets, int64_t n_patterns, int64_t ld,
                                     int elem_bits, sp_dmatrix **out) {
    if (!ctx) return SP_ERR_INVALID;
    if (!out || (!dev_ptr && n_targets * n_patterns > 0) || n_targets < 0 || n_patterns < 0 || ld < n_targets ||
        (elem_bits != 16 && elem_bits != 32))
        return fail(ctx, SP_ERR_INVALID, "sp_dmatrix_wrap: bad argument");
    sp_dmatrix *d = new (std::nothrow) sp_dmatrix();
    if (!d) return fail(ctx, SP_ERR_NOMEM, "out of host memory");
    d->ctx = ctx; d->d = dev_ptr; d->nt = n_targets; d->np = n_patterns; d->ld = ld; d->elem_bits = elem_bits;
    d->owned = false;
    *out = d;
    return SP_OK;
}

extern "C" sp_status sp_dmatrix_to_host(sp_ctx *ctx, const sp_dmatrix *d, int32_t *D, int32_t *end_col) {
    if (!ctx) return SP_ERR_INVALID;
    if (!d || (!D && !end_col)) return fail(ctx, SP_ERR_INVALID, "sp_dmatrix_to_host: NULL argument");
    if (end_col && !d->d_end) return fail(ctx, SP_ERR_INVALID, "matrix was scored without end columns");
    if (d->nt == 0 || d->np == 0) return SP_OK;
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = static_cast<size_t>(d->nt * d->np);
    int32_t *rows = nullptr;
    SP_CUDA(ctx, ctx_scratch(ctx, n * 4, reinterpret_cast<void **>(&rows)));
    const dim3 grid(static_cast<unsigned>((d->nt + 31) / 32), static_cast<unsigned>((d->np + 31) / 32)), blk(32, 8);
    cudaError_t e = cudaSuccess;
    if (D) {
        if (d->elem_bits == 16)
            dmatrix_to_rows<uint16_t, int32_t><<<grid, blk, 0, ctx->stream>>>(static_cast<const uint16_t *>(d->d), d->ld,
                                                                              static_cast<int>(d->nt), static_cast<int>(d->np), rows);
        else
            dmatrix_to_rows<int32_t, int32_t><<<grid, blk, 0, ctx->stream>>>(static_cast<const int32_t *>(d->d), d->ld,
                                                                             static_cast<int>(d->nt), static_cast<int>(d->np), rows);
        ++ctx->launches;
        e = cudaMemcpyAsync(D, rows, n * 4, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    }
    if (e == cudaSuccess && end_col) {
        dmatrix_to_rows<int32_t, int32_t><<<grid, blk, 0, ctx->stream>>>(d->d_end, d->ld, static_cast<int>(d->nt),
                                                                         static_cast<int>(d->np), rows);
        ++ctx->launches;
        e = cudaMemcpyAsync(end_col, rows, n * 4, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    }
    if (e != cudaSuccess) return fail(ctx, SP_ERR_CUDA, std::string("sp_dmatrix_to_host: ") + cudaGetErrorString(e));
    return SP_OK;
}

extern "C" sp_status sp_dmatrix_to_host_u16(sp_ctx *ctx, const sp_dmatrix *d, uint16_t *D) {
    if (!ctx) return SP_ERR_INVALID;
    if (!d || !D) return fail(ctx, SP_ERR_INVALID, "sp_dmatrix_to_host_u16: NULL argument");
    if (d->elem_bits != 16) return fail(ctx, SP_ERR_INVALID, "sp_dmatrix_to_host_u16: matrix is not 16-bit");
    if (d->nt == 0 || d->np == 0) return SP_OK;
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = static_cast<size_t>(d->nt * d->np);
    uint16_t *rows = nullptr;
    SP_CUDA(ctx, ctx_scratch(ctx, n * 2, reinterpret_cast<void **>(&rows)));
    const dim3 grid(static_cast<unsigned>((d->nt + 31) / 32), static_cast<unsigned>((d->np + 31) / 32)), blk(32, 8);
    dmatrix_to_rows<uint16_t, uint16_t><<<grid, blk, 0, ctx->stream>>>(static_cast<const uint16_t *>(d->d), d->ld,
                                                                       static_cast<int>(d->nt), static_cast<int>(d->np), rows);
    ++ctx->launches;
    cudaError_t e = cudaMemcpyAsync(D, rows, n * 2, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return fail(ctx, SP_ERR_CUDA, std::string("sp_dmatrix_to_host_u16: ") + cudaGetErrorString(e));
    return SP_OK;
}

// pinned host memory for callers that want full-speed PCIe copies into / out of the library
extern "C" sp_status sp_host_alloc(sp_ctx *ctx, size_t bytes, void **out) {
    if (!ctx) return SP_ERR_INVALID;
    if (!out) return fail(ctx, SP_ERR_INVALID, "sp_host_alloc: out is NULL");
    *out = nullptr;
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaError_t e = cudaHostAlloc(out, std::max<size_t>(bytes, 1), cudaHostAllocDefault);
    if (e != cudaSuccess) return fail(ctx, SP_ERR_NOMEM, std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
    return SP_OK;
}
extern "C" void sp_host_free(sp_ctx *ctx, void *ptr) {
    if (!ctx || !ptr) return;
    cudaSetDevice(ctx->device);
    cudaFreeHost(ptr);
}

extern "C" sp_status sp_score_batch(sp_ctx *ctx, const sp_seqset *targets, const sp_seqset *patterns, sp_mode mode,
                                    int32_t *D, int32_t *end_col) {
    if (!ctx) return SP_ERR_INVALID;
    if (!D) return fail(ctx, SP_ERR_INVALID, "sp_score_batch: D is NULL");
    sp_patterns *p = nullptr; sp_targets *t = nullptr; sp_dmatrix *d = nullptr;
    sp_status st = sp_patterns_create(ctx, patterns, mode, &p);
    if (st == SP_OK) st = sp_targets_create(ctx, targets, &t);
    if (st == SP_OK) st = sp_score_device(ctx, t, p, 32, end_col != nullptr, &d);
    if (st == SP_OK) st = sp_dmatrix_to_host(ctx, d, D, end_col);
    sp_dmatrix_destroy(d); sp_targets_destroy(t); sp_patterns_destroy(p);
    return st;
}

// ------------------------------------------------------------------------------------------
// K3 spans: distance + [start, end) of the optimal placement on the text
// ------------------------------------------------------------------------------------------
extern "C" sp_status sp_score_spans(sp_ctx *ctx, const sp_seqset *targets, const sp_seqset *patterns, int32_t *D,
                                    int32_t *start_col, int32_t *end_col) {
    return sp_score_spans_filtered(ctx, targets, patterns, -1, D, start_col, end_col);
}

extern "C" sp_status sp_score_spans_filtered(sp_ctx *ctx, const sp_seqset *targets, const sp_seqset *patterns, int max_dist_permille,
                                             int32_t *D, int32_t *start_col, int32_t *end_col) {
    if (!ctx) return SP_ERR_INVALID;
    if (!D || !start_col || !end_col) return fail(ctx, SP_ERR_INVALID, "sp_score_spans: NULL output");
    if (max_dist_permille > 1000) return fail(ctx, SP_ERR_INVALID, "sp_score_spans_filtered: max_dist_permille must be <= 1000 (or negative: no filter)");
    sp_patterns *p = nullptr; sp_targets *t = nullptr; sp_dmatrix *d = nullptr;
    uint8_t *d_bases = nullptr; long long *d_offs = nullptr;
    int32_t *d_lane_pat = nullptr, *d_lane_row0 = nullptr, *d_S = nullptr, *d_plen = nullptr;
    uint32_t *d_lane_info1 = nullptr, *d_blobs = nullptr;
    unsigned long long *d_next = nullptr;
    auto cleanup = [&]() {
        dev_free(ctx, d_bases); dev_free(ctx, d_offs); dev_free(ctx, d_lane_pat); dev_free(ctx, d_lane_row0); dev_free(ctx, d_lane_info1);
        dev_free(ctx, d_blobs); dev_free(ctx, d_S); dev_free(ctx, d_plen); dev_free(ctx, d_next);
        sp_dmatrix_destroy(d); sp_targets_destroy(t); sp_patterns_destroy(p);
    };
    // forward pass: distances and the smallest end column of a best placement
    sp_status st = sp_patterns_create(ctx, patterns, SP_INFIX, &p);
    if (st == SP_OK) st = sp_targets_create(ctx, targets, &t);
    if (st == SP_OK) st = sp_score_device(ctx, t, p, 32, 1, &d);
    if (st != SP_OK) { cleanup(); return st; }
    const int64_t np = patterns->n, nt = targets->n;
    if (np == 0 || nt == 0) { cleanup(); return SP_OK; }
    auto cu = [&](cudaError_t e, const char *what) -> sp_status {
        if (e != cudaSuccess) return fail(ctx, SP_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
        return SP_OK;
    };
#define SP_TRY(x)                                   \
    do {                                            \
        sp_status s__ = (x);                        \
        if (s__ != SP_OK) { cleanup(); return s__; } \
    } while (0)
    // reversed patterns, one per bin, anchored (prefix) pad rows
    int64_t longest = 0;
    for (int64_t i = 0; i < np; ++i) longest = std::max(longest, patterns->offsets[i + 1] - patterns->offsets[i]);
    const int span_u = longest > 32ll * 32 * SPAN_U ? SPAN_U_LONG : SPAN_U;
    const int64_t rows = 32ll * span_u;
    const size_t tab = static_cast<size_t>(np) * 32;
    LaneTables lanes;
    lanes.resize(static_cast<int>(np));
    for (int64_t i = 0; i < np; ++i) {
        const int64_t m = patterns->offsets[i + 1] - patterns->offsets[i];
        if (m > 0)  // nl <= 32: checked by sp_patterns_create
            lanes.place(static_cast<int>(i), 0, static_cast<int>((m + rows - 1) / rows), static_cast<int32_t>(i), m, span_u);
    }
    SP_TRY(upload_seqset(ctx, patterns, &d_bases, &d_offs));
    SP_TRY(cu(dev_malloc(ctx, reinterpret_cast<void **>(&d_lane_pat), tab * 4), "cudaMalloc"));
    SP_TRY(cu(dev_malloc(ctx, reinterpret_cast<void **>(&d_lane_row0), tab * 4), "cudaMalloc"));
    SP_TRY(cu(dev_malloc(ctx, reinterpret_cast<void **>(&d_lane_info1), tab * 4), "cudaMalloc"));
    SP_TRY(cu(dev_malloc(ctx, reinterpret_cast<void **>(&d_blobs), static_cast<size_t>(np) * blob_words(span_u) * 4), "cudaMalloc span blobs"));
    SP_TRY(cu(dev_malloc(ctx, reinterpret_cast<void **>(&d_S), static_cast<size_t>(np * d->ld) * 4), "cudaMalloc span starts"));
    SP_TRY(cu(cudaMemsetAsync(d_S, 0, static_cast<size_t>(np * d->ld) * 4, ctx->stream), "memset"));
    std::vector<int32_t> plen(static_cast<size_t>(np));
    for (int64_t i = 0; i < np; ++i) plen[static_cast<size_t>(i)] = static_cast<int32_t>(patterns->offsets[i + 1] - patterns->offsets[i]);
    SP_TRY(cu(dev_malloc(ctx, reinterpret_cast<void **>(&d_plen), static_cast<size_t>(np) * 4), "cudaMalloc"));
    SP_TRY(cu(cudaMemcpyAsync(d_plen, plen.data(), static_cast<size_t>(np) * 4, cudaMemcpyHostToDevice, ctx->stream), "H2D"));
    SP_TRY(cu(dev_malloc(ctx, reinterpret_cast<void **>(&d_next), sizeof(unsigned long long)), "cudaMalloc"));
    SP_TRY(cu(cudaMemsetAsync(d_next, 0, sizeof(unsigned long long), ctx->stream), "memset"));
    SP_TRY(cu(cudaMemcpyAsync(d_lane_pat, lanes.pat.data(), tab * 4, cudaMemcpyHostToDevice, ctx->stream), "H2D"));
    SP_TRY(cu(cudaMemcpyAsync(d_lane_row0, lanes.row0.data(), tab * 4, cudaMemcpyHostToDevice, ctx->stream), "H2D"));
    SP_TRY(cu(cudaMemcpyAsync(d_lane_info1, lanes.info1.data(), tab * 4, cudaMemcpyHostToDevice, ctx->stream), "H2D"));
    SP_TRY(sp_internal_pack_blobs(ctx, d_bases, d_offs, d_lane_pat, d_lane_row0, d_lane_info1, d_blobs, static_cast<int>(np), span_u, 1, 1));
    {
        SpanParams prm;
        prm.blobs = d_blobs; prm.tbases = t->d_bases; prm.toffs = t->d_offs;
        prm.D = static_cast<const int32_t *>(d->d); prm.E = d->d_end; prm.S = d_S; prm.ld = d->ld;
        prm.nt = static_cast<int>(nt); prm.np = static_cast<int>(np); prm.one = 1u; prm.m1 = 0xFFFFFFFFu;
        prm.max_dist_permille = max_dist_permille; prm.plen = d_plen; prm.next_pair = d_next;
        const size_t smem = static_cast<size_t>(K1_WARPS) * blob_words(span_u) * 4;
        const long long total = nt * np;
        const int grid = static_cast<int>(std::min<long long>(2ll * ctx->num_sms, (total + K1_WARPS - 1) / K1_WARPS));
        if (span_u == SPAN_U) {
            SP_TRY(cu(cudaFuncSetAttribute(k3_span_starts<SPAN_U>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)), "k3_span_starts smem"));
            k3_span_starts<SPAN_U><<<grid, K1_THREADS, smem, ctx->stream>>>(prm);
        } else {
            SP_TRY(cu(cudaFuncSetAttribute(k3_span_starts<SPAN_U_LONG>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)), "k3_span_starts smem"));
            k3_span_starts<SPAN_U_LONG><<<grid, K1_THREADS, smem, ctx->stream>>>(prm);
        }
        ++ctx->launches;
        SP_TRY(cu(cudaGetLastError(), "k3_span_starts launch"));
    }
    SP_TRY(sp_dmatrix_to_host(ctx, d, D, end_col));
    {
        sp_dmatrix view = *d;  // same geometry, start columns as the payload
        view.d = d_S; view.d_end = nullptr; view.owned = false;
        SP_TRY(sp_dmatrix_to_host(ctx, &view, start_col, nullptr));
    }
#undef SP_TRY
    cleanup();
    return SP_OK;
}

// ------------------------------------------------------------------------------------------
// K5: row top-k of a device distance matrix
// ------------------------------------------------------------------------------------------
extern "C" sp_status sp_row_topk_biased(sp_ctx *ctx, const sp_dmatrix *d, const int32_t *pattern_bias, int k, int32_t *idx,
                                        int32_t *dist) {
    return sp_row_topk_weighted(ctx, d, 1, pattern_bias, k, idx, dist);
}

extern "C" sp_status sp_row_topk_weighted(sp_ctx *ctx, const sp_dmatrix *d, int dist_weight, const int32_t *pattern_bias, int k,
                                          int32_t *idx, int32_t *dist) {
    if (!ctx) return SP_ERR_INVALID;
    // the 32-bit key weight * distance + bias must not wrap: K1 distances are <= SP_MAX_PATTERN_LEN (< 2^15), biases < 2^30
    if (dist_weight < 1 || dist_weight > 64) return fail(ctx, SP_ERR_INVALID, "sp_row_topk_weighted: dist_weight must be in [1, 64]");
    if (!d || !idx || !dist) return fail(ctx, SP_ERR_INVALID, "sp_row_topk: NULL argument");
    if (k < 1 || k > 16) return fail(ctx, SP_ERR_INVALID, "sp_row_topk: k must be in [1, 16]");
    if (d->nt > 0x7FFFFFF0ll || d->np > 0x7FFFFFF0ll) return fail(ctx, SP_ERR_RANGE, "sp_row_topk: matrix too large");
    if (d->nt == 0) return SP_OK;
    if (pattern_bias)
        for (int64_t p = 0; p < d->np; ++p)
            if (pattern_bias[p] < 0 || pattern_bias[p] > 0x3FFFFFFF) return fail(ctx, SP_ERR_INVALID, "sp_row_topk_biased: bias must be in [0, 2^30)");
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = static_cast<size_t>(d->nt) * static_cast<size_t>(k);
    void *buf = nullptr;
    SP_CUDA(ctx, ctx_scratch(ctx, 2 * n * sizeof(int32_t), &buf));
    int32_t *d_idx = static_cast<int32_t *>(buf), *d_dist = d_idx + n;
    int32_t *d_bias = nullptr;
    if (pattern_bias && d->np > 0) {
        SP_CUDA(ctx, dev_malloc(ctx, &d_bias, static_cast<size_t>(d->np) * sizeof(int32_t)));
        cudaError_t e = cudaMemcpyAsync(d_bias, pattern_bias, static_cast<size_t>(d->np) * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) { dev_free(ctx, d_bias); SP_CUDA(ctx, e); }
    }
    const int nt = static_cast<int>(d->nt), np = static_cast<int>(d->np);
    const unsigned grid = static_cast<unsigned>((nt + 127) / 128);
    if (d->elem_bits == 16) {
        if (k <= 8) k5_row_topk<uint16_t, 8><<<grid, 128, 0, ctx->stream>>>(static_cast<const uint16_t *>(d->d), d->ld, nt, np, k, d_bias, static_cast<uint32_t>(dist_weight), d_idx, d_dist);
        else k5_row_topk<uint16_t, 16><<<grid, 128, 0, ctx->stream>>>(static_cast<const uint16_t *>(d->d), d->ld, nt, np, k, d_bias, static_cast<uint32_t>(dist_weight), d_idx, d_dist);
    } else {
        if (k <= 8) k5_row_topk<int32_t, 8><<<grid, 128, 0, ctx->stream>>>(static_cast<const int32_t *>(d->d), d->ld, nt, np, k, d_bias, static_cast<uint32_t>(dist_weight), d_idx, d_dist);
        else k5_row_topk<int32_t, 16><<<grid, 128, 0, ctx->stream>>>(static_cast<const int32_t *>(d->d), d->ld, nt, np, k, d_bias, static_cast<uint32_t>(dist_weight), d_idx, d_dist);
    }
    ++ctx->launches;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(idx, d_idx, n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dist, d_dist, n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    dev_free(ctx, d_bias);
    SP_CUDA(ctx, e);
    return SP_OK;
}

extern "C" sp_status sp_row_topk(sp_ctx *ctx, const sp_dmatrix *d, int k, int32_t *idx, int32_t *dist) {
    return sp_row_topk_biased(ctx, d, nullptr, k, idx, dist);
}

// ------------------------------------------------------------------------------------------
// K6: allele-vector match
// ------------------------------------------------------------------------------------------
extern "C" sp_status sp_variant_match(sp_ctx *ctx, int64_t n_seq, int64_t n_hap, int64_t n_var, const uint8_t *seq_alleles,
                                      const uint8_t *hap_alleles, const uint8_t *is_vi, uint32_t *vi_match, uint32_t *all_match) {
    if (!ctx) return SP_ERR_INVALID;
    if (n_seq < 0 || n_hap < 0 || n_var < 0) return fail(ctx, SP_ERR_INVALID, "sp_variant_match: negative size");
    if (n_seq * n_hap > 0 && (!vi_match || !all_match)) return fail(ctx, SP_ERR_INVALID, "sp_variant_match: NULL output");
    if (n_var > 0 && ((n_seq > 0 && !seq_alleles) || (n_hap > 0 && !hap_alleles) || !is_vi))
        return fail(ctx, SP_ERR_INVALID, "sp_variant_match: NULL input");
    if (n_seq > 0x3FFFFFFFll || n_hap > 0x3FFFFFFFll || n_var > 0x3FFFFFFFll || n_seq * n_hap > 0x7FFFFFFF0ll)
        return fail(ctx, SP_ERR_RANGE, "sp_variant_match: problem too large");
    if (n_seq == 0 || n_hap == 0) return SP_OK;
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int W = static_cast<int>((n_var + 31) / 32);
    const size_t cells = static_cast<size_t>(n_seq) * static_cast<size_t>(n_hap);
    if (W == 0) {  // no sites: nothing matches
        std::fill(vi_match, vi_match + cells, 0u);
        std::fill(all_match, all_match + cells, 0u);
        return SP_OK;
    }
    uint8_t *d_seq = nullptr, *d_hap = nullptr, *d_vi = nullptr;
    uint32_t *d_sp = nullptr, *d_hp = nullptr, *d_vp = nullptr, *d_out = nullptr;
    int *d_bad = nullptr;
    auto cleanup = [&]() {
        dev_free(ctx, d_seq); dev_free(ctx, d_hap); dev_free(ctx, d_vi); dev_free(ctx, d_sp); dev_free(ctx, d_hp); dev_free(ctx, d_vp);
        dev_free(ctx, d_out); dev_free(ctx, d_bad);
    };
    auto cu = [&](cudaError_t e, const char *what) -> sp_status {
        if (e != cudaSuccess)
            return fail(ctx, e == cudaErrorMemoryAllocation ? SP_ERR_NOMEM : SP_ERR_CUDA,
                        std::string("sp_variant_match: ") + what + ": " + cudaGetErrorString(e));
        return SP_OK;
    };
#define SP_TRY(x)                                   \
    do {                                            \
        sp_status s__ = (x);                        \
        if (s__ != SP_OK) { cleanup(); return s__; } \
    } while (0)
    auto up = [&](uint8_t **dst, const uint8_t *src, size_t bytes) -> sp_status {
        sp_status st = cu(dev_malloc(ctx, dst, bytes), "cudaMalloc");
        if (st == SP_OK) st = cu(cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream), "H2D");
        return st;
    };
    SP_TRY(up(&d_seq, seq_alleles, static_cast<size_t>(n_seq) * n_var));
    SP_TRY(up(&d_hap, hap_alleles, static_cast<size_t>(n_hap) * n_var));
    SP_TRY(up(&d_vi, is_vi, static_cast<size_t>(n_var)));
    SP_TRY(cu(dev_malloc(ctx, &d_sp, static_cast<size_t>(n_seq) * 3 * W * 4), "cudaMalloc"));
    SP_TRY(cu(dev_malloc(ctx, &d_hp, static_cast<size_t>(n_hap) * 2 * W * 4), "cudaMalloc"));
    SP_TRY(cu(dev_malloc(ctx, &d_vp, static_cast<size_t>(2) * W * 4), "cudaMalloc"));
    SP_TRY(cu(dev_malloc(ctx, &d_out, 2 * cells * 4), "cudaMalloc"));
    SP_TRY(cu(dev_malloc(ctx, &d_bad, sizeof(int)), "cudaMalloc"));
    SP_TRY(cu(cudaMemsetAsync(d_bad, 0, sizeof(int), ctx->stream), "memset"));
    const int nv = static_cast<int>(n_var);
    k6_pack_states<<<static_cast<unsigned>((n_seq + 7) / 8), 256, 0, ctx->stream>>>(d_seq, static_cast<int>(n_seq), nv, W, 3, 3, d_sp, d_bad);
    k6_pack_states<<<static_cast<unsigned>((n_hap + 7) / 8), 256, 0, ctx->stream>>>(d_hap, static_cast<int>(n_hap), nv, W, 2, 1, d_hp, d_bad);
    k6_pack_states<<<1, 256, 0, ctx->stream>>>(d_vi, 1, nv, W, 2, 1, d_vp, d_bad);
    k6_variant_match<<<static_cast<unsigned>((cells + 255) / 256), 256, 0, ctx->stream>>>(d_sp, d_hp, d_vp, static_cast<int>(n_seq),
                                                                                        static_cast<int>(n_hap), W, d_out, d_out + cells);
    ctx->launches += 4;
    SP_TRY(cu(cudaGetLastError(), "k6 launch"));
    int bad = 0;
    SP_TRY(cu(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream), "D2H"));
    SP_TRY(cu(cudaMemcpyAsync(vi_match, d_out, cells * 4, cudaMemcpyDeviceToHost, ctx->stream), "D2H"));
    SP_TRY(cu(cudaMemcpyAsync(all_match, d_out + cells, cells * 4, cudaMemcpyDeviceToHost, ctx->stream), "D2H"));
    SP_TRY(cu(cudaStreamSynchronize(ctx->stream), "k6_variant_match"));
#undef SP_TRY
    cleanup();
    if (bad) return fail(ctx, SP_ERR_INVALID, "sp_variant_match: site state outside 0..3 (sequences) or 0..1 (haplotypes, is_vi)");
    return SP_OK;
}

// ------------------------------------------------------------------------------------------
// K3 chain windows
// ------------------------------------------------------------------------------------------
extern "C" sp_status sp_chain_window_scores(sp_ctx *ctx, int64_t n_chains, const int32_t *chain_off,
                                            const int32_t *chain_items, int64_t n_reads, const int32_t *seg_off,
                                            const uint32_t *W, int64_t n_haps, sp_dmatrix **out) {
    if (!ctx) return SP_ERR_INVALID;
    if (!out || n_chains < 0 || n_reads < 0 || n_haps < 0 || (n_chains > 0 && (!chain_off || !chain_items)) ||
        (n_reads > 0 && (!seg_off || !W)))
        return fail(ctx, SP_ERR_INVALID, "sp_chain_window_scores: bad argument");
    *out = nullptr;
    if (n_chains > 0x7FFFFFF0ll || n_reads > 0x7FFFFFF0ll || n_haps > 0x7FFFFFF0ll)
        return fail(ctx, SP_ERR_RANGE, "sp_chain_window_scores: too many chains / reads");
    const int64_t n_items = n_chains ? chain_off[n_chains] : 0, n_segs = n_reads ? seg_off[n_reads] : 0;
    for (int64_t c = 0; c < n_chains; ++c)
        if (chain_off[c + 1] < chain_off[c]) return fail(ctx, SP_ERR_INVALID, "chain offsets must be non-decreasing");
    for (int64_t r = 0; r < n_reads; ++r)
        if (seg_off[r + 1] < seg_off[r]) return fail(ctx, SP_ERR_INVALID, "segment offsets must be non-decreasing");
    for (int64_t q = 0; q < n_items; ++q)
        if (chain_items[q] < 0 || chain_items[q] >= n_haps) return fail(ctx, SP_ERR_INVALID, "chain item outside [0, n_haps)");
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    sp_dmatrix *d = new (std::nothrow) sp_dmatrix();
    if (!d) return fail(ctx, SP_ERR_NOMEM, "out of host memory");
    d->ctx = ctx; d->nt = n_reads; d->np = n_chains; d->elem_bits = 32; d->ld = (n_reads + 63) / 64 * 64;
    int32_t *d_coff = nullptr, *d_items = nullptr, *d_soff = nullptr; uint32_t *d_W = nullptr;
    auto cleanup = [&]() { dev_free(ctx, d_coff); dev_free(ctx, d_items); dev_free(ctx, d_soff); dev_free(ctx, d_W); };
    auto up = [&](void **dst, const void *src, size_t bytes) -> cudaError_t {
        cudaError_t e = dev_malloc(ctx, dst, std::max<size_t>(bytes, 16));
        if (e == cudaSuccess && bytes) e = cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream);
        return e;
    };
    const size_t elems = static_cast<size_t>(std::max<int64_t>(d->np * d->ld, 1));
    cudaError_t e = dev_malloc(ctx, &d->d, elems * 4);
    if (e == cudaSuccess) e = cudaMemsetAsync(d->d, 0, elems * 4, ctx->stream);
    if (e == cudaSuccess) e = up(reinterpret_cast<void **>(&d_coff), chain_off, static_cast<size_t>(n_chains + 1) * 4 * (n_chains > 0));
    if (e == cudaSuccess) e = up(reinterpret_cast<void **>(&d_items), chain_items, static_cast<size_t>(n_items) * 4);
    if (e == cudaSuccess) e = up(reinterpret_cast<void **>(&d_soff), seg_off, static_cast<size_t>(n_reads + 1) * 4 * (n_reads > 0));
    if (e == cudaSuccess) e = up(reinterpret_cast<void **>(&d_W), W, static_cast<size_t>(n_segs * n_haps) * 4);
    if (e == cudaSuccess && n_chains > 0 && n_reads > 0) {
        ChainWinParams prm;
        prm.chain_off = d_coff; prm.chain_items = d_items; prm.seg_off = d_soff; prm.W = d_W;
        prm.B = static_cast<int32_t *>(d->d); prm.ld = d->ld;
        prm.n_chains = static_cast<int>(n_chains); prm.n_reads = static_cast<int>(n_reads); prm.n_haps = static_cast<int>(n_haps);
        const dim3 grid(static_cast<unsigned>((n_reads + 255) / 256), static_cast<unsigned>(std::min<int64_t>(n_chains, 65535)));
        k3_chain_windows<<<grid, 256, 0, ctx->stream>>>(prm);
        ++ctx->launches;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);  // the caller's host arrays may go away
    cleanup();
    if (e != cudaSuccess) {
        sp_dmatrix_destroy(d);
        return fail(ctx, e == cudaErrorMemoryAllocation ? SP_ERR_NOMEM : SP_ERR_CUDA,
                    std::string("sp_chain_window_scores: ") + cudaGetErrorString(e));
    }
    *out = d;
    return SP_OK;
}

// ------------------------------------------------------------------------------------------
// K2
// ------------------------------------------------------------------------------------------
static sp_status k2_check(sp_ctx *ctx, const sp_dmatrix *d) {
    if (!d) return fail(ctx, SP_ERR_INVALID, "K2: matrix is NULL");
    if (d->np > 0x7FFFFFFFll || d->nt > 0x7FFFFFFFll) return fail(ctx, SP_ERR_RANGE, "K2: matrix too large");
    return SP_OK;
}

template <typename T>
static void launch_k2_topk(const K2Params &prm, unsigned n_ctas, bool dual, cudaStream_t st) {
    if (dual) k2_pair_minsum<T, false, true><<<n_ctas, K2_THREADS, 0, st>>>(prm);
    else k2_pair_minsum<T, false, false><<<n_ctas, K2_THREADS, 0, st>>>(prm);
}

extern "C" sp_status sp_pair_minsum_topk(sp_ctx *ctx, const sp_dmatrix *d, const sp_dmatrix *d2, int64_t i_begin,
                                         int64_t i_end, int k, sp_pair_rec *out, int *n_out) {
    if (!ctx) return SP_ERR_INVALID;
    sp_status st = k2_check(ctx, d);
    if (st != SP_OK) return st;
    if (d2 && (d2->nt != d->nt || d2->np != d->np || d2->elem_bits != d->elem_bits))
        return fail(ctx, SP_ERR_INVALID, "K2: secondary matrix must have the geometry and element type of the primary");
    if (!out || !n_out || k < 1 || k > K2_MAXK) return fail(ctx, SP_ERR_INVALID, "K2: bad k / NULL output");
    if (d->elem_bits == 16 && d->nt > 65536) return fail(ctx, SP_ERR_RANGE, "K2: more than 65536 reads need a 32-bit matrix");
    *n_out = 0;
    const int A = static_cast<int>(d->np);
    i_begin = std::max<int64_t>(i_begin, 0);
    i_end = std::min<int64_t>(i_end, A);
    if (i_begin >= i_end) return SP_OK;
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    K2Params prm;
    prm.D = d->d; prm.ld = d->ld; prm.D2 = d2 ? d2->d : nullptr; prm.ld2 = d2 ? d2->ld : 0;
    prm.R = static_cast<int>(d->nt); prm.A = A;
    prm.i_begin = static_cast<int>(i_begin); prm.i_end = static_cast<int>(i_end);
    prm.tile_i0 = prm.i_begin / K2_TILE;
    prm.n_tiles_j = (A + K2_TILE - 1) / K2_TILE;
    prm.k = k; prm.S = nullptr;
    const int tile_i1 = (prm.i_end + K2_TILE - 1) / K2_TILE;
    long long n_ctas = 0;
    for (int I = prm.tile_i0; I < tile_i1; ++I) n_ctas += prm.n_tiles_j - I;
    if (n_ctas > 0x7FFFFFFFll) return fail(ctx, SP_ERR_RANGE, "K2: too many tiles");
    SP_CUDA(ctx, dev_malloc(ctx, reinterpret_cast<void **>(&prm.cand), static_cast<size_t>(n_ctas) * k * sizeof(PairKey)));
    ev_begin(ctx, 1);
    if (d->elem_bits == 16) launch_k2_topk<uint16_t>(prm, static_cast<unsigned>(n_ctas), d2 != nullptr, ctx->stream);
    else launch_k2_topk<int32_t>(prm, static_cast<unsigned>(n_ctas), d2 != nullptr, ctx->stream);
    ev_end(ctx, 1);
    ++ctx->launches;
    std::vector<PairKey> cand(static_cast<size_t>(n_ctas) * k);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(cand.data(), prm.cand, cand.size() * sizeof(PairKey), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    dev_free(ctx, prm.cand);
    if (e != cudaSuccess) return fail(ctx, SP_ERR_CUDA, std::string("K2: ") + cudaGetErrorString(e));
    // merge of the per-tile lists: same (score, score2, i, j) order, so any sharding gives the same answer
    auto less = [](const PairKey &a, const PairKey &b) {
        if (a.score != b.score) return a.score < b.score;
        if (a.score2 != b.score2) return a.score2 < b.score2;
        return a.ij < b.ij;
    };
    cand.erase(std::remove_if(cand.begin(), cand.end(), [](const PairKey &c) { return c.ij == ~0ull; }), cand.end());
    const size_t kk = std::min<size_t>(static_cast<size_t>(k), cand.size());
    std::partial_sort(cand.begin(), cand.begin() + static_cast<std::ptrdiff_t>(kk), cand.end(), less);
    if (kk == 0) return SP_OK;
    std::vector<uint32_t> ij(2 * kk), c1(kk);
    for (size_t q = 0; q < kk; ++q) {
        ij[2 * q] = static_cast<uint32_t>(cand[q].ij >> 32);
        ij[2 * q + 1] = static_cast<uint32_t>(cand[q].ij & 0xFFFFFFFFu);
    }
    uint32_t *d_ij = nullptr, *d_c1 = nullptr;
    e = dev_malloc(ctx, reinterpret_cast<void **>(&d_ij), ij.size() * 4);
    if (e == cudaSuccess) e = dev_malloc(ctx, reinterpret_cast<void **>(&d_c1), c1.size() * 4);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_ij, ij.data(), ij.size() * 4, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        if (d->elem_bits == 16)
            k2_count_c1<uint16_t><<<static_cast<unsigned>(kk), 256, 0, ctx->stream>>>(
                static_cast<const uint16_t *>(d->d), d->ld, d2 ? static_cast<const uint16_t *>(d2->d) : nullptr, prm.ld2, prm.R, d_ij, d_c1);
        else
            k2_count_c1<int32_t><<<static_cast<unsigned>(kk), 256, 0, ctx->stream>>>(
                static_cast<const int32_t *>(d->d), d->ld, d2 ? static_cast<const int32_t *>(d2->d) : nullptr, prm.ld2, prm.R, d_ij, d_c1);
        ++ctx->launches;
        e = cudaMemcpyAsync(c1.data(), d_c1, c1.size() * 4, cudaMemcpyDeviceToHost, ctx->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    dev_free(ctx, d_ij); dev_free(ctx, d_c1);
    if (e != cudaSuccess) return fail(ctx, SP_ERR_CUDA, std::string("K2 c1: ") + cudaGetErrorString(e));
    for (size_t q = 0; q < kk; ++q) {
        out[q].score = cand[q].score; out[q].score2 = cand[q].score2;
        out[q].i = ij[2 * q]; out[q].j = ij[2 * q + 1]; out[q].c1 = c1[q]; out[q]._pad = 0;
    }
    *n_out = static_cast<int>(kk);
    return SP_OK;
}

extern "C" sp_status sp_pair_minsum_full(sp_ctx *ctx, const sp_dmatrix *d, uint64_t *S) {
    if (!ctx) return SP_ERR_INVALID;
    sp_status st = k2_check(ctx, d);
    if (st != SP_OK) return st;
    if (!S) return fail(ctx, SP_ERR_INVALID, "K2: S is NULL");
    const int A = static_cast<int>(d->np);
    if (A == 0) return SP_OK;
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    K2Params prm;
    prm.D = d->d; prm.ld = d->ld; prm.D2 = nullptr; prm.ld2 = 0; prm.R = static_cast<int>(d->nt); prm.A = A;
    if (d->elem_bits == 16 && d->nt > 65536) return fail(ctx, SP_ERR_RANGE, "K2: more than 65536 reads need a 32-bit matrix");
    prm.i_begin = 0; prm.i_end = A; prm.tile_i0 = 0; prm.n_tiles_j = (A + K2_TILE - 1) / K2_TILE;
    prm.k = 0; prm.cand = nullptr;
    const long long n_ctas = static_cast<long long>(prm.n_tiles_j) * (prm.n_tiles_j + 1) / 2;
    const size_t bytes = static_cast<size_t>(A) * A * sizeof(unsigned long long);
    SP_CUDA(ctx, dev_malloc(ctx, reinterpret_cast<void **>(&prm.S), bytes));
    cudaError_t e = cudaMemsetAsync(prm.S, 0, bytes, ctx->stream);
    if (e == cudaSuccess) {
        ev_begin(ctx, 1);
        if (d->elem_bits == 16) k2_pair_minsum<uint16_t, true, false><<<static_cast<unsigned>(n_ctas), K2_THREADS, 0, ctx->stream>>>(prm);
        else k2_pair_minsum<int32_t, true, false><<<static_cast<unsigned>(n_ctas), K2_THREADS, 0, ctx->stream>>>(prm);
        ev_end(ctx, 1);
        ++ctx->launches;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(S, prm.S, bytes, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    dev_free(ctx, prm.S);
    if (e != cudaSuccess) return fail(ctx, SP_ERR_CUDA, std::string("K2 full: ") + cudaGetErrorString(e));
    return SP_OK;
}

// host rows [R][A] int32 -> temporary device matrix
static sp_status upload_rows(sp_ctx *ctx, const int32_t *D, int64_t R, int64_t A, sp_dmatrix **out) {
    if (!D || R < 0 || A < 0) return fail(ctx, SP_ERR_INVALID, "K2 host: bad argument");
    if (R > 0x7FFFFFF0ll || A > 0x7FFFFFF0ll) return fail(ctx, SP_ERR_RANGE, "K2 host: matrix too large");
    // K2 adds the minima of 32 reads in a 32-bit partial sum before widening: 32 x 2^27 = 2^32.  Distances (at most the pattern
    // length) and chain-window scores are far below that; anything else is a caller error, reported instead of wrapped around
    for (int64_t i = 0; i < R * A; ++i)
        if (static_cast<uint32_t>(D[i]) >= (1u << 27))
            return fail(ctx, SP_ERR_RANGE, "K2 host: matrix values must lie in [0, 2^27)");
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    sp_dmatrix *d = new (std::nothrow) sp_dmatrix();
    if (!d) return fail(ctx, SP_ERR_NOMEM, "out of host memory");
    d->ctx = ctx; d->nt = R; d->np = A; d->ld = (R + 63) / 64 * 64; d->elem_bits = 32;
    int32_t *rows = nullptr;
    const size_t n = static_cast<size_t>(std::max<int64_t>(R * A, 1));
    cudaError_t e = dev_malloc(ctx, &d->d, static_cast<size_t>(std::max<int64_t>(A * d->ld, 1)) * 4);
    if (e == cudaSuccess) e = dev_malloc(ctx, reinterpret_cast<void **>(&rows), n * 4);
    if (e == cudaSuccess) e = cudaMemsetAsync(d->d, 0, static_cast<size_t>(std::max<int64_t>(A * d->ld, 1)) * 4, ctx->stream);
    if (e == cudaSuccess && R * A > 0) {
        e = cudaMemcpyAsync(rows, D, static_cast<size_t>(R * A) * 4, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) {
            const dim3 grid(static_cast<unsigned>((A + 31) / 32), static_cast<unsigned>((R + 31) / 32)), blk(32, 8);
            rows_to_dmatrix<<<grid, blk, 0, ctx->stream>>>(rows, static_cast<int>(R), static_cast<int>(A), d->ld,
                                                           static_cast<int32_t *>(d->d));
            ++ctx->launches;
            e = cudaGetLastError();
        }
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    dev_free(ctx, rows);
    if (e != cudaSuccess) { sp_dmatrix_destroy(d); return fail(ctx, SP_ERR_CUDA, std::string("K2 host upload: ") + cudaGetErrorString(e)); }
    *out = d;
    return SP_OK;
}

extern "C" sp_status sp_pair_minsum_topk_host(sp_ctx *ctx, const int32_t *D, const int32_t *D2, int64_t R, int64_t A,
                                              int k, sp_pair_rec *out, int *n_out) {
    if (!ctx) return SP_ERR_INVALID;
    sp_dmatrix *d = nullptr, *d2 = nullptr;
    sp_status st = upload_rows(ctx, D, R, A, &d);
    if (st == SP_OK && D2) st = upload_rows(ctx, D2, R, A, &d2);
    if (st == SP_OK) st = sp_pair_minsum_topk(ctx, d, d2, 0, A, k, out, n_out);
    sp_dmatrix_destroy(d); sp_dmatrix_destroy(d2);
    return st;
}

extern "C" sp_status sp_pair_minsum_full_host(sp_ctx *ctx, const int32_t *D, int64_t R, int64_t A, uint64_t *S) {
    if (!ctx) return SP_ERR_INVALID;
    sp_dmatrix *d = nullptr;
    sp_status st = upload_rows(ctx, D, R, A, &d);
    if (st == SP_OK) st = sp_pair_minsum_full(ctx, d, S);
    sp_dmatrix_destroy(d);
    return st;
}

// ------------------------------------------------------------------------------------------
// integer pipe peak
// ------------------------------------------------------------------------------------------
extern "C" sp_status sp_int_peak(sp_ctx *ctx, int kind, double *ops_per_s) {
    if (!ctx) return SP_ERR_INVALID;
    if (!ops_per_s || kind < 0 || kind > 5) return fail(ctx, SP_ERR_INVALID, "sp_int_peak: bad argument");
    SP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int grid = ctx->num_sms * 8, iters = 8192;
    uint32_t *d_out = nullptr;
    SP_CUDA(ctx, dev_malloc(ctx, reinterpret_cast<void **>(&d_out), static_cast<size_t>(grid) * 256 * 4));
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    float best_ms = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
        cudaEventRecord(a, ctx->stream);
        switch (kind) {
            case 0: int_peak_kernel<0><<<grid, 256, 0, ctx->stream>>>(d_out, iters); break;
            case 1: int_peak_kernel<1><<<grid, 256, 0, ctx->stream>>>(d_out, iters); break;
            case 2: int_peak_kernel<2><<<grid, 256, 0, ctx->stream>>>(d_out, iters); break;
            case 3: int_peak_kernel<3><<<grid, 256, 0, ctx->stream>>>(d_out, iters); break;
            case 4: int_peak_kernel<4><<<grid, 256, 0, ctx->stream>>>(d_out, iters); break;
            default: int_peak_kernel<5><<<grid, 256, 0, ctx->stream>>>(d_out, iters); break;
        }
        cudaEventRecord(b, ctx->stream);
        ++ctx->launches;
        cudaEventSynchronize(b);
        float ms = 0;
        cudaEventElapsedTime(&ms, a, b);
        if (rep > 0) best_ms = std::min(best_ms, ms);
    }
    cudaEventDestroy(a); cudaEventDestroy(b);
    cudaError_t e = cudaGetLastError();
    dev_free(ctx, d_out);
    if (e != cudaSuccess) return fail(ctx, SP_ERR_CUDA, std::string("sp_int_peak: ") + cudaGetErrorString(e));
    const double ops = static_cast<double>(grid) * 256.0 * iters * 64.0;
    *ops_per_s = ops / (best_ms * 1e-3);
    return SP_OK;
}
