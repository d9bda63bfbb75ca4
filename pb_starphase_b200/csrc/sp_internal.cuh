// sp_internal.cuh -- handles and helpers shared by the translation units of libstarphase_gpu.so
// (starphase_gpu.cu: context, K1/K2/K3/K5/K6; sp_align.cu: K4; sp_affine.cu: K9; sp_comm.cu: multi-GPU).  Not part of the ABI.
#pragma once
#include "../../include/starphase_gpu.h"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <new>
#include <string>
#include <vector>

#include <cuda_runtime.h>

// ------------------------------------------------------------------------------------------
// handles
// ------------------------------------------------------------------------------------------
struct sp_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int num_sms = 0;
    int smem_optin = 0;
    std::string err;
    cudaEvent_t ev[5][2] = {};
    bool ev_valid[5] = {false, false, false, false, false};
    uint64_t launches = 0;
    // grow-only device buffers reused across calls (cudaMalloc / cudaFree of large blocks cost up to a second each):
    // pool 0 = staging (transposed result rows, K5 lists, K4 traceback scratch), 1 = K4 CIGAR regions, 2 = K4 blobs, 3 = K4 dense CIGAR
    void *pool[4] = {nullptr, nullptr, nullptr, nullptr};
    size_t pool_bytes[4] = {0, 0, 0, 0};
    int *d_counter = nullptr;  // K1's work counter
    cudaMemPool_t mempool = nullptr;  // private stream-ordered pool (release threshold lifted on it, not on the device's default pool)
    // grow-only page-locked staging for the small per-call tables (plan tables of K4): pageable H2D copies are staged by the
    // driver one by one and cost more than the kernels they feed
    void *h_stage = nullptr;
    size_t h_stage_bytes = 0;
    size_t free_mem_cached = 0;  // cudaMemGetInfo is slow (~1 ms): asked once per context, refreshed when a pool has to grow
    // side streams for kernels that are independent of each other inside one call (K9's band classes): forked from and joined
    // back into `stream` with events, created on first use
    cudaStream_t aux[3] = {nullptr, nullptr, nullptr};
    cudaEvent_t aux_fork = nullptr, aux_join[3] = {nullptr, nullptr, nullptr};
    // sp_ctx_share_device: several contexts drive this GPU from concurrent host threads.  Long K1 launches then go to `bulk`, a
    // stream of the lowest priority, one CTA per work item, forked from / joined into `stream` (created at the highest priority)
    bool share_device = false;
    cudaStream_t bulk = nullptr;
    cudaEvent_t bulk_fork = nullptr, bulk_join = nullptr;
};

static inline cudaError_t ctx_bulk(sp_ctx *ctx) {
    if (ctx->bulk) return cudaSuccess;
    int lo = 0, hi = 0;  // numerically: lo = least priority, hi = greatest
    cudaError_t e = cudaDeviceGetStreamPriorityRange(&lo, &hi);
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&ctx->bulk, cudaStreamNonBlocking, lo);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->bulk_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->bulk_join, cudaEventDisableTiming);
    return e;
}

static inline cudaError_t ctx_aux(sp_ctx *ctx) {
    if (ctx->aux_fork) return cudaSuccess;
    cudaError_t e = cudaSuccess;
    for (int i = 0; i < 3 && e == cudaSuccess; ++i) {
        e = cudaStreamCreateWithFlags(&ctx->aux[i], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->aux_join[i], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->aux_fork, cudaEventDisableTiming);
    return e;
}

static inline cudaError_t ctx_stage(sp_ctx *ctx, size_t bytes, void **out) {
    if (bytes > ctx->h_stage_bytes) {
        cudaStreamSynchronize(ctx->stream);
        cudaFreeHost(ctx->h_stage);
        ctx->h_stage = nullptr; ctx->h_stage_bytes = 0;
        const size_t want = bytes + bytes / 2;
        cudaError_t e = cudaHostAlloc(&ctx->h_stage, want, cudaHostAllocDefault);
        if (e != cudaSuccess) return e;
        ctx->h_stage_bytes = want;
    }
    *out = ctx->h_stage;
    return cudaSuccess;
}

// stream-ordered reuse is safe: every user synchronises the context stream before it returns
static inline cudaError_t ctx_pool(sp_ctx *ctx, int which, size_t bytes, void **out) {
    if (bytes > ctx->pool_bytes[which]) {
        cudaStreamSynchronize(ctx->stream);
        cudaFree(ctx->pool[which]);
        ctx->pool[which] = nullptr; ctx->pool_bytes[which] = 0;
        const size_t want = bytes + bytes / 4;  // head-room: sizes creep up from call to call
        cudaError_t e = cudaMalloc(&ctx->pool[which], want);
        if (e != cudaSuccess) {
            cudaGetLastError();
            e = cudaMalloc(&ctx->pool[which], bytes);
            if (e != cudaSuccess) return e;
            ctx->pool_bytes[which] = bytes;
        } else {
            ctx->pool_bytes[which] = want;
        }
    }
    *out = ctx->pool[which];
    return cudaSuccess;
}
static inline cudaError_t ctx_scratch(sp_ctx *ctx, size_t bytes, void **out) { return ctx_pool(ctx, 0, bytes, out); }

// Every other device buffer is stream-ordered (cudaMallocFromPoolAsync / cudaFreeAsync on the context stream, from a memory
// pool the context owns, its release threshold lifted in sp_ctx_create): plain cudaFree synchronises the device and was
// measured at up to 450 ms per call next to multi-GB allocations.
template <typename T>
static inline cudaError_t dev_malloc(sp_ctx *ctx, T **p, size_t bytes) {
    // the context's own pool when it could be created (freed blocks stay with this library and nobody else's pool is touched)
    if (ctx->mempool) return cudaMallocFromPoolAsync(reinterpret_cast<void **>(p), bytes, ctx->mempool, ctx->stream);
    return cudaMallocAsync(reinterpret_cast<void **>(p), bytes, ctx->stream);
}
static inline void dev_free(sp_ctx *ctx, void *p) {
    if (p) cudaFreeAsync(p, ctx->stream);
}

extern thread_local std::string g_create_err;  // starphase_gpu.cu

// One lane-width class of a pattern set: every warp of the class holds 32 lanes x U words x 32 rows.
struct PatClass {
    int U = 0;
    int n_bins = 0;    // warps incl. the fillers that pad the last group
    int n_groups = 0;  // CTAs' worth of warps (K1_WARPS each)
    uint32_t *d_blobs = nullptr;
};

struct sp_patterns {
    sp_ctx *ctx = nullptr;
    int64_t n = 0, total_len = 0, padded_rows = 0;
    sp_mode mode = SP_INFIX;
    std::vector<PatClass> classes;
};

struct TextPack {
    int tc = 0;  // tile capacity in chunks
    int n_tiles = 0;
    int64_t total_chunks = 0;
    uint2 *d_text = nullptr;
    int32_t *d_tile_off = nullptr;
    int32_t *d_tile_text0 = nullptr;
};

struct sp_targets {
    sp_ctx *ctx = nullptr;
    int64_t n = 0, total_len = 0;
    uint8_t *d_bases = nullptr;
    long long *d_offs = nullptr;
    std::vector<int64_t> h_offs;  // host copy of the rebased offsets (n + 1 entries, h_offs[0] == 0): K4 plans from the lengths
    std::vector<int32_t> nch;  // chunks per text
    int32_t max_nch = 0;
    int64_t sum_nch = 0;
    std::map<int, TextPack> packs;
};

struct sp_dmatrix {
    sp_ctx *ctx = nullptr;
    void *d = nullptr;
    int32_t *d_end = nullptr;
    int64_t nt = 0, np = 0, ld = 0;
    int elem_bits = 32;
    bool owned = true;
};

// ------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------
static inline sp_status fail(sp_ctx *ctx, sp_status st, const std::string &msg) {
    if (ctx) ctx->err = msg;
    else g_create_err = msg;
    return st;
}
#define SP_CUDA(ctx, call)                                                                         \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return fail(ctx, SP_ERR_CUDA,                                                          \
                        std::string(#call) + ": " + cudaGetErrorString(e__) + " (" __FILE__ ":" +   \
                            std::to_string(__LINE__) + ")");                                       \
    } while (0)

static inline void ev_begin(sp_ctx *ctx, int which) { cudaEventRecord(ctx->ev[which][0], ctx->stream); }
static inline void ev_end(sp_ctx *ctx, int which) {
    cudaEventRecord(ctx->ev[which][1], ctx->stream);
    ctx->ev_valid[which] = true;
}

// SP_TIMING=1: wall-clock phases of the host side to stderr (diagnostic only)
struct PhaseTimer {
    bool on;
    std::chrono::steady_clock::time_point t0;
    explicit PhaseTimer() : on(getenv("SP_TIMING") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void mark(const char *what) {
        if (!on) return;
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[sp_timing] %-28s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

// a failed CUDA call inside entry point `fn` as a status: SP_ERR_NOMEM for an allocation failure, SP_ERR_CUDA otherwise
static inline sp_status cuda_status(sp_ctx *ctx, const char *fn, cudaError_t e, const char *what) {
    if (e == cudaSuccess) return SP_OK;
    return fail(ctx, e == cudaErrorMemoryAllocation ? SP_ERR_NOMEM : SP_ERR_CUDA, std::string(fn) + ": " + what + ": " + cudaGetErrorString(e));
}

// defined in starphase_gpu.cu
sp_status check_seqset(sp_ctx *ctx, const sp_seqset *s, const char *what);
sp_status upload_seqset(sp_ctx *ctx, const sp_seqset *s, uint8_t **d_bases, long long **d_offs);
// launches pack_patterns (sp_kernels.cuh) on the context stream: blobs of n_bins warps of lane width U
sp_status sp_internal_pack_blobs(sp_ctx *ctx, const uint8_t *d_bases, const long long *d_offs, const int32_t *d_lane_pat,
                                 const int32_t *d_lane_row0, const uint32_t *d_lane_info1, uint32_t *d_blobs, int n_bins, int U,
                                 int prefix_mode, int reverse);

// Lane layout of pattern blobs (what pack_patterns and the K1 / K3 / K4 kernels read): bin b, lane l is entry b * 32 + l of
// each table.  A pattern of m rows over nl lanes of width U fills them bottom-aligned: lane li holds rows from
// li * 32 * U - pad on (pad = nl * 32 * U - m leading wildcard rows) and info1 = m | INFO_FIRST (li == 0) | INFO_LAST
// (li == nl - 1).  An unused lane holds no pattern.
struct LaneTables {
    std::vector<int32_t> pat, row0;
    std::vector<uint32_t> info1;
    void resize(int n_bins);  // new lanes are unused
    void place(int bin, int lane0, int nl, int32_t p, int64_t m, int U);
};
// Best-fit decreasing: items of lanes[k] lanes (1..32), taken in the caller's order, each go to the fullest 32-lane bin that
// still has room (a new bin if none has).  Fills slots[k] = (bin, first lane) when slots is given; returns the bin count.
struct LaneSlot { int bin, lane0; };
int sp_internal_pack_lanes(const std::vector<int> &lanes, std::vector<LaneSlot> *slots);

// defined in sp_align.cu: the pair-call contract of K4 (sp_align_resident / sp_align_windows) and K9
// (sp_align_affine_resident), include/starphase_gpu.h
namespace sp { struct AlignRecDev; }
// the arguments both entry points take; sets *cigar_used = 0 once they pass
sp_status pair_call_check(sp_ctx *ctx, const char *fn, const void *texts, const void *patterns, int64_t n_pairs, const int32_t *pair_text,
                          const int32_t *pair_pattern, const int32_t *win_begin, const int32_t *win_end, const sp_align_rec *recs,
                          const uint32_t *cigar, int64_t cigar_cap, int64_t *cigar_used);
// pair q: first text byte in the text set's device buffer, text (window) length, pattern length
sp_status pair_resolve(sp_ctx *ctx, const char *fn, const sp_targets *texts, const sp_targets *patterns, int64_t q, const int32_t *pair_text,
                       const int32_t *pair_pattern, const int32_t *win_begin, const int32_t *win_end, int64_t &t_off, int64_t &n, int64_t &m);
// The device buffers of one call, freed (stream-ordered) with it.
struct PairCall {
    sp_ctx *ctx;
    const char *fn;
    uint32_t *cigar = nullptr;           // the pairs' CIGAR regions, written backwards (pool 1)
    uint32_t *dense = nullptr;           // the dense CIGAR pool handed to the caller (pool 3)
    sp::AlignRecDev *recs = nullptr;     // zeroed: a pair no kernel visits reads back as the empty placement
    int32_t *scores = nullptr;           // K9 only
    unsigned long long *used = nullptr;  // [0] = dense pool fill, then the kernels' work counters (zeroed)
    PairCall(sp_ctx *c, const char *f) : ctx(c), fn(f) {}
    ~PairCall();
    sp_status alloc(int64_t n_pairs, int64_t cig_total, int64_t cigar_cap, bool with_scores, int n_used);
    // Reads the call back after its launches: records (and scores) and the pool fill, *cigar_used; SP_ERR_RANGE past
    // cigar_cap without touching recs / scores / cigar, else the pool, then the records and scores.
    sp_status finish(int64_t n_pairs, sp_align_rec *recs, int32_t *scores, uint32_t *cigar, int64_t cigar_cap, int64_t *cigar_used,
                     PhaseTimer &tm);
};
// adopts device-resident bases / offsets as a text set (sp_comm.cu: read sets received by broadcast)
sp_status sp_internal_targets_adopt(sp_ctx *ctx, uint8_t *d_bases, long long *d_offs, const int64_t *host_offsets, int64_t n,
                                    sp_targets **out);
