// sp_consensus.cuh -- K7: batched extension of growing consensus sequences against a read set (row N1 of SURVEY.md 8f).
//
// The reference builds its HLA / CYP2D6 consensuses with waffle_con's dynamic-WFA search (src/hla/caller.rs:1097-1219,
// :727-755; src/cyp2d6/caller.rs:145-280): candidate consensus prefixes are extended one symbol at a time and every read keeps
// its edit distance to the growing prefix; reads vote for the next symbol with the bases that follow their best-scoring
// prefixes.  The data-parallel part of that search is "extend candidate X by symbol s for every read", and that is this
// kernel: one warp per (task, read).  A track holds, for every read, the last DP column of
//     E[i] = edit distance between the consensus so far and the read prefix r[0, i)
// restricted to a band of 2W + 1 rows around the read's nominal diagonal i = L - offset (HiFi reads drift by a few indels; the
// window of uncertainty of the offset widens the band).  Appending symbol s turns column L into column L + 1:
//     E'[i] = min(E[i-1] + (r[i-1] != s),  E[i] + 1,  E'[i-1] + 1)
// In band coordinates (k = i - (L - offset) + W) the diagonal neighbour keeps its k, the horizontal one is k + 1, and the
// vertical dependency is a min-plus prefix scan over k (per lane sequentially, across lanes with five shuffles).
// Row 0 (no read base used yet) costs max(0, L - (offset + window / 2)): the read may start anywhere inside its offset window
// for free.  A read becomes active at L = max(0, offset - window / 2); before that it has no cost and no vote.
// Per (task, read) the kernel reports ed = min_i E'[i] (end-free in the read: it continues), the set of next read bases at
// the rows reaching that minimum (the read's vote), whether the read is consumed at such a row, and the running minimum of
// E'[|r|] over all columns so far (the read's final cost once the consensus has passed its end).
//
// Integer DP on the INT32 pipe; the work per step is tiny (reads x band cells), so the kernel is written for batches: many
// tasks -- candidate extensions of many consensus problems -- per launch.
#pragma once
#include <cstdint>
#include <cooperative_groups.h>
#include <cuda_runtime.h>

namespace sp {

constexpr int CONS_INF = 0x3FFFFFFF;
constexpr uint8_t VOTE_FINISHED = 1u << 5;  // the read is consumed at a row reaching the minimum
constexpr uint8_t VOTE_INACTIVE = 1u << 6;  // the consensus has not reached the read's window yet
constexpr uint32_t CODE_WILDCARD = 5;       // read byte '*': matches every consensus symbol at no cost, votes for none

// one extension task: the read set and tracks of its handle, and where its rows go
struct K7Task {
    const uint8_t *codes;      // read bases as codes 0..3 (ACGT), 4 = other (matches nothing), 5 = wildcard '*'; concatenated
    const long long *roffs;    // [n_reads + 1]
    const int32_t *offset;     // [n_reads] nominal start of the read inside the consensus; < 0 = exactly at its start, no window
    int32_t *band;             // [n_tracks][n_reads][band_cells] last column, band coordinates
    int32_t *best_full;        // [n_tracks][n_reads] min over columns so far of E[|r|]
    int32_t *track_len;        // [n_tracks] consensus length of the track
    long long warp0;           // first warp of the task (its read r is warp warp0 + r) = first output row
    int n_reads, W, half_window, src, dst;
    uint32_t sym;              // code of the appended symbol (0..4), 255 = report only
};

struct ConsParams {
    const K7Task *tasks;       // [n_tasks], ascending warp0
    int32_t *out_ed;           // [n_warps]
    uint8_t *out_votes;        // [n_warps]
    int32_t *out_full;         // [n_warps]
    int n_tasks;
    long long n_warps;
};

// Column L0 of a read at band index k: CONS_INF outside the band / the read; the activating column (L0 == start) is E[i] = i by
// definition -- read bases before the window start are unaligned -- and is synthesised instead of stored, so a fresh track needs
// no initial columns.  stored(c, ln): the kept value of band cell ln * CELLS + c (= k), asked only for cells of the band when
// L0 > start; the caller names the cell by owner lane and slot so that the address needs no division.
template <typename Stored>
__device__ __forceinline__ int k7_old_at(int k, int c, int ln, int nb, int W, int L0, int off, int start, int m, Stored stored) {
    if (k < 0 || k >= nb) return CONS_INF;
    const int i_old = (L0 - off) + (k - W);
    if (i_old < 0 || i_old > m) return CONS_INF;
    return L0 == start ? i_old : stored(c, ln);
}

// Column L = L0 + 1 (>= start) of one read after appending symbol code s: e[c] = band cell lane * CELLS + c.
// base(x): code of read base x (0 <= x < m).
template <int CELLS, typename Base, typename Stored>
__device__ __forceinline__ void k7_next_column(int (&e)[CELLS], int lane, int W, int nb, int L0, int off, int hw, int start, int m,
                                               Base base, uint32_t s, Stored stored) {
    const int L = L0 + 1, k0 = lane * CELLS, ibase = (L - off) - W;
    if (L == start) {  // this step reaches the read's window: the activating column
#pragma unroll
        for (int c = 0; c < CELLS; ++c) {
            const int k = k0 + c, i = ibase + k;
            e[c] = (k < nb && i >= 0 && i <= m) ? i : CONS_INF;
        }
        return;
    }
    // base[k] = min(diagonal, horizontal); then the vertical min-plus scan
    const int row0_cost = max(0, L - (off + hw));  // E'[0]: the read may start anywhere inside its window for free
#pragma unroll
    for (int c = 0; c < CELLS; ++c) {
        const int k = k0 + c, i = ibase + k;
        int v = CONS_INF;
        if (k < nb && i >= 0 && i <= m) {
            if (i == 0) {
                v = row0_cost;
            } else {
                const int diag = k7_old_at(k, c, lane, nb, W, L0, off, start, m, stored);  // E[i-1] of column L0 has the same band index
                const int horiz = c + 1 < CELLS ? k7_old_at(k + 1, c + 1, lane, nb, W, L0, off, start, m, stored)
                                                : k7_old_at(k + 1, 0, lane + 1, nb, W, L0, off, start, m, stored);  // E[i] of column L0
                const uint32_t rb = base(i - 1);
                const int sub = (s < 4u && (rb == s || rb == CODE_WILDCARD)) ? 0 : 1;
                v = min(diag < CONS_INF ? diag + sub : CONS_INF, horiz < CONS_INF ? horiz + 1 : CONS_INF);
            }
        }
        e[c] = v;
    }
    // x[k] = e[k] - k; inclusive prefix min over k; e[k] = prefmin + k
    int run = CONS_INF;
#pragma unroll
    for (int c = 0; c < CELLS; ++c) {
        const int x = e[c] < CONS_INF ? e[c] - (k0 + c) : CONS_INF;
        run = min(run, x);
        e[c] = run;  // lane-local prefix min of x for now
    }
    int carry = run;  // lane total, then inclusive scan across lanes
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int up = __shfl_up_sync(0xffffffffu, carry, d);
        if (lane >= d) carry = min(carry, up);
    }
    int prev = __shfl_up_sync(0xffffffffu, carry, 1);  // prefix min of all lower lanes
    if (lane == 0) prev = CONS_INF;
#pragma unroll
    for (int c = 0; c < CELLS; ++c) {
        const int k = k0 + c, i = ibase + k;
        const int x = min(e[c], prev);
        e[c] = (k < nb && i >= 0 && i <= m && x < CONS_INF) ? x + k : CONS_INF;
    }
}

// What a column reports: its minimum, the next read bases at the rows reaching it (+ VOTE_FINISHED when the read is consumed
// there), and E[|r|].
template <int CELLS, typename Base>
__device__ __forceinline__ void k7_reduce_column(const int (&e)[CELLS], int lane, int nb, int ibase, int m, Base base, int &mn, int &full,
                                                 uint32_t &votes) {
    const int k0 = lane * CELLS;
    mn = CONS_INF; full = CONS_INF;
#pragma unroll
    for (int c = 0; c < CELLS; ++c) {
        const int k = k0 + c, i = ibase + k;
        mn = min(mn, e[c]);
        if (k < nb && i == m) full = e[c];
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, d));
        full = min(full, __shfl_xor_sync(0xffffffffu, full, d));
    }
    votes = 0;
#pragma unroll
    for (int c = 0; c < CELLS; ++c) {
        const int k = k0 + c, i = ibase + k;
        if (k < nb && e[c] == mn && mn < CONS_INF && i >= 0 && i <= m) votes |= i == m ? VOTE_FINISHED : ((1u << base(i)) & 31u);  // a wildcard (code 5) names no symbol
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) votes |= __shfl_xor_sync(0xffffffffu, votes, d);
}

// one warp per (task, read), over the tasks of many handles; CELLS * 32 >= 2W + 1 of every task.  A task whose band needs fewer
// cells per lane gives the same result: the cells are numbered k = lane * CELLS + c whatever CELLS is, and the scan runs over k.
template <int CELLS>
__global__ void __launch_bounds__(128) k7_extend(const ConsParams p) {
    const long long warp = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= p.n_warps) return;
    int lo = 0, hi = p.n_tasks - 1;  // the task holding this warp: the last one with warp0 <= warp
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (p.tasks[mid].warp0 <= warp) lo = mid; else hi = mid - 1;
    }
    const K7Task &t = p.tasks[lo];
    const int r = static_cast<int>(warp - t.warp0), W = t.W, n_reads = t.n_reads;
    const int src = t.src, dst = t.dst;
    const uint32_t s = t.sym;
    const bool extend = s != 255u;
    const int nb = 2 * W + 1;
    const int L0 = t.track_len[src];        // consensus length before the step
    const int L = L0 + (extend ? 1 : 0);    // after
    const int off_raw = t.offset[r];             // < 0: the read starts exactly at the consensus start (add_sequence without offset)
    const int off = max(off_raw, 0);
    const int hw = off_raw < 0 ? 0 : t.half_window;
    const int m = static_cast<int>(t.roffs[r + 1] - t.roffs[r]);
    const uint8_t *R = t.codes + t.roffs[r];
    const int32_t *old = t.band + (static_cast<size_t>(src) * n_reads + r) * nb;
    int32_t *nw = t.band + (static_cast<size_t>(dst) * n_reads + r) * nb;
    const size_t o = static_cast<size_t>(warp);
    const int start = max(0, off - hw);  // first column at which the read is active
    int32_t *best_full = t.best_full;
    int bf = best_full[static_cast<size_t>(src) * n_reads + r];

    if (L < start) {  // not active yet: the state stays "column `start` not reached"
        if (lane == 0) {
            p.out_ed[o] = 0; p.out_votes[o] = VOTE_INACTIVE; p.out_full[o] = CONS_INF;
            best_full[static_cast<size_t>(dst) * n_reads + r] = CONS_INF;
        }
        return;
    }
    int e[CELLS];
    const int k0 = lane * CELLS;
    const int ibase = (L - off) - W;  // row index of band cell k at column L:  i = ibase + k
    // column L0 of the parent track as stored (asked only for 0 <= k < nb when L0 > start)
    auto stored = [&](int c, int ln) -> int { return old[ln * CELLS + c]; };
    auto base = [&](int x) -> uint32_t { return R[x]; };
    if (!extend) {  // report the state of column L0 (>= start here)
#pragma unroll
        for (int c = 0; c < CELLS; ++c) e[c] = k7_old_at(k0 + c, c, lane, nb, W, L0, off, start, m, stored);
    } else {
        k7_next_column<CELLS>(e, lane, W, nb, L0, off, hw, start, m, base, s, stored);
    }
    // store the column, reduce: minimum, votes at the minimum, distance with the read consumed
#pragma unroll
    for (int c = 0; c < CELLS; ++c)
        if (k0 + c < nb) nw[k0 + c] = e[c];
    int mn, full;
    uint32_t votes;
    k7_reduce_column<CELLS>(e, lane, nb, ibase, m, base, mn, full, votes);
    bf = min(bf, full);
    if (lane == 0) {
        p.out_ed[o] = mn; p.out_votes[o] = static_cast<uint8_t>(votes); p.out_full[o] = bf;
        best_full[static_cast<size_t>(dst) * n_reads + r] = bf;
    }
}

// fresh tracks: empty consensus, no read consumed yet
__global__ void k7_reset(int32_t *best_full, int32_t *track_len, int track, int n_reads) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n_reads) best_full[static_cast<size_t>(track) * n_reads + r] = CONS_INF;
    if (r == 0) track_len[track] = 0;
}

// sets track_len[dst] = track_len[src] + 1 (or keeps it for report-only tasks) after the extension kernel has read the old lengths
__global__ void k7_bump_lengths(const ConsParams p) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= p.n_tasks) return;
    const K7Task &t = p.tasks[q];
    t.track_len[t.dst] = t.track_len[t.src] + (t.sym != 255u ? 1 : 0);
}

// ---------------------------------------------------------------------------------------------------------------
// K7 in a loop on the device.  The host search spends most of its steps on stretches where the reads agree: the node it pops has
// exactly one symbol with the votes, gets one child, and that child is popped next.  Each such step is a launch, two copies and
// a synchronisation (~25 us) for ~1 us of arithmetic.  k7_run takes a node -- one consensus or a dual pair -- and keeps extending
// it while that is what the host would do: one passing symbol per side (the host's vote rule, below), the child ahead of the
// best competitor in the host's queue (cheaper, or as cheap and longer), fewer than max_steps steps.  It returns the last child with its per-read state and
// the symbols it appended.
//
// One thread-block cluster per node (job): the grid holds one cluster per job of a batch, job = cluster index, and clusters do not
// wait on each other, so the grid may hold more of them than fit on the GPU at once.  A cluster larger than its job needs gives
// the same result: the items are only dealt over more warps.  An item = (read, side), one warp per item at a time, items dealt
// round-robin over the warps of the cluster.  The DP columns stay in shared memory (u16, cell-major: conflict-free) for the whole run; the per-read results
// (ed, votes, full) are replicated in every CTA through distributed shared memory, so every CTA takes the decision of a step
// for itself from its own copy: one cluster barrier + one CTA barrier per step.  The result arrays are double-buffered by step
// parity (a fast CTA may write step n + 1's results while a slow one still reads step n's).
//
// Vote rule (pb_starphase_b200/host/sp_host_consensus.cpp: tally / passing): a read votes when it is active and not already
// consumed at a better column (full >= ed), with 12 units split evenly over its candidate symbols (votes & 15); in a dual node a
// read counts towards, and votes for, the side(s) it is closest to (cost = inactive ? 0 : min(ed, full)); a symbol passes with
// >= 12 min_count units and a min_af share of the side's units; when none passes, the first best-voted one does; a side with
// no units at all is finished.
// ---------------------------------------------------------------------------------------------------------------
struct ConsRunParams {
    const uint8_t *codes;
    const long long *roffs;
    const int32_t *offset;
    int32_t *band, *best_full, *track_len;
    int n_reads, W, half_window, n_sides;
    int src[2], dst[2];
    int32_t *ed;       // [n_sides][n_reads]  in: the start node, out: the node returned
    uint8_t *votes;
    int32_t *full;
    int min_units;     // 12 * min_count
    int permille;      // min_af * 1000
    long long cost_limit, size_limit, cost_cap;  // go on while (cost, size) orders before the limit (cheaper, or as cheap and longer) and cost <= cap
    int max_steps;
    // one byte per round: low nibble = code appended to side 0, high nibble = side 1; 15 = side not extended
    uint8_t *log_head;  // rounds [0, 256)
    uint8_t *log_rest;  // rounds [256, max_steps)
    int *n_steps;
};

constexpr int K7_RUN_THREADS = 512;

// per item (read, side) in shared memory: what a step needs about its read, so that the loop never loads from global memory
// (cluster.sync invalidates L1: every global load inside the loop would be an L2 round trip on the critical path)
struct K7Item {
    long long roff;  // first code of the read
    int32_t off_raw, m;
    int32_t filled;  // read bases [.., filled) are in the item's code ring
    int32_t side;
};

// one block per SM stated outright: without it ptxas held k7_run<16> to 64 registers and spilled
template <int CELLS>
__global__ void __launch_bounds__(K7_RUN_THREADS, 1) k7_run(const ConsRunParams *jobs) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int n_cta = static_cast<int>(cluster.num_blocks()), cta = static_cast<int>(cluster.block_rank());
    // the job's parameters, read once into shared memory: kernel parameters live in the constant bank, a global array would be
    // reloaded through the L1 that every cluster.sync invalidates, and registers are spent (121 at CELLS = 16)
    __shared__ ConsRunParams p;
    if (threadIdx.x == 0) p = jobs[blockIdx.x / n_cta];
    __syncthreads();
    const int R = p.n_reads, NS = p.n_sides, items = R * NS, nb = 2 * p.W + 1;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = K7_RUN_THREADS / 32;
    const int gwarp = cta * nwarps + warp, total_warps = n_cta * nwarps;
    const int my_items = (items - gwarp + total_warps - 1) / total_warps;  // items gwarp, gwarp + total_warps, ...
    constexpr int COLW = CELLS * 32, RING = 2 * COLW;  // band cells per item (padded); code ring: the band's rows + a refill of 32
    extern __shared__ __align__(16) uint8_t smem[];
    // state[parity][items]: ed, full (i32), votes (u8); then this CTA's items: slot = warp * per_warp + j
    const int per_warp = (items + total_warps - 1) / total_warps, slots = nwarps * per_warp;
    K7Item *s_item = reinterpret_cast<K7Item *>(smem);                          // [slots]
    int32_t *s_ed = reinterpret_cast<int32_t *>(s_item + slots);                // [2][items]
    int32_t *s_full = s_ed + 2 * items;                                         // [2][items]
    uint16_t *col = reinterpret_cast<uint16_t *>(s_full + 2 * items);           // [slots][COLW] columns, cell-major
    uint8_t *ring = reinterpret_cast<uint8_t *>(col + static_cast<size_t>(slots) * COLW);  // [slots][RING] read codes
    uint8_t *s_votes = ring + static_cast<size_t>(slots) * RING;                // [2][items]
    __shared__ int s_dec[3];  // symbol of side 0 / 1 (-1: none), go
    __shared__ uint8_t s_log[256];  // the last <= 256 log bytes (CTA 0), written out in blocks: no global store inside a step

    for (int i = threadIdx.x; i < items; i += K7_RUN_THREADS) { s_ed[i] = p.ed[i]; s_full[i] = p.full[i]; s_votes[i] = p.votes[i]; }
    // scalars, not arrays: a run-time index puts them (and the parameter arrays) into local memory, and cluster.sync invalidates the
    // L1 that serves it
    int len0 = p.track_len[p.src[0]], len1 = NS == 2 ? p.track_len[p.src[1]] : 0;
    // this warp's items: metadata, and the columns from the source tracks (reads the consensus has not reached keep no column)
    for (int j = 0; j < my_items; ++j) {
        const int it = gwarp + j * total_warps, side = it / R, r = it - side * R, slot = warp * per_warp + j;
        const int off_raw = p.offset[r], off = max(off_raw, 0), hw = off_raw < 0 ? 0 : p.half_window, start = max(0, off - hw);
        if (lane == 0) {
            K7Item m;
            m.roff = p.roffs[r]; m.off_raw = off_raw; m.m = static_cast<int>(p.roffs[r + 1] - p.roffs[r]);
            m.filled = max(0, ((side ? len1 : len0) + 1 - off) - p.W - 1);  // nothing below the first row the next column can touch is ever read
            m.side = side;
            s_item[slot] = m;
        }
        uint16_t *c16 = col + static_cast<size_t>(slot) * COLW;
        const int32_t *old = p.band + (static_cast<size_t>(side ? p.src[1] : p.src[0]) * R + r) * nb;
#pragma unroll
        for (int c = 0; c < CELLS; ++c) {
            const int k = lane * CELLS + c;
            const int v = ((side ? len1 : len0) > start && k < nb) ? old[k] : CONS_INF;
            c16[c * 32 + lane] = static_cast<uint16_t>(min(v, 0xFFFF));
        }
    }
    cluster.sync();  // every CTA of the cluster runs and has its copy of the state before anyone writes into a peer
    int step = 0;
    for (;;) {
        const int cur = step & 1, nxt = cur ^ 1;
        const int32_t *ed = s_ed + cur * items, *fu = s_full + cur * items;
        const uint8_t *vo = s_votes + cur * items;
        if (warp == 0) {  // the decision, from this CTA's copy of the node's state
            int t0[4] = {0, 0, 0, 0}, t1[4] = {0, 0, 0, 0};
            long long cost = 0;
            for (int r = lane; r < R; r += 32) {
                const int c1 = (vo[r] & VOTE_INACTIVE) ? 0 : min(ed[r], fu[r]);
                int c2 = 0x7FFFFFFF;
                if (NS == 2) c2 = (vo[R + r] & VOTE_INACTIVE) ? 0 : min(ed[R + r], fu[R + r]);
                cost += min(c1, c2);
                if (c1 <= c2 && !(vo[r] & VOTE_INACTIVE) && fu[r] >= ed[r]) {  // the read votes on side 0
                    const uint32_t v = vo[r] & 15u;
                    const int w = (0x346C0 >> (4 * __popc(v))) & 15;  // 12 / candidates: 12, 6, 4, 3 (0 for none)
#pragma unroll
                    for (int k = 0; k < 4; ++k) t0[k] += (v >> k & 1u) ? w : 0;
                }
                if (NS == 2 && c2 <= c1 && !(vo[R + r] & VOTE_INACTIVE) && fu[R + r] >= ed[R + r]) {  // ... on side 1
                    const uint32_t v = vo[R + r] & 15u;
                    const int w = (0x346C0 >> (4 * __popc(v))) & 15;
#pragma unroll
                    for (int k = 0; k < 4; ++k) t1[k] += (v >> k & 1u) ? w : 0;
                }
            }
            // sums over the warp with the hardware reduction (costs are below 2^31: <= 2,048 read-sides x 60,000 bases)
            cost = __reduce_add_sync(0xffffffffu, static_cast<int>(cost));
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                t0[k] = __reduce_add_sync(0xffffffffu, t0[k]);
                if (NS == 2) t1[k] = __reduce_add_sync(0xffffffffu, t1[k]);
            }
            if (lane == 0) {
                // one side's verdict: number of passing symbols (1 when only the best-voted one goes on, 0 = finished) and the symbol
                auto verdict = [&](int a, int c, int g, int t, int &n_pass, int &sym) {
                    const int v[4] = {a, c, g, t};
                    const long long total = static_cast<long long>(a) + c + g + t;
                    n_pass = 0; sym = -1;
                    if (total == 0) return;
                    int best = 0, first = -1;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (v[k] >= p.min_units && static_cast<long long>(v[k]) * 1000 >= total * p.permille) {
                            if (n_pass++ == 0) first = k;
                        }
                    }
                    int bv = a;  // first best-voted symbol
                    if (c > bv) { best = 1; bv = c; }
                    if (g > bv) { best = 2; bv = g; }
                    if (t > bv) { best = 3; bv = t; }
                    sym = n_pass ? first : best;
                    n_pass = n_pass ? n_pass : 1;
                };
                int sym[2] = {-1, -1}, n_pass[2] = {0, 0};
                verdict(t0[0], t0[1], t0[2], t0[3], n_pass[0], sym[0]);
                if (NS == 2) verdict(t1[0], t1[1], t1[2], t1[3], n_pass[1], sym[1]);
                const long long size = len0 + (NS == 2 ? len1 : 0);
                const bool one_each = n_pass[0] <= 1 && n_pass[1] <= 1 && n_pass[0] + n_pass[1] >= 1;
                const bool before = cost < p.cost_limit || (cost == p.cost_limit && size > p.size_limit);
                const bool may = step < p.max_steps && (step == 0 || (before && cost <= p.cost_cap));
                s_dec[0] = sym[0]; s_dec[1] = sym[1]; s_dec[2] = (one_each && may) ? 1 : 0;
            }
        }
        __syncthreads();
        if (!s_dec[2]) break;
        const int sym0 = s_dec[0], sym1 = s_dec[1];
        for (int j = 0; j < my_items; ++j) {
            const int it = gwarp + j * total_warps, slot = warp * per_warp + j;
            const K7Item im = s_item[slot];
            __syncwarp();  // every lane has its copy before lane 0 updates `filled` below (racecheck: read here / write there)
            const int side = im.side, s = side ? sym1 : sym0;
            int o_ed = ed[it], o_full = fu[it];
            uint32_t o_votes = vo[it];
            if (s >= 0) {
                const int off = max(im.off_raw, 0), hw = im.off_raw < 0 ? 0 : p.half_window, start = max(0, off - hw);
                const int L0 = side ? len1 : len0, L = L0 + 1, m = im.m;
                if (L < start) {
                    o_ed = 0; o_votes = VOTE_INACTIVE; o_full = CONS_INF;
                } else {
                    const int ibase = (L - off) - p.W;
                    uint8_t *rg = ring + static_cast<size_t>(slot) * RING;
                    // the column touches read bases [ibase - 1, ibase + nb); refill the ring 32 bases at a time (about every 32nd step)
                    int filled = im.filled;
                    const int need = min(m, ibase + nb);
                    if (filled < need) {
                        const uint8_t *codes = p.codes + im.roff;
                        const int upto = min(m, max(need, filled + 32));
                        for (int x = filled + lane; x < upto; x += 32) rg[x & (RING - 1)] = codes[x];
                        filled = upto;
                        if (lane == 0) s_item[slot].filled = filled;
                        __syncwarp();
                    }
                    uint16_t *c16 = col + static_cast<size_t>(slot) * COLW;
                    auto stored = [&](int c, int ln) -> int {
                        const int v = c16[c * 32 + ln];
                        return v == 0xFFFF ? CONS_INF : v;
                    };
                    auto base = [&](int x) -> uint32_t { return rg[x & (RING - 1)]; };
                    int e[CELLS];
                    k7_next_column<CELLS>(e, lane, p.W, nb, L0, off, hw, start, m, base, static_cast<uint32_t>(s), stored);
                    __syncwarp();  // every lane has read its neighbours' cells
#pragma unroll
                    for (int c = 0; c < CELLS; ++c) c16[c * 32 + lane] = static_cast<uint16_t>(min(e[c], 0xFFFF));
                    int mn, full;
                    k7_reduce_column<CELLS>(e, lane, nb, ibase, m, base, mn, full, o_votes);
                    o_ed = mn; o_full = min(o_full, full);
                }
            }
            // the item's state of the next step, into every CTA's copy
            if (lane < n_cta) {
                int32_t *r_ed = cluster.map_shared_rank(s_ed, lane), *r_full = cluster.map_shared_rank(s_full, lane);
                uint8_t *r_votes = cluster.map_shared_rank(s_votes, lane);
                r_ed[nxt * items + it] = o_ed; r_full[nxt * items + it] = o_full; r_votes[nxt * items + it] = static_cast<uint8_t>(o_votes);
            }
        }
        if (cta == 0) {
            if (threadIdx.x == 0) s_log[step & 255] = static_cast<uint8_t>((sym0 < 0 ? 15 : sym0) | ((sym1 < 0 ? 15 : sym1) << 4));
            if ((step & 255) == 255) {  // a full block: out with it
                __syncthreads();
                if (threadIdx.x < 256) (step < 256 ? p.log_head : p.log_rest + (step - 511))[threadIdx.x] = s_log[threadIdx.x];
            }
        }
        if (sym0 >= 0) ++len0;
        if (sym1 >= 0) ++len1;
        ++step;
        cluster.sync();
    }
    // hand the node back: columns into the destination tracks, per-read state, lengths
    const int cur = step & 1;
    for (int j = 0; j < my_items; ++j) {
        const int it = gwarp + j * total_warps, side = it / R, r = it - side * R;
        const uint16_t *c16 = col + static_cast<size_t>(warp * per_warp + j) * COLW;
        const int dtrack = side ? p.dst[1] : p.dst[0];
        int32_t *nw = p.band + (static_cast<size_t>(dtrack) * R + r) * nb;
#pragma unroll
        for (int c = 0; c < CELLS; ++c) {
            const int k = lane * CELLS + c;
            if (k < nb) { const int v = c16[c * 32 + lane]; nw[k] = v == 0xFFFF ? CONS_INF : v; }
        }
        if (lane == 0) p.best_full[static_cast<size_t>(dtrack) * R + r] = s_full[cur * items + it];
    }
    if (cta == 0) {
        for (int i = threadIdx.x; i < items; i += K7_RUN_THREADS) {
            p.ed[i] = s_ed[cur * items + i]; p.full[i] = s_full[cur * items + i]; p.votes[i] = s_votes[cur * items + i];
        }
        if (static_cast<int>(threadIdx.x) < (step & 255))  // the last, partial log block
            (step < 256 ? p.log_head : p.log_rest + ((step & ~255) - 256))[threadIdx.x] = s_log[threadIdx.x];
        if (threadIdx.x == 0) {
            *p.n_steps = step;
            p.track_len[p.dst[0]] = len0;
            if (NS == 2) p.track_len[p.dst[1]] = len1;
        }
    }
    cluster.sync();  // nobody leaves while a peer may still write into its shared memory
}

}  // namespace sp
