// sp_align.cuh -- K4: traceback alignment of selected (text, pattern) pairs (sm_100a only).
//
// Gives the host everything it reads from a minimap2::Mapping at the HLA call sites
// (src/hla/processed_match.rs:53-100 of the reference: query_start / query_end / target_start /
// target_end / nm / EQX cigar), so HlaProcessedMatch::add_mapping, process_mm_cigar (:210-263) and
// is_better_match (:103-184) run unchanged on GPU output, and MappingStats' (seq_len, nm, unmapped)
// split (src/data_types/mapping.rs:7-22) is available for the result JSON.  Row N2 of SURVEY.md §8f.
//
// Round 2 layout.  The forward pass is K1's recurrence (column_step) on pattern-stationary systolic warps, but a warp is
// now a BIN of several pairs, each pair with its own text: pair q owns the consecutive lanes [lane0_q, lane0_q + nl_q) and
// its lanes stream the columns of text q skewed by one 8-column chunk per lane.  The lane width U is picked per pair from
// the pattern length (U = 4 up to 4,096 rows, 8, 12, 16 up to 16,384), so a 3 kb allele keeps 24 of 32 lanes busy at 49
// ALU-pipe instructions per column instead of 6 lanes at 145 (round 1: one pattern per warp at U = 16), and three 1.1 kb
// cDNA alleles share a warp.  Every pair takes two passes.  Pass 1 over the whole text finds d and the smallest end column
// e of a best placement.  Pass 2 re-runs the window [e - (m + d), e) -- every optimal placement ending at e lies inside it,
// and it is at most 2m columns wide -- and keeps, per column, Hyyro's diagonal-zero vector D0 and ~Pv in HBM scratch, but
// only the words inside the diagonal band the walk back can reach.  (A single pass keeping every word of every column
// wrote 12 GB of HBM for the 8,000 pairs of a score_read call and took 7.7 ms, write-bound; the two passes take 3.5 ms.)
// Walk back (warp-cooperative, one pair at a time): from (m, e) the diagonal when it explains the cell ('=' or 'X'), else
// up ('I', a pattern base without a text base), else left ('D'); before the first diagonal / 'D' step up wins ties, so a
// pattern end hanging over the text end is one trailing 'I' run (a clip).  Taking the diagonal first while walking
// backwards left-aligns gaps, the convention of minimap2's ksw2.  Lane k inspects the k-th cell down the diagonal, so a run
// of up to 32 diagonal steps costs one round of (L2-latency-bound) loads.  Leading / trailing 'I' runs are the clipped
// pattern ends (query_start, query_len - query_end).  The run-length CIGAR -- BAM style, (len << 4) | op with op 1 = I,
// 2 = D, 7 = '=', 8 = X -- is written backwards into the pair's region and then copied by the warp into a dense pool whose
// space it takes with one atomicAdd, so the host needs one copy of the records and one of the pool.
#pragma once
#include "sp_kernels.cuh"

namespace sp {

constexpr uint32_t CIG_I = 1, CIG_D = 2, CIG_EQ = 7, CIG_X = 8;
constexpr int K4_WARPS = 4;  // warps per CTA

struct AlignRecDev {  // layout of sp_align_rec (include/starphase_gpu.h)
    int32_t dist, nm, p_start, p_end, t_start, t_end, n_cigar, pad_;
    long long cigar_off;
};

struct AlignPairDev {   // one pair as the kernel sees it
    long long t_off;    // first text byte (window begin already added)
    long long scr_off;  // words, inside the warp's scratch slot
    long long cig_off;  // first entry of the pair's backwards region; the region ends at cig_off + cig_len
    int32_t n;          // text (window) length
    int32_t m;          // pattern length
    int32_t cig_len;
    int32_t out;        // index into recs
};

struct AlignParams {
    const uint32_t *blobs;       // [n_bins] bins of lane width U: forward rows, infix (wildcard) pad rows
    const uint8_t *tbases;       // ASCII texts
    const int32_t *lane_pair;    // [n_bins][32] pair of each lane (-1: unused lane)
    const int32_t *lane_first;   // [n_bins][32] first lane of that pair inside the bin
    const AlignPairDev *pairs;
    uint32_t *cigar;             // backwards regions
    uint32_t *dense;             // dense pool
    unsigned long long *dense_used;
    unsigned long long dense_cap;
    uint32_t *scratch;           // [n_slots][slot_words]
    long long slot_words;
    AlignRecDev *recs;
    int n_bins;
    int *next_bin;               // work counter
    uint32_t one, m1;
};

// 32-byte store (STG.256): one full L2 sector per lane and word group, so no sector is ever written in halves
__device__ __forceinline__ void st_v8(uint32_t *dst, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1,
                                      uint32_t b2, uint32_t b3) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst), "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0),
                 "r"(b1), "r"(b2), "r"(b3)
                 : "memory");
}

// ASCII -> base code table in shared memory (one LDS per column on the LSU pipe instead of a compare chain on the ALU pipe)
__device__ __forceinline__ void fill_code_lut(uint8_t *lut) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) lut[i] = static_cast<uint8_t>(base_code(static_cast<uint8_t>(i)));
}

// One forward pass of this lane over ncols columns of T.  STORE (pass 2) keeps (D0, ~Pv) of the words the lane owns for every
// column where the lane's rows [row_lo, row_lo + 32 U) touch the diagonal band [band_lo, band_hi] of i - j (cell coordinates).
// Scratch layout: column j = 2 * Wp words, as groups of eight: [D0 x 4 | ~Pv x 4] of four consecutive pattern words.
// The text bytes of the NEXT step are fetched before the current step's eight dependent column steps, so their latency
// (L2 or HBM) hides behind ~400 issue cycles of arithmetic.
// Columns past ncols in the last chunk match nothing; such a column never lowers the score of any row, so with the strict
// comparison of the arg-min they cannot move (best, best_col).
template <int U, bool STORE>
__device__ __forceinline__ void k4_forward(const uint32_t *blob, const uint8_t *lut, const uint8_t *T, int ncols, int rel, int nsteps,
                                           const AlignParams &p, bool first, bool owns, int m, int &best, int &best_col, uint32_t *scr,
                                           int Wp, int wf4, int row_lo, int band_lo, int band_hi) {
    const int lane = threadIdx.x & 31;
    const int row_hi = row_lo + 32 * U - 1;
    uint32_t npv[U], mv[U], d0[U];
    load_row<U>(blob + 5 * (32 * U), lane, npv);
#pragma unroll
    for (int u = 0; u < U; ++u) { npv[u] = ~npv[u]; mv[u] = 0; d0[u] = 0; }
    int score = m, col = 0;
    best = m; best_col = 0;
    uint32_t carry_out = 0;
    const int nch = (ncols + K1_CHUNK - 1) / K1_CHUNK;
    uint32_t nxt[K1_CHUNK];
    auto fetch = [&](int idx) {
        const bool in = owns && static_cast<unsigned>(idx) < static_cast<unsigned>(nch);
        const int j0 = idx * K1_CHUNK;
#pragma unroll
        for (int c = 0; c < K1_CHUNK; ++c) nxt[c] = (in && j0 + c < ncols) ? static_cast<uint32_t>(__ldg(T + j0 + c)) : 0u;  // 0 -> code 4
    };
    fetch(-rel);
    for (int s = 0; s < nsteps; ++s) {
        uint32_t cin = __shfl_up_sync(0xffffffffu, carry_out, 1);
        if (first) cin = 0u;  // infix: the row above the pattern is free
        const int idx = s - rel;
        uint32_t cur[K1_CHUNK];
#pragma unroll
        for (int c = 0; c < K1_CHUNK; ++c) cur[c] = nxt[c];
        fetch(idx + 1);
        if (owns && static_cast<unsigned>(idx) < static_cast<unsigned>(nch)) {
            const int j0 = idx * K1_CHUNK;
            uint32_t X = cin << 24, Y = cin << 16;
            uint32_t cph = 0, cmh = 0;
#pragma unroll
            for (int c = 0; c < K1_CHUNK; ++c) {
                const int j = j0 + c;
                column_step<U, true, STORE>(blob, lane, lut[cur[c]], p.one, p.m1, npv, mv, X, Y, cph, cmh, score, best, col,
                                            best_col, d0);
                if (STORE && j < ncols && row_hi >= j + 1 + band_lo && row_lo <= j + 1 + band_hi) {
                    uint32_t *dst = scr + static_cast<size_t>(j) * 2 * Wp + 2 * (rel * U - wf4);
#pragma unroll
                    for (int q = 0; q < U / 4; ++q)
                        if (rel * U + 4 * q >= wf4)
                            st_v8(dst + 8 * q, d0[4 * q], d0[4 * q + 1], d0[4 * q + 2], d0[4 * q + 3], npv[4 * q], npv[4 * q + 1], npv[4 * q + 2],
                                  npv[4 * q + 3]);
                }
            }
            carry_out = cph | (cmh << 8);
        }
    }
}

__device__ __forceinline__ int warp_max(int v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, off));
    return v;
}

template <int U>
__global__ void __launch_bounds__(32 * K4_WARPS) k4_align(const AlignParams p) {
    static_assert(U % 4 == 0, "the column store moves whole uint4 groups");
    constexpr int BW = blob_words(U);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t *blob = reinterpret_cast<uint32_t *>(smem_raw) + warp * BW;
    __shared__ uint8_t lut[256];
    fill_code_lut(lut);
    __syncthreads();
    const int slot = blockIdx.x * K4_WARPS + warp;
    uint32_t *scr_slot = p.scratch + static_cast<size_t>(slot) * p.slot_words;
    for (;;) {
        int bin = 0;
        if (lane == 0) bin = atomicAdd(p.next_bin, 1);
        bin = __shfl_sync(0xffffffffu, bin, 0);
        if (bin >= p.n_bins) break;
        __syncwarp();
        {
            const uint32_t *src = p.blobs + static_cast<size_t>(bin) * BW;
            for (int i = lane; i < BW; i += 32) blob[i] = src[i];
        }
        __syncwarp();
        const int q = p.lane_pair[bin * 32 + lane];
        const int lane0 = p.lane_first[bin * 32 + lane];
        const bool owns = q >= 0;
        const uint32_t info1 = blob[PEQ_ROWS * 32 * U + 32 + lane];
        const bool first = !owns || (info1 & INFO_FIRST) != 0, last = owns && (info1 & INFO_LAST) != 0;
        AlignPairDev pr = {0, 0, 0, 0, 0, 0, 0};
        if (owns) pr = p.pairs[q];
        const int m = pr.m, rel = lane - lane0;
        const int nl = (m + 32 * U - 1) / (32 * U);
        const int pad = nl * 32 * U - m;
        const int wf4 = (pad >> 5) & ~3, Wp = nl * U - wf4;
        const uint8_t *T = p.tbases + pr.t_off;
        uint32_t *scr = scr_slot + pr.scr_off;
        const int row_lo = rel * 32 * U - pad + 1;         // first pattern row (cell coordinates) of this lane
        const int last_lane = owns ? lane0 + nl - 1 : lane;  // lane holding the pair's last row
        int best, best_col;
        const int nch = (pr.n + K1_CHUNK - 1) / K1_CHUNK;
        const int nsteps = warp_max(owns ? nch + rel : 0);
        k4_forward<U, false>(blob, lut, T, pr.n, rel, nsteps, p, first, owns, m, best, best_col, nullptr, 0, 0, 0, 0, 0);
        const int d = __shfl_sync(0xffffffffu, best, last_lane);
        const int e = __shfl_sync(0xffffffffu, best_col, last_lane);
        const int w0 = max(0, e - (m + d)), ncols = e - w0;
        // d is known here: the walk back cannot leave the diagonal band |i - j - (m - ncols)| <= d (each edit moves i - j
        // by at most one), so only the lanes touching the band keep their columns
        const int delta_end = m - ncols;
        const int nsteps2 = warp_max(owns ? (ncols + K1_CHUNK - 1) / K1_CHUNK + rel : 0);
        k4_forward<U, true>(blob, lut, T + w0, ncols, rel, nsteps2, p, first, owns, m, best, best_col, scr, Wp, wf4, row_lo, delta_end - d - 1,
                            delta_end + d + 1);
        __threadfence_block();
        __syncwarp();
        // walk back, one pair of the bin at a time; the pair's parameters come from its last lane
        uint32_t todo = __ballot_sync(0xffffffffu, last);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const int w_m = __shfl_sync(0xffffffffu, m, src), w_lane0 = __shfl_sync(0xffffffffu, lane0, src);
            const int w_pad = __shfl_sync(0xffffffffu, pad, src), w_wf4 = __shfl_sync(0xffffffffu, wf4, src), w_Wp = __shfl_sync(0xffffffffu, Wp, src);
            const int w_d = __shfl_sync(0xffffffffu, d, src), w_e = __shfl_sync(0xffffffffu, e, src);
            const int w_w0 = __shfl_sync(0xffffffffu, w0, src), w_ncols = __shfl_sync(0xffffffffu, ncols, src);
            const int w_out = __shfl_sync(0xffffffffu, pr.out, src), w_cig_len = __shfl_sync(0xffffffffu, pr.cig_len, src);
            const long long w_scr_off = __shfl_sync(0xffffffffu, pr.scr_off, src), w_t_off = __shfl_sync(0xffffffffu, pr.t_off, src);
            const long long w_cig_off = __shfl_sync(0xffffffffu, pr.cig_off, src);
            const uint32_t *w_scr = scr_slot + w_scr_off;
            const uint8_t *w_T = p.tbases + w_t_off;
            // lane k looks at the diagonal cell (i - k, j - k); the leading run of cells the diagonal explains is taken in one
            // round (HiFi-like pairs are long '=' runs), anything else is one step.  (i, j, cur_op, cur_len, pos) are computed
            // from ballots only, so they stay uniform across the warp.
            const long long cig_end = w_cig_off + w_cig_len;
            long long pos = cig_end;
            uint32_t cur_op = 0, cur_len = 0;
            int i = w_m, j = w_ncols;
            bool started = false;  // a diagonal or 'D' step has been taken: until then 'I' wins ties (trailing clip in one run)
            auto emit = [&](uint32_t op, uint32_t n) {
                if (op == cur_op) { cur_len += n; return; }
                if (cur_len) { --pos; if (lane == 0) p.cigar[pos] = (cur_len << 4) | cur_op; }
                cur_op = op; cur_len = n;
            };
            while (i > 0) {
                if (j == 0) { emit(CIG_I, static_cast<uint32_t>(i)); i = 0; break; }
                const int ci = i - lane, cj = j - lane;
                bool diag_ok = false, is_eq = false, pv = false;
                if (ci >= 1 && cj >= 1) {
                    const int rr = ci - 1 + w_pad, w = rr >> 5, b = rr & 31;
                    const uint32_t *colp = w_scr + static_cast<size_t>(cj - 1) * 2 * w_Wp + 2 * ((w & ~3) - w_wf4) + (w & 3);
                    const uint32_t d0w = __ldcg(colp), npvw = __ldcg(colp + 4);  // same 32-byte sector
                    const uint32_t code = lut[__ldg(w_T + w_w0 + cj - 1)];
                    is_eq = code < 4 && ((blob[code * 32 * U + row_word(U, w_lane0 + w / U, w % U)] >> b) & 1u);
                    diag_ok = is_eq || !((d0w >> b) & 1u);  // the diagonal explains the cell ('=' or a substitution)
                    pv = !((npvw >> b) & 1u);                // vertical delta +1: the cell above explains it ('I')
                }
                const uint32_t ok_mask = __ballot_sync(0xffffffffu, diag_ok);
                const uint32_t eq_mask = __ballot_sync(0xffffffffu, is_eq);
                const bool pv0 = __shfl_sync(0xffffffffu, pv ? 1 : 0, 0) != 0;
                if (!started && pv0) { emit(CIG_I, 1); --i; continue; }
                started = true;
                const int n_diag = ok_mask == 0xffffffffu ? 32 : __ffs(~ok_mask) - 1;
                if (n_diag == 0) {
                    if (pv0) { emit(CIG_I, 1); --i; } else { emit(CIG_D, 1); --j; }
                    continue;
                }
                int done = 0;
                while (done < n_diag) {  // runs of '=' / 'X' among the first n_diag lanes, in walk order
                    const bool eq = (eq_mask >> done) & 1u;
                    const uint32_t rest = (eq ? ~eq_mask : eq_mask) >> done;  // first lane of the other kind
                    int run = rest ? __ffs(rest) - 1 : 32;
                    run = min(run, n_diag - done);
                    emit(eq ? CIG_EQ : CIG_X, static_cast<uint32_t>(run));
                    done += run;
                }
                i -= n_diag; j -= n_diag;
            }
            if (cur_len) { --pos; if (lane == 0) p.cigar[pos] = (cur_len << 4) | cur_op; }
            __threadfence_block();
            __syncwarp();
            // record + dense copy of the kept entries (leading / trailing 'I' runs are the clipped pattern ends)
            int ncig = static_cast<int>(cig_end - pos), clip_s = 0, clip_e = 0;
            long long from = pos;
            if (ncig > 0) {
                const uint32_t head = __ldcg(p.cigar + pos), tail = __ldcg(p.cigar + cig_end - 1);
                if ((head & 15u) == CIG_I) { clip_s = static_cast<int>(head >> 4); ++from; --ncig; }
                if (ncig > 0 && (tail & 15u) == CIG_I) { clip_e = static_cast<int>(tail >> 4); --ncig; }
            }
            unsigned long long at = 0;
            if (lane == 0 && ncig > 0) at = atomicAdd(p.dense_used, static_cast<unsigned long long>(ncig));
            at = __shfl_sync(0xffffffffu, at, 0);
            if (at + static_cast<unsigned long long>(ncig) <= p.dense_cap)
                for (int k = lane; k < ncig; k += 32) p.dense[at + k] = __ldcg(p.cigar + from + k);
            if (lane == 0) {
                AlignRecDev rec;
                rec.dist = w_d; rec.nm = w_d - clip_s - clip_e;
                rec.p_start = clip_s; rec.p_end = w_m - clip_e;
                rec.t_start = w_w0 + j; rec.t_end = w_e;
                rec.n_cigar = ncig; rec.pad_ = 0; rec.cigar_off = static_cast<long long>(at);
                p.recs[w_out] = rec;
            }
            __syncwarp();
        }
        __syncwarp();
    }
}

}  // namespace sp
