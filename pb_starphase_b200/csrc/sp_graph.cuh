// sp_graph.cuh -- K8: end-to-end alignment of sequences to variant graphs (row N3 of SURVEY.md 8f).
//
// Cyp2d6Extractor::assign_haplotype (src/cyp2d6/haplotyper.rs:371-468 of the reference) aligns every consensus to a graph of the
// CYP2D6 backbone with one bubble per database variant (hiphase's WFAGraph) and reads the allele of every variant off the nodes
// the optimal alignments pass through.  K8 is the forward half: the unit-cost DP over the graph, one warp per (graph, sequence)
// problem.  The graph arrives linearised: position = one character, predecessors = the previous character of its node or the
// last characters of the predecessor nodes (-1 = the start column), `diag` = the row the position is expected to align to.
//     D[pos][i] = min( min over preds q of { D[q][i-1] + (g[pos] != s[i-1]),  D[q][i] + 1 },  D[pos][i-1] + 1 )
// for the rows |i - diag[pos]| <= W.  Inside a node the predecessor is the previous position and the band moves down by one
// row, so the diagonal neighbour is the lane's own previous value and the horizontal one the next cell (one shuffle): no memory
// traffic except the column store; at node starts the predecessor columns are read back from the column matrix.  The vertical
// term is the same min-plus prefix scan as in K7.  Every column is written out.  K8's backward half (k8_graph_mark) walks the
// column matrix in descending position order, marks the cells that lie on optimal alignments and reports, per position, whether
// any of its cells is marked (the traversed nodes of sp_graph_traverse).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace sp {

constexpr int GRAPH_INF = 0x3FFFFFFF;

struct GraphParams {
    const uint8_t *gcodes;       // graph characters as codes 0..3, 4 = other
    const long long *goff;       // [n_problems + 1] positions of each problem
    const int32_t *pred_off;     // [total_positions + 1]
    const int32_t *preds;        // problem-local position ids, -1 = start column
    const int32_t *diag;         // [total_positions]
    const int32_t *end_off;      // [n_problems + 1]
    const int32_t *ends;
    const uint8_t *scodes;       // sequences as codes
    const long long *soff;       // [n_problems + 1]
    int32_t *columns;            // [total_positions][2W + 1]
    int32_t *score;              // [n_problems]
    // k8_graph_mark only
    uint8_t *marks;              // [total_positions][2W + 1] zeroed: marks pushed to a column by a successor off the fast path
    uint8_t *hit;                // [total_positions] zeroed: 1 = the column received such marks
    uint8_t *on_path;            // [total_positions] out
    int n_problems, W;
};

template <int CELLS>
__global__ void __launch_bounds__(128) k8_graph_forward(const GraphParams p) {
    const int prob = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (prob >= p.n_problems) return;
    const int nb = 2 * p.W + 1, W = p.W;
    const long long g0 = p.goff[prob];
    const int npos = static_cast<int>(p.goff[prob + 1] - g0);
    const uint8_t *S = p.scodes + p.soff[prob];
    const int m = static_cast<int>(p.soff[prob + 1] - p.soff[prob]);
    const int k0 = lane * CELLS;
    int e[CELLS];  // column of the previous position (valid when the fast path applies)
    int prev_diag = 0, prev_pos = -2;
    // value of row i in the column of predecessor q (-1 = start column: D = i for i <= W)
    auto col_at = [&](int q, int i) -> int {
        if (i < 0 || i > m) return GRAPH_INF;
        if (q < 0) return i <= W ? i : GRAPH_INF;
        const int k = i - p.diag[g0 + q] + W;
        if (k < 0 || k >= nb) return GRAPH_INF;
        return p.columns[(g0 + q) * nb + k];
    };
    for (int pos = 0; pos < npos; ++pos) {
        const int d = p.diag[g0 + pos];
        const uint32_t ch = p.gcodes[g0 + pos];
        const int pb = p.pred_off[g0 + pos], pe = p.pred_off[g0 + pos + 1];
        const bool fast = pe - pb == 1 && p.preds[pb] == prev_pos && d == prev_diag + 1 && prev_pos >= 0;
        int nw[CELLS];
        if (fast) {
            // diagonal neighbour = own previous value (same band index), horizontal = the next band cell of the previous column
            const int from_next_lane = __shfl_down_sync(0xffffffffu, e[0], 1);
#pragma unroll
            for (int c = 0; c < CELLS; ++c) {
                const int k = k0 + c, i = d - W + k;
                int v = GRAPH_INF;
                if (k < nb && i >= 0 && i <= m) {
                    const int horiz = c + 1 < CELLS ? e[c + 1] : (lane < 31 ? from_next_lane : GRAPH_INF);
                    const int hz = (k + 1 < nb && horiz < GRAPH_INF) ? horiz + 1 : GRAPH_INF;
                    int dg = GRAPH_INF;
                    if (i > 0 && e[c] < GRAPH_INF) dg = e[c] + ((ch < 4u && S[i - 1] == ch) ? 0 : 1);
                    v = min(hz, dg);
                }
                nw[c] = v;
            }
        } else {
            __syncwarp();  // the columns this position reads were written by this warp
#pragma unroll
            for (int c = 0; c < CELLS; ++c) {
                const int k = k0 + c, i = d - W + k;
                int v = GRAPH_INF;
                if (k < nb && i >= 0 && i <= m) {
                    for (int q = pb; q < pe; ++q) {
                        const int pr = p.preds[q];
                        const int h = col_at(pr, i);
                        if (h < GRAPH_INF) v = min(v, h + 1);
                        if (i > 0) {
                            const int dg = col_at(pr, i - 1);
                            if (dg < GRAPH_INF) v = min(v, dg + ((ch < 4u && S[i - 1] == ch) ? 0 : 1));
                        }
                    }
                }
                nw[c] = v;
            }
        }
        // vertical: x[k] = v[k] - k, inclusive prefix min, back to values
        int run = GRAPH_INF;
#pragma unroll
        for (int c = 0; c < CELLS; ++c) {
            const int x = nw[c] < GRAPH_INF ? nw[c] - (k0 + c) : GRAPH_INF;
            run = min(run, x);
            nw[c] = run;
        }
        int carry = run;
#pragma unroll
        for (int dd = 1; dd < 32; dd <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, carry, dd);
            if (lane >= dd) carry = min(carry, up);
        }
        int before = __shfl_up_sync(0xffffffffu, carry, 1);
        if (lane == 0) before = GRAPH_INF;
#pragma unroll
        for (int c = 0; c < CELLS; ++c) {
            const int k = k0 + c, i = d - W + k;
            const int x = min(nw[c], before);
            e[c] = (k < nb && i >= 0 && i <= m && x < GRAPH_INF) ? x + k : GRAPH_INF;
            if (k < nb) p.columns[(g0 + pos) * nb + k] = e[c];
        }
        prev_diag = d; prev_pos = pos;
    }
    __syncwarp();
    // best end: min over the end positions of D[end][m]
    int best = GRAPH_INF;
    for (int q = p.end_off[prob] + lane; q < p.end_off[prob + 1]; q += 32) best = min(best, col_at(p.ends[q], m));
#pragma unroll
    for (int dd = 16; dd > 0; dd >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, dd));
    if (lane == 0) p.score[prob] = best;
}

// K8 backward, on the columns k8_graph_forward wrote: marks the cells with forward + backward == score, i.e. the closure of the
// end cells (e, m) with D[e][m] == score under the moves of the recurrence taken backwards:
//     (q, i) -> (q, i-1)   when D[q][i-1] + 1 == D[q][i]
//     (q, i) -> (pr, i)    when D[pr][i] + 1 == D[q][i]          for every predecessor pr >= 0
//     (q, i) -> (pr, i-1)  when D[pr][i-1] + sub(q, i) == D[q][i]
// and writes on_path[q] = 1 when a cell of column q is marked.  Positions go in descending order, so every successor of q has
// pushed its marks when q is processed.  Where the forward kernel took its fast path (single predecessor q - 1, band one row
// lower), the marks for q - 1 stay in registers: the diagonal move keeps the band index, the horizontal one goes up one index
// (one shuffle).  Elsewhere they go to `marks`, and the receiving column reads them back when its `hit` flag is set.  Inside a
// column the vertical move is a segmented scan, lane-local and then across lanes as a carry chain over two ballots.  Marked cells
// are finite, so an INF neighbour never matches.
template <int CELLS>
__global__ void __launch_bounds__(128, 4) k8_graph_mark(const GraphParams p) {
    constexpr int PREFETCH = 8;  // columns ahead pulled into L2: the matrix of a batch is larger than the L2
    const int prob = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (prob >= p.n_problems) return;
    const int nb = 2 * p.W + 1, W = p.W;
    const long long g0 = p.goff[prob];
    const int npos = static_cast<int>(p.goff[prob + 1] - g0);
    const uint8_t *S = p.scodes + p.soff[prob];
    const int m = static_cast<int>(p.soff[prob + 1] - p.soff[prob]);
    const int32_t *cols = p.columns + g0 * nb, *diag = p.diag + g0, *pred_off = p.pred_off + g0;
    const uint8_t *gc = p.gcodes + g0;
    uint8_t *marks = p.marks + g0 * nb, *hit = p.hit + g0, *on_path = p.on_path + g0;
    const int score = p.score[prob];
    if (score >= GRAPH_INF) {  // the band excludes every path
        for (int q = lane; q < npos; q += 32) on_path[q] = 0;
        return;
    }
    const int k0 = lane * CELLS;
    auto col_at = [&](int q, int i) -> int {
        if (i < 0 || i > m) return GRAPH_INF;
        if (q < 0) return i <= W ? i : GRAPH_INF;
        const int k = i - diag[q] + W;
        if (k < 0 || k >= nb) return GRAPH_INF;
        return cols[static_cast<long long>(q) * nb + k];
    };
    auto push = [&](int pr, int i) {
        marks[static_cast<long long>(pr) * nb + i - diag[pr] + W] = 1;
        hit[pr] = 1;
    };
    // seeds: the end cells that reach the score (-1 = the start column, never marked)
    for (int t = p.end_off[prob] + lane; t < p.end_off[prob + 1]; t += 32) {
        const int e = p.ends[t];
        if (e >= 0 && col_at(e, m) == score) push(e, m);
    }
    __syncwarp();
    int cur[CELLS], nxt[CELLS];
#pragma unroll
    for (int c = 0; c < CELLS; ++c) cur[c] = npos > 0 && k0 + c < nb ? cols[static_cast<long long>(npos - 1) * nb + k0 + c] : GRAPH_INF;
    uint32_t carry = 0;  // marks of column q brought in registers by the fast step of q + 1 (bit c = band index k0 + c)
    bool pushed = npos > 0 && hit[npos - 1];
    for (int q = npos - 1; q >= 0; --q) {
        const int d = diag[q], pb = pred_off[q], pe = pred_off[q + 1];
        const uint32_t ch = gc[q];
        const bool fast = q > 0 && pe - pb == 1 && p.preds[pb] == q - 1 && d == diag[q - 1] + 1;
        const bool pushed_next = q > 0 && hit[q - 1];  // from the steps before this one; this step's own pushes are added below
#pragma unroll
        for (int c = 0; c < CELLS; ++c) nxt[c] = q > 0 && k0 + c < nb ? cols[static_cast<long long>(q - 1) * nb + k0 + c] : GRAPH_INF;
        if (q >= PREFETCH && k0 < nb) asm volatile("prefetch.global.L2 [%0];" ::"l"(cols + static_cast<long long>(q - PREFETCH) * nb + k0));
        uint32_t mk = carry;
        if (pushed) {
#pragma unroll
            for (int c = 0; c < CELLS; ++c)
                if (k0 + c < nb && marks[static_cast<long long>(q) * nb + k0 + c]) mk |= 1u << c;
        }
        // vertical closure: link bit c (D[k-1] + 1 == D[k], k = k0 + c) carries a mark from band index k to k - 1
        const int below = __shfl_up_sync(0xffffffffu, cur[CELLS - 1], 1);
        uint32_t link = lane > 0 && below + 1 == cur[0] ? 1u : 0u;
#pragma unroll
        for (int c = 1; c < CELLS; ++c) link |= cur[c - 1] + 1 == cur[c] ? 1u << c : 0u;
#pragma unroll
        for (int c = CELLS - 2; c >= 0; --c) mk |= (mk & link) >> 1 & 1u << c;
        // across lanes, from lane 31 down: lane j passes a mark to lane j - 1 when it generates one at its index 0 (g) or when
        // one enters at its top and every link of the lane holds (p).  Bit-reversed, that is the carry chain of G + (G | P).
        const uint32_t G = __brev(__ballot_sync(0xffffffffu, mk & link & 1u)), Y = G | __brev(__ballot_sync(0xffffffffu, link == (1u << CELLS) - 1));
        if (((G + Y) ^ G ^ Y) >> (31 - lane) & 1u) {
            mk |= 1u << (CELLS - 1);
#pragma unroll
            for (int c = CELLS - 2; c >= 0; --c) mk |= (mk & link) >> 1 & 1u << c;
        }
        const bool any = __any_sync(0xffffffffu, mk != 0);
        if (lane == 0) on_path[q] = any ? 1 : 0;
        carry = 0;
        bool self = false;  // this step pushed into column q - 1
        if (fast) {
            const int top_of_below = __shfl_up_sync(0xffffffffu, mk >> (CELLS - 1) & 1u ? cur[CELLS - 1] : -1, 1);
#pragma unroll
            for (int c = 0; c < CELLS; ++c) {
                const int i = d - W + k0 + c;
                const int left = c > 0 ? (mk >> (c - 1) & 1u ? cur[c - 1] : -1) : (lane > 0 ? top_of_below : -1);
                const int sub = ch < 4u && i >= 1 && i <= m && S[i - 1] == ch ? 0 : 1;
                if ((mk >> c & 1u) && nxt[c] + sub == cur[c]) carry |= 1u << c;  // diagonal: (q, i) -> (q - 1, i - 1), same index
                if (nxt[c] + 1 == left) carry |= 1u << c;                        // horizontal: (q, i) -> (q - 1, i), one index up
            }
        } else {
#pragma unroll
            for (int c = 0; c < CELLS; ++c) {
                if (!(mk >> c & 1u)) continue;
                const int i = d - W + k0 + c, v = cur[c];
                const int sub = ch < 4u && i >= 1 && S[i - 1] == ch ? 0 : 1;
                for (int t = pb; t < pe; ++t) {
                    const int pr = p.preds[t];
                    if (pr < 0) continue;
                    if (col_at(pr, i) + 1 == v) { push(pr, i); self |= pr == q - 1; }
                    if (i > 0 && col_at(pr, i - 1) + sub == v) { push(pr, i - 1); self |= pr == q - 1; }
                }
            }
            self = __any_sync(0xffffffffu, self);
            __syncwarp();  // the next steps read these marks back
        }
        pushed = pushed_next || self;
#pragma unroll
        for (int c = 0; c < CELLS; ++c) cur[c] = nxt[c];
    }
}

}  // namespace sp
