"""tests/graph_walk.py -- the checker of sp_graph_traverse (K8's marking pass).  TEST INFRASTRUCTURE ONLY.

`traverse` is the walk back of graph_oracle.align restated over graph_oracle.forward's columns, returning the marked positions
instead of the nodes: the end cells (e, m) that reach the score and, from each marked (q, i), the neighbours whose step into
(q, i) is tight; the start column is never marked.  tests/test_graph_traverse_cpu.py pins it to graph_oracle.align and to brute
force over every path."""
from __future__ import annotations

import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "oracle"))

import graph_oracle as go  # noqa: E402


def traverse(g: go.Graph, seq: bytes, band: int = 1 << 20):
    """(score, linearise(g), sorted positions with a cell on an optimal alignment); an unreachable problem (score INF) marks
    nothing."""
    lin, cols, score = go.forward(g, seq, band)
    chars, preds, diag, node_of, ends = lin
    m = len(seq)
    start = {i: i for i in range(0, min(m, band) + 1)}

    def col(q):
        return start if q < 0 else cols[q]

    if score >= go.INF:
        return go.INF, lin, []
    marked = [set() for _ in chars]
    stack = [(e, m) for e in ends if col(e).get(m, go.INF) == score]
    seen_start = False
    while stack:
        pos, i = stack.pop()
        if pos < 0:
            seen_start = True
            continue
        if i in marked[pos]:
            continue
        marked[pos].add(i)
        v = cols[pos][i]
        if i > 0 and cols[pos].get(i - 1, go.INF) + 1 == v:
            stack.append((pos, i - 1))
        for q in preds[pos]:
            cq = col(q)
            if cq.get(i, go.INF) + 1 == v:
                stack.append((q, i))
            if i > 0 and cq.get(i - 1, go.INF) < go.INF and cq[i - 1] + (0 if seq[i - 1] == chars[pos] and chars[pos] in b"ACGT" else 1) == v:
                stack.append((q, i - 1))
    assert seen_start
    return score, lin, [q for q, cells in enumerate(marked) if cells]
