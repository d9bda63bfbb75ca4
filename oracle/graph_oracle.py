"""oracle/graph_oracle.py -- CPU ORACLE for row N3 (sequence-to-variant-graph alignment).  TEST INFRASTRUCTURE ONLY.

PARITY STATUS: "parity unpinned".  Cyp2d6Extractor::assign_haplotype (src/cyp2d6/haplotyper.rs:371-468) builds a variant graph
with hiphase v1.2.1 (`WFAGraph::from_reference_variants`, git dependency, Cargo.lock:812-814, not vendored, not buildable here),
aligns the consensus to it end to end (`edit_distance_with_pruning`) and turns the traversed nodes into a 0/1/2/3 allele vector
(:452-468; restated in starphase_oracle.alleles_from_traversal).  What is restated here is the published behaviour the reference
relies on -- reference backbone with one bubble per variant site, node -> (variant, allele) labels, unit-cost end-to-end
alignment, "traversed" = the nodes some optimal alignment passes through -- NOT hiphase's code: how overlapping variants are
grouped into one site and which labels an ALT branch gives to the other variants of its site are choices of this repository.
Pinned by properties (tests/test_graph_cpu.py): a sequence spelled from the backbone with chosen alleles has distance 0 and
traverses exactly those allele nodes; on small graphs the DP equals brute force over every path; a site whose alleles cannot
be told apart by the sequence comes out ambiguous.

`build_graph` and `align` are the checkers of VariantGraph / graph_edit_distance in pb_starphase_b200/host/sp_host_graph.cpp
and of the K8 kernel behind them (same banded recurrence)."""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Sequence, Tuple

INF = 0x3FFFFFFF


@dataclass
class Graph:
    seqs: List[bytes] = field(default_factory=list)              # node sequences (only the unlabelled source / sink may be empty)
    preds: List[List[int]] = field(default_factory=list)         # predecessor nodes
    coord: List[int] = field(default_factory=list)               # backbone offset at which the node starts (band centre)
    node_to_alleles: Dict[int, List[Tuple[int, int]]] = field(default_factory=dict)
    sink: int = -1

    def add(self, seq: bytes, preds: Sequence[int], coord: int) -> int:
        self.seqs.append(seq); self.preds.append(list(preds)); self.coord.append(coord)
        return len(self.seqs) - 1


def build_graph(backbone: bytes, region_start: int, variants: Sequence[Tuple[int, bytes, bytes]]) -> Graph:
    """backbone = reference[region_start, region_start + len); variants = (position, ref allele, alt allele) in reference
    coordinates, in the order that defines their indices (src/cyp2d6/haplotyper.rs:452: `ordered_variants`).  Variants not wholly
    inside the region are left out (their allele stays 3 = unset).  Overlapping variants form one site: a REF branch labelled
    (v, 0) for every variant of the site and one ALT branch per variant, labelled (v, 1) and (u, 0) for the others."""
    g = Graph()
    n = len(backbone)
    inside = [(p - region_start, r, a, k) for k, (p, r, a) in enumerate(variants)
              if p - region_start >= 0 and p - region_start + len(r) <= n and backbone[p - region_start:p - region_start + len(r)] == r]
    inside.sort(key=lambda v: (v[0], v[3]))
    sites, cur, cur_end = [], [], -1
    for v in inside:
        if cur and v[0] < cur_end or (cur and v[0] == cur[0][0]):
            cur.append(v); cur_end = max(cur_end, v[0] + len(v[1]))
        else:
            if cur:
                sites.append(cur)
            cur, cur_end = [v], v[0] + len(v[1])
    if cur:
        sites.append(cur)
    last, pos = [g.add(b"", [], 0)], 0  # node 0: empty source
    for site in sites:
        s0 = site[0][0]
        s1 = max(v[0] + len(v[1]) for v in site)
        # every branch keeps at least one character: a bare deletion (no anchor base in the record) takes the backbone base before
        # it into the site, or the one after it at the very start
        if any(len(backbone[s0:v[0]] + v[2] + backbone[v[0] + len(v[1]):s1]) == 0 for v in site):
            if s0 > pos:
                s0 -= 1
            elif s1 < n:
                s1 += 1
        if s0 > pos:
            last = [g.add(backbone[pos:s0], last, pos)]
        branches = []
        ref = g.add(backbone[s0:s1], last, s0)
        g.node_to_alleles[ref] = [(v[3], 0) for v in site]
        branches.append(ref)
        for v in site:
            alt = g.add(backbone[s0:v[0]] + v[2] + backbone[v[0] + len(v[1]):s1], last, s0)
            g.node_to_alleles[alt] = [(v[3], 1)] + [(u[3], 0) for u in site if u[3] != v[3]]
            branches.append(alt)
        last, pos = branches, s1
    g.sink = g.add(backbone[pos:], last, pos)
    return g


def linearise(g: Graph):
    """Positions = the characters of all nodes in node order (a topological order); preds of a position = the previous character
    of its node, or the last characters of the predecessor nodes (through empty nodes); -1 = the start column.
    Returns (chars, pred lists, nominal row of each position, node of each position, end positions of the sink)."""
    first, lastpos = {}, {}
    chars, preds, diag, node_of = [], [], [], []

    def tails(node):  # positions at which a path can stand after node `node`
        if g.seqs[node]:
            return [lastpos[node]]
        if not g.preds[node]:
            return [-1]
        out = []
        for p in g.preds[node]:
            out += tails(p)
        return sorted(set(out))

    for node, seq in enumerate(g.seqs):
        for c, ch in enumerate(seq):
            pid = len(chars)
            if c == 0:
                first[node] = pid
                pr = []
                for p in g.preds[node]:
                    pr += tails(p)
                preds.append(sorted(set(pr)) if g.preds[node] else [-1])
            else:
                preds.append([pid - 1])
            chars.append(ch); diag.append(g.coord[node] + c + 1); node_of.append(node)
        if seq:
            lastpos[node] = len(chars) - 1
    return bytes(chars), preds, diag, node_of, tails(g.sink)


def forward(g: Graph, seq: bytes, band: int = 1 << 20):
    """The forward DP of `align`: (linearise(g), cols, score).  cols[pos] maps row i -> D[pos][i] for the band rows
    |i - diag[pos]| <= band inside [0, len(seq)] (INF where no path reaches); score = min over the end positions of D[end][m]."""
    lin = linearise(g)
    chars, preds, diag, node_of, ends = lin
    m = len(seq)

    def rows(d):
        return range(max(0, d - band), min(m, d + band) + 1)

    start = {i: i for i in rows(0)}
    cols: List[Dict[int, int]] = []

    def col(q):
        return start if q < 0 else cols[q]

    for pos, ch in enumerate(chars):
        c, prev = {}, INF
        for i in rows(diag[pos]):
            best = prev + 1 if prev < INF else INF
            for q in preds[pos]:
                cq = col(q)
                h = cq.get(i, INF)
                if h < INF:
                    best = min(best, h + 1)
                if i > 0:
                    d = cq.get(i - 1, INF)
                    if d < INF:
                        best = min(best, d + (0 if seq[i - 1] == ch and ch in b"ACGT" else 1))
            c[i] = best
            prev = best
        cols.append(c)
    score = min((col(e).get(m, INF) for e in ends), default=INF)
    return lin, cols, score


def align(g: Graph, seq: bytes, band: int = 1 << 20):
    """(edit distance, sorted traversed nodes): end-to-end alignment of seq to a source -> sink path, unit costs; rows outside
    |i - nominal row| <= band are not computed (the product's band; the default is "no band")."""
    (chars, preds, diag, node_of, ends), cols, score = forward(g, seq, band)
    m = len(seq)

    def rows(d):
        return range(max(0, d - band), min(m, d + band) + 1)

    start = {i: i for i in rows(0)}

    def col(q):
        return start if q < 0 else cols[q]

    if score >= INF:
        return INF, []
    # backward: cells on optimal alignments
    marked = [set() for _ in chars]
    stack = [(e, m) for e in ends if col(e).get(m, INF) == score]
    nodes = set()
    seen_start = False
    while stack:
        pos, i = stack.pop()
        if pos < 0:
            seen_start = True
            continue
        if i in marked[pos]:
            continue
        marked[pos].add(i)
        nodes.add(node_of[pos])
        v = cols[pos][i]
        if i > 0 and cols[pos].get(i - 1, INF) + 1 == v:
            stack.append((pos, i - 1))
        for q in preds[pos]:
            cq = col(q)
            if cq.get(i, INF) + 1 == v:
                stack.append((q, i))
            if i > 0 and cq.get(i - 1, INF) < INF and cq[i - 1] + (0 if seq[i - 1] == chars[pos] and chars[pos] in b"ACGT" else 1) == v:
                stack.append((q, i - 1))
    assert seen_start
    return score, sorted(nodes)


def brute_force(g: Graph, seq: bytes):
    """Every source -> sink path spelled out and aligned globally with a plain DP: (min distance, nodes on the optimal paths)."""
    paths = []

    def walk(node, acc):
        acc = acc + [node]
        succ = [k for k, pr in enumerate(g.preds) if node in pr]
        if node == g.sink:
            paths.append(acc)
            return
        for s in succ:
            walk(s, acc)

    walk(0, [])

    def ed(a: bytes, b: bytes) -> int:
        prev = list(range(len(b) + 1))
        for i, ca in enumerate(a, 1):
            cur = [i]
            for j, cb in enumerate(b, 1):
                cur.append(min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (0 if ca == cb and ca in b"ACGT" else 1)))
            prev = cur
        return prev[-1]

    scored = [(ed(b"".join(g.seqs[k] for k in p), seq), p) for p in paths]
    best = min(s for s, _ in scored)
    nodes = sorted({k for s, p in scored if s == best for k in p if g.seqs[k]})
    return best, nodes
