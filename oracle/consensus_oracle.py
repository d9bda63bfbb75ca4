"""oracle/consensus_oracle.py -- CPU ORACLE for row N1 (consensus).  TEST INFRASTRUCTURE ONLY.

PARITY STATUS: "parity unpinned".  The reference takes its consensus sequences from waffle_con v0.4.4 (git dependency,
Cargo.lock:2246-2248; not vendored, not buildable here: no Rust toolchain, no network) through ConsensusDWFA / DualConsensusDWFA /
PriorityConsensusDWFA (src/hla/caller.rs:1097-1219, :727-755; src/cyp2d6/caller.rs:145-280).  What is restated here is the
published outline of that algorithm -- a best-first search over consensus prefixes in which every read keeps its edit distance
to the growing prefix (end-free in the read), reads vote for the next symbol with the bases following their best prefixes,
symbols need min_count votes and a min_af share, the queue holds at most max_queue_size nodes and max_capacity_per_size nodes
are expanded per consensus length, a dual node carries two consensuses and every read counts towards the closer one
(CdwfaConfig as set at src/hla/caller.rs:1103-1116) -- NOT waffle_con's code: tie orders, the offset search inside
offset_window and the pruning details are choices of this repository.  The reference's tests hold no consensus vectors for this
path, so the restatement is pinned only by properties (error-free reads => the source sequence; a majority out-votes errors;
two alleles => both come back with the right read split): tests/test_consensus_cpu.py, tests/test_consensus_gpu.py.

Two layers, mirroring the product: `extend` is the checker of the K7 kernel (same banded recurrence, same outputs, bit for
bit); `consensus` / `dual_consensus` are the checker of the host search in pb_starphase_b200/host/sp_host_consensus.cpp.
"""
from __future__ import annotations

import heapq
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

INF = 0x3FFFFFFF
VOTE_FINISHED, VOTE_INACTIVE = 1 << 5, 1 << 6
_CODE = {65: 0, 67: 1, 71: 2, 84: 3, 97: 0, 99: 1, 103: 2, 116: 3, 42: 5}  # '*' = wildcard: matches every symbol, votes for none
VOTE_UNIT = 12  # one read's vote, split evenly over its 1..4 candidate symbols


@dataclass
class Config:  # the members of waffle_con's CdwfaConfig the reference sets (src/hla/caller.rs:1103-1116)
    min_count: int = 3
    min_af: float = 0.10
    allow_early_termination: bool = False
    max_queue_size: int = 20
    max_capacity_per_size: int = 10
    offset_window: int = 0
    band: int = 32


class Track:
    """The DP column of every read against one consensus prefix (what one K7 track holds)."""

    def __init__(self, n_reads: int):
        self.length = 0
        self.cols: List[Optional[Dict[int, int]]] = [None] * n_reads  # row i -> E[i], band rows only
        self.best_full = [INF] * n_reads


def extend(reads: Sequence[bytes], offsets: Sequence[int], cfg: Config, src: Track, symbol: int) -> Tuple[Track, List[int], List[int], List[int]]:
    """K7 restated: (new track, ed[r], votes[r], full[r]).  symbol 0 = report only."""
    W = cfg.band + cfg.offset_window // 2
    out = Track(len(reads))
    ext = symbol != 0
    L0 = src.length
    L = L0 + (1 if ext else 0)
    out.length = L
    s = min(_CODE.get(symbol, 4), 4)
    eds, votes, fulls = [], [], []
    for r, read in enumerate(reads):
        off, m = max(offsets[r], 0), len(read)
        hw = 0 if offsets[r] < 0 else cfg.offset_window // 2  # offset None (< 0): anchored at the consensus start, no window
        start = max(0, off - hw)
        if L < start:
            eds.append(0); votes.append(VOTE_INACTIVE); fulls.append(INF)
            continue

        def rows(col):  # band rows of column `col`
            c = col - off
            return range(max(0, c - W), min(m, c + W) + 1)

        def old_at(i):  # column L0
            if i < 0 or i > m or abs(i - (L0 - off)) > W:
                return INF
            return i if L0 == start else src.cols[r].get(i, INF)

        if not ext:
            col = {i: old_at(i) for i in rows(L)}
        elif L == start:
            col = {i: i for i in rows(L)}
        else:
            col, prev = {}, INF  # prev = E'[i-1]
            for i in rows(L):
                if i == 0:
                    v = max(0, L - (off + hw))
                else:
                    d, h = old_at(i - 1), old_at(i)
                    sub = 0 if (s < 4 and _CODE.get(read[i - 1], 4) in (s, 5)) else 1
                    v = min(d + sub if d < INF else INF, h + 1 if h < INF else INF, prev + 1 if prev < INF else INF)
                col[i] = v
                prev = v
        out.cols[r] = col
        mn = min(col.values()) if col else INF
        bf = min(src.best_full[r], col.get(m, INF))
        out.best_full[r] = bf
        vt = 0
        if mn < INF:
            for i, v in col.items():
                if v == mn:
                    vt |= VOTE_FINISHED if i == m else ((1 << _CODE.get(read[i], 4)) & 31)
        eds.append(mn); votes.append(vt); fulls.append(bf)
    return out, eds, votes, fulls


# ---------------------------------------------------------------------------------------------------------------
# search policy (restated outline of ConsensusDWFA / DualConsensusDWFA; see the header for what is and is not pinned)
# ---------------------------------------------------------------------------------------------------------------
def read_costs(eds, votes, fulls, reads):
    """Cost of every read against one consensus: its best prefix so far, or the best column at which it was consumed."""
    return [0 if v & VOTE_INACTIVE else min(e, f) for e, v, f in zip(eds, votes, fulls)]


def tally(eds, votes, fulls, voters=None):
    """Votes per symbol (A, C, G, T) in units of VOTE_UNIT / candidates; a read whose best state is 'already consumed' is silent."""
    t = [0, 0, 0, 0]
    for r, (e, v, f) in enumerate(zip(eds, votes, fulls)):
        if voters is not None and not voters[r]:
            continue
        if v & VOTE_INACTIVE or f < e:
            continue
        cands = [k for k in range(4) if v >> k & 1]
        for k in cands:
            t[k] += VOTE_UNIT // len(cands)
    return t


def passing(t, cfg: Config) -> List[int]:
    total = sum(t)
    if total == 0:
        return []
    permille = int(round(cfg.min_af * 1000))
    ok = [k for k in range(4) if t[k] >= VOTE_UNIT * cfg.min_count and t[k] * 1000 >= total * permille]
    return ok if ok else [max(range(4), key=lambda k: (t[k], -k))]


def run(reads: Sequence[bytes], offsets: Sequence[int], cfg: Config, tracks: Sequence[Track], state: Sequence[tuple], min_count: int,
        min_af_permille: int, cost_limit: int, size_limit: int, cost_cap: int, max_steps: int):
    """sp_consensus_run (the K7 loop on the device) restated from extend / tally / passing / read_costs.  tracks[s] and
    state[s] = (eds, votes, fulls) describe side s of the start node (one or two sides).  Keep extending while every side has at
    most one passing symbol and one side has one, the node orders before (cost_limit, size_limit) -- cheaper, or as cheap and
    longer -- its cost is <= cost_cap, and fewer than max_steps rounds were done; round 0 is exempt from the limits.  A side
    with no votes stays as it is.  Returns (tracks, state, steps, costs): the last node, one log byte per round (low nibble:
    code appended to side 0, high nibble: side 1, 15: not extended) and the node cost seen at every decision."""
    pcfg = Config(min_count=min_count, min_af=min_af_permille / 1000)
    assert int(round(pcfg.min_af * 1000)) == min_af_permille
    tracks, state = list(tracks), [tuple(list(x) for x in s) for s in state]
    ns = len(tracks)
    steps, costs = [], []
    while True:
        c = [read_costs(*state[s], reads) for s in range(ns)]
        cost = sum(c[0]) if ns == 1 else sum(min(a, b) for a, b in zip(c[0], c[1]))
        costs.append(cost)
        if ns == 1:
            voters = [None]
        else:
            voters = [[a <= b for a, b in zip(c[0], c[1])], [b <= a for a, b in zip(c[0], c[1])]]
        syms = [passing(tally(*state[s], voters[s]), pcfg) for s in range(ns)]
        size = sum(t.length for t in tracks)
        one_each = all(len(p) <= 1 for p in syms) and any(len(p) == 1 for p in syms)
        before = cost < cost_limit or (cost == cost_limit and size > size_limit)
        may = len(steps) < max_steps and (not steps or (before and cost <= cost_cap))
        if not (one_each and may):
            break
        log = 0
        for s in range(ns):
            if syms[s]:
                k = syms[s][0]
                t, e, v, f = extend(reads, offsets, cfg, tracks[s], b"ACGT"[k])
                tracks[s], state[s] = t, (e, v, f)
            log |= (syms[s][0] if syms[s] else 15) << (4 * s)
        if ns == 1:
            log |= 15 << 4
        steps.append(log)
    return tracks, state, steps, costs


@dataclass(order=True)
class _Node:
    key: tuple
    cons: Tuple[bytes, Optional[bytes]] = field(compare=False)
    state: tuple = field(compare=False)  # ((track, eds, votes, fulls), same for side 2 or None)
    cost: int = field(compare=False, default=0)


def _side_cost(side, reads):
    return read_costs(side[1], side[2], side[3], reads)


def _node(cons, s1, s2, reads) -> _Node:
    c1 = _side_cost(s1, reads)
    if s2 is None:
        cost = sum(c1)
    else:
        c2 = _side_cost(s2, reads)
        cost = sum(min(a, b) for a, b in zip(c1, c2))
    length = len(cons[0]) + (len(cons[1]) if cons[1] is not None else 0)
    return _Node((cost, -length, cons[0], cons[1] if cons[1] is not None else b""), cons, (s1, s2), cost)


def _search(reads, offsets, cfg: Config, allow_dual: bool):
    root_t, e, v, f = extend(reads, offsets, cfg, Track(len(reads)), 0)
    queue = [_node((b"", None), (root_t, e, v, f), None, reads)]
    best, best_cost, expanded = [], None, {}
    while queue:
        node = heapq.heappop(queue)
        if best_cost is not None and node.cost > best_cost:
            break
        s1, s2 = node.state
        if s2 is None:
            t1 = tally(s1[1], s1[2], s1[3])
            p1, p2 = passing(t1, cfg), [None]
            strict = [k for k in p1 if t1[k] >= VOTE_UNIT * cfg.min_count and t1[k] * 1000 >= sum(t1) * int(round(cfg.min_af * 1000))]
        else:
            c1, c2 = _side_cost(s1, reads), _side_cost(s2, reads)
            t1 = tally(s1[1], s1[2], s1[3], [a <= b for a, b in zip(c1, c2)])
            t2 = tally(s2[1], s2[2], s2[3], [b <= a for a, b in zip(c1, c2)])
            p1, p2 = passing(t1, cfg) or [None], passing(t2, cfg) or [None]
            strict = []
        if (s2 is None and not p1) or (s2 is not None and p1 == [None] and p2 == [None]):  # nobody wants to go on: complete
            if s2 is not None:
                n1 = sum(a <= b for a, b in zip(c1, c2))
                n2 = len(reads) - n1
                if min(n1, n2) < cfg.min_count or min(n1, n2) * 1000 < (n1 + n2) * int(round(cfg.min_af * 1000)):
                    continue  # one side is not supported by enough reads: not a valid dual solution
            if best_cost is None or node.cost < best_cost:
                best, best_cost = [node], node.cost
            elif node.cost == best_cost:
                best.append(node)
            continue
        size = len(node.cons[0]) + (len(node.cons[1]) if node.cons[1] is not None else 0)
        if expanded.get(size, 0) >= cfg.max_capacity_per_size:
            continue
        expanded[size] = expanded.get(size, 0) + 1
        children = []
        if s2 is None:
            ext = {k: extend(reads, offsets, cfg, s1[0], b"ACGT"[k]) for k in p1}
            for k in p1:
                children.append(_node((node.cons[0] + b"ACGT"[k:k + 1], None), ext[k], None, reads))
            if allow_dual and len(strict) >= 2:
                for ia in range(len(strict)):
                    for ib in range(ia + 1, len(strict)):
                        a, b = strict[ia], strict[ib]
                        children.append(_node((node.cons[0] + b"ACGT"[a:a + 1], node.cons[0] + b"ACGT"[b:b + 1]), ext[a], ext[b], reads))
        else:
            e1 = {k: (extend(reads, offsets, cfg, s1[0], b"ACGT"[k]) if k is not None else s1) for k in p1}
            e2 = {k: (extend(reads, offsets, cfg, s2[0], b"ACGT"[k]) if k is not None else s2) for k in p2}
            for a in p1:
                for b in p2:
                    ca = node.cons[0] + (b"ACGT"[a:a + 1] if a is not None else b"")
                    cb = node.cons[1] + (b"ACGT"[b:b + 1] if b is not None else b"")
                    children.append(_node((ca, cb), e1[a], e2[b], reads))
        for ch in children:
            heapq.heappush(queue, ch)
        while len(queue) > cfg.max_queue_size:
            queue.remove(max(queue))
            heapq.heapify(queue)
    return best


def consensus(reads: Sequence[bytes], offsets: Optional[Sequence[int]] = None, cfg: Optional[Config] = None):
    """ConsensusDWFA::consensus(): [(sequence, scores[r])] of the best complete nodes (ties in key order)."""
    cfg = cfg or Config()
    offsets = [-1 if o is None else o for o in offsets] if offsets is not None else [-1] * len(reads)
    out = []
    for n in _search(list(reads), offsets, cfg, False):
        s1 = n.state[0]
        out.append((n.cons[0], _side_cost(s1, reads)))
    return out


def dual_consensus(reads: Sequence[bytes], offsets: Optional[Sequence[int]] = None, cfg: Optional[Config] = None):
    """DualConsensusDWFA::consensus(): [dict(consensus1, consensus2 | None, is_consensus1[r], scores1[r], scores2[r])]."""
    cfg = cfg or Config()
    offsets = [-1 if o is None else o for o in offsets] if offsets is not None else [-1] * len(reads)
    out = []
    for n in _search(list(reads), offsets, cfg, True):
        s1, s2 = n.state
        c1 = _side_cost(s1, reads)
        if s2 is None:
            out.append(dict(consensus1=n.cons[0], consensus2=None, is_consensus1=[True] * len(reads), scores1=c1, scores2=[None] * len(reads)))
        else:
            c2 = _side_cost(s2, reads)
            out.append(dict(consensus1=n.cons[0], consensus2=n.cons[1], is_consensus1=[a <= b for a, b in zip(c1, c2)], scores1=c1, scores2=c2))
    return out


def priority_consensus(chains: Sequence[Sequence[bytes]], offsets: Sequence[Sequence[Optional[int]]], seeds: Sequence[Optional[int]],
                       cfg: Optional[Config] = None):
    """PriorityConsensusDWFA as the CYP2D6 caller drives it (src/cyp2d6/caller.rs:145-280), restated outline (parity unpinned; the
    same policy as pb_starphase_b200/host/sp_host_consensus.cpp): inputs with different seeds never share a group; a group is
    examined level by level with dual_consensus -- a dual answer splits it in two (both examined again at the same level), a
    single answer moves it to the next level, after the last level it is final; groups ordered by their smallest input index.
    Returns (consensuses[group][level] = (sequence, scores), sequence_indices)."""
    cfg = cfg or Config()
    levels = len(chains[0])
    by_seed: Dict[tuple, List[int]] = {}
    for i, sd in enumerate(seeds):
        by_seed.setdefault((sd is not None, sd or 0), []).append(i)
    work = [dict(members=by_seed[k], level=0, known=[None] * levels) for k in sorted(by_seed, reverse=True)]
    done = []
    while work:
        g = work.pop()
        if g["level"] == levels:
            done.append(g)
            continue
        lv = g["level"]
        d = dual_consensus([chains[i][lv] for i in g["members"]], [offsets[i][lv] for i in g["members"]], cfg)[0]
        if d["consensus2"] is not None:
            a = [i for i, first in zip(g["members"], d["is_consensus1"]) if first]
            b = [i for i, first in zip(g["members"], d["is_consensus1"]) if not first]
            work.append(dict(members=b, level=lv, known=[None] * levels))
            work.append(dict(members=a, level=lv, known=[None] * levels))
        else:
            g["known"][lv] = (d["consensus1"], list(d["scores1"]))
            g["level"] += 1
            work.append(g)
    done.sort(key=lambda g: g["members"][0])
    cons, idx = [], [0] * len(chains)
    for gi, g in enumerate(done):
        for lv in range(levels):
            if g["known"][lv] is None:
                g["known"][lv] = consensus([chains[i][lv] for i in g["members"]], [offsets[i][lv] for i in g["members"]], cfg)[0]
        cons.append([tuple(x) for x in g["known"]])
        for i in g["members"]:
            idx[i] = gi
    return cons, idx
