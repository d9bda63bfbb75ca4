"""GPU suite, row N3: sp_graph_traverse (K8 forward + k8_graph_mark) through the C ABI.  Scores and on_path bit for bit against
graph_walk.traverse, and against the walk back over sp_graph_align's own columns (what graph_edit_distance did on the host
before the marking pass moved to the device), at both ends of every CELLS class, on random graphs with the shapes the kernel
treats differently, with unreachable problems mixed in, with more problems than resident warps, and at CYP2D6 size."""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "oracle"))

import graph_oracle as go  # noqa: E402
import graph_walk as gw  # noqa: E402
from test_graph_cpu import random_variants, rnd, spell  # noqa: E402

pytestmark = pytest.mark.gpu

SP_ERR_INVALID = 1


def pack(problems):
    """problems = [(linearisation, seq)] -> the C ABI arrays (empty arrays padded to one element)."""
    gch, goff, poff, preds, diag, eoff, ends, seqs, soff = [], [0], [0], [], [], [0], [], [], [0]
    for (chars, pr, dg, _, en), s in problems:
        gch += list(chars); goff.append(len(gch)); diag += dg
        for p in pr:
            preds += p; poff.append(len(preds))
        ends += en; eoff.append(len(ends))
        seqs += list(s); soff.append(len(seqs))
    a = lambda x, t: np.ascontiguousarray(x if len(x) else [0], dtype=t)  # noqa: E731
    return dict(gch=a(gch, np.uint8), goff=a(goff, np.int64), poff=a(poff, np.int32), preds=a(preds, np.int32), diag=a(diag, np.int32),
                eoff=a(eoff, np.int32), ends=a(ends, np.int32), seqs=a(seqs, np.uint8), soff=a(soff, np.int64), npos=len(gch))


def call(fn, arrays, n, band, out, with_out=True):
    from pb_starphase_b200 import binding

    lib = binding.load_library()
    x = arrays
    score = np.full(max(n, 1), -7, dtype=np.int32)
    ctx = binding.Context(0)
    st = getattr(lib, fn)(ctx._h, n, x["gch"].ctypes.data, x["goff"].ctypes.data, x["poff"].ctypes.data, x["preds"].ctypes.data,
                          x["diag"].ctypes.data, x["eoff"].ctypes.data, x["ends"].ctypes.data, x["seqs"].ctypes.data, x["soff"].ctypes.data,
                          band, score.ctypes.data, out.ctypes.data if with_out else None)
    ctx.close()
    return st, score[:n]


def traverse_raw(problems, band, with_on_path=True):
    x = pack(problems)
    on_path = np.full(max(x["npos"], 1), 7, dtype=np.uint8)
    st, score = call("sp_graph_traverse", x, len(problems), band, on_path, with_on_path)
    return st, score, on_path[:x["npos"]]


def align_raw(problems, band):
    x = pack(problems)
    cols = np.full((max(x["npos"], 1), 2 * band + 1), -7, dtype=np.int32)
    st, score = call("sp_graph_align", x, len(problems), band, cols)
    return st, score, cols


def walk_columns(lin, seq, cols, band, score):
    """The walk back over one problem's sp_graph_align columns, as graph_edit_distance did it on the host: marked positions."""
    chars, preds, diag, _, ends = lin
    m, nb = len(seq), 2 * band + 1

    def at(q, i):
        if i < 0 or i > m:
            return go.INF
        if q < 0:
            return i if i <= band else go.INF
        k = i - diag[q] + band
        return int(cols[q][k]) if 0 <= k < nb else go.INF

    def sub(q, i):
        g, c = chars[q], seq[i - 1]
        return 0 if g in b"ACGTacgt" and (g & ~0x20) == (c & ~0x20) else 1

    marked = set()
    if score >= go.INF:
        return marked
    stack = [(e, m) for e in ends if at(e, m) == score]
    while stack:
        q, i = stack.pop()
        if q < 0 or (q, i) in marked:
            continue
        marked.add((q, i))
        v = at(q, i)
        if i > 0 and at(q, i - 1) < go.INF and at(q, i - 1) + 1 == v:
            stack.append((q, i - 1))
        for pr in preds[q]:
            if at(pr, i) < go.INF and at(pr, i) + 1 == v:
                stack.append((pr, i))
            if i > 0 and at(pr, i - 1) < go.INF and at(pr, i - 1) + sub(q, i) == v:
                stack.append((pr, i - 1))
    return {q for q, _ in marked}


def upper(g: go.Graph) -> go.Graph:
    """graph_code_of folds case and sends every other character to a code that never matches: the oracle compares upper case."""
    return go.Graph([s.upper() for s in g.seqs], g.preds, g.coord, g.node_to_alleles, g.sink)


def oracle(g, seq, band):
    """(score, linearisation of g as the kernel gets it, on_path) from graph_walk.traverse."""
    score, lin, positions = gw.traverse(upper(g), seq.upper(), band)
    on = np.zeros(len(lin[0]), dtype=np.uint8)
    on[positions] = 1
    return score, go.linearise(g), on


def mutate(rng, s, band):
    s = bytearray(s)
    for _ in range(int(rng.integers(0, 6))):
        if len(s) > 1:
            q = int(rng.integers(0, len(s)))
            s[q:q + 1] = [b"", b"N", s[q:q + 1] + b"T", b"g", s[q:q + 1].lower()][int(rng.integers(0, 5))]
    return bytes(s)


def random_problem(rng, band, case):
    """One (graph, sequence) problem; `case` picks the shape."""
    kind = case % 8
    if kind == 0:  # a bubble whose two branches are equally good: the sequence drops the variant base
        bb = rnd(rng, int(rng.integers(12, 60)))
        p = int(rng.integers(3, len(bb) - 3))
        alt = bytes([b"ACGT"[(b"ACGT".index(bb[p]) + 1) % 4]])
        g = go.build_graph(bb, 100, [(100 + p, bb[p:p + 1], alt)])
        return g, bb[:p] + bb[p + 1:]
    if kind == 1:  # one site with many branches: the node after it has many predecessors
        bb = rnd(rng, int(rng.integers(10, 50)))
        p = int(rng.integers(1, len(bb) - 4))
        vs = [(200 + p, bb[p:p + 1], bb[p:p + 1] + rnd(rng, k)) for k in range(1, 7)] + [(200 + p, bb[p:p + 3], bb[p:p + 1])]
        g = go.build_graph(bb, 200, vs)
        return g, mutate(rng, spell(rng, g)[1], band)
    if kind == 2:  # single-character nodes: substitutions one base apart
        bb = rnd(rng, int(rng.integers(8, 40)))
        vs = [(300 + p, bb[p:p + 1], bytes([b"ACGT"[(b"ACGT".index(bb[p]) + 2) % 4]])) for p in range(1, len(bb) - 1, 2)]
        g = go.build_graph(bb, 300, vs)
        return g, mutate(rng, spell(rng, g)[1], band)
    if kind == 3:  # long in-node runs: nodes far longer than the band, so the band crosses every lane boundary
        bb = rnd(rng, int(rng.integers(band + 40, 2 * band + 120)))
        g = go.build_graph(bb, 0, random_variants(rng, bb, 0, int(rng.integers(0, 3))))
        return g, mutate(rng, spell(rng, g)[1], band)
    if kind == 4:  # ends that include -1: the sink can be reached straight from the empty source
        g = go.Graph()
        src = g.add(b"", [], 0)
        a = g.add(rnd(rng, int(rng.integers(1, 12))), [src], 0)
        b = g.add(rnd(rng, int(rng.integers(1, 12))), [a], len(g.seqs[a]))
        g.sink = g.add(b"", [src, b], len(g.seqs[a]) + len(g.seqs[b]))
        seq = [b"", g.seqs[a] + g.seqs[b], g.seqs[a][:1], rnd(rng, 3)][int(rng.integers(0, 4))]
        return g, seq
    if kind == 5:  # empty sequence
        bb = rnd(rng, int(rng.integers(1, min(band, 40) + 2)))
        return go.build_graph(bb, 0, random_variants(rng, bb, 0, int(rng.integers(0, 3)))), b""
    if kind == 6:  # non-ACGT and lower-case graph characters
        bb = rnd(rng, int(rng.integers(6, 60)))
        g = go.build_graph(bb, 0, random_variants(rng, bb, 0, int(rng.integers(0, 5))))
        s = spell(rng, g)[1]
        for k in range(len(g.seqs)):
            if g.seqs[k] and rng.random() < 0.5:
                node = bytearray(g.seqs[k])
                q = int(rng.integers(0, len(node)))
                node[q] = [ord("N"), ord("n"), ord("R"), node[q] | 0x20][int(rng.integers(0, 4))]
                g.seqs[k] = bytes(node)
        return g, mutate(rng, s, band)
    bb = rnd(rng, int(rng.integers(3, 90)))
    g = go.build_graph(bb, 500, random_variants(rng, bb, 500, int(rng.integers(0, 7))))
    return g, mutate(rng, spell(rng, g)[1], band)


def cells_class(band):
    c = -(-(2 * band + 1) // 32)
    return 3 if c <= 3 else 5 if c <= 5 else 9 if c <= 9 else 17


def check(problems, band):
    """sp_graph_traverse on `problems` = [(graph, seq)] against the oracle and against the walk over sp_graph_align's columns."""
    want = [oracle(g, s, band) for g, s in problems]
    lins = [(w[1], s) for w, (_, s) in zip(want, problems)]
    st, score, on_path = traverse_raw(lins, band)
    assert st == 0
    assert score.tolist() == [w[0] for w in want]
    assert on_path.tolist() == [int(x) for w in want for x in w[2]]
    st2, score2, cols = align_raw(lins, band)
    assert st2 == 0 and score2.tolist() == score.tolist()
    row = 0
    for (lin, s), sc in zip(lins, score2.tolist()):
        n = len(lin[0])
        walked = walk_columns(lin, s, cols[row:row + n], band, sc)
        assert on_path[row:row + n].tolist() == [int(q in walked) for q in range(n)]
        row += n
    return score, on_path


@pytest.mark.parametrize("band,cells", [(1, 3), (47, 3), (48, 5), (79, 5), (80, 9), (143, 9), (144, 17), (271, 17)])
def test_traverse_every_width(band, cells):
    """64 random graphs per call at both ends of the 3 / 5 / 9 / 17 cell classes; problems the band shuts out are mixed in."""
    assert cells_class(band) == cells
    rng = np.random.default_rng(900 + band)
    problems = []
    for case in range(64):
        g, s = random_problem(rng, band, case)
        if case % 16 == 15:
            s = spell(rng, g)[1] + rnd(rng, band + 60)  # longer than every path by more than the band: unreachable
        problems.append((g, s))
    score, on_path = check(problems, band)
    assert sum(x >= go.INF for x in score.tolist()) >= 4 and 0 < int(on_path.sum()) < len(on_path)


def test_traverse_both_branches_of_a_tie_marked():
    bb = b"ACGTACGTTTGACCAGTACCGGTTAACGT"
    g = go.build_graph(bb, 100, [(112, b"C", b"G")])
    score, on_path = check([(g, bb[:12] + bb[13:])], 16)
    lin = go.linearise(g)
    assert score.tolist() == [1] and {lin[3][q] for q in np.flatnonzero(on_path)} == {1, 2, 3, 4}


def test_traverse_more_problems_than_resident_warps():
    """4,096 small problems in one call (more warps than 148 SMs hold at once), unreachable ones interleaved: no problem's marks
    reach another's positions."""
    rng = np.random.default_rng(77)
    problems = []
    for case in range(4096):
        bb = rnd(rng, int(rng.integers(2, 14)))
        g = go.build_graph(bb, 0, random_variants(rng, bb, 0, int(rng.integers(0, 3))))
        s = spell(rng, g)[1]
        problems.append((g, s + rnd(rng, 12) if case % 3 == 1 else mutate(rng, s, 4)))
    score, on_path = check(problems, 4)
    assert int((score >= go.INF).sum()) > 1000


def cyp2d6_problems():
    rng = np.random.default_rng(4)
    bb = rnd(rng, 6200)
    pos = sorted(int(x) for x in rng.choice(np.arange(20, 6150, 14), size=380, replace=False))
    variants = []
    for k, p in enumerate(pos):
        if k % 5 == 4:
            variants.append((42_000_000 + p, bb[p:p + 3], bb[p:p + 1]))
        elif k % 5 == 3:
            variants.append((42_000_000 + p, bb[p:p + 1], bb[p:p + 1] + b"GA"))
        else:
            variants.append((42_000_000 + p, bb[p:p + 1], bytes([b"ACGT"[(b"ACGT".index(bb[p]) + 1 + k % 3) % 4]])))
    g = go.build_graph(bb, 42_000_000, variants)
    from pb_starphase_b200 import synth

    seqs = []
    for h in range(6):
        vec = [int(x) for x in (rng.random(len(variants)) < 0.03 * (h + 1))]
        path, cur = [0], 0
        while cur != g.sink:
            succ = [k for k, pr in enumerate(g.preds) if cur in pr]
            pick = succ[0]
            for k in succ:
                lab = g.node_to_alleles.get(k)
                if lab and all(vec[v] == a for v, a in lab):
                    pick = k
            path.append(pick)
            cur = pick
        noisy, _ = synth.hifi_reads(rng, [b"".join(g.seqs[k] for k in path)], 1, err=0.001, flank=0, lo=0, hi=1 << 20)
        seqs.append(noisy[0])
    return [(g, s) for s in seqs]


@pytest.mark.parametrize("band", [64, 128])
def test_traverse_cyp2d6_sized(band):
    """Six 6.2 kb consensuses on a backbone with 380 variant sites, one call."""
    problems = cyp2d6_problems()
    score, on_path = check(problems, band)
    assert all(x < go.INF for x in score.tolist())


def test_traverse_refusals():
    g = go.build_graph(b"ACGTACGT", 0, [])
    lin = go.linearise(g)
    assert traverse_raw([(lin, b"ACGT")], 1)[0] == 0
    assert traverse_raw([(lin, b"ACGT")], 271)[0] == 0
    assert traverse_raw([(lin, b"ACGT")], 0)[0] == SP_ERR_INVALID
    assert traverse_raw([(lin, b"ACGT")], 272)[0] == SP_ERR_INVALID
    assert traverse_raw([(lin, b"ACGT")], 8, with_on_path=False)[0] == SP_ERR_INVALID
    empty = go.linearise(go.build_graph(b"", 0, []))
    st, score, _ = traverse_raw([(empty, b"")], 8, with_on_path=False)  # no positions: on_path may be NULL
    assert empty[4] == [-1] and st == 0 and score.tolist() == [0]
    x = pack([(lin, b"ACGT"), (lin, b"ACG")])
    on = np.zeros(x["npos"], dtype=np.uint8)
    bad = dict(x, eoff=np.ascontiguousarray([0, 1, 1], dtype=np.int32))  # the second problem has no end
    assert call("sp_graph_traverse", bad, 2, 8, on)[0] == SP_ERR_INVALID
    bad = dict(x, goff=np.ascontiguousarray([1, 8, 16], dtype=np.int64))  # offsets must start at 0
    assert call("sp_graph_traverse", bad, 2, 8, on)[0] == SP_ERR_INVALID
    bad = dict(x, preds=np.ascontiguousarray([5] + x["preds"].tolist()[1:], dtype=np.int32))  # a predecessor that comes later
    assert call("sp_graph_traverse", bad, 2, 8, on)[0] == SP_ERR_INVALID


def test_context_graph_traverse():
    """binding.Context.graph_traverse returns the same (scores, on_path) as the raw call."""
    from pb_starphase_b200 import binding

    rng = np.random.default_rng(5)
    problems = [random_problem(rng, 24, case) for case in range(16)]
    lins = [(go.linearise(g), s) for g, s in problems]
    x = pack(lins)
    with binding.Context(0) as ctx:
        scores, on_path = ctx.graph_traverse(b"".join(lin[0] for lin, _ in lins), x["goff"], x["poff"], x["preds"], x["diag"], x["eoff"],
                                             x["ends"], b"".join(s for _, s in lins), x["soff"], 24)
    st, want_scores, want_on = traverse_raw(lins, 24)
    assert st == 0 and scores.tolist() == want_scores.tolist() and on_path.tolist() == want_on.tolist()
