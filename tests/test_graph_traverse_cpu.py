"""CPU suite: graph_walk.traverse, the walk back that sp_graph_traverse (K8's marking pass) is checked against.  On small random
graphs its positions, mapped to nodes, are align's nodes and brute force's nodes, and they are exactly the positions of the nodes
on some optimal source -> sink path."""
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "oracle"))

import graph_oracle as go  # noqa: E402
import graph_walk as gw  # noqa: E402
from test_graph_cpu import random_variants, rnd, spell  # noqa: E402


def paths(g: go.Graph):
    out = []

    def walk(node, acc):
        acc = acc + [node]
        if node == g.sink:
            out.append(acc)
            return
        for k, pr in enumerate(g.preds):
            if node in pr:
                walk(k, acc)

    walk(0, [])
    return out


def edit_distance(a: bytes, b: bytes) -> int:
    prev = list(range(len(b) + 1))
    for i, ca in enumerate(a, 1):
        cur = [i]
        for j, cb in enumerate(b, 1):
            cur.append(min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (0 if ca == cb and ca in b"ACGT" else 1)))
        prev = cur
    return prev[-1]


def test_traverse_positions_are_the_optimal_paths():
    rng = np.random.default_rng(11)
    for case in range(120):
        bb = rnd(rng, int(rng.integers(4, 30)))
        g = go.build_graph(bb, 300, random_variants(rng, bb, 300, int(rng.integers(0, 5))))
        seq = bytearray(spell(rng, g)[1])
        for _ in range(int(rng.integers(0, 4))):
            if len(seq) > 1:
                q = int(rng.integers(0, len(seq)))
                seq[q:q + 1] = [b"", b"N", seq[q:q + 1] + b"A", bytes([b"ACGT"[(b"ACGTN".index(seq[q]) + 1) % 4]])][int(rng.integers(0, 4))]
        if case % 10 == 7:
            seq = bytearray()
        seq = bytes(seq)
        score, lin, positions = gw.traverse(g, seq)
        node_of = lin[3]
        assert positions == sorted(set(positions))
        want_score, want_nodes = go.brute_force(g, seq)
        assert score == want_score, case
        assert sorted({node_of[q] for q in positions}) == want_nodes == go.align(g, seq)[1], case
        # every marked position lies on a path whose cost is the score, and every position of such a path is marked
        cost = {}
        for p in paths(g):
            c = edit_distance(b"".join(g.seqs[k] for k in p), seq)
            for k in p:
                cost[k] = min(cost.get(k, go.INF), c)
        assert all(cost[node_of[q]] == score for q in positions), case
        assert positions == [q for q, k in enumerate(node_of) if cost[k] == score], case


def test_traverse_unreachable_marks_nothing():
    g = go.build_graph(b"ACGTACGTAC", 0, [(3, b"T", b"G")])
    score, lin, positions = gw.traverse(g, b"ACGTACGTAC" + b"A" * 20, band=4)
    assert score == go.INF and positions == [] and len(lin[0]) == 11
    assert go.align(g, b"ACGTACGTAC" + b"A" * 20, band=4) == (go.INF, [])


def test_traverse_marks_both_branches_of_a_tie():
    # the sequence deletes the variant base: REF and ALT cost the same, so both branches carry marks
    bb = b"ACGTACGTTTGACCAGTACCGGTTAACGT"
    g = go.build_graph(bb, 100, [(112, b"C", b"G")])
    score, lin, positions = gw.traverse(g, bb[:12] + bb[13:])
    assert score == 1
    assert {lin[3][q] for q in positions} == set(range(1, len(g.seqs)))
