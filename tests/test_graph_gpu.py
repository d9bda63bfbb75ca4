"""GPU suite, row N3: K8 (sp_graph_align through the C++ host: VariantGraph::from_reference_variants, graph_edit_distance, the
walk back, graph_alleles) against the oracle (oracle/graph_oracle.py): same graph, same distance, same traversed nodes, same
allele vector -- and the hand-off to K6 (assign_haplotypes_from_alleles) end to end at CYP2D6 size."""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "oracle"))

import graph_oracle as go  # noqa: E402
import starphase_oracle as so  # noqa: E402
from test_graph_cpu import random_variants, rnd, spell  # noqa: E402

pytestmark = pytest.mark.gpu


def host_typing(bb, region_start, variants, seqs, band):
    from pb_starphase_b200 import _starphase_host as host

    gpu = host.GpuAligner(0)
    res, nodes, n2a, sink = host.graph_typing(gpu, bb.decode(), region_start, [(p, r.decode(), a.decode()) for p, r, a in variants],
                                              [s.decode() for s in seqs], band)
    return res, nodes, n2a, sink


def test_graph_and_alignment_vs_oracle_small():
    rng = np.random.default_rng(3)
    for case in range(40):
        bb = rnd(rng, int(rng.integers(5, 60)))
        variants = random_variants(rng, bb, 700, int(rng.integers(0, 6)))
        g = go.build_graph(bb, 700, variants)
        seqs = []
        for _ in range(3):
            s = bytearray(spell(rng, g)[1])
            for _ in range(int(rng.integers(0, 3))):
                if len(s) > 1:
                    q = int(rng.integers(0, len(s)))
                    s[q:q + 1] = [b"", b"N", s[q:q + 1] + b"C"][int(rng.integers(0, 3))]
            seqs.append(bytes(s))
        seqs.append(b"")
        for band in (4, 40):
            res, nodes, n2a, sink = host_typing(bb, 700, variants, seqs, band)
            assert [(n[0], list(n[1]), n[2]) for n in nodes] == [(g.seqs[k], g.preds[k], g.coord[k]) for k in range(len(g.seqs))], case
            assert {k: [tuple(x) for x in v] for k, v in n2a.items()} == g.node_to_alleles and sink == g.sink
            for s, (found, score, trav, alleles) in zip(seqs, res):
                want_score, want_nodes = go.align(g, s, band=band)
                assert found == (want_score < go.INF), (case, band)
                if found:
                    assert score == want_score and list(trav) == want_nodes, (case, band, s)
                    assert list(alleles) == so.alleles_from_traversal(len(variants), want_nodes, g.node_to_alleles)


def test_cyp2d6_sized_typing_and_k6_handoff():
    """A 6.2 kb backbone with 380 variant sites, consensuses carrying a known set of alleles plus HiFi-like errors: distance,
    traversed nodes and allele vectors equal the oracle's; the vectors then go through K6 (assign_haplotypes_from_alleles) and
    come back as the haplotype they were built from."""
    from pb_starphase_b200 import _starphase_host as host
    from pb_starphase_b200 import synth

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
    haps = {f"{h + 1}.001": [int(x) for x in (rng.random(len(variants)) < 0.03 * (h + 1))] for h in range(6)}
    seqs, truth = [], []
    for name, vec in haps.items():
        # spell the path that takes ALT where the haplotype says 1
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
        clean = b"".join(g.seqs[k] for k in path)
        noisy, _ = synth.hifi_reads(rng, [clean], 1, err=0.001, flank=0, lo=0, hi=1 << 20)
        seqs.append(noisy[0])
        truth.append(name)
    gpu = host.GpuAligner(0)
    res, nodes, n2a, sink = host.graph_typing(gpu, bb.decode(), 42_000_000, [(p, r.decode(), a.decode()) for p, r, a in variants],
                                              [s.decode() for s in seqs], 96)
    vectors = []
    for s, (found, score, trav, alleles) in zip(seqs, res):
        want_score, want_nodes = go.align(g, s, band=96)
        assert found and score == want_score and list(trav) == want_nodes
        assert list(alleles) == so.alleles_from_traversal(len(variants), want_nodes, g.node_to_alleles)
        vectors.append(list(alleles))
    # K6 hand-off: arg-max of (vi_match, all_match) over the haplotype definitions gives back the haplotype each consensus carries
    meta = [(f"rs{k}", k % 7 == 0) for k in range(len(variants))]
    out = host.assign_haplotypes_from_alleles(gpu, vectors, haps, meta, True)
    assert [o[0] for o in out] == truth
    for o, vec in zip(out, vectors):
        want = so.assign_haplotype_from_alleles(vec, haps, [m[0] for m in meta], [m[1] for m in meta], True)
        assert (o[0], tuple(o[2])) == (want[0], want[2])


def test_find_full_type_in_sequences_vs_oracle(oracle):
    """find_full_type_in_sequence end to end (src/cyp2d6/haplotyper.rs:326-361, :371-601): template search, consensus -> backbone
    mapping (K4 + K9), variant graph of the aligned stretch, K8, allele vector, K6 -- the C++ host against the same flow on
    oracle numbers; consensuses built from known haplotypes come back as those haplotypes."""
    import json

    import flow_oracle as fo
    from pb_starphase_b200 import _starphase_host as host
    from pb_starphase_b200 import synth

    c = synth.cyp2d6_diploid_sample(2001)
    templates = [(t, s, q) for (t, s), q in zip(c["template_labels"], c["templates"])]
    d6 = next(q for t, s, q in templates if t == "CYP2D6" and s is None)
    d7 = next(q for t, s, q in templates if t == "CYP2D7" and s is None)
    rng = np.random.default_rng(9)
    start = 42_100_000
    backbone = rnd(rng, 300) + d6 + rnd(rng, 300)
    pos = sorted(int(x) for x in rng.choice(np.arange(60, len(d6) - 60, 16), size=120, replace=False))
    variants = []
    for k, p in enumerate(pos):
        if k % 6 == 5:
            variants.append((start + 300 + p, d6[p:p + 3], d6[p:p + 1]))
        elif k % 6 == 4:
            variants.append((start + 300 + p, d6[p:p + 1], d6[p:p + 1] + b"TC"))
        else:
            variants.append((start + 300 + p, d6[p:p + 1], bytes([b"ACGT"[(b"ACGT".index(d6[p]) + 1 + k % 3) % 4]])))
    haps = {f"{h + 2}.001": [int(x) for x in (rng.random(len(variants)) < 0.03 * (h + 1))] for h in range(3)}
    haps["1.001"] = [0] * len(variants)
    seqs, truth = [], []
    for name, vec in haps.items():
        s = d6
        for (p, r, a), on in sorted(zip(variants, vec), reverse=True):
            if on:
                q = p - start - 300
                assert s[q:q + len(r)] == r
                s = s[:q] + a + s[q + len(r):]
        noisy, _ = synth.hifi_reads(rng, [s], 1, err=0.0005, flank=0, lo=0, hi=1 << 20)
        seqs.append(noisy[0])
        truth.append(("CYP2D6", name))
    seqs += [d7, rnd(rng, 3000), seqs[1][400:5200]]  # a D7 consensus, junk, an incomplete D6 consensus
    meta = [(f"rs{k}", k % 5 == 0) for k in range(len(variants))]
    mapped = [("CYP2D6", None), ("Hybrid", "CYP2D6::CYP2D7::exon9")]
    db = dict(backbone=backbone, backbone_start=start, variants=variants, metadata=meta, haplotype_lookup=haps, mapped_hybrids=mapped)
    want = fo.find_full_type_in_sequences(oracle, templates, seqs, 0.5, True, db, 96)
    gpu = host.GpuAligner(0)
    got = host.find_full_type_in_sequences(gpu, [(t, s, q.decode()) for t, s, q in templates], [s.decode() for s in seqs], 0.5, True,
                                           backbone.decode(), start, [(p, r.decode(), a.decode()) for p, r, a in variants], meta, haps, mapped, 96)
    assert len(got) == len(want) == len(seqs)
    for g, w in zip(got, want):
        if w is None:
            assert g is None
            continue
        assert (g[0], g[1]) == w[0]
        assert (json.loads(g[2]) if g[2] is not None else None) == w[1]
    assert [w[0] for w in want[:len(truth)]] == truth
    assert want[len(truth)][0] == ("CYP2D7", None) and want[len(truth) + 1] is None


def test_cyp2d6_consensus_stage_vs_oracle(oracle):
    """The consensus stage of the CYP2D6 caller (src/cyp2d6/caller.rs:145-310, :750-893) through the C++ host against the same flow
    on oracle numbers: the inputs the caller collects from the regions of interest (hpc_with_guide, offsets, seeds), the priority
    chain over them, and merge_consensus_results with every branch -- two consensuses with one HPC form and one type are re-solved
    as one (K7), a different type with the same HPC form stays apart, an untypable consensus joins its only typed HPC relative,
    is emptied when it has two, and stays an UNKNOWN pile when it has none."""
    import consensus_oracle as co
    import flow_oracle as fo
    from pb_starphase_b200 import _starphase_host as host
    from pb_starphase_b200 import synth
    from test_host_cpp_gpu import cyp_templates

    c = cyp_templates(seed=5, scale=240)
    templates = [(t, s, (seq if seq is not None else c["spacer" if t == "spacer" else "link"])) for t, s, seq in c["templates"]]
    cpp_templates = [(t, s, q.decode()) for t, s, q in templates]
    d6, d7 = c["d6"], c["d7"]
    rng = np.random.default_rng(31)
    gpu = host.GpuAligner(0)

    # -- hpc_with_guide: the reference's vector (src/util/homopolymers.rs:93-101) --
    assert host.hpc_with_guide("GAACCCGTTTT", "ATTGGGGGAACCCGTTTT", 6) == (b"GACGT", 2) == fo.hpc_with_guide(b"GAACCCGTTTT", b"ATTGGGGGAACCCGTTTT", 6)

    # -- the inputs of the priority chain: a full D6, a D6 whose first 90 template bases are clipped, a REP6, a mostly missing D7 --
    reads = {"m1/a": rnd(rng, 40) + c["rep6"] + d6 + rnd(rng, 30), "m1/b": d6[90:] + c["link"] + d7[:200]}
    n6, nr = len(d6), len(c["rep6"])
    roi = {"m1/a": [("REP6", None, 40, 40 + nr, (nr, 1, 0, 0, 0)), ("CYP2D6", None, 40 + nr, 40 + nr + n6, (n6, 2, 0, 0, 0))],
           "m1/b": [("CYP2D6", None, 0, n6 - 90, (n6, 0, 90, 90, 0)), ("CYP2D7", None, n6 - 90 + len(c["link"]), len(reads["m1/b"]), (len(d7), 0, len(d7) - 200, 0, len(d7) - 200))]}
    want_in = fo.cyp2d6_consensus_inputs(reads, roi, templates, 0.5)
    got_in = host.cyp2d6_consensus_inputs(gpu, {k: v.decode() for k, v in reads.items()}, roi, cpp_templates, 0.5)
    assert {k: list(got_in[k]) for k in want_in} == want_in
    assert want_in["seeds"] == [1, None, None] and want_in["base_offsets"] == [0, 0, 140]  # the clipped D6 may start 90 +- 50 into the consensus
    assert want_in["hpc_offsets"][2] == so.hpc_pos(d6, 90) + 50 and len(want_in["raw_sequences"]) == 3          # the D7 piece misses too much

    # -- the priority chain over such inputs (HPC level first, then the raw bases): three D6 reads, one of them clipped, and a REP6 --
    pr_reads = [d6, d6[90:], d6, c["rep6"]]
    chains = [[so.hpc(r), r] for r in pr_reads]
    offs = [[None, None], [so.hpc_pos(d6, 90) + 50, 140], [None, None], [None, None]]
    cfg = dict(allow_early_termination=True, offset_window=100, min_count=1)
    want_pc = co.priority_consensus(chains, offs, [None, None, None, 1], co.Config(**cfg))
    got_pc = host.priority_consensus(gpu, [[x.decode() for x in ch] for ch in chains], offs, [None, None, None, 1], cfg)
    assert list(got_pc[1]) == want_pc[1] == [0, 0, 0, 1]
    assert [[(s, list(sc)) for s, sc in lv] for lv in got_pc[0]] == [[(s, list(sc)) for s, sc in lv] for lv in want_pc[0]]
    assert want_pc[0][0][1][0] == d6 and want_pc[0][1][1][0] == c["rep6"]

    # -- merge_consensus_results --
    def dup(s, p):  # one more copy of base p: the homopolymer-compressed form stays the same
        return s[:p] + s[p:p + 1] + s[p:]

    def snv(s, p):
        return s[:p] + bytes([b"ACGT"[(b"ACGT".index(s[p]) + 1) % 4]]) + s[p + 1:]

    start, fl = 42_100_000, 100
    backbone = rnd(rng, fl) + d6 + rnd(rng, fl)
    p1, p2, p3, p4 = 120, 300, 470, 610  # V1, V2: homopolymer-length variants; V3: a substitution; p4: a length change the database does not know
    while d6[p3 - 1] == d6[p3] or d6[p3 + 1] == d6[p3] or snv(d6, p3)[p3] in (d6[p3 - 1], d6[p3 + 1]):
        p3 += 1
    variants = [(start + fl + p1, d6[p1:p1 + 1], d6[p1:p1 + 1] * 2), (start + fl + p2, d6[p2:p2 + 1], d6[p2:p2 + 1] * 2),
                (start + fl + p3, d6[p3:p3 + 1], snv(d6, p3)[p3:p3 + 1])]
    haps = {"1.001": [0, 0, 0], "2.001": [1, 0, 0], "3.001": [0, 1, 0], "4.001": [0, 1, 0], "5.001": [0, 0, 1]}  # *3.001 == *4.001: ambiguous
    meta = [("rs1", False), ("rs2", False), ("rs3", True)]
    mapped = [("CYP2D6", None)]
    db = dict(backbone=backbone, backbone_start=start, variants=variants, metadata=meta, haplotype_lookup=haps, mapped_hybrids=mapped)
    A, B = dup(d6, p1), d6
    fulls = [A, dup(A, p4), B, dup(d6, p2), rnd(rng, 500), d7, dup(snv(d6, p3), p2), snv(d6, p3)]
    assert len({so.hpc(x) for x in fulls[:4]}) == 1 and so.hpc(fulls[6]) == so.hpc(fulls[7]) != so.hpc(d6)
    sequences, offsets, raw_idx = [], [], []
    for gi, full in enumerate(fulls):
        noisy, _ = synth.hifi_reads(rng, [full], 3, err=0.003, flank=0, lo=0, hi=1 << 20)
        for k, r in enumerate(noisy):
            clipped = gi in (0, 7) and k == 2  # one read of two groups starts 60 bases into its region
            sequences.append(r[60:] if clipped else r)
            offsets.append(60 + 50 if clipped else 0)
            raw_idx.append(gi)
    raw = [[(so.hpc(full), [0, 0, 0]), (full, [1, 0, 2])] for full in fulls]
    raw[2][1] = (b"**" + B + b"*", [1, 0, 2])  # wildcards around a consensus are trimmed before typing
    want, want_idx = fo.merge_consensus_results(oracle, sequences, offsets, co.Config(**cfg), raw, raw_idx, templates, db, 0.1)
    got, got_idx = host.merge_consensus_results(gpu, [s.decode() for s in sequences], offsets, cfg, raw, raw_idx, cpp_templates, backbone.decode(), start,
                                                [(p, r.decode(), a.decode()) for p, r, a in variants], meta, haps, mapped, 0.1)
    assert list(got_idx) == want_idx
    assert [(s, list(sc)) for s, sc in got] == [(s, list(sc)) for s, sc in want]
    # what the branches must have done: groups 0 + 1 one consensus (= A, the majority), 2 alone, 3 emptied, 4 an unknown pile, 5 alone, 6 + 7 one
    assert want_idx[0] == want_idx[3] and want_idx[6] != want_idx[0] and want_idx[9] not in (want_idx[0], want_idx[6])
    assert want[want_idx[9]] == (b"", [0, 0, 0]) and want_idx[18] == want_idx[21] and len(want) == 6
    assert want[want_idx[6]][0] == b"**" + B + b"*" and want[want_idx[15]][0] == d7 and want[want_idx[12]][0] == fulls[4]
    assert want[want_idx[0]][0] in (A, dup(A, p4)) and want[want_idx[18]][0] in (fulls[6], fulls[7])


def graph_align_raw(problems, band, with_columns=True):
    """sp_graph_align through the C ABI on the oracle's linearisations: problems = [((chars, preds, diag, node_of, ends), seq)].
    Returns (status, scores, columns [total positions][2 band + 1] or None)."""
    import ctypes as C

    from pb_starphase_b200 import binding

    lib = binding.load_library()
    gch, goff, poff, preds, diag, eoff, ends, seqs, soff = [], [0], [0], [], [], [0], [], [], [0]
    for (chars, pr, dg, _, en), s in problems:
        gch += list(chars); goff.append(len(gch)); diag += dg
        for p in pr:
            preds += p; poff.append(len(preds))
        ends += en; eoff.append(len(ends))
        seqs += list(s); soff.append(len(seqs))
    a = lambda x, t: np.ascontiguousarray(x if len(x) else [0], dtype=t)  # noqa: E731
    gch_a, seq_a = a(gch, np.uint8), a(seqs, np.uint8)
    goff_a, soff_a = a(goff, np.int64), a(soff, np.int64)
    poff_a, preds_a, diag_a, eoff_a, ends_a = a(poff, np.int32), a(preds, np.int32), a(diag, np.int32), a(eoff, np.int32), a(ends, np.int32)
    score = np.full(len(problems), -7, dtype=np.int32)
    cols = np.full((max(len(gch), 1), 2 * band + 1), -7, dtype=np.int32) if with_columns else None
    ctx = binding.Context(0)
    st = lib.sp_graph_align(ctx._h, len(problems), gch_a.ctypes.data, goff_a.ctypes.data, poff_a.ctypes.data, preds_a.ctypes.data,
                            diag_a.ctypes.data, eoff_a.ctypes.data, ends_a.ctypes.data, seq_a.ctypes.data, soff_a.ctypes.data, band,
                            score.ctypes.data, cols.ctypes.data if cols is not None else None)
    ctx.close()
    return st, score, cols


@pytest.mark.parametrize("band", [1, 47, 48, 79, 80, 143, 144, 271])
def test_k8_columns_every_width(band):
    """K8 at both ends of its 3 / 5 / 9 / 17 cell classes: many random graphs in one call (several CTAs), every column cell
    -- INF included -- and every score against graph_oracle.forward.  Includes an empty sequence and one the band shuts out of
    every path; with columns = NULL the scores stay the same."""
    rng = np.random.default_rng(700 + band)
    problems = []
    for case in range(64):
        # every fourth graph is longer than the band, so that the top band cells (lane 0) hold rows of the matrix
        bb = rnd(rng, int(rng.integers(band + 20, band + 90) if case % 4 == 3 else rng.integers(3, 90)))
        g = go.build_graph(bb, 500, random_variants(rng, bb, 500, int(rng.integers(0, 7))))
        s = bytearray(spell(rng, g)[1])
        for _ in range(int(rng.integers(0, 6))):
            if len(s) > 1:
                q = int(rng.integers(0, len(s)))
                s[q:q + 1] = [b"", b"N", s[q:q + 1] + b"T", b"G"][int(rng.integers(0, 4))]
        if case == 5:
            s = b""
        elif case == 9:
            s = bytes(s) + rnd(rng, band + 60)  # longer than every path by more than the band: no path reaches row m
        problems.append((g, bytes(s)))
    want = [go.forward(g, s, band) for g, s in problems]
    st, score, cols = graph_align_raw([(w[0], s) for w, (_, s) in zip(want, problems)], band)
    assert st == 0
    assert score.tolist() == [w[2] for w in want]
    assert want[9][2] == go.INF
    nb, row = 2 * band + 1, 0
    for (lin, oc, _), (_, s) in zip(want, problems):
        for q, d in enumerate(lin[2]):
            exp = [oc[q].get(d - band + k, go.INF) for k in range(nb)]
            assert cols[row].tolist() == exp, (band, q)
            row += 1
    assert row == len(cols) or (row == 0 and len(cols) == 1)
    st2, score2, _ = graph_align_raw([(w[0], s) for w, (_, s) in zip(want, problems)], band, with_columns=False)
    assert st2 == 0 and score2.tolist() == score.tolist()


def test_k8_refuses_band_272():
    g = go.build_graph(b"ACGTACGT", 0, [])
    lin, _, _ = go.forward(g, b"ACGT", 8)
    assert graph_align_raw([(lin, b"ACGT")], 271)[0] == 0
    assert graph_align_raw([(lin, b"ACGT")], 272)[0] == 1  # SP_ERR_INVALID
