"""CPU suite: the consensus oracle (oracle/consensus_oracle.py, row N1) holds the properties that pin it -- waffle_con itself
cannot be run here (parity unpinned): error-free reads give back their source, a majority out-votes HiFi-like errors, two
alleles come back as a dual consensus with the right read split, reads with offsets assemble a longer consensus."""
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "oracle"))

import consensus_oracle as co  # noqa: E402
from pb_starphase_b200 import synth  # noqa: E402


def rnd(rng, n):
    return bytes(rng.choice(list(b"ACGT"), n).tolist())


def het_pair(rng, n, sites):
    a = rnd(rng, n)
    b = bytearray(a)
    for p in sites:
        b[p] = ord("A") if b[p] != ord("A") else ord("C")
    return a, bytes(b)


def test_error_free_reads_give_back_the_source():
    rng = np.random.default_rng(1)
    src = rnd(rng, 240)
    res = co.consensus([src] * 5)
    assert len(res) == 1 and res[0][0] == src and res[0][1] == [0] * 5
    dual = co.dual_consensus([src] * 5)
    assert len(dual) == 1 and dual[0]["consensus1"] == src and dual[0]["consensus2"] is None


def test_majority_outvotes_errors():
    rng = np.random.default_rng(2)
    src = rnd(rng, 300)
    reads, _ = synth.hifi_reads(rng, [src], 12, err=0.01, flank=0, lo=0, hi=1 << 20)
    res = co.consensus(reads)
    assert res[0][0] == src
    assert res[0][1] == [co.extend([r], [0], co.Config(band=64), co.Track(1), 0)[1][0] * 0 + s for r, s in zip(reads, res[0][1])]  # scores are per read
    assert sum(res[0][1]) > 0  # the reads do carry errors


def test_two_alleles_come_back_as_a_dual_consensus():
    rng = np.random.default_rng(3)
    a, b = het_pair(rng, 320, (40, 170, 290))
    ra, _ = synth.hifi_reads(rng, [a], 7, err=0.004, flank=0, lo=0, hi=1 << 20)
    rb, _ = synth.hifi_reads(rng, [b], 6, err=0.004, flank=0, lo=0, hi=1 << 20)
    reads = [x for pair in zip(ra, rb) for x in pair] + ra[6:]
    truth = [True, False] * 6 + [True]
    d = co.dual_consensus(reads)[0]
    assert {d["consensus1"], d["consensus2"]} == {a, b}
    first_is_a = d["consensus1"] == a
    assert d["is_consensus1"] == [t == first_is_a for t in truth]
    # a single allele with one odd read stays single: the minor side would have fewer than min_count reads
    d = co.dual_consensus(ra + rb[:1])[0]
    assert d["consensus2"] is None and d["consensus1"] == a


def test_offsets_assemble_partial_reads():
    """src/hla/caller.rs:1150-1219: reads that start later carry an offset (add_sequence_offset) and may end early."""
    rng = np.random.default_rng(4)
    src = rnd(rng, 400)
    reads = [src[:300], src[:320], src[:310], src[100:], src[120:], src[90:], src[:400]]
    offsets = [None, None, None, 100, 120, 90, None]
    res = co.consensus(reads, offsets, co.Config(allow_early_termination=True))
    assert res[0][0] == src and res[0][1] == [0] * 7
    # an offset that is 15 bases off is absorbed by the window
    offsets[3] = 115
    res = co.consensus(reads, offsets, co.Config(allow_early_termination=True, offset_window=40))
    assert res[0][0] == src and res[0][1] == [0] * 7


def test_priority_consensus_groups_by_source():
    """The priority chain (HPC first, then raw): sources that differ only in a homopolymer length are split at the second level,
    a seeded input never joins the others, wildcards cost nothing."""
    sys.path.insert(0, str(ROOT / "tests"))
    import starphase_oracle as so
    from test_consensus_gpu import priority_case

    sources, chains, offsets, seeds, truth = priority_case(np.random.default_rng(21))
    cons, idx = co.priority_consensus(chains, offsets, seeds)
    assert len(cons) == 4 and [idx[k] for k in range(4)] == [0, 1, 2, 3]
    for k, g in enumerate(idx):
        assert g == idx[k % 4] and cons[g][1][0] == sources[truth[k]] and cons[g][0][0] == so.hpc(sources[truth[k]])
        assert cons[g][1][1] == [0] * 5
    # a read whose first 40 bases are wildcards votes with the rest and costs nothing
    src = sources[0]
    res = co.consensus([src, src, src, b"*" * 40 + src[40:]])
    assert res[0][0] == src and res[0][1] == [0, 0, 0, 0]


def _root(reads, offsets, cfg):
    t, e, v, f = co.extend(reads, offsets, cfg, co.Track(len(reads)), 0)
    return t, (e, v, f)


def test_run_spells_error_free_reads_and_stops_when_they_are_consumed():
    """co.run (the restatement of sp_consensus_run): error-free reads of one source spell it, one round per base, and the run
    stops when every read is consumed (nobody votes any more)."""
    rng = np.random.default_rng(11)
    src = rnd(rng, 150)
    reads, offsets, cfg = [src] * 4 + [src[:70]], [-1] * 5, co.Config(band=8)
    t, st = _root(reads, offsets, cfg)
    tracks, state, steps, costs = co.run(reads, offsets, cfg, [t], [st], 3, 100, 1 << 40, 0, 1 << 40, 10_000)
    assert bytes(b"ACGT"[s & 15] for s in steps) == src and all(s >> 4 == 15 for s in steps)
    assert tracks[0].length == len(src) and costs == [0] * (len(src) + 1)
    e, v, f = state[0]
    assert f == [0] * 5 and e == [0] * 4 + [co.INF]  # the short read left the band long ago: consumed, its cost is `full`
    assert all(x == co.VOTE_FINISHED for x in v[:4]) and v[4] == 0


def test_run_single_side_stops_at_the_first_het_site():
    rng = np.random.default_rng(12)
    a, b = het_pair(rng, 200, (57, 120))
    reads, offsets, cfg = [a] * 4 + [b] * 4, [-1] * 8, co.Config(band=16)
    t, st = _root(reads, offsets, cfg)
    tracks, state, steps, _ = co.run(reads, offsets, cfg, [t], [st], 3, 100, 1 << 40, 0, 1 << 40, 10_000)
    assert len(steps) == 57 and bytes(b"ACGT"[s & 15] for s in steps) == a[:57]
    assert sorted(co.passing(co.tally(*state[0]), co.Config(min_count=3, min_af=0.1))) == sorted(b"ACGT".index(x) for x in {a[57], b[57]})
    # a dual node split at the site goes on past it, every read on its own side
    ta, ea, va, fa = co.extend(reads, offsets, cfg, tracks[0], a[57])
    tb, eb, vb, fb = co.extend(reads, offsets, cfg, tracks[0], b[57])
    tr, _, steps2, _ = co.run(reads, offsets, cfg, [ta, tb], [(ea, va, fa), (eb, vb, fb)], 3, 100, 1 << 40, 0, 1 << 40, 10_000)
    assert len(steps2) == 200 - 58 and tr[0].length == tr[1].length == 200


def test_run_chained_equals_one_run():
    rng = np.random.default_rng(13)
    src = rnd(rng, 160)
    reads, _ = synth.hifi_reads(rng, [src], 7, err=0.01, flank=0, lo=0, hi=1 << 20)
    offsets, cfg = [-1] * 7, co.Config(band=12)
    t, st = _root(reads, offsets, cfg)
    whole = co.run(reads, offsets, cfg, [t], [st], 3, 100, 1 << 40, 0, 1 << 40, 90)
    first = co.run(reads, offsets, cfg, [t], [st], 3, 100, 1 << 40, 0, 1 << 40, 35)
    second = co.run(reads, offsets, cfg, first[0], first[1], 3, 100, 1 << 40, 0, 1 << 40, 55)
    assert len(whole[2]) == 90 and first[2] + second[2] == whole[2]
    assert second[1] == whole[1] and second[0][0].cols == whole[0][0].cols and second[0][0].best_full == whole[0][0].best_full
    # the limits cut at the step the cost trajectory says: the first node whose cost reaches the limit is not extended
    costs = whole[3]
    q = next(k for k in range(1, 90) if costs[k] > costs[0])
    cut = co.run(reads, offsets, cfg, [t], [st], 3, 100, costs[q], 1 << 40, 1 << 40, 90)
    assert len(cut[2]) == q
