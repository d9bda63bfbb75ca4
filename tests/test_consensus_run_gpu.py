"""GPU suite, row N1: K7's on-device loop (sp_consensus_run, `k7_run`) at every cluster shape and item count, and K7's extension
step (`k7_extend`) at every compiled band width, against the oracle (oracle/consensus_oracle.py: `run` and `extend`), bit for bit.

k7_run deals items -- (read, side) pairs -- round-robin over the 16 warps of each CTA of one cluster; a warp owns ceil(items /
warps) shared-memory slots, each with a u16 DP column and a ring of read codes refilled 32 bases at a time; per-read results go
to every CTA through distributed shared memory.  Every k7_run test first asserts the shape it exists for (cluster size, items
per warp), then compares the step log, the returned node state and the handed-back tracks: a report-only extension of every
destination track and one extension by each of A / C / G / T pin the whole column, best_full and the track length."""
import ctypes as C
import os
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "oracle"))

import consensus_oracle as co  # noqa: E402
from pb_starphase_b200 import synth  # noqa: E402
from test_consensus_cpu import rnd  # noqa: E402

pytestmark = pytest.mark.gpu
SKIP_LARGE = pytest.mark.skipif(os.environ.get("SP_SKIP_LARGE") == "1", reason="large case skipped")

WARPS = 16  # k7_run: 512 threads per CTA
BIG = 1 << 40  # a limit that never binds
SP_ERR_INVALID, SP_ERR_RANGE = 1, 5


def plan(items, force=None):
    """plan_run's shape (sp_consensus.cu): the smallest power of two n_cta with n_cta x 16 warps >= items, at most 8, unless
    SP_K7_RUN_CTAS forces it; then items per warp."""
    n_cta = 1
    while n_cta < 8 and n_cta * WARPS < items:
        n_cta *= 2
    if force is not None:
        n_cta = max(1, min(8, force))
    return n_cta, -(-items // (WARPS * n_cta))


def cells_of(W):
    """k7_run's CELLS class: band cells per lane rounded up to 2 / 4 / 8 / 16."""
    nb = 2 * W + 1
    return 2 if nb < 64 else 4 if nb < 128 else 8 if nb < 256 else 16


class Mirror:
    """A K7 handle and the oracle's copy of its tracks; every extension is compared on the way."""

    def __init__(self, ctx, reads, offsets, band, window, max_tracks=16):
        import pb_starphase_b200 as sp

        self.reads, self.offsets = list(reads), list(offsets)
        self.cfg = co.Config(band=band, offset_window=window)
        self.W = band + window // 2
        self.gpu = sp.Consensus(ctx, self.reads, self.offsets, offset_window=window, band=band, max_tracks=max_tracks)
        self.tr = {}

    def extend(self, src, symbols, dst):
        ed, votes, full = self.gpu.extend(src, symbols, dst)
        out = []
        for q, (s, y, d) in enumerate(zip(src, symbols, dst)):
            t, e, v, f = co.extend(self.reads, self.offsets, self.cfg, self.tr[s], y)
            assert ed[q].tolist() == e and votes[q].tolist() == v and full[q].tolist() == f, (s, y, d)
            out.append((t, (e, v, f)))
        for d, (t, _) in zip(dst, out):
            self.tr[d] = t
        return [st for _, st in out]

    def fresh(self, track):
        """Track `track` = the empty consensus; returns its state (the report of column 0)."""
        self.gpu.reset(track)
        self.tr[track] = co.Track(len(self.reads))
        return self.extend([track], [0], [track])[0]

    def grow(self, track, seq):
        st = self.fresh(track)
        for b in seq:
            st = self.extend([track], [b], [track])[0]
        return st

    def run(self, src, dst, state, min_count=3, permille=100, cost_limit=BIG, size_limit=0, cost_cap=BIG, max_steps=10_000,
            scratch=(12, 13, 14, 15)):
        """sp_consensus_run against co.run: steps, node state, and the destination tracks through follow-on extensions.
        Returns (n_steps, the oracle's per-decision costs, the state of the last node)."""
        n = len(src)
        ed = np.array([s[0] for s in state], dtype=np.int32)
        votes = np.array([s[1] for s in state], dtype=np.uint8)
        full = np.array([s[2] for s in state], dtype=np.int32)
        keep = (ed.copy(), votes.copy(), full.copy())
        e, v, f, steps = self.gpu.run(src, dst, ed, votes, full, min_count, permille, cost_limit, size_limit, cost_cap, max_steps)
        assert np.array_equal(ed, keep[0]) and np.array_equal(votes, keep[1]) and np.array_equal(full, keep[2])
        tracks, ost, osteps, costs = co.run(self.reads, self.offsets, self.cfg, [self.tr[s] for s in src], state, min_count, permille,
                                            cost_limit, size_limit, cost_cap, max_steps)
        assert steps.tolist() == osteps
        for s in range(n):
            assert e[s].tolist() == ost[s][0] and v[s].tolist() == ost[s][1] and f[s].tolist() == ost[s][2], s
        for s in range(n):
            self.tr[dst[s]] = tracks[s]
        # the handed-back tracks: report them, then extend each by every symbol (the extension reads the whole stored column)
        self.extend(list(dst), [0] * n, list(dst))
        for d in dst:
            self.extend([d] * 4, b"ACGT", list(scratch))
        return len(osteps), costs, ost


def allele_reads(rng, src, n, err=0.01):
    reads, _ = synth.hifi_reads(rng, [src], n, err=err, flank=0, lo=0, hi=1 << 20)
    return reads


def het(src, sites):
    b = bytearray(src)
    for p in sites:
        b[p] = b"ACGT"[(b"ACGT".index(src[p]) + 1) % 4]
    return bytes(b)


KINDS = ("anchored", "anchored", "wildcard", "anchored", "consumed", "anchored", "offset0", "anchored", "short", "anchored", "midrun",
         "anchored", "never", "anchored", "empty", "anchored")


def mixed_reads(rng, src, n, run_len, band, window):
    """n reads of src of every kind the loop treats apart, half of them anchored reads with errors (offset reads vote for
    whatever follows their window start until the consensus reaches them, so they stay a minority): wildcards and N, reads
    consumed mid-run (`full < ed` silences them), offset reads that activate at round 0, mid-run or never, reads shorter than
    the band, an empty read."""
    hw = window // 2
    reads, offsets = [], []
    for k in range(n):
        kind = KINDS[k % len(KINDS)]
        o = -1
        if kind == "anchored":
            r = allele_reads(rng, src, 1)[0]
        elif kind == "wildcard":
            r = b"*" * 17 + src[17:60] + b"N" + src[61:90] + b"**" + src[92:]
        elif kind == "consumed":
            r = src[: int(rng.integers(band + 10, max(run_len // 2, band + 12)))]
        elif kind == "offset0":
            o = int(rng.integers(0, hw + 1))
            r = src[o:]
        elif kind == "midrun":
            o = hw + int(rng.integers(3, max(4, run_len // 2)))
            r = allele_reads(rng, src[o:], 1)[0]
        elif kind == "never":
            o, r = hw + run_len + 50, src[:40]
        elif kind == "short":
            r = src[: max(1, band // 2)]
        else:
            r = b"" if k % 32 == 14 else src[: int(rng.integers(1, 5))]
        reads.append(r)
        offsets.append(o)
    return reads, offsets


# ---------------------------------------------------------------------------------------------------------------
# cluster shapes: forced and default cluster sizes, one, two and >= 5 items per warp, idle warps, ragged item counts
# ---------------------------------------------------------------------------------------------------------------
SHAPES = [  # (SP_K7_RUN_CTAS, reads, sides, max_steps)
    (None, 5, 1, 10_000),    # 5 items on 16 warps: idle warps
    (None, 14, 2, 10_000),   # 28 items: 2 CTAs
    (None, 30, 2, 10_000),   # 60 items: 4 CTAs
    (None, 70, 2, 80),       # 140 items: 8 CTAs, 2 per warp
    (1, 40, 1, 10_000),      # 3 per warp
    (1, 45, 2, 10_000),      # 90 items on one CTA: 6 per warp
    (2, 21, 2, 10_000),      # 42 items: 2 per warp, ragged
    (3, 50, 2, 120),         # a cluster of 3: 100 items on 48 warps
    (3, 7, 1, 10_000),
    (4, 33, 1, 10_000),      # 33 items on 64 warps
    (4, 160, 2, 40),         # 5 per warp
    (5, 41, 2, 10_000),      # a cluster of 5: 82 items on 80 warps, 2 per warp
    (5, 200, 2, 40),         # 5 per warp
    (8, 3, 1, 10_000),       # 3 items on 8 CTAs
    (8, 129, 2, 40),         # 258 items: 3 per warp
]


@pytest.mark.parametrize("force,n_reads,n_sides,max_steps", SHAPES)
def test_k7_run_cluster_shapes(ctx, monkeypatch, force, n_reads, n_sides, max_steps):
    items = n_reads * n_sides
    n_cta, per_warp = plan(items, force)
    if force is not None:
        monkeypatch.setenv("SP_K7_RUN_CTAS", str(force))
    assert (n_cta, per_warp) == {
        (None, 5, 1): (1, 1), (None, 14, 2): (2, 1), (None, 30, 2): (4, 1), (None, 70, 2): (8, 2), (1, 40, 1): (1, 3), (1, 45, 2): (1, 6),
        (2, 21, 2): (2, 2), (3, 50, 2): (3, 3), (3, 7, 1): (3, 1), (4, 33, 1): (4, 1), (4, 160, 2): (4, 5), (5, 41, 2): (5, 2),
        (5, 200, 2): (5, 5), (8, 3, 1): (8, 1), (8, 129, 2): (8, 3)}[(force, n_reads, n_sides)]
    rng = np.random.default_rng(1001 + items + (force or 0))
    band, window = 24, 16
    a = rnd(rng, 190)
    if n_sides == 1:
        reads, offsets = mixed_reads(rng, a, n_reads, 180, band, window)
        m = Mirror(ctx, reads, offsets, band, window)
        n, _, _ = m.run([0], [0], [m.fresh(0)], max_steps=max_steps)  # dst == src
    else:
        # side 1 ends first and finishes while side 0 goes on.  Reads that do not cover the first site (wildcards, offsets)
        # count towards both sides until the next one, so the share a symbol needs is raised to 35 %.
        b = het(a, (0, 70, 150))[:175]
        ha = n_reads // 2 + n_reads % 2
        ra, oa = mixed_reads(rng, a, ha, 180, band, window)
        m = Mirror(ctx, ra + allele_reads(rng, b, n_reads - ha), oa + [-1] * (n_reads - ha), band, window)
        m.fresh(0)
        s1, s2 = m.extend([0, 0], a[:1] + b[:1], [1, 2])
        n, _, _ = m.run([1, 2], [3, 4], [s1, s2], permille=350, max_steps=max_steps)
        if max_steps > 180:
            assert m.tr[3].length > m.tr[4].length  # one side stopped, the other went on
    assert n >= min(max_steps, 40)


# ---------------------------------------------------------------------------------------------------------------
# band classes: both sides of every k7_run<CELLS> boundary, and the production settings
# ---------------------------------------------------------------------------------------------------------------
BANDS = [(31, 0), (32, 0), (63, 0), (64, 0), (127, 0), (128, 0), (55, 400), (32, 100), (32, 400)]  # W = band + window / 2


@pytest.mark.parametrize("band,window", BANDS)
def test_k7_run_band_classes(ctx, band, window):
    W = band + window // 2
    rng = np.random.default_rng(2000 + W)
    L = 2 * W + 70  # the consensus passes W, so every band cell holds a row
    a = rnd(rng, L)
    b = het(a, (0, L // 3))
    reads = allele_reads(rng, a, 4, 0.01) + allele_reads(rng, b, 3, 0.01) + [a[: W // 2], b"", a[W + 5:]]
    offsets = [-1] * 9 + [W + 5]
    m = Mirror(ctx, reads, offsets, band, window)
    n_cta, per_warp = plan(2 * len(reads))
    assert cells_of(m.W) == {31: 2, 32: 4, 63: 4, 64: 8, 82: 8, 127: 8, 128: 16, 232: 16, 255: 16}[m.W] and (n_cta, per_warp) == (2, 1)
    m.fresh(0)
    s1, s2 = m.extend([0, 0], a[:1] + b[:1], [1, 2])
    steps = W + 40 if W > 200 else 10_000
    n, _, _ = m.run([1, 2], [1, 2], [s1, s2], max_steps=steps)
    assert n >= min(steps, L - 1)


# ---------------------------------------------------------------------------------------------------------------
# the stop rule
# ---------------------------------------------------------------------------------------------------------------
def stop_case(ctx):
    rng = np.random.default_rng(31)
    a = rnd(rng, 700)
    reads = allele_reads(rng, a, 9, 0.02)
    m = Mirror(ctx, reads, [-1] * 9, 12, 0)
    return m, a


def test_k7_run_het_site_stops(ctx):
    rng = np.random.default_rng(32)
    a = rnd(rng, 260)
    b = het(a, (97,))
    m = Mirror(ctx, allele_reads(rng, a, 5, 0.005) + allele_reads(rng, b, 5, 0.005), [-1] * 10, 16, 0)
    n, _, _ = m.run([0], [1], [m.fresh(0)])
    assert n == 97  # two passing symbols at the het site


@pytest.mark.parametrize("max_steps", [1, 255, 256, 257, 512, 513])
def test_k7_run_max_steps_around_log_blocks(ctx, max_steps):
    m, a = stop_case(ctx)
    n, _, _ = m.run([0], [1], [m.fresh(0)], max_steps=max_steps)
    assert n == max_steps


def test_k7_run_limits(ctx):
    """Limits taken from the oracle's cost trajectory, so that each cuts at a known round: cost_limit with the size tie on both
    sides, cost_cap equal to the cost and one below, the exemption of round 0, and a start node that does not qualify."""
    m, a = stop_case(ctx)
    root = m.fresh(0)
    _, costs, _ = m.run([0], [1], [root], max_steps=600)
    # the first round q at which the cost grows, with a flat stretch before it
    q = next(k for k in range(2, 600) if costs[k] > costs[k - 1] and costs[k] > costs[0])
    c = costs[q]
    # cost_limit == the cost of node q: node q goes on only while its size is above size_limit (the tie)
    assert m.run([0], [2], [root], cost_limit=c, size_limit=q, max_steps=600)[0] == q  # size q is not > q: stop at q
    n_tie, _, _ = m.run([0], [2], [root], cost_limit=c, size_limit=q - 1, max_steps=600)
    assert n_tie > q
    # cost_cap: equal to the cost goes on, one below stops there
    n_cap, _, _ = m.run([0], [2], [root], cost_cap=c, max_steps=600)
    assert n_cap > q
    assert m.run([0], [2], [root], cost_cap=c - 1, max_steps=600)[0] == q
    # round 0 is exempt: a start node above every limit still takes one round
    assert m.run([0], [2], [root], cost_limit=-1, cost_cap=-1)[0] == 1
    # n_steps == 0: the start node has two passing symbols; dst comes back as a copy of src
    h = Mirror(ctx, [a[:50] + b"A" + a[51:300]] * 4 + [a[:50] + b"C" + a[51:300]] * 4, [-1] * 8, 12, 0)
    assert h.run([0], [5], [h.grow(0, a[:50])])[0] == 0 and h.tr[5].length == 50


def test_k7_run_chained(ctx):
    """A run, an extension step, another run: the second run starts from the state the step returned."""
    m, a = stop_case(ctx)
    n1, _, st = m.run([0], [1], [m.fresh(0)], max_steps=150)
    s = m.extend([1], a[150:151], [2])[0]
    n2, _, _ = m.run([2], [3], [s], max_steps=200)
    assert (n1, n2, m.tr[3].length) == (150, 200, 351)


# ---------------------------------------------------------------------------------------------------------------
# the fit boundary and refusals
# ---------------------------------------------------------------------------------------------------------------
def _supported(ctx, n_reads, band, window, read_len=60, n_sides=2):
    import pb_starphase_b200 as sp

    c = sp.Consensus(ctx, [b"A" * read_len] * n_reads, None, offset_window=window, band=band, max_tracks=2)
    ok = c.run_supported(n_sides)
    c.close()
    return ok


def _raw_run(cons, n_sides, src, dst, ed, votes, full, min_count=3, permille=100, max_steps=100):
    lib = cons.ctx._lib
    s = np.ascontiguousarray(src, dtype=np.int32)
    d = np.ascontiguousarray(dst, dtype=np.int32)
    log = np.zeros(max(max_steps, 1), dtype=np.uint8)
    n = C.c_int32(7)
    st = lib.sp_consensus_run(cons._h, n_sides, s.ctypes.data, d.ctypes.data, ed.ctypes.data, votes.ctypes.data, full.ctypes.data,
                              min_count, permille, BIG, 0, BIG, max_steps, log.ctypes.data, C.byref(n))
    return st, n.value


@SKIP_LARGE
def test_k7_run_fit_boundary(ctx):
    """W = 255, two sides: the largest read count run_supported accepts puts > 128 items on 8 CTAs and runs >= 40 rounds (a
    ring refill) against the oracle; one read more is refused by run_supported and by run, which then writes nothing."""
    band, window = 55, 400
    lo, hi = 64, 2048
    assert _supported(ctx, lo, band, window) and not _supported(ctx, hi, band, window)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if _supported(ctx, mid, band, window) else (lo, mid)
    R = lo
    print(f"largest read set k7_run takes at W = 255, two sides: {R} reads")
    n_cta, per_warp = plan(2 * R)
    assert n_cta == 8 and 2 * R > 128 and per_warp >= 2
    rng = np.random.default_rng(41)
    a = rnd(rng, 400)
    b = het(a, (0, 200))
    reads = [r[:300] for r in allele_reads(rng, a, R // 2, 0.01) + allele_reads(rng, b, R - R // 2, 0.01)]
    m = Mirror(ctx, reads, [-1] * R, band, window)
    assert m.W == 255 and m.gpu.run_supported(2) and not m.gpu.run_supported(3)
    m.fresh(0)
    s1, s2 = m.extend([0, 0], a[:1] + b[:1], [1, 2])
    n, _, _ = m.run([1, 2], [3, 4], [s1, s2], max_steps=40)
    assert n == 40
    m.gpu.close()
    # R + 1 reads: refused, nothing written
    import pb_starphase_b200 as sp

    big = sp.Consensus(ctx, reads + reads[:1], None, offset_window=window, band=band, max_tracks=4)
    assert not big.run_supported(2) and big.run_supported(1)
    big.reset(0)
    big.reset(1)
    e0, v0, f0 = big.extend([0, 1], [0, 0], [0, 1])
    ed, votes, full = e0.copy(), v0.copy(), f0.copy()
    st, n = _raw_run(big, 2, [0, 1], [2, 3], ed, votes, full)
    assert (st, n) == (SP_ERR_RANGE, 0)
    assert np.array_equal(ed, e0) and np.array_equal(votes, v0) and np.array_equal(full, f0)
    with pytest.raises(sp.SpError) as ex:
        big.run([0, 1], [2, 3], e0, v0, f0, 3, 100, BIG, 0, BIG, 10)
    assert ex.value.status == SP_ERR_RANGE
    big.close()


def test_k7_run_refusals(ctx):
    import pb_starphase_b200 as sp

    # more than 2,048 read-sides, a read over 60,000 bases
    assert _supported(ctx, 1024, 8, 0) and not _supported(ctx, 1025, 8, 0)
    assert _supported(ctx, 2048, 8, 0, n_sides=1) and not _supported(ctx, 2049, 8, 0, n_sides=1)
    assert _supported(ctx, 2, 8, 0, read_len=60_000) and not _supported(ctx, 2, 8, 0, read_len=60_001)
    c = sp.Consensus(ctx, [b"ACGT" * 10] * 3, None, band=8, max_tracks=4)
    assert not c.run_supported(0) and not c.run_supported(3)
    c.reset(0)
    c.reset(1)
    e0, v0, f0 = c.extend([0, 1], [0, 0], [0, 1])
    bad = [
        dict(n_sides=0), dict(n_sides=3), dict(max_steps=0), dict(permille=1001), dict(permille=-1), dict(min_count=-1),
        dict(src=[-1, 1]), dict(dst=[2, 4]), dict(dst=[2, 2]), dict(dst=[1, 3]), dict(dst=[2, 0]),
    ]
    for kw in bad:
        args = dict(n_sides=2, src=[0, 1], dst=[2, 3], min_count=3, permille=100, max_steps=10)
        args.update(kw)
        ed, votes, full = e0.copy(), v0.copy(), f0.copy()
        st, n = _raw_run(c, args["n_sides"], args["src"], args["dst"], ed, votes, full, args["min_count"], args["permille"], args["max_steps"])
        assert st == SP_ERR_INVALID, kw
        assert np.array_equal(ed, e0) and np.array_equal(votes, v0) and np.array_equal(full, f0), kw
    with pytest.raises(sp.SpError) as ex:
        c.run([0, 1], [2, 2], e0, v0, f0, 3, 100, BIG, 0, BIG, 10)
    assert ex.value.status == SP_ERR_INVALID
    with pytest.raises(sp.SpError):
        c.run([0], [1], e0[:1], v0[:1], f0[:1], 3, 100, BIG, 0, BIG, 0)
    c.close()


# ---------------------------------------------------------------------------------------------------------------
# the host search with and without the device loop, at a size the oracle's own search cannot reach
# ---------------------------------------------------------------------------------------------------------------
@SKIP_LARGE
def test_host_dual_consensus_large_run_equals_stepped(monkeypatch):
    from pb_starphase_b200 import _starphase_host as host

    rng = np.random.default_rng(51)
    a = rnd(rng, 1200)
    b = het(a, (150, 600, 1050))
    reads = allele_reads(rng, a, 80, 0.004) + allele_reads(rng, b, 80, 0.004)
    gpu = host.GpuAligner(0)
    rs, cfg = [r.decode() for r in reads], dict(offset_window=400)
    got_run, calls_run = host.dual_consensus(gpu, rs, [], cfg)
    monkeypatch.setenv("SP_CONSENSUS_NO_RUN", "1")
    got_step, calls_step = host.dual_consensus(gpu, rs, [], cfg)
    assert calls_step > calls_run
    assert len(got_run) == len(got_step) >= 1
    for g, w in zip(got_run, got_step):
        assert (g["consensus1"], g["consensus2"]) == (w["consensus1"], w["consensus2"])
        assert list(g["is_consensus1"]) == list(w["is_consensus1"]) and list(g["scores1"]) == list(w["scores1"])
        assert list(g["scores2"]) == list(w["scores2"])
    # both alleles come back through every het site (a read set may append a base that only a few reads carry at the very end)
    assert sorted(c[:1100] for c in (got_run[0]["consensus1"], got_run[0]["consensus2"])) == sorted([a[:1100], b[:1100]])


# ---------------------------------------------------------------------------------------------------------------
# k7_extend at both ends of every CELLS class
# ---------------------------------------------------------------------------------------------------------------
WIDTHS = sorted({w for c in range(1, 33) for w in (max(1, 16 * (c - 1)), 16 * c - 1)})


@pytest.mark.parametrize("W", WIDTHS)
def test_k7_extend_every_width(ctx, W):
    """k7_extend<CELLS> at both ends of its class: reads long enough that the upper half of the band holds read rows, and per
    launch the right symbol, a wrong one and a report of the parent (as test_k7_extend_vs_oracle walks)."""
    cells = -(-(2 * W + 1) // 32)
    assert W in (max(1, 16 * (cells - 1)), 16 * cells - 1)
    rng = np.random.default_rng(3000 + W)
    src = rnd(rng, W + 60)
    reads = allele_reads(rng, src, 2, 0.03) + [src[5:], b"*" * 9 + src[9:40] + b"N" + src[41:]]
    m = Mirror(ctx, reads, [-1, -1, 3, -1], W, 0, max_tracks=8)
    m.fresh(0)
    cur = 0
    for pos, base in enumerate(src[:40]):
        free = [t for t in range(8) if t != cur][:3]
        wrong = b"ACGT"[(b"ACGT".index(base) + 1 + pos % 3) % 4]
        m.extend([cur] * 3, [base, wrong, 0], free)
        cur = free[0]


def test_k7_extend_refuses_w512(ctx):
    import pb_starphase_b200 as sp

    sp.Consensus(ctx, [b"ACGT"], None, band=511, max_tracks=1).close()
    with pytest.raises(sp.SpError) as ex:
        sp.Consensus(ctx, [b"ACGT"], None, band=512, max_tracks=1)
    assert ex.value.status == SP_ERR_RANGE
    with pytest.raises(sp.SpError):
        sp.Consensus(ctx, [b"ACGT"], None, band=312, offset_window=400, max_tracks=1)
