"""GPU suite, row N1: many independent consensus searches in one device pass.  sp_consensus_run_batch (one `k7_run` cluster per
job, one launch per CELLS class) and sp_consensus_extend_batch (every (task, read) of every list in one `k7_extend` launch) against
single sp_consensus_run / sp_consensus_extend calls on fresh handles built from the same inputs, bit for bit; then the C++ host's
batch driver (ConsensusDWFA / DualConsensusDWFA::consensus_batch) against each search run alone."""
import ctypes as C
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "oracle"))

import consensus_oracle as co  # noqa: E402
from test_consensus_cpu import rnd  # noqa: E402
from test_consensus_run_gpu import BIG, allele_reads, cells_of, het, plan  # noqa: E402

pytestmark = pytest.mark.gpu
SP_ERR_INVALID, SP_ERR_RANGE = 1, 5


class Case:
    """One read set: how to build its handle, and the preparation (resets, extensions) that makes its start nodes."""

    def __init__(self, reads, offsets, band, window, prep, max_tracks=16):
        self.reads, self.offsets, self.band, self.window, self.prep, self.max_tracks = reads, offsets, band, window, prep, max_tracks

    def build(self, ctx):
        import pb_starphase_b200 as sp

        c = sp.Consensus(ctx, self.reads, self.offsets, offset_window=self.window, band=self.band, max_tracks=self.max_tracks)
        states = {}
        for track, seq in self.prep:  # track := the root extended by seq; its state
            c.reset(track)
            st = c.extend([track], [0], [track])
            for b in seq:
                st = c.extend([track], [b], [track])
            states[track] = tuple(a[0] for a in st)
        return c, states


def job(cons, states, src, dst, max_steps=10_000, min_count=3, permille=100):
    ed = np.stack([states[s][0] for s in src])
    votes = np.stack([states[s][1] for s in src])
    full = np.stack([states[s][2] for s in src])
    return (cons, list(src), list(dst), ed, votes, full, min_count, permille, BIG, 0, BIG, max_steps)


def single(case, ctx, src, dst, **kw):
    """The job alone, on a fresh handle: its outputs and the handle (for the follow-on extensions)."""
    c, states = case.build(ctx)
    j = job(c, states, src, dst, **kw)
    return c.run(*j[1:]), c


def same_tracks(a, b, tracks, scratch):
    """Report each track, then extend it by A / C / G / T: equal on both handles (the whole column, best_full, the length)."""
    for t in tracks:
        for x, y in zip(a.extend([t], [0], [t]), b.extend([t], [0], [t])):
            assert np.array_equal(x, y), t
        for x, y in zip(a.extend([t] * 4, b"ACGT", list(scratch)), b.extend([t] * 4, b"ACGT", list(scratch))):
            assert np.array_equal(x, y), t


def same_run(got, want):
    for x, y in zip(got, want):
        assert np.array_equal(x, y)


def cases(rng):
    a = rnd(rng, 300)
    b = het(a, (40, 110, 170, 220, 260))
    single16 = Case(allele_reads(rng, a, 16), [-1] * 16, 32, 0, [(0, b""), (2, a[:20])])
    dual30 = Case(allele_reads(rng, a, 15, 0.004) + allele_reads(rng, b, 15, 0.004), [-1] * 30, 8, 0, [(0, b""), (1, b"")])
    o = [-1 if k % 3 == 0 else int(rng.integers(0, 120)) for k in range(20)]
    offset20 = Case([a if x < 0 else a[x:] for x in o], o, 16, 200, [(0, b"")])
    wild = Case([b"*" * 25 + a[25:], a[:150] + b"**" + a[152:], a, a, b"*" * 300, a], [-1] * 6, 32, 0, [(0, b"")])
    split = Case([b"A" + a] * 8 + [b"C" + a] * 8, [-1] * 16, 32, 0, [(0, b"")])
    return single16, dual30, offset20, wild, split


def test_run_batch_mixed_jobs(ctx):
    """One call: a single 16-read consensus, a 30-read dual across het sites, offset reads in a wider CELLS class, wildcard reads, a
    start node that does not qualify (n_steps == 0) and two jobs on one handle with disjoint tracks (one crossing a log block)."""
    import pb_starphase_b200 as sp

    single16, dual30, offset20, wild, split = cases(np.random.default_rng(7))
    assert len({cells_of(c.band + c.window // 2) for c in (single16, dual30, offset20)}) == 3
    specs = [(single16, [0], [1], {}), (single16, [2], [3], {"max_steps": 40}), (dual30, [0, 1], [2, 3], {}), (offset20, [0], [1], {}),
             (wild, [0], [1], {}), (split, [0], [1], {})]
    built = {}
    jobs = []
    for case, src, dst, kw in specs:
        if id(case) not in built:
            built[id(case)] = case.build(ctx)
        c, states = built[id(case)]
        jobs.append(job(c, states, src, dst, **kw))
    got = sp.Consensus.run_batch(ctx, jobs)
    assert len(got[0][3]) > 256  # the log beyond its first block comes back too
    assert len(got[5][3]) == 0 and len(got[2][3]) > 0
    for (case, src, dst, kw), g in zip(specs, got):
        want, fresh = single(case, ctx, src, dst, **kw)
        same_run(g, want)
        same_tracks(built[id(case)][0], fresh, dst, (12, 13, 14, 15))


def test_run_batch_cluster_shapes(ctx):
    """Jobs of one CELLS class whose plans need 4 and 8 CTAs share one launch (clusters of 8) and equal their single runs."""
    import pb_starphase_b200 as sp

    rng = np.random.default_rng(8)
    a = rnd(rng, 120)
    small = Case(allele_reads(rng, a, 40), [-1] * 40, 16, 0, [(0, b"")], max_tracks=8)
    large = Case(allele_reads(rng, a, 900), [-1] * 900, 16, 0, [(0, b"")], max_tracks=8)
    assert plan(40)[0] == 4 and plan(900)[0] == 8
    cs, ss = small.build(ctx)
    cl, sl = large.build(ctx)
    n0 = ctx.launch_count()
    got = sp.Consensus.run_batch(ctx, [job(cs, ss, [0], [1]), job(cl, sl, [0], [1])])
    assert ctx.launch_count() - n0 == 1
    for case, c, g in ((small, cs, got[0]), (large, cl, got[1])):
        want, fresh = single(case, ctx, [0], [1])
        same_run(g, want)
        assert len(g[3]) > 0
        same_tracks(c, fresh, [1], (4, 5, 6, 7))


def test_run_batch_many_clusters(ctx):
    """64 jobs of 8-CTA clusters (512 CTAs: more than the GPU holds at once) in one call, each equal to its single run."""
    import pb_starphase_b200 as sp

    rng = np.random.default_rng(9)
    handles = []
    for h in range(8):
        a = rnd(rng, 150)
        prep = [(2 * k, a[: 3 * k]) for k in range(8)]
        handles.append(Case(allele_reads(rng, a, 70), [-1] * 70, 16, 0, prep, max_tracks=20))
    assert plan(70)[0] == 8
    built = [c.build(ctx) for c in handles]
    jobs = [job(c, st, [2 * k], [2 * k + 1]) for c, st in built for k in range(8)]
    got = sp.Consensus.run_batch(ctx, jobs)
    for h, case in enumerate(handles):
        fresh, fst = case.build(ctx)
        for k in range(8):
            want = fresh.run(*job(fresh, fst, [2 * k], [2 * k + 1])[1:])
            same_run(got[8 * h + k], want)
        same_tracks(built[h][0], fresh, [2 * k + 1 for k in range(8)], (16, 17, 18, 19))


def test_extend_batch_vs_single(ctx):
    """Lists on handles of different CELLS classes in one launch, with in-place tasks and report-only tasks (symbol 0)."""
    import pb_starphase_b200 as sp

    single16, dual30, offset20, wild, _ = cases(np.random.default_rng(10))
    specs = [(single16, [0, 2, 0], b"A\x00G", [4, 2, 5]), (offset20, [0, 0, 0], b"ACT", [1, 2, 3]), (wild, [0], b"C", [0]),
             (dual30, [0, 1], b"\x00T", [0, 1])]
    built = [case.build(ctx)[0] for case, *_ in specs]
    n0 = ctx.launch_count()
    got = sp.Consensus.extend_batch(ctx, [(c, src, sym, dst) for c, (_, src, sym, dst) in zip(built, specs)])
    assert ctx.launch_count() - n0 == 2  # k7_extend + the length update
    for c, (case, src, sym, dst), g in zip(built, specs, got):
        fresh = case.build(ctx)[0]
        same_run(g, fresh.extend(src, sym, dst))
        same_tracks(c, fresh, sorted(set(dst)), (10, 11, 12, 13))


def test_batch_refusals(ctx):
    """Each refusal returns its status and writes nothing, not even for the valid jobs of the same call."""
    import pb_starphase_b200 as sp
    from pb_starphase_b200.binding import ConsensusExt, ConsensusJob

    lib = ctx._lib
    rng = np.random.default_rng(11)
    a = rnd(rng, 80)
    c = sp.Consensus(ctx, allele_reads(rng, a, 6), None, band=16, max_tracks=4)
    for t in range(4):
        c.reset(t)
    other_ctx = sp.Context(ctx.device)
    other = sp.Consensus(other_ctx, allele_reads(rng, a, 6), None, band=16, max_tracks=4)
    huge = sp.Consensus(ctx, [b"A" * 30] * 1100, None, band=16, max_tracks=4)
    assert not huge.run_supported(2)

    bufs = []

    def mk(cons, src, dst, n_reads, max_steps=50):
        j = ConsensusJob()
        n = len(src)
        e = np.full(n * n_reads, 77, np.int32); v = np.full(n * n_reads, 77, np.uint8); f = np.full(n * n_reads, 77, np.int32)
        steps = np.full(max_steps, 77, np.uint8); ns = np.full(1, 77, np.int32)
        bufs.append((e, v, f, steps, ns))
        j.c, j.n_sides = cons._h, n
        for s in range(n):
            j.src[s], j.dst[s] = src[s], dst[s]
        j.ed, j.votes, j.full, j.steps, j.n_steps = e.ctypes.data, v.ctypes.data, f.ctypes.data, steps.ctypes.data, ns.ctypes.data
        j.min_count, j.min_af_permille, j.cost_limit, j.size_limit, j.cost_cap, j.max_steps = 3, 100, BIG, 0, BIG, max_steps
        return j

    def untouched():
        return all((x == 77).all() for b in bufs for x in b)

    def call(js, n=None):
        arr = (ConsensusJob * max(len(js), 1))(*js)
        return lib.sp_consensus_run_batch(ctx._h, len(js) if n is None else n, C.cast(arr, C.c_void_p))

    ok = mk(c, [0], [1], 6)
    assert lib.sp_consensus_run_batch(ctx._h, 1, None) == SP_ERR_INVALID and untouched()
    assert call([ok], -1) == SP_ERR_INVALID and untouched()
    assert call([ok, mk(other, [0], [1], 6)]) == SP_ERR_INVALID and untouched()
    assert call([ok, mk(c, [2], [4], 6)]) == SP_ERR_INVALID and untouched()
    assert call([ok, mk(c, [2], [1], 6)]) == SP_ERR_INVALID and untouched()  # two jobs write track 1
    assert call([ok, mk(c, [0], [3], 6)]) == SP_ERR_INVALID and untouched()  # ... or share track 0
    assert call([ok, mk(huge, [0, 1], [2, 3], 1100)]) == SP_ERR_RANGE and untouched()
    assert call([ok, mk(c, [2], [3], 6)]) == 0 and int(bufs[0][4][0]) != 77  # disjoint tracks: both run

    e = np.full(6, 77, np.int32); v = np.full(6, 77, np.uint8); f = np.full(6, 77, np.int32)
    src, dst, sym = np.array([0], np.int32), np.array([1], np.int32), np.array([ord("A")], np.uint8)
    x = ConsensusExt(other._h, 1, src.ctypes.data, sym.ctypes.data, dst.ctypes.data, e.ctypes.data, v.ctypes.data, f.ctypes.data)
    assert lib.sp_consensus_extend_batch(ctx._h, 1, C.byref(x)) == SP_ERR_INVALID
    assert lib.sp_consensus_extend_batch(ctx._h, 1, None) == SP_ERR_INVALID
    assert lib.sp_consensus_extend_batch(ctx._h, -1, C.byref(x)) == SP_ERR_INVALID
    x2 = ConsensusExt(c._h, 1, src.ctypes.data, sym.ctypes.data, dst.ctypes.data, e.ctypes.data, v.ctypes.data, f.ctypes.data)
    arr = (ConsensusExt * 2)(x2, x2)  # two lists write track 1 of one handle
    assert lib.sp_consensus_extend_batch(ctx._h, 2, C.cast(arr, C.c_void_p)) == SP_ERR_INVALID
    assert (e == 77).all() and (v == 77).all() and (f == 77).all()
    other.close(); huge.close(); c.close()
    other_ctx.close()


# ---------------------------------------------------------------------------------------------------------------
# the C++ host: batches of searches
# ---------------------------------------------------------------------------------------------------------------
def host_groups(rng):
    a = rnd(rng, 400)
    b = het(a, (60, 200, 330))
    c = rnd(rng, 250)
    return [
        ([r.decode() for r in allele_reads(rng, a, 10, 0.004) + allele_reads(rng, b, 10, 0.004)], []),
        ([r.decode() for r in allele_reads(rng, c, 12)], []),
        ([a.decode()[x:] for x in (0, 30, 0, 55, 0, 10)], [None, 30 + 50, None, 55 + 50, None, 10 + 50]),
    ]


def test_host_consensus_batch_equals_single():
    """consensus_batch / dual_consensus_batch return exactly what each search returns alone, a failing search (no reads) does
    not stop the others, and the batch takes fewer kernel launches than the searches one by one."""
    from pb_starphase_b200 import _starphase_host as host

    gpu = host.GpuAligner(0)
    groups = host_groups(np.random.default_rng(12))
    cfg = dict(offset_window=100)
    for batch_fn, one_fn in ((host.consensus_batch, host.consensus), (host.dual_consensus_batch, host.dual_consensus)):
        n0 = gpu.launch_count()
        got = batch_fn(gpu, groups + [([], [])], cfg)
        batch_launches = gpu.launch_count() - n0
        assert got[3][2] is not None and "no sequences" in got[3][2]
        n0 = gpu.launch_count()
        for (reads, offs), (sols, calls, err) in zip(groups, got):
            assert err is None
            want_sols, want_calls = one_fn(gpu, reads, offs, cfg)
            assert len(sols) == len(want_sols) >= 1 and calls == want_calls
            for g, w in zip(sols, want_sols):
                if isinstance(g, dict):
                    assert {k: (list(v) if isinstance(v, list) else v) for k, v in g.items()} == {k: (list(v) if isinstance(v, list) else v) for k, v in w.items()}
                else:
                    assert (g[0], list(g[1])) == (w[0], list(w[1]))
        assert batch_launches < gpu.launch_count() - n0
    assert got[0][0][0]["consensus2"] is not None  # the het group is dual


def chain_one_by_one(host, gpu, chains, offsets, seeds, cfg):
    """PriorityConsensusDWFA's outline (starphase_host.hpp) with one search at a time."""
    levels = len(chains[0])
    by_seed = {}
    for i, s in enumerate(seeds):
        by_seed.setdefault((s is not None, s or 0), []).append(i)
    work = [[by_seed[k], 0, [None] * levels] for k in sorted(by_seed, reverse=True)]
    done = []
    while work:
        members, level, known = work.pop()
        if level == levels:
            done.append((members, known))
            continue
        sols, _ = host.dual_consensus(gpu, [chains[i][level] for i in members], [offsets[i][level] for i in members], cfg)
        d = sols[0]
        if d["consensus2"] is not None:
            a = [m for m, one in zip(members, d["is_consensus1"]) if one]
            b = [m for m, one in zip(members, d["is_consensus1"]) if not one]
            work += [[b, level, [None] * levels], [a, level, [None] * levels]]
        else:
            known[level] = (d["consensus1"], [x or 0 for x in d["scores1"]])
            work.append([members, level + 1, known])
    done.sort(key=lambda g: g[0][0])
    idx = [0] * len(chains)
    for gi, (members, known) in enumerate(done):
        for lv in range(levels):
            if known[lv] is None:
                sols, _ = host.consensus(gpu, [chains[i][lv] for i in members], [offsets[i][lv] for i in members], cfg)
                known[lv] = (sols[0][0], list(sols[0][1]))
        for m in members:
            idx[m] = gi
    return [[(s, list(sc)) for s, sc in known] for _, known in done], idx


def test_host_priority_chain_batched():
    """The priority chain on four groups (seeds plus a split at the second level) equals the oracle's restatement and the same
    chain run one search at a time, with fewer kernel launches."""
    from pb_starphase_b200 import _starphase_host as host
    from test_consensus_gpu import priority_case

    sources, chains, offsets, seeds, truth = priority_case(np.random.default_rng(21))
    want_cons, want_idx = co.priority_consensus(chains, offsets, seeds)
    assert len(want_cons) == 4
    gpu = host.GpuAligner(0)
    str_chains = [[x.decode() for x in ch] for ch in chains]
    n0 = gpu.launch_count()
    got_cons, got_idx = host.priority_consensus(gpu, str_chains, offsets, seeds, {})
    batched = gpu.launch_count() - n0
    assert list(got_idx) == want_idx
    got = [[(s, list(sc)) for s, sc in levels] for levels in got_cons]
    assert got == [[(s, list(sc)) for s, sc in levels] for levels in want_cons]
    n0 = gpu.launch_count()
    seq_cons, seq_idx = chain_one_by_one(host, gpu, str_chains, offsets, seeds, {})
    one_by_one = gpu.launch_count() - n0
    assert (seq_cons, seq_idx) == (got, list(got_idx))
    assert batched < one_by_one
