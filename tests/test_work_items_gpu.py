"""GPU parity tests for the dynamically scheduled paths of K1, K4 and K9: one persistent CTA or warp running many work items.

K1's persistent CTAs take (pattern group, text tile) items from an atomic counter and reset the column state at every text end
inside a tile; K4 and K9 warps take bins / pairs from a counter and reuse one traceback slot each.  Every test first asserts that
the device really runs more items than it has CTAs or warps for (bounds from torch.cuda.get_device_properties), so that it cannot
pass on a configuration where every item gets fresh state; then it compares everything the kernel writes with the CPU oracle,
bit for bit."""
import math
import os
import re

import numpy as np
import pytest

import oracle_util as ou
import pb_starphase_b200 as sp
from pb_starphase_b200 import synth
from pb_starphase_b200.binding import plan_lane_classes
from test_k1_gpu import noisy_copy, rnd

pytestmark = pytest.mark.gpu
SKIP_LARGE = pytest.mark.skipif(os.environ.get("SP_SKIP_LARGE") == "1", reason="large case skipped")

K1_CHUNK = 8                    # text columns per K1 chunk
K1_THREADS = 256                # threads per K1 CTA (8 warps)
ROWS_U16 = 32 * 16              # pattern rows per lane at the widest ordinary lane width
OP_I, OP_D, OP_EQ, OP_X = 1, 2, 7, 8


@pytest.fixture(scope="module")
def dev():
    import torch

    p = torch.cuda.get_device_properties(0)
    return {"sms": p.multi_processor_count, "warps_per_sm": p.max_threads_per_multi_processor // 32,
            "k1_ctas_per_sm": p.max_threads_per_multi_processor // K1_THREADS, "smem_optin": p.shared_memory_per_block_optin}


def chunks(n: int) -> int:
    return max(1, -(-n // K1_CHUNK))


def effective_tc(text_lens, force_tc: int) -> int:
    """run_k1's tile capacity under SP_FORCE_TC: at least 64 and the longest text, rounded up to even."""
    tc = max(64, force_tc, max(chunks(n) for n in text_lens))
    return (tc + 1) // 2 * 2


def n_tiles(text_lens, tc: int) -> int:
    """get_text_pack's packing rule: whole texts per tile, a tile closes when the next text would not fit (the even-count
    padding comes after the fill test, so it does not change the tile count)."""
    tiles, fill = 0, None
    for n in text_lens:
        c = chunks(n)
        if fill is None or fill + c > tc:
            tiles, fill = tiles + 1, 0
        fill += c
    return tiles


def k1_items_lower_bound(text_lens, pat_lens, tc: int) -> int:
    """Work items of one K1 call, from below: every class has at least ceil(lanes / 256) groups of 8 warps x 32 lanes, and a
    pattern takes the fewest lanes at U = 16."""
    lanes = sum(-(-m // ROWS_U16) for m in pat_lens if m)
    return n_tiles(text_lens, tc) * -(-lanes // 256)


# ---------------------------------------------------------------------------------------------------------------------------
# 1. K1: many items per persistent CTA, forced tile shapes
# ---------------------------------------------------------------------------------------------------------------------------
FORCED_TC = (64, 66, 130, 4096)


def tile_fills(text_lens, tc: int):
    """(chunks in each tile, chunks of the text that closed each full tile) under get_text_pack's packing rule."""
    fills, closers, fill = [], [], None
    for n in text_lens:
        c = chunks(n)
        if fill is not None and fill + c > tc:
            fills.append(fill); closers.append(c); fill = None
        fill = c if fill is None else fill + c
    return fills + [fill], closers


def k1_text_set(rng, pats):
    """~3,000 texts of 0-512 bases (at most 64 chunks, so that SP_FORCE_TC=64 really gives 64-chunk tiles): lengths of every
    residue mod 8, empty and all-N texts, texts of exactly 64 chunks, a fifth carrying noisy pattern copies, and runs of texts
    that fill a tile of each forced capacity exactly or overflow it by one chunk."""
    texts = [rnd(rng, int(n)) for n in rng.integers(0, 513, size=2600)]
    texts += [rnd(rng, n) for n in (0, 1, 7, 8, 9, 15, 16, 17, 255, 256, 257, 504, 505, 511, 512) for _ in range(3)]
    texts += [b"", b"", b"", b"N" * 8, b"N" * 63, b"N" * 512, b"ACGTN" * 60, b"acgt" * 40] * 3
    for i in range(0, len(texts), 5):   # noisy pattern copies: distances spread from 0 to m
        p = pats[int(rng.integers(0, len(pats)))]
        if len(texts[i]) > len(p) + 8:
            s = int(rng.integers(0, len(texts[i]) - len(p) + 1))
            texts[i] = (texts[i][:s] + noisy_copy(rng, p.upper(), int(rng.integers(0, 8))) + texts[i][s + len(p):])[:512]
    texts = [texts[i] for i in rng.permutation(len(texts))]
    for tc in FORCED_TC[:3]:
        for total in (tc, tc + 1):
            for _ in range(12):
                parts = [64] * (total // 64 - 1) + [total % 64 + 64] if total > 64 else [total]
                parts = [x for y in parts for x in ((y // 2, y - y // 2) if y > 64 or rng.random() < 0.7 else (y,))]
                run = [rnd(rng, 8 * c - int(rng.integers(0, 8))) for c in parts]
                at = int(rng.integers(0, len(texts)))
                texts[at:at] = [rnd(rng, 512)] * int(rng.integers(0, 3)) + run
    return texts


def k1_pattern_set(rng):
    pats = [rnd(rng, int(m)) for m in rng.integers(1, 2201, size=380)]
    for k in range(0, 380, 19):
        b = bytearray(pats[k])
        for pos in rng.integers(0, len(b), size=max(1, len(b) // 50)):
            b[int(pos)] = ord("N")
        pats[k] = bytes(b)
    for k in range(7, 380, 23):
        pats[k] = pats[k].lower()
    pats += [b"N" * 33, b"A", b"ACGT" * 128, b"acgtn" * 100, rnd(rng, 2200), rnd(rng, 512), rnd(rng, 513), rnd(rng, 1024),
             rnd(rng, 1025), rnd(rng, 2048), rnd(rng, 2049), b"T" * 70]
    pats += [rnd(rng, int(m)) for m in rng.integers(1, 200, size=8)]
    return pats


@pytest.fixture(scope="module")
def k1_sets(oracle):
    rng = np.random.default_rng(2024)
    pats = k1_pattern_set(rng)
    texts = k1_text_set(rng, pats)
    assert 2800 <= len(texts) <= 3200 and 390 <= len(pats) <= 410
    ref = {prefix: oracle.score_batch(texts, pats, prefix=prefix, impl="myers", want_end_col=True) for prefix in (False, True)}
    return texts, pats, ref


def assert_same(got, want, what):
    bad = np.argwhere(got != want)
    assert len(bad) == 0, (what, len(bad), [(int(t), int(p), int(got[t, p]), int(want[t, p])) for t, p in bad[:8]])


@pytest.mark.parametrize("prefix", [False, True], ids=["infix", "prefix"])
@pytest.mark.parametrize("force_tc", FORCED_TC)
def test_k1_forced_tiles_full_matrix(ctx, dev, k1_sets, monkeypatch, force_tc, prefix):
    """Whole matrix and end columns equal the oracle at every forced tile capacity, for 16- and 32-bit output, with and without
    end columns."""
    texts, pats, ref = k1_sets
    lens = [len(t) for t in texts]
    tc = effective_tc(lens, force_tc)
    assert tc == force_tc, "the text set must not raise the forced tile capacity"
    items = k1_items_lower_bound(lens, [len(p) for p in pats], tc)
    if force_tc == 64:
        assert items > 2 * dev["sms"] * dev["k1_ctas_per_sm"], (items, dev)
    if force_tc != 4096:   # tiles filled to exactly tc, and tiles closed by a text that overflows them by one chunk
        fills, closers = tile_fills(lens, tc)
        assert tc in fills and any(f + c == tc + 1 for f, c in zip(fills, closers))
    monkeypatch.setenv("SP_FORCE_TC", str(force_tc))
    Dw, Ew = ref[prefix]
    T = ctx.targets(texts)
    P = ctx.patterns(pats, mode=sp.SP_PREFIX if prefix else sp.SP_INFIX)
    for bits in (16, 32):
        for want_end in (False, True):
            M = ctx.score_device(T, P, elem_bits=bits, want_end_col=want_end)
            if want_end:
                D, E = M.to_host(want_end_col=True)
                assert_same(E, Ew, ("end", bits))
            else:
                D = M.to_host()
            assert_same(D, Dw, ("dist", bits, want_end))
            M.close()
    P.close(); T.close()


@pytest.mark.parametrize("prefix", [False, True], ids=["infix", "prefix"])
def test_k1_many_items_vs_dp_rows(ctx, oracle, k1_sets, monkeypatch, prefix):
    """The plain DP (not the oracle's Myers) on a seeded sample of rows, 64-chunk tiles."""
    texts, pats, ref = k1_sets
    rows = sorted(np.random.default_rng(7).choice(len(texts), size=10, replace=False).tolist())
    rows += [i for i, t in enumerate(texts) if t in (b"", b"N" * 512)][:3]
    Dd, Ed = oracle.score_batch([texts[r] for r in rows], pats, prefix=prefix, impl="dp", want_end_col=True)
    assert (Dd == ref[prefix][0][rows]).all() and (Ed == ref[prefix][1][rows]).all()  # the two oracle paths agree
    monkeypatch.setenv("SP_FORCE_TC", "64")
    D, E = ctx.score_batch(texts, pats, mode=sp.SP_PREFIX if prefix else sp.SP_INFIX, want_end_col=True)
    assert_same(D[rows], Dd, "dist")
    assert_same(E[rows], Ed, "end")


@pytest.mark.parametrize("env", [{"SP_MAX_CLASSES": "1"}, {"SP_MAX_CLASSES": "4"}, {"SP_FORCE_U": "4"}, {"SP_FORCE_U": "16"}],
                         ids=["classes1", "classes4", "u4", "u16"])
def test_k1_lane_classes_identical(ctx, k1_sets, monkeypatch, env):
    """One class, up to four classes, and every pattern at U = 4 or U = 16: the same matrix (64-chunk tiles)."""
    texts, pats, ref = k1_sets
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv("SP_FORCE_TC", "64")
    classes, _ = plan_lane_classes([len(p) for p in pats], int(env.get("SP_MAX_CLASSES", 4)))
    if "SP_FORCE_U" in env:
        assert [c[0] for c in classes] == [int(env["SP_FORCE_U"])]
    elif env["SP_MAX_CLASSES"] == "1":
        assert len(classes) == 1
    D, E = ctx.score_batch(texts, pats, want_end_col=True)
    assert_same(D, ref[False][0], "dist")
    assert_same(E, ref[False][1], "end")


def test_k1_share_device_full_matrix(dev, k1_sets, monkeypatch):
    """sp_ctx_share_device: one CTA per item on the low-priority side stream (more items than 2 x SMs x resident CTAs, so the
    bulk route is taken) gives the oracle's whole matrix and end columns."""
    texts, pats, ref = k1_sets
    monkeypatch.setenv("SP_FORCE_TC", "64")
    assert k1_items_lower_bound([len(t) for t in texts], [len(p) for p in pats], 64) > 2 * dev["sms"] * dev["k1_ctas_per_sm"]
    for prefix in (False, True):
        with sp.Context(0) as c:
            c.share_device(True)
            D, E = c.score_batch(texts, pats, mode=sp.SP_PREFIX if prefix else sp.SP_INFIX, want_end_col=True)
        assert_same(D, ref[prefix][0], ("dist", prefix))
        assert_same(E, ref[prefix][1], ("end", prefix))


@pytest.mark.parametrize("bits", [16, 32])
def test_k1_score_into_row_offset(ctx, oracle, k1_sets, monkeypatch, bits):
    """score_into at pattern_row0 > 0 of a wider matrix writes rows [row0, row0 + n) and leaves every other row as it was."""
    texts, pats, ref = k1_sets
    monkeypatch.setenv("SP_FORCE_TC", "64")
    rng = np.random.default_rng(bits)
    sub = [rnd(rng, int(m)) for m in rng.integers(1, 2201, size=45)] + [b"", b"NNNN", pats[3]]
    T, P, S = ctx.targets(texts), ctx.patterns(pats), ctx.patterns(sub)
    M = ctx.score_device(T, P, elem_bits=bits)
    row0 = 123
    ctx.score_into(T, S, M, pattern_row0=row0)
    got = M.to_host()
    want = ref[False][0].copy()
    want[:, row0:row0 + len(sub)] = oracle.score_batch(texts, sub)
    assert_same(got, want, "score_into")
    ctx.score_into(T, S, M, pattern_row0=len(pats) - len(sub))   # the last rows of the matrix
    want[:, len(pats) - len(sub):] = want[:, row0:row0 + len(sub)]
    assert_same(M.to_host(), want, "score_into at the end")
    with pytest.raises(sp.SpError):
        ctx.score_into(T, S, M, pattern_row0=len(pats) - len(sub) + 1)
    M.close(); S.close(); P.close(); T.close()


# ---------------------------------------------------------------------------------------------------------------------------
# 2. K1: long texts and the tile budget
# ---------------------------------------------------------------------------------------------------------------------------
def long_text(rng, pats, n):
    """n bases of random text carrying noisy copies of some patterns, the last one ending at the text's end."""
    parts, size = [], 0
    while size < n:
        p = pats[int(rng.integers(0, len(pats)))]
        s = rnd(rng, int(rng.integers(100, 3000))) + noisy_copy(rng, p, int(rng.integers(0, 30)))
        parts.append(s)
        size += len(s)
    t = b"".join(parts)[:n]
    tail = noisy_copy(rng, pats[0], 3)[-min(n, len(pats[0])):]
    return t[:n - len(tail)] + tail


def hla_patterns(n_alleles):
    alleles, _, _ = synth.hla_gene(synth.DEFAULT_SEED, "HLA-A", n_alleles=n_alleles, n_reads=2)
    return list(alleles)


@pytest.mark.parametrize("n", [40_000, pytest.param(100_000, marks=SKIP_LARGE)])
def test_k1_long_texts(ctx, oracle, n):
    """Texts above one default tile (4,096 chunks): the tile grows to the longest text and occupancy drops; distances and end
    columns bit-exact, next to short texts in the same call."""
    rng = np.random.default_rng(n)
    pats = hla_patterns(120)
    texts = [long_text(rng, pats, n), rnd(rng, 300), b"", long_text(rng, pats, n // 2 + 3), b"N" * 40]
    assert max(chunks(len(t)) for t in texts) > 4096
    D, E = ctx.score_batch(texts, pats, want_end_col=True)
    Dw, Ew = oracle.score_batch(texts, pats, want_end_col=True)
    assert_same(D, Dw, "dist")
    assert_same(E, Ew, "end")


def test_k1_long_text_widest_lane(ctx, oracle, monkeypatch):
    """SP_FORCE_U=24 with a 17 kb pattern: the largest blob (one CTA per SM) next to a tile of more than 4,096 chunks."""
    monkeypatch.setenv("SP_FORCE_U", "24")
    rng = np.random.default_rng(24)
    big = rnd(rng, 17011)
    pats = [big] + hla_patterns(30) + [noisy_copy(rng, big, 50)[:16500], b"ACGTN" * 20]
    texts = [long_text(rng, pats, 40_000), rnd(rng, 200) + noisy_copy(rng, big, 40) + rnd(rng, 24_000), rnd(rng, 1000)]
    assert max(chunks(len(t)) for t in texts) > 4096
    assert [c[0] for c in plan_lane_classes([len(p) for p in pats])[0]] == [24]
    D, E = ctx.score_batch(texts, pats, want_end_col=True)
    Dw, Ew = oracle.score_batch(texts, pats, want_end_col=True)
    assert_same(D, Dw, "dist")
    assert_same(E, Ew, "end")


def test_k1_text_beyond_budget_is_refused(ctx):
    with pytest.raises(sp.SpError) as ei:
        ctx.score_batch([b"ACGT" * 250_000], [b"ACGTACGT"])
    assert ei.value.status == 3 and "tile budget" in ei.value.message
    assert ctx.score_batch([b"TTACGT"], [b"ACGT"]).tolist() == [[0]]   # the context is still usable


@pytest.mark.parametrize("u", [4, 24])
def test_k1_tile_budget_boundary(ctx, oracle, dev, monkeypatch, u):
    """A text of exactly the budget N (from the refusal's message) is scored correctly, with a pattern copy ending in its last
    column; N + 1 bases are refused."""
    monkeypatch.setenv("SP_FORCE_U", str(u))
    rng = np.random.default_rng(u)
    pats = [rnd(rng, 17011)] if u == 24 else []
    tail = rnd(rng, 300)
    pats += [rnd(rng, int(m)) for m in rng.integers(1, 1500, size=12)] + [tail, b"ACGTN" * 30]
    with pytest.raises(sp.SpError) as ei:
        ctx.score_batch([b"A" * 10_000_000], pats)
    assert ei.value.status == 3
    N = int(re.search(r"tile budget \((\d+)\)", ei.value.message).group(1))
    assert N % (2 * K1_CHUNK) == 0 and 4096 * K1_CHUNK < N < dev["smem_optin"]
    text = rnd(rng, N - 2000) + noisy_copy(rng, pats[1], 2)
    text = (text + rnd(rng, N))[:N - len(tail)] + tail   # a copy of `tail` ends in the last column
    assert len(text) == N
    texts = [rnd(rng, 100), text, b""]
    D, E = ctx.score_batch(texts, pats, want_end_col=True)
    Dw, Ew = oracle.score_batch(texts, pats, want_end_col=True)
    assert_same(D, Dw, "dist")
    assert_same(E, Ew, "end")
    assert D[1, len(pats) - 2] == 0 and E[1, len(pats) - 2] == N
    with pytest.raises(sp.SpError) as ei:
        ctx.score_batch([text + b"A"], pats)
    assert ei.value.status == 3


# ---------------------------------------------------------------------------------------------------------------------------
# 3. K4: reused traceback scratch slots
# ---------------------------------------------------------------------------------------------------------------------------
_CODE = np.full(256, 4, dtype=np.uint8)
for _k, _c in enumerate(b"ACGT"):
    _CODE[_c] = _CODE[_c + 32] = _k


def check_cigar(p: bytes, t: bytes, r: dict):
    """The CIGAR is an alignment of P[p_start, p_end) with T[t_start, t_end): '=' runs match (N matches nothing), 'X' runs do
    not, the lengths cover both spans; dist = edits + clipped pattern ends, nm = everything but '='."""
    pc, tc = _CODE[np.frombuffer(p, np.uint8)], _CODE[np.frombuffer(t, np.uint8)]
    i, j, edits, nm = r["p_start"], r["t_start"], 0, 0
    for ln, op in r["cigar"]:
        assert ln > 0
        if op in (OP_EQ, OP_X):
            a, b = pc[i:i + ln], tc[j:j + ln]
            assert len(a) == ln and len(b) == ln
            eq = (a == b) & (a < 4)
            assert eq.all() if op == OP_EQ else not eq.any(), (op, i, j, ln)
            i, j = i + ln, j + ln
        elif op == OP_I:
            i += ln
        elif op == OP_D:
            j += ln
        else:
            raise AssertionError(f"op {op}")
        if op != OP_EQ:
            edits += ln
            nm += ln
    assert (i, j) == (r["p_end"], r["t_end"])
    assert 0 <= r["p_start"] <= r["p_end"] <= len(p) and 0 <= r["t_start"] <= r["t_end"] <= len(t)
    assert r["dist"] == edits + r["p_start"] + len(p) - r["p_end"]
    assert r["nm"] == nm


@pytest.fixture(scope="module")
def k4_workload(dev):
    """>= 1.25 x SMs x resident warps per SM pairs, one pair per bin: patterns of 2,049-2,176 bases take 17 lanes at U = 4."""
    n_pairs = math.ceil(1.25 * dev["sms"] * dev["warps_per_sm"])
    rng = np.random.default_rng(404)
    pats = [rnd(rng, int(m)) for m in rng.integers(2049, 2177, size=512)]
    texts, pairs = [], []
    for q in range(n_pairs):
        pi = int(rng.integers(0, len(pats)))
        p, kind = pats[pi], q % 10
        if kind < 7:     # noisy copy with random flanks
            t = rnd(rng, int(rng.integers(0, 61))) + noisy_copy(rng, p, int(rng.integers(0, 60))) + rnd(rng, int(rng.integers(0, 61)))
        elif kind == 7:  # the pattern's head hangs off the text's start
            t = noisy_copy(rng, p[int(rng.integers(1, 400)):], int(rng.integers(0, 20))) + rnd(rng, int(rng.integers(0, 61)))
        elif kind == 8:  # its tail hangs off the text's end
            t = rnd(rng, int(rng.integers(0, 61))) + noisy_copy(rng, p[:len(p) - int(rng.integers(1, 400))], int(rng.integers(0, 20)))
        else:            # unrelated
            t = rnd(rng, int(rng.integers(1500, 2300)))
        texts.append(t)
        pairs.append((q, pi))
    assert all(-(-len(p) // 128) == 17 for p in pats)   # 17 lanes of 4 x 32 rows: no two pairs share a bin
    assert n_pairs >= 1.25 * dev["sms"] * dev["warps_per_sm"]
    return texts, pats, pairs


def test_k4_reused_slots_vs_oracle(ctx, oracle, k4_workload):
    """Every pair: dist / t_end equal the oracle's Myers, the CIGAR is a valid alignment worth dist; a seeded sample of ~300
    pairs equals the oracle's canonical traceback in full."""
    texts, pats, pairs = k4_workload
    got = ctx.align_pairs(texts, pats, pairs)
    assert len(got) == len(pairs)
    for (t, p), g in zip(pairs, got):
        d, e = oracle.infix(pats[p], texts[t], impl="myers")
        assert (g["dist"], g["t_end"]) == (d, e), (t, p, g["dist"], d, g["t_end"], e)
        check_cigar(pats[p], texts[t], g)
    for q in np.random.default_rng(5).choice(len(pairs), size=300, replace=False):
        t, p = pairs[int(q)]
        want = oracle.align(pats[p], texts[t])
        assert got[int(q)] == want, (int(q), {k: (got[int(q)][k], want[k]) for k in want if k != "cigar" and got[int(q)][k] != want[k]})


def test_k4_sliced_submission_identical(ctx, dev, k4_workload):
    """The same pairs in calls of fewer pairs than SMs (a slot per pair, no reuse) give byte-identical records and CIGARs."""
    texts, pats, pairs = k4_workload
    whole = ctx.align_pairs(texts, pats, pairs)
    step = dev["sms"]
    for lo in range(0, len(pairs), step):
        part = ctx.align_pairs(texts, pats, pairs[lo:lo + step])
        assert part == whole[lo:lo + step], lo


# ---------------------------------------------------------------------------------------------------------------------------
# 4. K9: reused trace slots, four width classes at volume
# ---------------------------------------------------------------------------------------------------------------------------
K9_CLASSES = ((1, 31), (32, 63), (64, 127), (128, 255))


def k9_pair(rng, W):
    """(pattern, text, centre) of one of several shapes; W is the pair's band half-width."""
    kind = int(rng.integers(0, 12))
    m = int(rng.integers(100, 401))
    p = rnd(rng, m)
    left = int(rng.integers(0, 61))
    if kind <= 3:          # noisy copy inside flanks, band centred on its start diagonal
        t = rnd(rng, left) + noisy_copy(rng, p, int(rng.integers(0, 12))) + rnd(rng, int(rng.integers(0, 61)))
        c = left + int(rng.integers(-3, 4))
    elif kind == 4:        # a gap of 19, 20 or 21 bases: either side of the two-piece crossover 6 + 2k = 26 + k at k = 20
        k, a = int(rng.integers(19, 22)), int(rng.integers(30, m - 40))
        t = rnd(rng, left) + (p[:a] + p[a + k:] if rng.random() < 0.5 else p[:a] + rnd(rng, k) + p[a:]) + rnd(rng, 20)
        c = left
    elif kind == 5:        # N in pattern and text
        b = bytearray(p)
        for pos in rng.integers(0, m, size=m // 30):
            b[int(pos)] = ord("N")
        p = bytes(b)
        tb = bytearray(noisy_copy(rng, p, 5))
        for pos in rng.integers(0, max(len(tb), 1), size=len(tb) // 40):
            tb[int(pos)] = ord("N")
        t, c = rnd(rng, left) + bytes(tb), left
    elif kind == 6:        # band partly outside the matrix: centre near -m or near n
        t = rnd(rng, left) + noisy_copy(rng, p, 4)
        c = -m + int(rng.integers(0, W + 1)) if rng.random() < 0.5 else len(t) - int(rng.integers(0, W + 1))
    elif kind == 7:        # best score 0: no base in the band can match
        t = b"N" * int(rng.integers(0, 300)) if rng.random() < 0.5 else rnd(rng, 200)
        c = 0 if t[:1] in (b"", b"N") else len(t) + W + 1 + int(rng.integers(0, 5))
    elif kind == 8:        # periodic: equal maxima on several diagonals (the end-cell tie rule decides)
        unit = rnd(rng, int(rng.integers(2, 6)))
        p = (unit * 100)[:m]
        t = (unit * 200)[:m + int(rng.integers(0, 2 * W + 1))]
        c = int(rng.integers(0, W + 1))
    elif kind == 9:        # two equally good copies of a short pattern inside one band
        p = p[:100]
        gap = int(rng.integers(0, W + 1))
        t = rnd(rng, left) + p + rnd(rng, gap) + p + rnd(rng, left)
        c = left + (100 + gap) // 2
    elif kind == 10:       # unrelated
        t, c = rnd(rng, int(rng.integers(50, 450))), int(rng.integers(-50, 100))
    else:                  # the pattern overhangs both text ends
        s = int(rng.integers(10, 60))
        t = noisy_copy(rng, p[s:m - s], 6)
        c = -s
    return p, t, c


@pytest.fixture(scope="module")
def k9_workload(dev):
    """Per width class more pairs than SMs x resident warps per SM (an upper bound on its trace slots)."""
    per_class = dev["sms"] * dev["warps_per_sm"] + dev["sms"]
    rng = np.random.default_rng(909)
    pats, texts, pairs, centres, bands = [], [], [], [], []
    for q in range(per_class * len(K9_CLASSES)):
        lo, hi = K9_CLASSES[q % 4]
        W = (lo, hi)[q // 4 % 2] if q < 64 else int(rng.integers(lo, hi + 1))
        p, t, c = k9_pair(rng, W)
        pats.append(p); texts.append(t); pairs.append((q, q)); centres.append(c); bands.append(W)
    per = np.bincount([next(k for k, (lo, hi) in enumerate(K9_CLASSES) if lo <= w <= hi) for w in bands], minlength=4)
    assert (per > dev["sms"] * dev["warps_per_sm"]).all(), per
    return texts, pats, pairs, centres, bands


def k9_expected(aff, pats, texts, pairs, centres, bands):
    out = []
    for (t, p), c, b in zip(pairs, centres, bands):
        want = aff.align(pats[p], texts[t], centre=c, band=b)
        out.append(dict(want, dist=len(pats[p])) if want["score"] == 0 else want)
        aff.cache.clear()
    return out


@SKIP_LARGE
def test_k9_reused_slots_four_classes(ctx, k9_workload):
    """All four width classes side by side in one call, sharing one record array and one dense CIGAR pool: every record, score
    and CIGAR entry equals the banded CPU model; map-hifi costs on a quarter of the pairs."""
    texts, pats, pairs, centres, bands = k9_workload
    T, P = ctx.targets(texts), ctx.targets(pats)
    for costs, take in ((ou.COSTS_ALLELE_SCORING, slice(None)), (ou.COSTS_MAP_HIFI, slice(0, None, 4))):
        pr, ce, bd = pairs[take], centres[take], bands[take]
        got = ctx.align_affine(T, P, pr, costs, centres=ce, bands=bd)
        want = k9_expected(ou.AffineOracle(costs), pats, texts, pr, ce, bd)
        bad = [q for q in range(len(pr)) if got[q] != want[q]]
        assert not bad, (costs, len(bad), [(q, bd[q], ce[q], {k: (got[q][k], want[q][k]) for k in want[q] if k != "cigar" and got[q][k] != want[q][k]})
                                           for q in bad[:5]])
        assert sum(g["score"] == 0 for g in got) > 0 and sum(g["score"] > 0 for g in got) > len(got) // 2
    T.close(); P.close()


@SKIP_LARGE
def test_k9_sliced_submission_identical(ctx, dev, k9_workload):
    """The same pairs in calls of fewer than SMs pairs per class (a slot per pair) give identical records, scores and CIGARs."""
    texts, pats, pairs, centres, bands = k9_workload
    T, P = ctx.targets(texts), ctx.targets(pats)
    costs = ou.COSTS_ALLELE_SCORING
    whole = ctx.align_affine(T, P, pairs, costs, centres=centres, bands=bands)
    step = 4 * dev["sms"] - 4
    for lo in range(0, len(pairs), step):
        sl = slice(lo, lo + step)
        assert ctx.align_affine(T, P, pairs[sl], costs, centres=centres[sl], bands=bands[sl]) == whole[sl], lo
    T.close(); P.close()
