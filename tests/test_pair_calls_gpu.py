"""GPU suite: the pair-call contract K4 (sp_align_resident) and K9 (sp_align_affine_resident) share (include/starphase_gpu.h).
Both refuse the same bad pair lists, and when the CIGARs need more than cigar_cap entries both fail with SP_ERR_RANGE, report the
need in *cigar_used and leave recs, scores and cigar exactly as they were."""
import ctypes as C

import numpy as np
import pytest

import oracle_util as ou
import pb_starphase_b200 as sp
from pb_starphase_b200.binding import AlignRec
from test_k3_gpu import noisy, rnd

pytestmark = pytest.mark.gpu

SP_ERR_INVALID, SP_ERR_RANGE = 1, 5
FILL = 0xA5  # sentinel byte of every output buffer


@pytest.fixture(scope="module")
def seqs():
    """Texts holding noisy copies of three patterns of different lane widths, and an empty pattern."""
    rng = np.random.default_rng(77)
    pats = [rnd(rng, m) for m in (150, 900, 5000)] + [b""]
    texts = [rnd(rng, 40) + noisy(rng, p, 6) + rnd(rng, 60) for p in pats[:3]]
    pairs = [(0, 0), (1, 1), (2, 2), (0, 3), (1, 0), (2, 1), (2, 3)]
    return texts, pats, pairs


def align(ctx, kernel, texts, pats, pairs, windows=None):
    if kernel == "k4":
        return ctx.align_pairs(texts, pats, pairs, windows=windows)
    T, P = ctx.targets(texts), ctx.targets(pats)
    try:
        return ctx.align_affine(T, P, pairs, ou.COSTS_MAP_HIFI, windows=windows)
    finally:
        T.close(); P.close()


@pytest.mark.parametrize("kernel", ["k4", "k9"])
def test_same_refusals(ctx, seqs, kernel):
    texts, pats, _ = seqs
    with pytest.raises(sp.SpError) as ei:
        align(ctx, kernel, texts, pats, [(len(texts), 0)])
    assert ei.value.status == SP_ERR_INVALID
    with pytest.raises(sp.SpError) as ei:
        align(ctx, kernel, texts, pats, [(0, len(pats))])
    assert ei.value.status == SP_ERR_INVALID
    for bad in ((-1, 10), (10, 5), (0, len(texts[0]) + 1)):
        with pytest.raises(sp.SpError) as ei:
            align(ctx, kernel, texts, pats, [(0, 0)], windows=[bad])
        assert ei.value.status == SP_ERR_INVALID, bad
    assert align(ctx, kernel, texts, pats, []) == []


def raw_call(ctx, kernel, T, P, pairs, cap):
    """One call through the C ABI into buffers filled with FILL: (status, cigar_used, recs bytes, scores, cigar)."""
    n = len(pairs)
    pt = np.ascontiguousarray([t for t, _ in pairs], dtype=np.int32)
    pp = np.ascontiguousarray([p for _, p in pairs], dtype=np.int32)
    recs = (AlignRec * n)()
    C.memset(recs, FILL, C.sizeof(recs))
    scores = np.full(4 * n, FILL, dtype=np.uint8).view(np.int32)
    cig = np.full(4 * max(cap, 1), FILL, dtype=np.uint8).view(np.uint32)
    used = C.c_int64(-1)
    if kernel == "k4":
        st = ctx._lib.sp_align_resident(ctx._h, T._h, P._h, n, pt.ctypes.data, pp.ctypes.data, None, None, recs, cig.ctypes.data, cap,
                                        C.byref(used))
    else:
        costs = np.ascontiguousarray(ou.COSTS_MAP_HIFI, dtype=np.int32)
        st = ctx._lib.sp_align_affine_resident(ctx._h, T._h, P._h, n, pt.ctypes.data, pp.ctypes.data, None, None, None, 64, None,
                                               costs.ctypes.data, recs, scores.ctypes.data, cig.ctypes.data, cap, C.byref(used))
    return st, used.value, bytes(recs), scores, cig


def per_pair(recs_bytes, cig):
    """Every record without cigar_off, and its CIGAR entries (the order of the pairs inside the pool is unspecified)."""
    recs = (AlignRec * (len(recs_bytes) // C.sizeof(AlignRec))).from_buffer_copy(recs_bytes)
    return [((r.dist, r.nm, r.p_start, r.p_end, r.t_start, r.t_end, r.n_cigar, r._pad), cig[r.cigar_off:r.cigar_off + r.n_cigar].tolist())
            for r in recs]


@pytest.mark.parametrize("kernel", ["k4", "k9"])
def test_range_error_writes_nothing(ctx, seqs, kernel):
    texts, pats, pairs = seqs
    T, P = ctx.targets(texts), ctx.targets(pats)
    try:
        st, need, recs0, scores0, cig0 = raw_call(ctx, kernel, T, P, pairs, 1 << 20)
        assert st == 0 and 0 < need < 1 << 20
        want = per_pair(recs0, cig0)
        for q, (t, p) in enumerate(pairs):
            if not pats[p]:  # empty pattern: the empty placement, score 0
                assert want[q] == ((0,) * 8, [])
                assert kernel == "k4" or scores0[q] == 0

        st, used, recs, scores, cig = raw_call(ctx, kernel, T, P, pairs, need - 1)
        assert st == SP_ERR_RANGE and used == need
        assert recs == bytes([FILL]) * len(recs)
        assert scores.view(np.uint8).tolist() == [FILL] * scores.nbytes
        assert cig.view(np.uint8).tolist() == [FILL] * cig.nbytes

        st, used, recs, scores, cig = raw_call(ctx, kernel, T, P, pairs, need)
        assert st == 0 and used == need
        assert per_pair(recs, cig) == want
        if kernel == "k9":
            assert scores.tolist() == scores0.tolist()
    finally:
        T.close(); P.close()
