"""ctypes mirror of include/starphase_gpu.h.

This is the binding a Python host would use; the Rust host of the reference binds the same
symbols through rust/starphase-gpu-sys (see INTEGRATION.md).  Nothing here computes on the
CPU: a missing library or a missing GPU raises SpError.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path
from typing import Optional, Sequence, Tuple

import numpy as np

SP_INFIX, SP_PREFIX = 0, 1
_STATUS = {0: "SP_OK", 1: "SP_ERR_INVALID", 2: "SP_ERR_CUDA", 3: "SP_ERR_TOO_LONG", 4: "SP_ERR_NOMEM", 5: "SP_ERR_RANGE"}


class SpError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"{_STATUS.get(status, status)}: {message}")
        self.status = status
        self.message = message


class SeqSet(C.Structure):
    _fields_ = [("bases", C.c_void_p), ("offsets", C.c_void_p), ("n", C.c_int64)]


class PairRec(C.Structure):
    _fields_ = [("score", C.c_uint64), ("score2", C.c_uint64), ("i", C.c_uint32), ("j", C.c_uint32), ("c1", C.c_uint32), ("_pad", C.c_uint32)]


class AlignRec(C.Structure):
    _fields_ = [("dist", C.c_int32), ("nm", C.c_int32), ("p_start", C.c_int32), ("p_end", C.c_int32),
                ("t_start", C.c_int32), ("t_end", C.c_int32), ("n_cigar", C.c_int32), ("_pad", C.c_int32),
                ("cigar_off", C.c_int64)]


def lib_path() -> Path:
    # $SP_GPU_LIB: another build of the same library (A/B runs of a kernel variant on the GPU box)
    over = os.environ.get("SP_GPU_LIB")
    return Path(over) if over else Path(__file__).resolve().parent / "libstarphase_gpu.so"


_lib = None

# name -> (restype, argtypes); every symbol include/starphase_gpu.h declares
_P = C.c_void_p
SIGNATURES = {
    "sp_ctx_create": (C.c_int, [C.c_int, _P, C.POINTER(_P)]),
    "sp_ctx_destroy": (None, [_P]),
    "sp_last_error": (C.c_char_p, [_P]),
    "sp_last_kernel_ms": (C.c_float, [_P, C.c_int]),
    "sp_launch_count": (C.c_uint64, [_P]),
    "sp_ctx_synchronize": (C.c_int, [_P]),
    "sp_ctx_share_device": (C.c_int, [_P, C.c_int]),
    "sp_pinned_alloc": (C.c_int, [_P, C.c_size_t, C.POINTER(_P)]),
    "sp_pinned_free": (None, [_P, _P]),
    "sp_patterns_create": (C.c_int, [_P, C.POINTER(SeqSet), C.c_int, C.POINTER(_P)]),
    "sp_patterns_destroy": (None, [_P]),
    "sp_patterns_count": (C.c_int64, [_P]),
    "sp_patterns_total_len": (C.c_int64, [_P]),
    "sp_patterns_padded_rows": (C.c_int64, [_P]),
    "sp_plan_lane_classes": (C.c_int, [_P, C.c_int64, C.c_int, C.POINTER(C.c_int), _P, _P, _P, C.POINTER(C.c_int64)]),
    "sp_targets_create": (C.c_int, [_P, C.POINTER(SeqSet), C.POINTER(_P)]),
    "sp_targets_derive": (C.c_int, [_P, _P, C.c_int64, _P, _P, _P, _P, _P, C.POINTER(_P)]),
    "sp_targets_read": (C.c_int, [_P, _P, _P]),
    "sp_targets_destroy": (None, [_P]),
    "sp_targets_count": (C.c_int64, [_P]),
    "sp_targets_total_len": (C.c_int64, [_P]),
    "sp_score_device": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(_P)]),
    "sp_score_into": (C.c_int, [_P, _P, _P, _P, C.c_int64]),
    "sp_dmatrix_destroy": (None, [_P]),
    "sp_dmatrix_to_host": (C.c_int, [_P, _P, _P, _P]),
    "sp_dmatrix_to_host_u16": (C.c_int, [_P, _P, _P]),
    "sp_host_alloc": (C.c_int, [_P, C.c_size_t, C.POINTER(_P)]),
    "sp_host_free": (None, [_P, _P]),
    "sp_dmatrix_device_ptr": (_P, [_P]),
    "sp_dmatrix_ld": (C.c_int64, [_P]),
    "sp_dmatrix_elem_bits": (C.c_int, [_P]),
    "sp_dmatrix_wrap": (C.c_int, [_P, _P, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.POINTER(_P)]),
    "sp_score_batch": (C.c_int, [_P, C.POINTER(SeqSet), C.POINTER(SeqSet), C.c_int, _P, _P]),
    "sp_score_spans": (C.c_int, [_P, C.POINTER(SeqSet), C.POINTER(SeqSet), _P, _P, _P]),
    "sp_score_spans_filtered": (C.c_int, [_P, C.POINTER(SeqSet), C.POINTER(SeqSet), C.c_int, _P, _P, _P]),
    "sp_align_pairs": (C.c_int, [_P, C.POINTER(SeqSet), C.POINTER(SeqSet), C.c_int64, _P, _P, C.POINTER(AlignRec), _P, C.c_int64,
                                 C.POINTER(C.c_int64)]),
    "sp_align_windows": (C.c_int, [_P, C.POINTER(SeqSet), C.POINTER(SeqSet), C.c_int64, _P, _P, _P, _P, C.POINTER(AlignRec), _P, C.c_int64,
                                   C.POINTER(C.c_int64)]),
    "sp_align_resident": (C.c_int, [_P, _P, _P, C.c_int64, _P, _P, _P, _P, C.POINTER(AlignRec), _P, C.c_int64, C.POINTER(C.c_int64)]),
    "sp_align_affine_resident": (C.c_int, [_P, _P, _P, C.c_int64, _P, _P, _P, _P, _P, C.c_int32, _P, _P, C.POINTER(AlignRec), _P, _P, C.c_int64,
                                           C.POINTER(C.c_int64)]),
    "sp_row_topk": (C.c_int, [_P, _P, C.c_int, _P, _P]),
    "sp_row_topk_biased": (C.c_int, [_P, _P, _P, C.c_int, _P, _P]),
    "sp_row_topk_weighted": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, _P]),
    "sp_variant_match": (C.c_int, [_P, C.c_int64, C.c_int64, C.c_int64, _P, _P, _P, _P, _P]),
    "sp_chain_window_scores": (C.c_int, [_P, C.c_int64, _P, _P, C.c_int64, _P, _P, C.c_int64, C.POINTER(_P)]),
    "sp_pair_minsum_topk": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, C.c_int, C.POINTER(PairRec), C.POINTER(C.c_int)]),
    "sp_pair_minsum_full": (C.c_int, [_P, _P, _P]),
    "sp_pair_minsum_topk_host": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, C.c_int, C.POINTER(PairRec), C.POINTER(C.c_int)]),
    "sp_pair_minsum_full_host": (C.c_int, [_P, _P, C.c_int64, C.c_int64, _P]),
    "sp_consensus_create": (C.c_int, [_P, C.POINTER(SeqSet), _P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_P)]),
    "sp_consensus_destroy": (None, [_P]),
    "sp_consensus_num_reads": (C.c_int32, [_P]),
    "sp_consensus_num_tracks": (C.c_int32, [_P]),
    "sp_consensus_reset": (C.c_int, [_P, C.c_int32]),
    "sp_consensus_extend": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "sp_consensus_run_supported": (C.c_int32, [_P, C.c_int32]),
    "sp_consensus_run": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_int64, C.c_int32, _P,
                         C.POINTER(C.c_int32)]),
    "sp_graph_align": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int32, _P, _P]),
    "sp_comm_unique_id": (C.c_int, [_P]),
    "sp_comm_create": (C.c_int, [_P, _P, C.c_int, C.c_int, C.POINTER(_P)]),
    "sp_comm_destroy": (None, [_P]),
    "sp_comm_rank": (C.c_int, [_P]),
    "sp_comm_world": (C.c_int, [_P]),
    "sp_comm_barrier": (C.c_int, [_P]),
    "sp_shard_plan": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int, _P, C.POINTER(C.c_int64)]),
    "sp_triangle_rows": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "sp_comm_bcast_targets": (C.c_int, [_P, C.POINTER(SeqSet), C.c_int, C.POINTER(_P)]),
    "sp_comm_score_allgather": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int, C.POINTER(_P)]),
    "sp_comm_pair_minsum_topk": (C.c_int, [_P, _P, _P, C.c_int, C.POINTER(PairRec), C.POINTER(C.c_int)]),
    "sp_int_peak": (C.c_int, [_P, C.c_int, C.POINTER(C.c_double)]),
    "sp_version": (C.c_char_p, []),
}


def load_library():
    """Loads libstarphase_gpu.so (built in-tree by pb_starphase_b200.build).  Fails loudly if it
    is missing: there is no eager / CPU path to fall back to."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not path.exists():
        raise SpError(2, f"{path} is missing -- run `python -m pb_starphase_b200.build` (there is no CPU fallback)")
    lib = C.CDLL(str(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def pack_sequences(seqs: Sequence[bytes]) -> Tuple[np.ndarray, np.ndarray]:
    """list of bytes -> (uint8 bases, int64 offsets[n+1]) in the sp_seqset layout."""
    offs = np.zeros(len(seqs) + 1, dtype=np.int64)
    if len(seqs):
        np.cumsum([len(s) for s in seqs], out=offs[1:])
    joined = b"".join(bytes(s) for s in seqs)
    bases = np.frombuffer(joined, dtype=np.uint8).copy() if joined else np.zeros(1, dtype=np.uint8)
    return bases, offs


def plan_lane_classes(lens, max_classes: int = 4):
    """Host-only: the lane-width classes sp_patterns_create would use for patterns of these lengths.
    Returns ([(width, n_patterns, n_warps), ...], padded_rows)."""
    lib = load_library()
    a = np.ascontiguousarray(lens, dtype=np.int64)
    nc = C.c_int(0)
    w = np.zeros(max_classes, dtype=np.int32)
    npat = np.zeros(max_classes, dtype=np.int64)
    nw = np.zeros(max_classes, dtype=np.int64)
    padded = C.c_int64(0)
    st = lib.sp_plan_lane_classes(a.ctypes.data, len(a), max_classes, C.byref(nc), w.ctypes.data, npat.ctypes.data,
                                  nw.ctypes.data, C.byref(padded))
    if st != 0:
        raise SpError(st, "sp_plan_lane_classes failed")
    return [(int(w[k]), int(npat[k]), int(nw[k])) for k in range(nc.value)], int(padded.value)


def shard_plan(lens, world: int, rank: int) -> np.ndarray:
    """Host-only (sp_shard_plan): ascending database indices of the patterns rank `rank` of `world` owns."""
    lib = load_library()
    a = np.ascontiguousarray(lens, dtype=np.int64)
    idx = np.zeros(max(len(a), 1), dtype=np.int64)
    n = C.c_int64(0)
    st = lib.sp_shard_plan(a.ctypes.data, len(a), world, rank, idx.ctypes.data, C.byref(n))
    if st != 0:
        raise SpError(st, "sp_shard_plan failed")
    return idx[: n.value].copy()


def triangle_rows(n: int, world: int, rank: int) -> Tuple[int, int]:
    """Host-only (sp_triangle_rows): row range of the pair triangle scored by `rank`."""
    lib = load_library()
    lo, hi = C.c_int64(0), C.c_int64(0)
    st = lib.sp_triangle_rows(n, world, rank, C.byref(lo), C.byref(hi))
    if st != 0:
        raise SpError(st, "sp_triangle_rows failed")
    return int(lo.value), int(hi.value)


def comm_unique_id() -> bytes:
    """sp_comm_unique_id: 128 bytes drawn on rank 0, to be carried to the other ranks by the host program."""
    lib = load_library()
    buf = (C.c_uint8 * 128)()
    st = lib.sp_comm_unique_id(buf)
    if st != 0:
        raise SpError(st, lib.sp_last_error(None).decode())
    return bytes(buf)


def _seqset(bases: np.ndarray, offs: np.ndarray) -> SeqSet:
    assert bases.dtype == np.uint8 and offs.dtype == np.int64 and bases.flags.c_contiguous and offs.flags.c_contiguous
    return SeqSet(bases.ctypes.data, offs.ctypes.data, len(offs) - 1)


class Context:
    """sp_ctx: one per process per GPU."""

    def __init__(self, device: int = 0, stream: Optional[int] = None):
        self._lib = load_library()
        h = _P()
        st = self._lib.sp_ctx_create(device, _P(stream) if stream else None, C.byref(h))
        if st != 0:
            raise SpError(st, self._lib.sp_last_error(None).decode())
        self._h = h
        self.device = device
        self._pinned = []

    def _check(self, st: int):
        if st != 0:
            raise SpError(st, self._lib.sp_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None):
            for ptr in self._pinned:
                self._lib.sp_host_free(self._h, ptr)
            self._pinned = []
            self._lib.sp_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- K1 ---------------------------------------------------------------------------------
    def patterns(self, seqs, mode: int = SP_INFIX) -> "PatternSet":
        return PatternSet(self, seqs, mode)

    def targets(self, seqs) -> "TargetSet":
        return TargetSet(self, seqs)

    def score_device(self, targets: "TargetSet", patterns: "PatternSet", elem_bits: int = 16,
                     want_end_col: bool = False) -> "DMatrix":
        h = _P()
        self._check(self._lib.sp_score_device(self._h, targets._h, patterns._h, elem_bits, int(want_end_col), C.byref(h)))
        return DMatrix(self, h, targets.n, patterns.n, want_end_col)

    def score_into(self, targets: "TargetSet", patterns: "PatternSet", dst: "DMatrix", pattern_row0: int = 0):
        self._check(self._lib.sp_score_into(self._h, targets._h, patterns._h, dst._h, pattern_row0))

    def score_batch(self, targets, patterns, mode: int = SP_INFIX, want_end_col: bool = False):
        """Host buffers in, host int32 matrix out: D[t, p] (and end columns).  One C-ABI call."""
        tb, to = targets if isinstance(targets, tuple) else pack_sequences(targets)
        pb, po = patterns if isinstance(patterns, tuple) else pack_sequences(patterns)
        nt, np_ = len(to) - 1, len(po) - 1
        D = np.empty((nt, np_), dtype=np.int32)
        E = np.empty((nt, np_), dtype=np.int32) if want_end_col else None
        ts, ps = _seqset(tb, to), _seqset(pb, po)
        self._check(self._lib.sp_score_batch(self._h, C.byref(ts), C.byref(ps), mode, D.ctypes.data,
                                             E.ctypes.data if E is not None else None))
        return (D, E) if want_end_col else D

    def score_spans(self, targets, patterns, max_dist_permille: int = -1):
        """K3: (D, start_col, end_col), each [n_targets, n_patterns] int32; the optimal placement of pattern p
        covers text columns [start, end) of target t.  With max_dist_permille >= 0, pairs with D * 1000 > |P| * that
        get start_col = -1 (no reverse pass)."""
        tb, to = targets if isinstance(targets, tuple) else pack_sequences(targets)
        pb, po = patterns if isinstance(patterns, tuple) else pack_sequences(patterns)
        nt, np_ = len(to) - 1, len(po) - 1
        D, S, E = (np.zeros((nt, np_), dtype=np.int32) for _ in range(3))
        ts, ps = _seqset(tb, to), _seqset(pb, po)
        self._check(self._lib.sp_score_spans_filtered(self._h, C.byref(ts), C.byref(ps), int(max_dist_permille), D.ctypes.data,
                                                      S.ctypes.data, E.ctypes.data))
        return D, S, E

    def align_pairs(self, targets, patterns, pairs, windows=None):
        """K4: traceback alignment of the listed (target index, pattern index) pairs.  Returns one dict per pair with
        the minimap2::Mapping fields the reference reads (src/hla/processed_match.rs:53-100): dist, nm,
        p_start/p_end (pattern = minimap2's query), t_start/t_end (text = its target) and cigar = [(len, op), ...]
        with BAM op codes 1 = I, 2 = D, 7 = '=', 8 = X.  windows (optional, [n_pairs, 2] = begin, end): align inside that
        part of the text only (sp_align_windows); t_start / t_end are then relative to begin."""
        tb, to = targets if isinstance(targets, tuple) else pack_sequences(targets)
        pb, po = patterns if isinstance(patterns, tuple) else pack_sequences(patterns)
        pairs = np.ascontiguousarray(np.asarray(pairs, dtype=np.int32).reshape(-1, 2))
        n = len(pairs)
        pt, pp = np.ascontiguousarray(pairs[:, 0]), np.ascontiguousarray(pairs[:, 1])
        tl, pl = np.diff(to), np.diff(po)
        ok = n and pt.min() >= 0 and pt.max() < len(tl) and pp.min() >= 0 and pp.max() < len(pl)  # else the library rejects it
        wb = we = None
        if windows is not None:
            w = np.ascontiguousarray(np.asarray(windows, dtype=np.int32).reshape(-1, 2))
            if len(w) != n:
                raise ValueError("align_pairs: one window per pair expected")
            wb, we = np.ascontiguousarray(w[:, 0]), np.ascontiguousarray(w[:, 1])
        nl = (we - wb).astype(np.int64) if wb is not None else (tl[pt] if ok else None)
        cap = int((pl[pp] + np.minimum(np.maximum(nl, 0), 2 * pl[pp]) + 1).sum()) if ok else 0
        recs = (AlignRec * max(n, 1))()
        cig = np.zeros(max(cap, 1), dtype=np.uint32)
        used = C.c_int64(0)
        ts, ps = _seqset(tb, to), _seqset(pb, po)
        self._check(self._lib.sp_align_windows(self._h, C.byref(ts), C.byref(ps), n, pt.ctypes.data, pp.ctypes.data,
                                               wb.ctypes.data if wb is not None else None, we.ctypes.data if we is not None else None,
                                               recs, cig.ctypes.data, cap, C.byref(used)))
        out = []
        for r in recs[:n]:
            c = cig[r.cigar_off:r.cigar_off + r.n_cigar]
            out.append({"dist": r.dist, "nm": r.nm, "p_start": r.p_start, "p_end": r.p_end, "t_start": r.t_start,
                        "t_end": r.t_end, "cigar": [(int(x) >> 4, int(x) & 15) for x in c]})
        return out

    def align_affine(self, texts: "TargetSet", patterns: "TargetSet", pairs, costs, band: int = 64, centres=None, windows=None, bands=None):
        """K9: best local alignment of each (text index, pattern index) pair under two-piece affine costs (a, b, q, e, q2, e2), inside
        the diagonal band |(j - i) - centre| <= band (`bands`: one half width per pair instead).  Returns dicts like align_pairs
        plus `score`."""
        pairs = np.ascontiguousarray(np.asarray(pairs, dtype=np.int32).reshape(-1, 2))
        n = len(pairs)
        pt, pp = np.ascontiguousarray(pairs[:, 0]), np.ascontiguousarray(pairs[:, 1])
        cen = np.ascontiguousarray(centres, dtype=np.int32) if centres is not None else None
        pb = np.ascontiguousarray(bands, dtype=np.int32) if bands is not None else None
        if pb is not None and pb.shape != (n,):
            raise ValueError("align_affine: one band per pair expected")
        wb = we = None
        if windows is not None:
            w = np.ascontiguousarray(np.asarray(windows, dtype=np.int32).reshape(-1, 2))
            wb, we = np.ascontiguousarray(w[:, 0]), np.ascontiguousarray(w[:, 1])
        cst = np.ascontiguousarray(costs, dtype=np.int32)
        recs = (AlignRec * max(n, 1))()
        scores = np.zeros(max(n, 1), dtype=np.int32)
        cap = max(1 << 16, n * 1024)
        for _ in range(2):
            cig = np.zeros(cap, dtype=np.uint32)
            used = C.c_int64(0)
            st = self._lib.sp_align_affine_resident(self._h, texts._h, patterns._h, n, pt.ctypes.data, pp.ctypes.data,
                                                    wb.ctypes.data if wb is not None else None, we.ctypes.data if we is not None else None,
                                                    cen.ctypes.data if cen is not None else None, band, pb.ctypes.data if pb is not None else None,
                                                    cst.ctypes.data, recs, scores.ctypes.data,
                                                    cig.ctypes.data, cap, C.byref(used))
            if st == 5 and used.value > cap:
                cap = used.value
                continue
            self._check(st)
            break
        out = []
        for q, r in enumerate(recs[:n]):
            c = cig[r.cigar_off:r.cigar_off + r.n_cigar]
            out.append({"dist": r.dist, "nm": r.nm, "p_start": r.p_start, "p_end": r.p_end, "t_start": r.t_start, "t_end": r.t_end,
                        "cigar": [(int(x) >> 4, int(x) & 15) for x in c], "score": int(scores[q])})
        return out

    def row_topk(self, d: "DMatrix", k: int = 5, bias=None, weight: int = 1):
        """K5: (idx, dist), each [n_targets, k] int32: the k best patterns of every target by (weight * distance [+ bias[p]], index)."""
        idx = np.zeros((d.n_targets, k), dtype=np.int32)
        dist = np.zeros((d.n_targets, k), dtype=np.int32)
        if weight != 1:
            b = np.ascontiguousarray(bias if bias is not None else np.zeros(d.n_patterns), dtype=np.int32)
            if b.shape != (d.n_patterns,):
                raise ValueError("row_topk: bias must have one entry per pattern")
            self._check(self._lib.sp_row_topk_weighted(self._h, d._h, int(weight), b.ctypes.data, k, idx.ctypes.data, dist.ctypes.data))
        elif bias is None:
            self._check(self._lib.sp_row_topk(self._h, d._h, k, idx.ctypes.data, dist.ctypes.data))
        else:
            b = np.ascontiguousarray(bias, dtype=np.int32)
            if b.shape != (d.n_patterns,):
                raise ValueError("row_topk: bias must have one entry per pattern")
            self._check(self._lib.sp_row_topk_biased(self._h, d._h, b.ctypes.data, k, idx.ctypes.data, dist.ctypes.data))
        return idx, dist

    def variant_match(self, seq_alleles, hap_alleles, is_vi):
        """K6: (vi_match, all_match), each [n_seq, n_hap] uint32, for site-state rows seq_alleles [n_seq, n_var] (0 REF, 1 ALT,
        2 ambiguous, 3 unset), haplotype definitions hap_alleles [n_hap, n_var] (0 / 1) and the VI flags is_vi [n_var]."""
        sa = np.ascontiguousarray(seq_alleles, dtype=np.uint8)
        ha = np.ascontiguousarray(hap_alleles, dtype=np.uint8)
        vi = np.ascontiguousarray(is_vi, dtype=np.uint8)
        if sa.ndim != 2 or ha.ndim != 2 or vi.ndim != 1 or sa.shape[1] != vi.shape[0] or ha.shape[1] != vi.shape[0]:
            raise ValueError("variant_match: expected [n_seq, n_var], [n_hap, n_var], [n_var]")
        vm = np.zeros((sa.shape[0], ha.shape[0]), dtype=np.uint32)
        am = np.zeros((sa.shape[0], ha.shape[0]), dtype=np.uint32)
        self._check(self._lib.sp_variant_match(self._h, sa.shape[0], ha.shape[0], vi.shape[0], sa.ctypes.data, ha.ctypes.data,
                                               vi.ctypes.data, vm.ctypes.data, am.ctypes.data))
        return vm, am

    def chain_window_scores(self, chains, read_weights, n_haps: int) -> "DMatrix":
        """K3 chain windows.  chains: list of lists of haplotype indices; read_weights: per read an array
        [n_segments_of_read, n_haps] of edit distances.  Returns the device matrix B (chains x reads)."""
        coff = np.zeros(len(chains) + 1, dtype=np.int32)
        if len(chains):
            np.cumsum([len(c) for c in chains], out=coff[1:])
        items = np.ascontiguousarray(np.concatenate([np.asarray(c, dtype=np.int32) for c in chains]) if len(chains) and coff[-1] else np.zeros(1, np.int32), dtype=np.int32)
        soff = np.zeros(len(read_weights) + 1, dtype=np.int32)
        if len(read_weights):
            np.cumsum([len(w) for w in read_weights], out=soff[1:])
        W = (np.ascontiguousarray(np.concatenate([np.asarray(w, dtype=np.uint32).reshape(-1, n_haps) for w in read_weights]), dtype=np.uint32)
             if len(read_weights) and soff[-1] else np.zeros((1, max(n_haps, 1)), np.uint32))
        h = _P()
        self._check(self._lib.sp_chain_window_scores(self._h, len(chains), coff.ctypes.data, items.ctypes.data, len(read_weights),
                                                     soff.ctypes.data, W.ctypes.data, n_haps, C.byref(h)))
        return DMatrix(self, h, len(read_weights), len(chains), False)

    # -- K2 ---------------------------------------------------------------------------------
    def pair_minsum_topk(self, d, k: int = 10, i_begin: int = 0, i_end: Optional[int] = None, d2=None):
        """d (and optional secondary d2): DMatrix (device) or host int32 array [R, A].
        Returns a list of (score, i, j, c1) -- or (score, score2, i, j, c1) when d2 is given."""
        recs = (PairRec * k)()
        n = C.c_int(0)
        if isinstance(d, DMatrix):
            self._check(self._lib.sp_pair_minsum_topk(self._h, d._h, d2._h if d2 is not None else None, i_begin,
                                                      d.n_patterns if i_end is None else i_end, k, recs, C.byref(n)))
        else:
            a = np.ascontiguousarray(d, dtype=np.int32)
            a2 = np.ascontiguousarray(d2, dtype=np.int32) if d2 is not None else None
            self._check(self._lib.sp_pair_minsum_topk_host(self._h, a.ctypes.data, a2.ctypes.data if a2 is not None else None,
                                                           a.shape[0], a.shape[1], k, recs, C.byref(n)))
        if d2 is None:
            return [(int(r.score), int(r.i), int(r.j), int(r.c1)) for r in recs[: n.value]]
        return [(int(r.score), int(r.score2), int(r.i), int(r.j), int(r.c1)) for r in recs[: n.value]]

    def pair_minsum_full(self, d) -> np.ndarray:
        if isinstance(d, DMatrix):
            A = d.n_patterns
            S = np.zeros((A, A), dtype=np.uint64)
            self._check(self._lib.sp_pair_minsum_full(self._h, d._h, S.ctypes.data))
        else:
            a = np.ascontiguousarray(d, dtype=np.int32)
            S = np.zeros((a.shape[1], a.shape[1]), dtype=np.uint64)
            self._check(self._lib.sp_pair_minsum_full_host(self._h, a.ctypes.data, a.shape[0], a.shape[1], S.ctypes.data))
        return S

    # -- misc -------------------------------------------------------------------------------
    def last_kernel_ms(self, which: int) -> float:
        return float(self._lib.sp_last_kernel_ms(self._h, which))

    def launch_count(self) -> int:
        return int(self._lib.sp_launch_count(self._h))

    def synchronize(self):
        self._check(self._lib.sp_ctx_synchronize(self._h))

    def share_device(self, on: bool = True):
        """Several contexts on one GPU, one host thread each: K1 runs one CTA per item at the lowest stream priority."""
        self._check(self._lib.sp_ctx_share_device(self._h, 1 if on else 0))

    def int_peak(self, kind: int = 0) -> float:
        v = C.c_double(0)
        self._check(self._lib.sp_int_peak(self._h, kind, C.byref(v)))
        return v.value

    def pinned_empty(self, shape, dtype) -> np.ndarray:
        """numpy array backed by page-locked memory from sp_host_alloc (freed with the context)."""
        dt = np.dtype(dtype)
        n = int(np.prod(shape)) * dt.itemsize
        ptr = _P()
        self._check(self._lib.sp_host_alloc(self._h, n, C.byref(ptr)))
        self._pinned.append(ptr)
        buf = (C.c_uint8 * max(n, 1)).from_address(ptr.value)
        return np.frombuffer(buf, dtype=dt, count=int(np.prod(shape))).reshape(shape)

    def wrap_dmatrix(self, dev_ptr: int, n_targets: int, n_patterns: int, ld: int, elem_bits: int) -> "DMatrix":
        h = _P()
        self._check(self._lib.sp_dmatrix_wrap(self._h, _P(dev_ptr), n_targets, n_patterns, ld, elem_bits, C.byref(h)))
        return DMatrix(self, h, n_targets, n_patterns, False)


class Consensus:
    """sp_consensus (K7): device-resident banded DP columns of a read set against growing consensus prefixes ("tracks")."""

    def __init__(self, ctx: Context, reads, offsets=None, offset_window: int = 0, band: int = 32, max_tracks: int = 64):
        self.ctx = ctx
        bases, offs = reads if isinstance(reads, tuple) else pack_sequences(reads)
        ss = _seqset(bases, offs)
        o = np.ascontiguousarray([-1 if x is None else int(x) for x in offsets], dtype=np.int32) if offsets is not None else None  # None / < 0: anchored at the start
        h = _P()
        ctx._check(ctx._lib.sp_consensus_create(ctx._h, C.byref(ss), o.ctypes.data if o is not None else None, offset_window, band, max_tracks,
                                                C.byref(h)))
        self._h, self.n_reads, self.n_tracks = h, len(offs) - 1, max_tracks

    def reset(self, track: int):
        self.ctx._check(self.ctx._lib.sp_consensus_reset(self._h, track))

    def extend(self, src, symbols, dst):
        """symbols: bytes / list of ints, 0 = report only.  Returns (ed, votes, full), each [n_tasks, n_reads]."""
        s = np.ascontiguousarray(src, dtype=np.int32)
        d = np.ascontiguousarray(dst, dtype=np.int32)
        y = np.ascontiguousarray(list(symbols), dtype=np.uint8)
        n = len(s)
        ed = np.zeros((n, self.n_reads), dtype=np.int32)
        full = np.zeros((n, self.n_reads), dtype=np.int32)
        votes = np.zeros((n, self.n_reads), dtype=np.uint8)
        self.ctx._check(self.ctx._lib.sp_consensus_extend(self._h, n, s.ctypes.data, y.ctypes.data, d.ctypes.data, ed.ctypes.data,
                                                          votes.ctypes.data, full.ctypes.data))
        return ed, votes, full

    def run_supported(self, n_sides: int) -> bool:
        """Whether run() fits this read set on chip for n_sides sides."""
        return bool(self.ctx._lib.sp_consensus_run_supported(self._h, n_sides))

    def run(self, src, dst, ed, votes, full, min_count: int, min_af_permille: int, cost_limit: int, size_limit: int, cost_cap: int,
            max_steps: int):
        """sp_consensus_run (K7 in a loop on the device) from the node with tracks src[] and per-read state ed / votes / full
        ([n_sides, n_reads]).  Returns (ed, votes, full, steps): the state of the last node and one log byte per round (low
        nibble: code 0..3 appended to side 0, high nibble: side 1, 15: side not extended).  The inputs are not changed."""
        s = np.ascontiguousarray(src, dtype=np.int32)
        d = np.ascontiguousarray(dst, dtype=np.int32)
        n = len(s)
        if len(d) != n:
            raise ValueError("src and dst need one track per side")
        e = np.array(ed, dtype=np.int32).reshape(n, self.n_reads)
        v = np.array(votes, dtype=np.uint8).reshape(n, self.n_reads)
        f = np.array(full, dtype=np.int32).reshape(n, self.n_reads)
        steps = np.zeros(max(int(max_steps), 1), dtype=np.uint8)
        n_steps = C.c_int32(0)
        self.ctx._check(self.ctx._lib.sp_consensus_run(self._h, n, s.ctypes.data, d.ctypes.data, e.ctypes.data, v.ctypes.data, f.ctypes.data,
                                                       min_count, min_af_permille, cost_limit, size_limit, cost_cap, max_steps,
                                                       steps.ctypes.data, C.byref(n_steps)))
        return e, v, f, steps[: n_steps.value].copy()

    def close(self):
        if getattr(self, "_h", None) and self.ctx._h:
            self.ctx._lib.sp_consensus_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Comm:
    """sp_comm: this rank's end of a communicator over the GPUs of one box; every method is a collective."""

    def __init__(self, ctx: Context, unique_id: bytes, rank: int, world: int):
        self.ctx, self.rank, self.world = ctx, rank, world
        buf = (C.c_uint8 * 128).from_buffer_copy(bytes(unique_id).ljust(128, b"\0")[:128])
        h = _P()
        ctx._check(ctx._lib.sp_comm_create(ctx._h, buf, rank, world, C.byref(h)))
        self._h = h

    def barrier(self):
        self.ctx._check(self.ctx._lib.sp_comm_barrier(self._h))

    def bcast_targets(self, seqs, root: int = 0) -> "TargetSet":
        """seqs is read on `root` only (None elsewhere)."""
        ss = None
        if self.rank == root:
            bases, offs = seqs if isinstance(seqs, tuple) else pack_sequences(seqs)
            ss = _seqset(bases, offs)
        h = _P()
        self.ctx._check(self.ctx._lib.sp_comm_bcast_targets(self._h, C.byref(ss) if ss is not None else None, root, C.byref(h)))
        return TargetSet._adopt(self.ctx, h)

    def score_allgather(self, targets: "TargetSet", shard: "PatternSet", shard_idx, n_total: int, elem_bits: int = 16) -> "DMatrix":
        idx = np.ascontiguousarray(shard_idx, dtype=np.int64)
        h = _P()
        self.ctx._check(self.ctx._lib.sp_comm_score_allgather(self._h, targets._h, shard._h, idx.ctypes.data, n_total, elem_bits, C.byref(h)))
        return DMatrix(self.ctx, h, targets.n, n_total, False)

    def pair_minsum_topk(self, d: "DMatrix", k: int = 10, d2: Optional["DMatrix"] = None):
        recs = (PairRec * k)()
        n = C.c_int(0)
        self.ctx._check(self.ctx._lib.sp_comm_pair_minsum_topk(self._h, d._h, d2._h if d2 is not None else None, k, recs, C.byref(n)))
        if d2 is None:
            return [(int(r.score), int(r.i), int(r.j), int(r.c1)) for r in recs[: n.value]]
        return [(int(r.score), int(r.score2), int(r.i), int(r.j), int(r.c1)) for r in recs[: n.value]]

    def close(self):
        if getattr(self, "_h", None) and self.ctx._h:
            self.ctx._lib.sp_comm_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PatternSet:
    def __init__(self, ctx: Context, seqs, mode: int = SP_INFIX):
        self.ctx = ctx
        bases, offs = seqs if isinstance(seqs, tuple) else pack_sequences(seqs)
        ss = _seqset(bases, offs)
        h = _P()
        ctx._check(ctx._lib.sp_patterns_create(ctx._h, C.byref(ss), mode, C.byref(h)))
        self._h = h
        self.n = len(offs) - 1
        self.total_len = int(ctx._lib.sp_patterns_total_len(h))
        self.padded_rows = int(ctx._lib.sp_patterns_padded_rows(h))

    def close(self):
        if getattr(self, "_h", None) and self.ctx._h:
            self.ctx._lib.sp_patterns_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class TargetSet:
    def __init__(self, ctx: Context, seqs):
        self.ctx = ctx
        bases, offs = seqs if isinstance(seqs, tuple) else pack_sequences(seqs)
        ss = _seqset(bases, offs)
        h = _P()
        ctx._check(ctx._lib.sp_targets_create(ctx._h, C.byref(ss), C.byref(h)))
        self._h = h
        self.n = len(offs) - 1
        self.total_len = int(ctx._lib.sp_targets_total_len(h))

    @classmethod
    def _adopt(cls, ctx: Context, h) -> "TargetSet":
        self = cls.__new__(cls)
        self.ctx, self._h = ctx, h
        self.n = int(ctx._lib.sp_targets_count(h))
        self.total_len = int(ctx._lib.sp_targets_total_len(h))
        return self

    def derive(self, pieces, revcomp=None) -> "TargetSet":
        """A new resident set built on the device: pieces[q] = (source index, [(begin, end), ...]) -- the concatenation of those
        intervals of that sequence -- reverse-complemented as a whole where revcomp[q] is true (sp_targets_derive)."""
        n = len(pieces)
        src = np.ascontiguousarray([p[0] for p in pieces] or [0], dtype=np.int32)
        off = np.zeros(n + 1, dtype=np.int64)
        for q, p in enumerate(pieces):
            off[q + 1] = off[q] + len(p[1])
        iv = [iv for p in pieces for iv in p[1]] or [(0, 0)]
        b = np.ascontiguousarray([x[0] for x in iv], dtype=np.int32)
        e = np.ascontiguousarray([x[1] for x in iv], dtype=np.int32)
        rc = np.ascontiguousarray(revcomp, dtype=np.uint8) if revcomp is not None else None
        h = _P()
        self.ctx._check(self.ctx._lib.sp_targets_derive(self.ctx._h, self._h, n, src.ctypes.data, off.ctypes.data, b.ctypes.data, e.ctypes.data,
                                                        rc.ctypes.data if rc is not None else None, C.byref(h)))
        return TargetSet._adopt(self.ctx, h)

    def read(self):
        """The sequences back as a list of bytes (sp_targets_read)."""
        bases = np.zeros(max(self.total_len, 1), dtype=np.uint8)
        offs = np.zeros(self.n + 1, dtype=np.int64)
        self.ctx._check(self.ctx._lib.sp_targets_read(self._h, bases.ctypes.data, offs.ctypes.data))
        raw = bases.tobytes()
        return [raw[int(offs[i]):int(offs[i + 1])] for i in range(self.n)]

    def close(self):
        if getattr(self, "_h", None) and self.ctx._h:
            self.ctx._lib.sp_targets_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DMatrix:
    """Device-resident distance matrix, allele-major: D[p * ld + t]."""

    def __init__(self, ctx: Context, h, n_targets: int, n_patterns: int, has_end: bool):
        self.ctx, self._h = ctx, h
        self.n_targets, self.n_patterns, self.has_end = n_targets, n_patterns, has_end

    @property
    def device_ptr(self) -> int:
        return int(self.ctx._lib.sp_dmatrix_device_ptr(self._h) or 0)

    @property
    def ld(self) -> int:
        return int(self.ctx._lib.sp_dmatrix_ld(self._h))

    @property
    def elem_bits(self) -> int:
        return int(self.ctx._lib.sp_dmatrix_elem_bits(self._h))

    def to_host_u16(self, out: Optional[np.ndarray] = None) -> np.ndarray:
        """16-bit read-back (the matrix must be 16-bit); `out` may be a pinned array from Context.pinned_empty."""
        D = out if out is not None else np.empty((self.n_targets, self.n_patterns), dtype=np.uint16)
        assert D.dtype == np.uint16 and D.shape == (self.n_targets, self.n_patterns) and D.flags.c_contiguous
        self.ctx._check(self.ctx._lib.sp_dmatrix_to_host_u16(self.ctx._h, self._h, D.ctypes.data))
        return D

    def to_host(self, want_end_col: bool = False, out: Optional[np.ndarray] = None):
        if out is not None and not want_end_col:
            assert out.dtype == np.int32 and out.shape == (self.n_targets, self.n_patterns) and out.flags.c_contiguous
            self.ctx._check(self.ctx._lib.sp_dmatrix_to_host(self.ctx._h, self._h, out.ctypes.data, None))
            return out
        D = np.zeros((self.n_targets, self.n_patterns), dtype=np.int32)
        E = np.zeros((self.n_targets, self.n_patterns), dtype=np.int32) if want_end_col else None
        self.ctx._check(self.ctx._lib.sp_dmatrix_to_host(self.ctx._h, self._h, D.ctypes.data,
                                                         E.ctypes.data if E is not None else None))
        return (D, E) if want_end_col else D

    def close(self):
        if getattr(self, "_h", None) and self.ctx._h:
            self.ctx._lib.sp_dmatrix_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
