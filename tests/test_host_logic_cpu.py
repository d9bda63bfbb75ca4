"""CPU suite: pins oracle/starphase_oracle.py (the restated in-tree integer/float logic of the reference) against
the known-answer vectors of the reference's own unit tests, re-expressed here (SURVEY.md §4).  Each test names
the reference test it mirrors (paths relative to /root/reference)."""
import math
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "oracle"))

import starphase_oracle as so  # noqa: E402


# ---- src/hla/processed_match.rs:269-328 -----------------------------------------------------------
CIGAR = [(2, 7), (1, 8), (2, 7), (1, 1), (2, 7), (1, 2), (2, 7)]  # ==X==I==D==


def test_process_mm_cigar():
    assert so.process_mm_cigar(CIGAR, 0, 10, 0, 0) == [0, 0, 0, 1, 1, 1, 2, 2, 3, 3, 3]
    assert so.process_mm_cigar(CIGAR, 3, 18, 2, 3) == [0, 0, 1, 2, 2, 2, 3, 3, 3, 4, 4, 5, 5, 5, 6, 7, 8, 8, 8]


def test_large_unmapped():
    assert so.process_mm_cigar([(2, 7)], 2, 4, 100, 0) == [0, 1, 2, 2, 2]
    assert so.process_mm_cigar([(2, 7)], 0, 4, 0, 100) == [0, 0, 0, 1, 2]


def test_process_mm_cigar_rejects_plain_m():
    with pytest.raises(ValueError):  # EQX flag required, processed_match.rs:244-246
        so.process_mm_cigar([(4, 0)], 0, 4, 0, 0)


# ---- src/data_types/mapping.rs:211-241, src/hla/mapping.rs:181-229 --------------------------------------
def test_mapping_stats_scores():
    assert so.MappingStats(10, 1, 0).mapping_score() == 0.1
    assert so.MappingStats(10, 0, 0).mapping_score() == 0.01  # 0.1 floor of score_value, mapping.rs:191-195
    assert so.MappingStats(10, 1, 5).custom_score(False) == 1 / 5
    assert so.harmonic_mean([0.2, 0.4, 0.2]) == pytest.approx(3.0 / (5.0 + 2.5 + 5.0), rel=0, abs=1e-15)


def test_hla_mapping_score_order():
    s = so.HlaMappingStats(so.MappingStats(10, 1, 0), so.MappingStats(20, 0, 1))
    assert s.mapping_score() == (0.1, 0.05)
    s1, s2, s3 = (1.0, 0.5), (0.9, 1.0), (1.0, 0.2)  # lexicographic, cDNA first
    assert min(s1, s2) == s2 and min(s1, s3) == s3 and min(s2, s3) == s2
    assert so.HlaMappingStats(None, None).mapping_score() == (1.0, 1.0)  # missing side = worst


# ---- src/util/mapping.rs:22-57 -----------------------------------------------------------------------
def test_select_best_mapping():
    m1 = so.Mapping(0, 90, 100, 10, 100, 200, nm=2)
    m2 = so.Mapping(0, 100, 100, 0, 100, 200, nm=3)
    idx, st = so.select_best_mapping([m1, m2], unmapped_from_target=False, penalize_unmapped=True)
    assert idx == 1 and (st.seq_len, st.nm, st.unmapped) == (100, 3, 0)  # (2 + 10)/100 vs 3/100
    idx, st = so.select_best_mapping([m1, m2], unmapped_from_target=True, penalize_unmapped=False)
    assert idx == 0 and (st.seq_len, st.nm, st.unmapped) == (200, 2, 110)  # 2/90 vs 3/100
    idx, st = so.select_best_mapping([], False, True)
    assert idx is None and st.mapping_score() == 1.0  # default best = (1, 1, 0)
    idx, _ = so.select_best_mapping([m2, m2], False, True)
    assert idx == 0  # strict <: the first of equals wins


# ---- src/hla/processed_match.rs:103-184 --------------------------------------------------------------
def _pm(hla_id, cdna, dna):
    pm = so.HlaProcessedMatch(hla_id)
    pm.add_mapping(cdna)
    pm.add_mapping(dna)
    return pm


def test_is_better_match_overlap_rule():
    full = so.Mapping(0, 10, 10, 0, 10, 10, nm=0, cigar=[(10, 7)])
    one_x = so.Mapping(0, 10, 10, 0, 10, 10, nm=1, cigar=[(4, 7), (1, 8), (5, 7)])
    a, b = _pm("A", full, full), _pm("B", one_x, full)
    assert a.is_better_match(b) and not b.is_better_match(a)
    worst = so.HlaProcessedMatch.worst_match(2)
    assert a.is_better_match(worst) and not worst.is_better_match(a)
    none = _pm("N", None, None)
    assert not none.is_better_match(worst)  # an all-absent candidate never replaces the initial worst
    # a short allele that is clean where it overlaps beats a longer one with an edit inside the overlap
    short = so.Mapping(0, 6, 6, 2, 8, 10, nm=0, cigar=[(6, 7)])
    c = _pm("C", short, None)
    d = _pm("D", one_x, None)
    assert c.is_better_match(d)


# ---- src/hla/realigner.rs:124-146 ------------------------------------------------------------------
def test_realign_select_thresholds():
    ok = so.Mapping(0, 3000, 12000, 0, 3000, 3000, nm=30)     # 1 % edits, fully mapped
    bad_ed = so.Mapping(0, 3000, 12000, 0, 3000, 3000, nm=100)  # 3.3 % > 0.03
    half = so.Mapping(0, 1400, 12000, 0, 1400, 3000, nm=0)    # (0 + 1600)/3000 > 0.5
    idx, st = so.realign_select(12000, [bad_ed, half, ok])
    assert idx == 2 and (st.seq_len, st.nm, st.unmapped) == (3000, 30, 0)
    idx, st = so.realign_select(12000, [bad_ed, half])
    assert idx is None and (st.seq_len, st.nm, st.unmapped) == (12000, 12000, 0)


# ---- src/hla/caller.rs:1836-1845 -------------------------------------------------------------------
def test_is_passing_dual():
    kw = dict(min_consensus_fraction=0.10, min_cdf=0.001, expected_maf=0.5)
    assert not so.is_passing_dual(3, 20, **kw) and not so.is_passing_dual(20, 3, **kw)
    assert so.is_passing_dual(10, 20, **kw) and so.is_passing_dual(20, 10, **kw)


def test_dual_passing_stats_reference_docs_vector():
    """docs/debug_outputs.md:128-135: the reference's own example hla_debug.json (default settings, expected MAF 0.45)."""
    want = """{
  "is_passing": true,
  "is_dual": true,
  "counts1": 27,
  "counts2": 10,
  "maf": 0.2702702702702703,
  "cdf": 0.019406414321609413
}"""
    assert so.serde_pretty(so.dual_passing_stats(True, 27, 10)) == want
    # the continued fraction against the exact rational sum
    for n, p, k in ((37, 0.45, 10), (23, 0.5, 3), (200, 0.45, 60), (5, 0.1, 0), (64, 0.45, 63)):
        assert so.binomial_cdf(n, p, k) == pytest.approx(so.binomial_cdf_exact(n, p, k), rel=1e-11)


# ---- src/util/stats.rs:45-70 -------------------------------------------------------------------------
def test_multinomial():
    assert so.multinomial_ln_pmf([1.0], [10]) == pytest.approx(0.0, abs=1e-9)
    assert so.multinomial_ln_pmf([0.25, 0.75], [1, 3]) == pytest.approx(math.log(4.0 * 0.25 * 0.75 ** 3), abs=1e-6)
    assert so.multinomial_ln_pmf([0.25, 0.75], [3, 1]) == pytest.approx(math.log(4.0 * 0.25 ** 3 * 0.75), abs=1e-6)
    assert so.multinomial_ln_pmf([0.25, 0.25, 0.5], [1, 1, 2]) == pytest.approx(math.log(12.0 * 0.25 * 0.25 * 0.25), abs=1e-6)
    assert so.multinomial_ln_pmf([0.25, 0.25, 0.5], [2, 2, 0]) == pytest.approx(math.log(6.0 * 0.25 ** 4), abs=1e-6)


# ---- src/cyp2d6/caller.rs:971-1006 -------------------------------------------------------------------
def test_convert_chain_to_hap():
    labels = [so.RegionLabel(so.CYP2D7), so.RegionLabel(so.CYP2D6, "1.001"), so.RegionLabel(so.CYP2D6, "10"),
              so.RegionLabel(so.CYP2D6, "1.002"), so.RegionLabel(so.CYP2D6, "1.002")]
    tr = so.Cyp2d6Config.default().cyp_translate
    assert so.convert_chain_to_hap([2, 2, 1, 0], labels, so.SUB, tr) == "*1.001 + *10x2"
    assert so.convert_chain_to_hap([3, 1, 0], labels, so.SUB, tr) == "*1.001 + *1.002"
    assert so.convert_chain_to_hap([3, 1, 0], labels, so.CORE, tr) == "*1x2"
    assert so.convert_chain_to_hap([3, 4], labels, so.SUB, tr) == "*1.002x2"


# ---- src/cyp2d6/chaining.rs:949-1195 -----------------------------------------------------------------
def _d6(name):
    return so.RegionLabel(so.CYP2D6, name)


def test_find_best_chain_pair():
    labels = [_d6("A"), _d6("B"), _d6("C"), _d6("D")]
    obs = {"seq_1": [[0, 2]], "seq_2": [[1, 1]]}
    one = 1.0
    scores = {"seq_1": [[(0, one), (1, one), (1, one), (1, one)], [(1, one), (1, one), (0, one), (1, one)]],
              "seq_2": [[(1, one), (0, one), (1, one), (1, one)], [(1, one), (0, one), (1, one), (1, one)]]}
    chains, danglers = so.find_best_chain_pair(so.Cyp2d6Config.default(), obs, scores, labels, False, True,
                                               so.ChainPenalties(), True)
    assert chains == [[0, 2], [1, 1]] and danglers == ["3_CYP2D6*D"]


def test_ambiguous_find_best_chain_pair():
    labels = [_d6("A"), _d6("B")]
    obs = {"seq_0": [[1]], "seq_1": [[1, 0]], "seq_2": [[0, 0]], "seq_3": [[0]], "seq_4": [[1]], "seq_5": [[1, 0]],
           "seq_6": [[0]]}
    a, b = [(0, 1.0), (10, 1.0)], [(10, 1.0), (0, 1.0)]  # best = hap 0 / best = hap 1
    scores = {"seq_0": [b], "seq_1": [b, a], "seq_2": [a, a], "seq_3": [a], "seq_4": [b], "seq_5": [b, a], "seq_6": [a]}
    cfg = so.Cyp2d6Config.default()
    pen = so.ChainPenalties(0.0, -math.log(0.01), 0.0, 2.0)
    chains, danglers = so.find_best_chain_pair(cfg, obs, scores, labels, False, True, pen, True)
    assert chains == [[1], [1, 0, 0, 0]] and danglers == []
    pen = so.ChainPenalties(3.0, -math.log(0.01), 0.0, 2.0)
    chains, danglers = so.find_best_chain_pair(cfg, obs, scores, labels, False, True, pen, True)
    assert chains == [[1], [1, 0, 0]] and danglers == []


def pairwise_chains(num_labels, chains):
    """create_pairwise_chains, src/cyp2d6/chaining.rs:918-947 (weights for every member of the chain, as there)."""
    obs, scores, idx = {}, {}, 0
    for chain in chains:
        for a, b in zip(chain, chain[1:]):
            name = f"read_{idx}"
            obs[name] = [[a, b]]
            w = []
            for h in chain:
                row = [(100, 1.0)] * num_labels
                row[h] = (0, 1.0)
                w.append(row)
            scores[name] = w
            idx += 1
    return obs, scores


def test_inferred_alleles():
    labels = [_d6("3"), so.RegionLabel(so.LINK), so.RegionLabel(so.REP7), so.RegionLabel(so.SPACER), so.RegionLabel(so.CYP2D7),
              _d6("4"), so.RegionLabel(so.HYBRID, "CYP2D6::CYP2D7::exon2")]
    obs, scores = pairwise_chains(len(labels), [[0, 1], [2, 3, 4], [5, 1], [2, 3, 6]])
    cfg = so.Cyp2d6Config.default()
    chains, danglers = so.find_best_chain_pair(cfg, obs, scores, labels, False, True, so.ChainPenalties(), False)
    assert chains == [[0, 1], [5, 1]]
    assert danglers == ["2_REP7", "3_spacer", "4_CYP2D7", "6_CYP2D6::CYP2D7::exon2"]
    chains, danglers = so.find_best_chain_pair(cfg, obs, scores, labels, True, True, so.ChainPenalties(), False)
    assert chains == [[0, 1, 2, 3, 4], [5, 1, 2, 3, 6]] and danglers == []


def test_chaining_errors():
    labels = [so.RegionLabel(so.CYP2D7), so.RegionLabel(so.LINK), so.RegionLabel(so.SPACER), so.RegionLabel(so.UNKNOWN)]
    with pytest.raises(so.NoChainingHead):
        so.find_best_chain_pair(so.Cyp2d6Config.default(), {}, {}, labels, False, True, so.ChainPenalties(), False)


def test_double5_targeted():
    labels = [so.RegionLabel(so.DELETION)]
    obs = {f"read{x}": [[0]] for x in range(2)}
    scores = {f"read{x}": [[(0, 1.0)]] for x in range(2)}
    chains, danglers = so.find_best_chain_pair(so.Cyp2d6Config.default(), obs, scores, labels, True, False,
                                               so.ChainPenalties(), False)
    assert chains == [[0], [0]] and danglers == []


def test_containment_score_is_min_of_per_chain_windows():
    """The identity the GPU path uses: containment(c1, c2) = min(B(c1), B(c2)) - optimum (chaining.rs:683-731)."""
    import random

    rnd = random.Random(4)
    for _ in range(200):
        n_haps = rnd.randint(1, 5)
        w = [[(rnd.randint(0, 30), 1.0) for _ in range(n_haps)] for _ in range(rnd.randint(1, 4))]
        c1 = [rnd.randrange(n_haps) for _ in range(rnd.randint(1, 6))]
        c2 = [rnd.randrange(n_haps) for _ in range(rnd.randint(1, 6))]
        opt = sum(min(x for x, _ in seg) for seg in w)
        score, _ = so.containment_score(c1, c2, w)
        assert score == min(so.chain_best_window(c1, w), so.chain_best_window(c2, w)) - opt


# ---- serde-pretty JSON writer (src/util/file_io.rs:37-52, src/data_types/starphase_json.rs) ------------------
def test_result_json_layout():
    stats = so.HlaMappingStats(None, so.MappingStats(3502, 2, 0))
    md = so.mapping_details_json("read/1", "HLA:HLA00001", "HLA-A*03:01:01:01", stats, False)
    gene = so.gene_details_from_mappings([so.diplotype_json("*03:01:01:01", "*03:01:01:01")], [md])
    meta = dict(pbstarphase_version="2.0.1-test", cpic_version="v", hla_version="3.62.0", pharmvar_version="6", build_time="t")
    text = so.starphase_json("2.0.1-test", meta, {"HLA-A": gene})
    assert text.startswith('{\n  "pbstarphase_version": "2.0.1-test",\n  "database_metadata": {\n    "pbstarphase_version"')
    assert '"cdna_stats": null' in text and '"clipped_start": null' in text
    assert '"diplotype": "*03:01:01:01/*03:01:01:01"' in text
    import json

    back = json.loads(text)
    assert list(back) == ["pbstarphase_version", "database_metadata", "gene_details"]
    assert back["gene_details"]["HLA-A"]["mapping_details"][0]["best_mapping_stats"]["dna_stats"]["nm"] == 2


def test_bench_clock_sampler_parses_nvidia_smi_rows():
    """bench.py's `clocks` key: median SM clock, its maximum and the active throttle reasons of the samples taken after mark()."""
    import importlib.util
    from pathlib import Path

    spec = importlib.util.spec_from_file_location("bench_for_test", Path(__file__).resolve().parent.parent / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    s = bench.ClockSampler(0)
    s.rows = [["1200", "1965", "Not Active", "Not Active", "Not Active", "Active"],      # warm-up: before mark()
              ["1965", "1965", "Not Active", "Not Active", "Not Active", "Not Active"]]
    s.mark()
    s.rows += [["1965", "1965", "Not Active", "Not Active", "Not Active", "Not Active"],
               ["1950", "1965", "Not Active", "Not Active", "Not Active", "Active"],
               ["1965", "1965", "Not Active", "Not Active", "Not Active", "Not Active"],
               ["[N/A]", "1965", "x"]]                                                        # a malformed row is skipped
    got = s.stop()
    assert got == dict(sm_mhz=1965.0, sm_max_mhz=1965.0, reasons=["sw_power_cap"], samples=3)
    assert bench.ClockSampler.Q.count(",") == 5 and "power.draw" not in bench.ClockSampler.Q


def test_bench_dump_outputs_writes_float_arrays_of_a_fixed_read_sample(tmp_path):
    """bench.py --dump-outputs: top pair records exactly, distance matrices on the same seeded rows every time, float dtypes only,
    and at most 64 MB at the bench's full allele count (12,451 DNA + 19,629 cDNA)."""
    import importlib.util

    import numpy as np

    spec = importlib.util.spec_from_file_location("bench_for_test", Path(__file__).resolve().parent.parent / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)

    class HostMatrix:  # the two members of DMatrix that dump_outputs reads
        def __init__(self, a):
            self.a, self.n_targets = a, a.shape[0]

        def to_host_u16(self):
            return self.a

    rng = np.random.default_rng(11)
    Dd = HostMatrix(rng.integers(0, 1 << 16, size=(bench.DUMP_READS + 44, 37)).astype(np.uint16))
    Dc = HostMatrix(rng.integers(0, 1 << 16, size=(bench.DUMP_READS + 44, 53)).astype(np.uint16))
    result = {"HLA-A": [(28141, 161162, 42, 2136, 932), (28150, 161000, 7, 9, 3)], "HLA-B": []}
    for out in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(out, result, Dd, Dc)
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == ["cdna_distances.npy", "dna_distances.npy", "top_pairs_HLA-A.npy", "top_pairs_HLA-B.npy"]
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64) and a.dtype == b.dtype and (a == b).all()
    assert np.load(tmp_path / "a" / "top_pairs_HLA-A.npy").tolist() == [list(map(float, r)) for r in result["HLA-A"]]
    assert np.load(tmp_path / "a" / "top_pairs_HLA-B.npy").shape == (0, 5)
    dna = np.load(tmp_path / "a" / "dna_distances.npy")
    assert dna.shape == (bench.DUMP_READS, 37)
    rows = [int(np.flatnonzero((Dd.a == r).all(axis=1))[0]) for r in dna.astype(np.uint16)]
    assert rows == sorted(set(rows)) and (np.load(tmp_path / "a" / "cdna_distances.npy") == Dc.a[rows]).all()
    assert bench.DUMP_READS * (12451 + 19629) * 4 + 2 * 16 * 5 * 8 <= 64 << 20
