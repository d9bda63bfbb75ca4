"""CPU suite: the lane-width planner of sp_patterns_create (sp_plan_lane_classes) on fixed length sets.  The expected classes
and padded rows are pinned, so a change to the class choice or to the best-fit-decreasing bin packer shows up here."""
import numpy as np
import pytest

from pb_starphase_b200 import binding, synth


@pytest.fixture(scope="module")
def bench_sets():
    return synth.hla_wgs_workload(synth.DEFAULT_SEED, 256, 1.0)


@pytest.mark.parametrize("gene, kind, classes, padded", [
    ("HLA-A", "dna", [(13, 5695, 1386)], 18_450_432),
    ("HLA-A", "cdna", [(9, 8949, 1114)], 10_266_624),
    ("HLA-B", "dna", [(12, 6756, 1721)], 21_147_648),
    ("HLA-B", "cdna", [(9, 10680, 1330)], 12_257_280),
])
def test_plan_of_the_bench_allele_sets(bench_sets, gene, kind, classes, padded):
    assert binding.plan_lane_classes([len(s) for s in bench_sets[gene][kind]]) == (classes, padded)


def _long_set():
    """Patterns up to 6 kb plus two of more than 16,384 rows (only U = 20 / 24 fit them) and an empty one."""
    rng = np.random.default_rng(11)
    return [int(x) for x in rng.integers(200, 6000, 300)] + [17000, 20000, 0]


def _bimodal_set():
    """cDNA-, DNA- and CYP-sized patterns in shuffled order, one empty."""
    rng = np.random.default_rng(5)
    lens = [int(x) for x in np.concatenate([rng.integers(500, 1300, 400), rng.integers(2800, 3600, 300), rng.integers(6000, 9000, 40)])] + [0]
    rng.shuffle(lens)
    return lens


@pytest.mark.parametrize("make, max_classes, classes, padded", [
    (_long_set, 4, [(20, 119, 15), (24, 183, 30)], 1_044_480),
    (_long_set, 1, [(20, 302, 52)], 1_064_960),
    (_bimodal_set, 4, [(13, 385, 55), (16, 355, 62)], 1_747_968),
    (_bimodal_set, 1, [(13, 740, 133)], 1_770_496),
])
def test_plan_of_seeded_sets(make, max_classes, classes, padded):
    assert binding.plan_lane_classes(make(), max_classes) == (classes, padded)
