#!/usr/bin/env python3
"""G independent HLA-sized dual consensuses (30 reads x 3.3 kb, 5 het sites: the tools/k7_bench.py generator, one seed per
problem), G = 1, 2, 4, 8: one after another (host.dual_consensus per problem) and as one batch (host.dual_consensus_batch).
Records per mode the wall time (every consensus call ends in a device synchronise), the host's device calls, the kernel
launches, and the k7_* kernel time from torch.profiler in a separate pass; checks that both modes return identical results; and
reads the card's name and power limit in the same run.  Usage: consensus_batch_bench.py OUT.json"""
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import numpy as np  # noqa: E402

from pb_starphase_b200 import _starphase_host as host  # noqa: E402
from pb_starphase_b200 import synth  # noqa: E402
from test_consensus_gpu import het_pair  # noqa: E402

REPEATS = 5


def problem(seed):
    rng = np.random.default_rng(seed)
    a, b = het_pair(rng, 3300, (200, 900, 1700, 2500, 3100))
    ra, _ = synth.hifi_reads(rng, [a], 16, err=0.002, flank=0, lo=0, hi=1 << 20)
    rb, _ = synth.hifi_reads(rng, [b], 14, err=0.002, flank=0, lo=0, hi=1 << 20)
    return [r.decode() for r in ra + rb]


def norm(sols):
    return [{k: (list(v) if isinstance(v, list) else v) for k, v in d.items()} for d in sols]


def one_by_one(gpu, probs):
    out, calls = [], 0
    for reads in probs:
        sols, n = host.dual_consensus(gpu, reads, [], {})
        out.append(norm(sols))
        calls += n
    return out, calls


def batched(gpu, probs):
    res = host.dual_consensus_batch(gpu, [(reads, []) for reads in probs], {})
    assert all(err is None for _, _, err in res), [err for _, _, err in res]
    return [norm(sols) for sols, _, _ in res], sum(n for _, n, _ in res)


def kernel_ms(fn):
    """k7_* kernel time of one call of fn, from torch.profiler (CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        fn()
    evs = [e for e in prof.key_averages() if "k7_" in e.key]
    return round(sum(e.device_time_total for e in evs) / 1e3, 3), sorted({e.key.split("(")[0] for e in evs})


def main():
    out_path = Path(sys.argv[1])
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    gpu = host.GpuAligner(0)
    # a second of K1 first: a lone small kernel on an idle GPU runs at idle clocks, which is not how the search runs inside a sample
    alleles, wreads, _ = synth.hla_gene(3, "HLA-A", n_alleles=3000, n_reads=256)
    gpu.score_batch([r.decode() for r in wreads], [x.decode() for x in alleles])
    probs_all = [problem(100 + k) for k in range(8)]
    one_by_one(gpu, probs_all[:1]), batched(gpu, probs_all[:2])  # warm-up of both paths
    rows = []
    for G in (1, 2, 4, 8):
        probs = probs_all[:G]
        times = {"one_by_one": [], "batch": []}
        results, calls, launches = {}, {}, {}
        for _ in range(REPEATS):  # the two modes alternate
            for mode, fn in (("one_by_one", one_by_one), ("batch", batched)):
                n0 = gpu.launch_count()
                t0 = time.perf_counter()
                res, n = fn(gpu, probs)
                times[mode].append(time.perf_counter() - t0)
                launches[mode] = gpu.launch_count() - n0
                results[mode], calls[mode] = res, n
        identical = results["one_by_one"] == results["batch"]
        row = {"G": G, "identical": identical, "dual_found": sum(1 for r in results["batch"] if r and r[0]["consensus2"] is not None)}
        for mode in times:
            ts = sorted(times[mode])
            row[mode] = {"wall_ms_min": round(1e3 * ts[0], 2), "wall_ms_median": round(1e3 * statistics.median(ts), 2),
                         "device_calls": calls[mode], "launches": launches[mode]}
        row["speedup_median"] = round(row["one_by_one"]["wall_ms_median"] / row["batch"]["wall_ms_median"], 3)
        rows.append(row)
        print(json.dumps(row), flush=True)
        assert identical, G
    doc = {"workload": "G independent dual consensuses, 30 reads x 3.3 kb, 5 het sites (tools/k7_bench.py generator, seeds 100..107)",
           "card": card, "repeats": REPEATS, "rows": rows}
    out_path.parent.mkdir(parents=True, exist_ok=True)
    out_path.write_text(json.dumps(doc, indent=1) + "\n")
    # kernel time in a pass of its own, after the timed runs (tracing slows the host)
    for row in rows:
        probs = probs_all[: row["G"]]
        for mode, fn in (("one_by_one", one_by_one), ("batch", batched)):
            row[mode]["k7_kernel_ms"], row[mode]["k7_kernels"] = kernel_ms(lambda: fn(gpu, probs))
        print(json.dumps({"G": row["G"], "k7_kernel_ms": {m: row[m]["k7_kernel_ms"] for m in ("one_by_one", "batch")}}), flush=True)
        out_path.write_text(json.dumps(doc, indent=1) + "\n")


if __name__ == "__main__":
    main()
