"""K8 end to end: graph_edit_distance (through the host module's graph_typing) on a batch of 20 CYP2D6-sized consensuses (6.2 kb
backbone, 380 variant sites) at W = 128, for two builds of the package, alternating in one run so both see the same machine.

    python tools/graph_bench.py --other <tree> [--rounds 5] [--reps 10] [--out graph_bench.json]

<tree> is another checkout of the repository with its package already built (for example the parent commit).  Per round and
tree a child process times `reps` calls after two warm-up calls (host clock around the whole call, which ends in a stream
synchronise).  One more child per tree runs a single call under torch.profiler and sums the device time of K8's kernels and of
the copies.  Both trees must return the same distances and traversed nodes.  The card's name and power limit are read in the
same run."""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def make_inputs(path: Path, n: int = 20):
    import numpy as np

    sys.path.insert(0, str(ROOT))
    from pb_starphase_b200 import synth

    rng = np.random.default_rng(4)
    bb = bytes(rng.choice(list(b"ACGT"), 6200).tolist())
    pos = sorted(int(x) for x in rng.choice(np.arange(20, 6150, 14), size=380, replace=False))
    variants = []
    for k, p in enumerate(pos):
        if k % 5 == 4:
            variants.append((42_000_000 + p, bb[p:p + 3], bb[p:p + 1]))
        elif k % 5 == 3:
            variants.append((42_000_000 + p, bb[p:p + 1], bb[p:p + 1] + b"GA"))
        else:
            variants.append((42_000_000 + p, bb[p:p + 1], bytes([b"ACGT"[(b"ACGT".index(bb[p]) + 1 + k % 3) % 4]])))
    seqs = []
    for h in range(n):
        s = bb
        for (p, r, a), on in sorted(zip(variants, rng.random(len(variants)) < 0.02 + 0.004 * h), reverse=True):
            if on and s[p - 42_000_000:p - 42_000_000 + len(r)] == r:
                s = s[:p - 42_000_000] + a + s[p - 42_000_000 + len(r):]
        noisy, _ = synth.hifi_reads(rng, [s], 1, err=0.001, flank=0, lo=0, hi=1 << 20)
        seqs.append(noisy[0].decode())
    path.write_text(json.dumps({"backbone": bb.decode(), "start": 42_000_000, "variants": [(p, r.decode(), a.decode()) for p, r, a in variants],
                                "seqs": seqs}))


def child(tree: str, inputs: str, reps: int, profile: bool):
    sys.path.insert(0, str(Path(tree).resolve()))
    from pb_starphase_b200 import _starphase_host as host

    d = json.loads(Path(inputs).read_text())
    gpu = host.GpuAligner(0)

    def run():
        return host.graph_typing(gpu, d["backbone"], d["start"], d["variants"], d["seqs"], 128)[0]

    res = run()
    run()
    digest = hashlib.sha256(repr([(f, s, list(t), list(a)) for f, s, t, a in res]).encode()).hexdigest()[:16]
    out = {"tree": tree, "digest": digest, "found": sum(bool(r[0]) for r in res)}
    if profile:
        import torch
        from torch.profiler import ProfilerActivity, profile as prof

        torch.cuda.init()
        with prof(activities=[ProfilerActivity.CUDA]) as p:
            run()
        k = {"forward_ms": 0.0, "mark_ms": 0.0, "memcpy_dtoh_ms": 0.0, "memcpy_htod_ms": 0.0, "memset_ms": 0.0}
        for e in p.events():
            name, dur = e.name, e.time_range.elapsed_us() / 1000.0
            if "k8_graph_forward" in name:
                k["forward_ms"] += dur
            elif "k8_graph_mark" in name:
                k["mark_ms"] += dur
            elif "Memcpy DtoH" in name:
                k["memcpy_dtoh_ms"] += dur
            elif "Memcpy HtoD" in name:
                k["memcpy_htod_ms"] += dur
            elif "Memset" in name:
                k["memset_ms"] += dur
        out.update({key: round(v, 3) for key, v in k.items()})
    else:
        times = []
        for _ in range(reps):
            t0 = time.perf_counter()
            run()
            times.append((time.perf_counter() - t0) * 1e3)
        out["call_ms"] = [round(t, 3) for t in times]
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--other", help="another built checkout to time against this one")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out")
    ap.add_argument("--child")
    ap.add_argument("--inputs")
    ap.add_argument("--profile", action="store_true")
    a = ap.parse_args()
    if a.child:
        child(a.child, a.inputs, a.reps, a.profile)
        return
    trees = {"this": str(ROOT)}
    if a.other:
        trees["other"] = str(Path(a.other).resolve())
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    with tempfile.TemporaryDirectory() as tmp:
        inputs = Path(tmp) / "inputs.json"
        make_inputs(inputs)

        def spawn(tree, profile=False):
            cmd = [sys.executable, __file__, "--child", tree, "--inputs", str(inputs), "--reps", str(a.reps)] + (["--profile"] if profile else [])
            r = subprocess.run(cmd, capture_output=True, text=True, env=dict(os.environ, PYTHONDONTWRITEBYTECODE="1"))
            if r.returncode:
                raise RuntimeError(f"child for {tree} failed:\n{r.stderr[-3000:]}")
            return json.loads(r.stdout.strip().splitlines()[-1])

        calls = {k: [] for k in trees}
        digests = {k: set() for k in trees}
        for _ in range(a.rounds):
            for k, tree in trees.items():
                r = spawn(tree)
                calls[k] += r["call_ms"]
                digests[k].add(r["digest"])
        profiles = {k: spawn(tree, profile=True) for k, tree in trees.items()}
    result = {"card": card, "batch": 20, "band": 128, "identical_results": len(set().union(*digests.values())) == 1}
    for k in trees:
        result[k] = {"tree": trees[k], "call_ms_median": round(statistics.median(calls[k]), 3), "call_ms_min": round(min(calls[k]), 3),
                     "calls": len(calls[k]), **{x: v for x, v in profiles[k].items() if x.endswith("_ms")}}
    print(json.dumps(result, indent=1))
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
