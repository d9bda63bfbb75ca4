#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200 scoring path (contract: see the task statement / DESIGN.md §6).

Metric (BASELINE.json): HLA read-allele GCUPS (+ samples/s).  Main leg = BASELINE.json configs[1], "HLA-A/HLA-B WGS 30x:
~2k synthetic HiFi reads x full IMGT/HLA allele set" (SURVEY.md §8(d).2): 2,048 reads per GPU against 12,451 DNA +
19,629 cDNA alleles.  One step = K1(DNA) + K1(cDNA) + K2 (cDNA,DNA)-lexicographic pair scoring per gene + top-k merge.
N > 1: reads = 2,048 x N (weak scaling), broadcast from rank 0; alleles dealt to the ranks by sp_shard_plan, D shards
all-gathered into database order, K2 row blocks per rank, per-rank top-k merged -- all through the library's own multi-GPU
C ABI (sp_comm_*, NCCL inside libstarphase_gpu.so); torch.distributed only carries the communicator id and the final timings.
Two more legs ride in the same JSON line: `panel` = configs[2] (40,960 fixed reads, alleles sharded N ways: STRONG scaling)
and `cohort` = configs[4] (independent samples through the C++ host, 125 per GPU = 1,000 on 8 GPUs; `samples_per_s`).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--panel-reads R] [--cohort-samples S]
                  [--dump-outputs DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

METRIC = "hla_read_allele_gcups"
UNIT = "GCUPS"
READS_PER_GPU = 2048
INT_OPS_PER_CELL = 23.0 / 64.0  # SURVEY.md §8(d): Hyyro block step = 23 INT32-pipe ops per 64 cells
TOPK = 16


PANEL_READS = 40960      # BASELINE configs[2]
COHORT_PER_GPU = 125     # BASELINE configs[4]: 1,000 samples on 8 GPUs
COHORT_WORKERS = 3        # host threads (one sp_ctx each) per GPU in the cohort leg
DUMP_READS = 256          # --dump-outputs: reads (rows) of the distance matrices written; 256 x 32,080 alleles x 4 B = 33 MB
DUMP_SEED = 7

# The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints "NCCL version ..." on the first communicator
# when NCCL_DEBUG=VERSION is set in the environment), so the process's fd 1 is pointed at stderr for its whole life and the
# result line goes to a private duplicate of the original stdout.
_RESULT_FD = None


def _claim_stdout():
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=float, default=float(os.environ.get("SP_BENCH_SCALE", "1.0")),
                    help="debug only: shrink the allele set (a scaled run is NOT a valid bench number)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="CPU-baseline budget")
    ap.add_argument("--cohort-samples", type=int, default=COHORT_PER_GPU,
                    help="samples per GPU for the cohort leg (BASELINE configs[4]: 125 x 8 GPUs = 1,000 samples); 0 disables it")
    ap.add_argument("--cohort-workers", type=int, default=COHORT_WORKERS,
                    help="host threads per GPU in the cohort leg, one sp_ctx each (sp_ctx_share_device); 1 = one sample at a time")
    ap.add_argument("--panel-reads", type=int, default=PANEL_READS,
                    help="reads of the strong-scaling panel leg (BASELINE configs[2]: 40,960); 0 disables it")
    ap.add_argument("--panel-steps", type=int, default=1, help="timed steps of the panel leg (one step is ~110 s on one GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy: the top pair records of "
                         "each gene and the DNA / cDNA distance matrices on a fixed, seeded sample of reads")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


# ---------------------------------------------------------------------------------------------
# workload
# ---------------------------------------------------------------------------------------------
def build_workload(n_gpus: int, scale: float, n_reads: int | None = None):
    from pb_starphase_b200 import synth

    genes = synth.hla_wgs_workload(synth.DEFAULT_SEED, READS_PER_GPU * n_gpus if n_reads is None else n_reads, scale)
    A, B = genes["HLA-A"], genes["HLA-B"]
    w = dict(
        dna=A["dna"] + B["dna"], cdna=A["cdna"] + B["cdna"],
        reads=A["reads"] + B["reads"], ctargets=A["ctargets"] + B["ctargets"],
        # per gene: (dna row0, cdna row0, n alleles with DNA, read col0, n reads)
        gene_views={
            "HLA-A": (0, 0, len(A["dna"]), 0, len(A["reads"])),
            "HLA-B": (len(A["dna"]), len(A["cdna"]), len(B["dna"]), len(A["reads"]), len(B["reads"])),
        },
    )
    w["cells_dna"] = sum(map(len, w["dna"])) * sum(map(len, w["reads"]))
    w["cells_cdna"] = sum(map(len, w["cdna"])) * sum(map(len, w["ctargets"]))
    return w


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    # SM clock, its maximum and the four throttle reasons the contract names, once a second.  (Polling every 200 ms with power.draw
    # in the query cost the timed steps 40-190 ms each in idle gaps between launches -- NVML queries contend with the CUDA calls
    # of the step for the driver; the e2e loop, which runs without the sampler, never showed them.)
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    PERIOD_MS = 1000

    def __init__(self, device: int):
        self.rows, self.proc, self.device, self.first = [], None, device, 0

    def mark(self):
        """The timed region starts here: only samples taken from now on are reported.  The process is started earlier (before
        the warm-up steps): nvidia-smi's start-up takes the driver's attention for a few hundred ms, which showed up as idle
        gaps between the launches of the first timed step when it was started inside the timed region."""
        self.first = len(self.rows)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", str(self.PERIOD_MS), "-i", str(self.device)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        rows = self.rows[self.first:] or self.rows
        sm = [float(r[0]) for r in rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in rows:
            if len(r) >= 6:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ---------------------------------------------------------------------------------------------
# CPU baseline (oracle port; the reference binary cannot be built here -- DESIGN.md §3)
# ---------------------------------------------------------------------------------------------
def cpu_sample(w, budget_s: float, steps: int = 1):
    """Times the oracle's 64-bit Myers on all host threads on a bounded sample of the same workload."""
    import oracle_util

    orc = oracle_util.Oracle()
    threads = os.cpu_count() or orc.num_threads()  # torchrun exports OMP_NUM_THREADS=1: ask for every host thread explicitly
    rng = np.random.default_rng(1)
    reads, ctargets = w["reads"], w["ctargets"]
    ridx = rng.choice(len(reads), size=min(8, len(reads)), replace=False)
    # calibrate on a tiny slice, then size the sample for ~budget_s of wall time per step
    aidx = rng.choice(len(w["dna"]), size=min(32, len(w["dna"])), replace=False)
    t0 = time.perf_counter()
    orc.score_batch([reads[i] for i in ridx], [w["dna"][i] for i in aidx], nthreads=threads)
    rate = orc.last_cells / max(time.perf_counter() - t0, 1e-6)
    want_cells = rate * budget_s
    per_allele = float(np.mean([len(reads[i]) for i in ridx])) * len(ridx) * float(np.mean([len(a) for a in w["dna"]]))
    n_alleles = int(max(32, min(len(w["dna"]), want_cells * 0.85 / per_allele)))
    aidx = rng.choice(len(w["dna"]), size=n_alleles, replace=False)
    cidx = rng.choice(len(w["cdna"]), size=min(len(w["cdna"]), max(32, int(n_alleles * 1.5))), replace=False)
    times, cells = [], 0
    for _ in range(steps):
        t0 = time.perf_counter()
        orc.score_batch([reads[i] for i in ridx], [w["dna"][i] for i in aidx], nthreads=threads)
        c = orc.last_cells
        orc.score_batch([ctargets[i] for i in ridx], [w["cdna"][i] for i in cidx], nthreads=threads)
        c += orc.last_cells
        times.append(time.perf_counter() - t0)
        cells = c
    sample = f"{len(ridx)} reads x {n_alleles} DNA + {len(cidx)} cDNA alleles of the same workload ({cells / 1e9:.1f} Gcells/step)"
    return dict(gcups=cells / float(np.mean(times)) / 1e9, cores=threads, sample=sample, ms_per_step=float(np.mean(times)) * 1e3)


# ---------------------------------------------------------------------------------------------
# shared pieces of the JSON line
# ---------------------------------------------------------------------------------------------
def workload_name(n):
    return f"hla_wgs30x: {READS_PER_GPU * n} reads x 12,451 DNA + 19,629 cDNA alleles (BASELINE configs[1]" + (")" if n == 1 else f", reads x{n}, alleles sharded {n} ways)")


def bench_config(n, scale):
    """`config` of the line; identical for both arms (the reference arm times a bounded sample of it, see cpu_baseline.sample)."""
    return dict(workload=workload_name(n), seed=20251106, l2="flushed between timed steps (256 MB write)",
                step="K1 DNA + K1 cDNA + K2 (cDNA,DNA) pair top-%d per gene" % TOPK, scale=scale)


def dump_outputs(out_dir, result, Dd, Dc):
    """--dump-outputs: one step's answers, so that two builds can be compared output for output on the same inputs.
    top_pairs_<gene>.npy: the step's result for that gene, one (score, score2, i, j, c1) record per row (float64 holds them
    exactly).  dna_distances.npy / cdna_distances.npy: the gathered u16 distance matrices [read][allele] as float32, all
    alleles of DUMP_READS reads drawn with a fixed seed (ascending), which keeps the files small at any read count."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for gene, recs in result.items():
        np.save(out / f"top_pairs_{gene}.npy", np.asarray(recs, dtype=np.float64).reshape(-1, 5))
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(Dd.n_targets, size=min(DUMP_READS, Dd.n_targets), replace=False))
    np.save(out / "dna_distances.npy", Dd.to_host_u16()[rows].astype(np.float32))
    np.save(out / "cdna_distances.npy", Dc.to_host_u16()[rows].astype(np.float32))


# ---------------------------------------------------------------------------------------------
# reference arm
# ---------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = build_workload(args.gpus, args.scale)
    for _ in range(min(args.warmup, 1)):
        cpu_sample(w, 1.0)
    res = cpu_sample(w, max(3.0, args.cpu_seconds / max(args.steps, 1)), steps=args.steps)
    cells_total = w["cells_dna"] + w["cells_cdna"]
    line = dict(metric=METRIC, value=res["gcups"], unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=res["ms_per_step"], higher_is_better=True, scaling="weak", vs_baseline=None, dtype="u32",
                data="synthetic", impl="reference", config=bench_config(args.gpus, args.scale),
                cpu_baseline=dict(value=res["gcups"], unit=UNIT, cores=res["cores"], kind="port", sample=res["sample"],
                                  note="oracle port of the reference's CPU path (64-bit Myers, OpenMP over pairs); the Rust reference + "
                                       "minimap2 cannot be built here.  Each step times the bounded sample and reports its rate",
                                  extrapolated_full_step_s=cells_total / (res["gcups"] * 1e9)),
                e2e=dict(value=res["gcups"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    _emit(line)


# ---------------------------------------------------------------------------------------------
# cohort leg (BASELINE configs[4], SURVEY.md 8(d).5): independent samples through the C++ host, one at a time per GPU
# ---------------------------------------------------------------------------------------------
def run_cohort(w, n_samples, rank, world, local_rank, workers=1):
    """Per sample the complete calls a pb-StarPhase run makes on this path, through the C++ host above the C ABI
    (pb_starphase_b200/host): HLA-A and HLA-B diplotypes (64 reads per gene, DNA + cDNA, against that gene's resident allele
    set: K1 x2, K2 pair ranking, het/hom decision, per-read database assignment via K5 + K4), CYP2D6 (39-template search over
    96 reads with K4 tracebacks, weight_sequence spans, chains, find_best_chain_pair) -- ending in the result JSON text of
    that sample.  Samples are independent: ranks work through disjoint samples with no exchange (replicas).  With
    workers > 1 the rank runs that many host threads, each with its own GpuAligner (sp_ctx) in sp_ctx_share_device mode
    and its own resident allele index, taking samples from one queue -- the way a cohort is run with the reference, many
    single-sample runs side by side: the latency-bound CYP2D6 / read-assignment phases of one sample fill the GPU and
    the host while another sample's K1 runs.
    Returns (seconds, samples, bytes of JSON, info)."""
    import threading

    from pb_starphase_b200 import _starphase_host as host
    from pb_starphase_b200 import synth

    settings = host.DiplotypeSettings()
    genes = list(w["gene_views"].items())
    rows = []
    for g, (gene, (drow, crow, na, _, _)) in enumerate(genes):
        for a in range(na):
            rows.append((f"HLA:HLA{g * 100000 + a:06d}", gene, [f"{1 + a // 400:02d}", f"{1 + (a // 20) % 20:02d}", f"{1 + a % 20:02d}", "01"],
                         w["dna"][drow + a].decode(), w["cdna"][crow + a].decode()))
    per_gene = 64
    meta = dict(pbstarphase_version="2.0.1", cpic_version="synthetic", hla_version="synthetic", pharmvar_version="synthetic", build_time="n/a")
    dbg = os.environ.get("SP_COHORT_DEBUG") == "1"

    class Worker:
        def __init__(self):
            self.gpu = host.GpuAligner(local_rank)
            if workers > 1 and os.environ.get("SP_COHORT_NOSHARE") != "1":  # experiment hook: persistent K1 grids side by side
                self.gpu.share_device(True)
            self.index = {gene: host.HlaGeneIndex(self.gpu, [r for r in rows if r[1] == gene], gene, settings) for gene, _ in genes}

        def one_sample(self, sid, cyp):
            gpu, details, marks = self.gpu, {}, [("start", time.perf_counter())]
            for gene, (_, _, _, col0, nr) in genes:
                lo = col0 + (sid * per_gene) % max(nr - per_gene, 1)
                reads = [(f"s{sid}/{gene}/{k}", w["reads"][lo + k].decode(), w["ctargets"][lo + k].decode()) for k in range(per_gene)]
                details[gene] = host.diplotype_hla_gene_indexed(gpu, self.index[gene], reads, settings)["gene_details"]
                marks.append((gene, time.perf_counter()))
            hits = host.find_base_type_in_sequences(gpu, cyp["templates"], cyp["reads"], False, 0.5)
            marks.append(("cyp_template_search", time.perf_counter()))
            call = host.call_cyp2d6_chains(gpu, cyp["consensuses"], cyp["regions"], cyp["roi"], False, True)
            marks.append(("cyp_chains", time.perf_counter()))
            details["CYP2D6"] = call["gene_details"]
            text = host.starphase_json("2.0.1", meta, details)
            marks.append(("json", time.perf_counter()))
            if dbg:
                print("cohort rank", rank, "sample", sid, " ".join(f"{b[0]}={1e3 * (b[1] - a[1]):.1f}ms" for a, b in zip(marks, marks[1:])), file=sys.stderr)
            return text, sum(len(h) for h in hits)

    def cyp_inputs(sid):
        c = synth.cyp2d6_diploid_sample(2000 + sid)
        return dict(templates=[(t, s, q.decode()) for (t, s), q in zip(c["template_labels"], c["templates"])],
                    reads=[r.decode() for r in c["reads"]], consensuses=[x.decode() for x in c["consensuses"]], regions=c["regions"],
                    roi={q: [(a, b, seq.decode()) for a, b, seq in regs] for q, regs in c["roi"].items()})

    sids = [rank + world * k for k in range(n_samples)]
    inputs = {sid: cyp_inputs(sid) for sid in sids}  # host-side inputs exist before the clock starts
    pool = [Worker() for _ in range(max(workers, 1))]
    results, errors, lock, nxt = {}, [], threading.Lock(), [0]
    start = threading.Barrier(len(pool) + 1)

    def work(wk, k0):
        try:
            for k in range(2):  # untimed: pools, plans and page-locked buffers of this worker's context reach their sizes
                sid = sids[(k0 + k) % len(sids)]
                wk.one_sample(sid, inputs[sid])
            start.wait()
            while True:
                with lock:
                    k = nxt[0]
                    nxt[0] += 1
                if k >= len(sids):
                    return
                results[sids[k]] = wk.one_sample(sids[k], inputs[sids[k]])
        except Exception as e:  # noqa: BLE001
            errors.append(e)
            start.abort()

    threads = [threading.Thread(target=work, args=(wk, 2 * i), daemon=True) for i, wk in enumerate(pool)]
    for th in threads:
        th.start()
    try:
        start.wait()
    except threading.BrokenBarrierError:
        pass
    t0 = time.perf_counter()
    for th in threads:
        th.join()
    dt = time.perf_counter() - t0
    if errors:
        raise errors[0]
    nbytes = sum(len(t) for t, _ in results.values())
    text, n_hits = results[sids[-1]]
    doc = json.loads(text)
    calls = {g: d["diplotypes"][0]["diplotype"] for g, d in doc["gene_details"].items()}
    return dt, n_samples, nbytes, dict(last_sample_calls=calls, cyp2d6_template_hits=n_hits, workers_per_gpu=len(pool),
                                       kernel_launches=int(sum(wk.gpu.launch_count() for wk in pool)))


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    import pb_starphase_b200 as sp
    from pb_starphase_b200 import binding, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the scoring path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n = max(args.gpus, world)
    w = build_workload(n, args.scale)

    # one explicit stream for everything: the library's kernels and collectives, torch's fills and events.
    # (The legacy default stream has handle 0 == NULL, which sp_ctx_create reads as "make a private stream".)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx = sp.Context(local_rank, stream=stream.cuda_stream)
    assert stream.cuda_stream != 0
    # the library's own communicator: rank 0 draws the id, torch.distributed only carries the 128 bytes
    uid = [binding.comm_unique_id() if rank == 0 and world > 1 else bytes(128)]
    if world > 1:
        dist.broadcast_object_list(uid, src=0, device=dev)
    comm = sp.Comm(ctx, uid[0], rank, world)
    int_peak = ctx.int_peak(0)       # ALU pipe alone (LOP3)
    int_peak2 = ctx.int_peak(2)      # ALU + FMA pipes (LOP3 + IMAD alternating)

    # ---- resident database: this rank's allele shards (prepared once, like HlaRealigner::new) ----
    n_dna, n_cdna = len(w["dna"]), len(w["cdna"])
    idx_d = binding.shard_plan([len(a) for a in w["dna"]], world, rank)
    idx_c = binding.shard_plan([len(a) for a in w["cdna"]], world, rank)
    P_dna = ctx.patterns([w["dna"][i] for i in idx_d])
    P_cdna = ctx.patterns([w["cdna"][i] for i in idx_c])
    sum_dna, sum_cdna = sum(map(len, w["dna"])), sum(map(len, w["cdna"]))
    sum_dna_local = sum(len(w["dna"][i]) for i in idx_d)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def pinned(arr):
        out = ctx.pinned_empty(arr.shape, arr.dtype)
        out[...] = arr
        return out

    k1_ms = []

    def gene_views(Dd, Dc, gv):
        """K2 inputs per gene: blocks of the gathered matrices (database order: one gene's alleles are consecutive rows)."""
        out = {}
        for gene, (drow, crow, na, col0, nr) in gv.items():
            vd = ctx.wrap_dmatrix(Dd.device_ptr + 2 * (drow * Dd.ld + col0), nr, na, Dd.ld, 16)
            vc = ctx.wrap_dmatrix(Dc.device_ptr + 2 * (crow * Dc.ld + col0), nr, na, Dc.ld, 16)
            out[gene] = (vc, vd)
        return out

    phases = os.environ.get("SP_BENCH_PHASES") == "1"  # debug: wall-clock phases of every step to stderr (synchronises each phase)

    def device_step(T_dna, T_cdna, gv, keep=False):
        marks = [time.perf_counter()]

        def mark():
            if phases:
                ctx.synchronize()
                marks.append(time.perf_counter())

        Dd = comm.score_allgather(T_dna, P_dna, idx_d, n_dna, 16)      # K1 on this rank's shard + ncclAllGather + row permutation
        k1_ms.append(ctx.last_kernel_ms(0))
        mark()
        Dc = comm.score_allgather(T_cdna, P_cdna, idx_c, n_cdna, 16)
        mark()
        out = {}
        views = gene_views(Dd, Dc, gv)
        for gene, (vc, vd) in views.items():
            out[gene] = comm.pair_minsum_topk(vc, TOPK, d2=vd)         # K2 on this rank's row block + record all-gather + merge
            vc.close(); vd.close()
            mark()
        if phases:
            print(f"rank {rank} step phases ms: dna+gather {1e3 * (marks[1] - marks[0]):.1f} (k1 {k1_ms[-1]:.1f}) cdna+gather {1e3 * (marks[2] - marks[1]):.1f} "
                  + " ".join(f"k2[{g}] {1e3 * (b - a):.1f}" for g, a, b in zip(views, marks[2:], marks[3:])), file=sys.stderr)
        if keep:
            return out, Dd, Dc
        Dd.close(); Dc.close()
        return out

    def barrier():
        comm.barrier()
        torch.cuda.synchronize()

    # ---- `value`: inputs resident in HBM.  The read set lives on rank 0 and is broadcast (the path's real exchange) ----
    reads_pack = tuple(pinned(a) for a in sp.binding.pack_sequences(w["reads"])) if rank == 0 else None
    ct_pack = tuple(pinned(a) for a in sp.binding.pack_sequences(w["ctargets"])) if rank == 0 else None
    T_dna, T_cdna = comm.bcast_targets(reads_pack, 0), comm.bcast_targets(ct_pack, 0)
    cells_dna, cells_cdna = sum_dna * T_dna.total_len, sum_cdna * T_cdna.total_len
    cells_total = cells_dna + cells_cdna
    cells_dna_local = sum_dna_local * T_dna.total_len
    gv = w["gene_views"]
    result = None
    sampler = ClockSampler(local_rank)
    sampler.start()  # polls once a second from here on; the samples of the timed region are the ones reported
    for _ in range(args.warmup):
        result = device_step(T_dna, T_cdna, gv)
    k1_ms.clear()
    launches0 = ctx.launch_count()
    barrier()
    sampler.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    kept = None
    for step in range(args.steps):
        flush.fill_(1)  # L2 flush between timed iterations (256 MB > 126 MB L2)
        if args.dump_outputs and step == args.steps - 1:  # the last step's distance matrices outlive it for the dump
            result, *kept = device_step(T_dna, T_cdna, gv, keep=True)
        else:
            result = device_step(T_dna, T_cdna, gv)
    e1.record(stream)
    barrier()
    clocks = sampler.stop()
    if kept:
        if rank == 0:
            dump_outputs(args.dump_outputs, result, *kept)
        for m in kept:
            m.close()
    ms_total = e0.elapsed_time(e1)
    launches = ctx.launch_count() - launches0
    k1_avg_ms = float(np.mean(k1_ms))

    # ---- `e2e`: pinned host buffers in, host results out, through the C-ABI calls a host program makes ----
    lo_d, hi_d = rank * n_dna // world, (rank + 1) * n_dna // world      # this rank hands back its block of rows: the whole
    lo_c, hi_c = rank * n_cdna // world, (rank + 1) * n_cdna // world    # matrix reaches host memory once per step
    R = T_dna.n
    host_dd = ctx.pinned_empty((R, hi_d - lo_d), np.uint16)
    host_dc = ctx.pinned_empty((R, hi_c - lo_c), np.uint16)

    def e2e_step():
        Td, Tc = comm.bcast_targets(reads_pack, 0), comm.bcast_targets(ct_pack, 0)  # H2D of the read set on rank 0 + broadcast
        res, Dd, Dc = device_step(Td, Tc, gv, keep=True)
        own_d = ctx.wrap_dmatrix(Dd.device_ptr + 2 * lo_d * Dd.ld, R, hi_d - lo_d, Dd.ld, 16)
        own_c = ctx.wrap_dmatrix(Dc.device_ptr + 2 * lo_c * Dc.ld, R, hi_c - lo_c, Dc.ld, 16)
        own_d.to_host_u16(host_dd); own_c.to_host_u16(host_dc)  # D2H of the distance matrices [read][allele]
        for h in (own_d, own_c, Dd, Dc, Td, Tc):
            h.close()
        return res, host_dd.nbytes + host_dc.nbytes

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    d2h = 0
    for _ in range(args.steps):
        res_e2e, d2h = e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    assert res_e2e == result, "e2e and device-resident runs disagree"
    h2d = int(sum(a.nbytes for a in reads_pack) + sum(a.nbytes for a in ct_pack)) if rank == 0 else 0
    T_dna.close(); T_cdna.close()

    # ---- panel leg: BASELINE configs[2], a FIXED read set, alleles sharded N ways (strong scaling) ----
    panel = None
    if args.panel_reads > 0:
        pr = args.panel_reads
        if rank == 0:
            # reads of the same two genes against the SAME database as the main leg (drawn from its alleles)
            rng = np.random.default_rng([synth.DEFAULT_SEED, 40960])
            p_reads, p_ct = [], []
            for gi, gene in enumerate(("HLA-A", "HLA-B")):
                drow, crow, na, _, _ = gv[gene]
                nr = pr // 2 if gi == 0 else pr - pr // 2
                rd, src = synth.hifi_reads(rng, w["dna"][drow:drow + na], nr)
                p_reads += rd
                p_ct += [synth.hifi_reads(rng, [w["cdna"][crow + int(s)]], 1, flank=50, lo=0, hi=1400)[0][0] for s in src]
            pp_r, pp_c = sp.binding.pack_sequences(p_reads), sp.binding.pack_sequences(p_ct)
        else:
            pp_r = pp_c = None
        Tp, Tpc = comm.bcast_targets(pp_r, 0), comm.bcast_targets(pp_c, 0)
        pgv = {"HLA-A": (gv["HLA-A"][0], gv["HLA-A"][1], gv["HLA-A"][2], 0, pr // 2),
               "HLA-B": (gv["HLA-B"][0], gv["HLA-B"][1], gv["HLA-B"][2], pr // 2, pr - pr // 2)}
        p_cells = sum_dna * Tp.total_len + sum_cdna * Tpc.total_len
        k1_keep = list(k1_ms)
        barrier()
        pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        pe0.record(stream)
        for _ in range(args.panel_steps):
            flush.fill_(1)
            p_res = device_step(Tp, Tpc, pgv)
        pe1.record(stream)
        barrier()
        p_ms = pe0.elapsed_time(pe1)
        p_k1 = float(np.mean(k1_ms[len(k1_keep):]))
        del k1_ms[len(k1_keep):]
        panel = dict(ms=p_ms, cells=p_cells, k1_ms=p_k1, best_pairs={g: (r[0][:4] if r else None) for g, r in p_res.items()},
                     launches=0)
        Tp.close(); Tpc.close()

    # ---- cohort leg ----
    host_s, host_n, host_bytes, host_info = 0.0, 0, 0, None
    if args.cohort_samples > 0:
        barrier()
        try:
            host_s, host_n, host_bytes, host_info = run_cohort(w, args.cohort_samples, rank, world, local_rank, args.cohort_workers)
        except Exception as e:  # the contract line must not depend on this leg
            host_info = dict(error=f"{type(e).__name__}: {e}")
        barrier()

    # max over ranks of every time, sums of the counts
    if world > 1:
        t = torch.tensor([ms_total, e2e_s, k1_avg_ms, host_s, panel["ms"] if panel else 0.0, panel["k1_ms"] if panel else 0.0],
                         dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, e2e_s, k1_avg_ms, host_s, p_ms_max, p_k1_max = (float(x) for x in t.cpu())
        if panel:
            panel["ms"], panel["k1_ms"] = p_ms_max, p_k1_max
        cnt = torch.tensor([host_n, launches, h2d, d2h], dtype=torch.int64, device=dev)
        dist.all_reduce(cnt)
        host_n, launches, h2d, d2h = (int(x) for x in cnt.cpu())

    if rank == 0:
        value = cells_total * args.steps / (ms_total * 1e-3) / 1e9
        e2e_val = cells_total * args.steps / e2e_s / 1e9
        achieved = INT_OPS_PER_CELL * cells_dna_local / (k1_avg_ms * 1e-3)
        hbm_bytes = (T_dna.total_len + P_dna.padded_rows * 0.75 + 2.0 * len(idx_d) * R)
        peaks, traffic = {}, {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:
            pass
        try:  # dram__bytes_read.sum + dram__bytes_write.sum of the K1 DNA launches of one step, from a committed ncu capture
            traffic = json.loads((ROOT / "profiles" / "k1_dram_traffic.json").read_text())
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        cpu = cpu_sample(w, args.cpu_seconds) if world == 1 else None  # the CPU baseline is an N=1 figure
        cohort = None
        if host_n and host_s > 0:
            cohort = dict(samples_per_s=host_n / host_s, samples=host_n, ms_per_sample_per_gpu=host_s / (host_n / world) * 1e3,
                          json_bytes_per_sample=host_bytes // max(host_n // world, 1), **host_info,
                          scaling="replicas: independent samples round-robin over ranks, no exchange (%d per GPU; 1,000 at 8 GPUs); per GPU %d host "
                                  "threads with one sp_ctx each (sp_ctx_share_device) take samples from one queue" % (host_n // world, host_info.get("workers_per_gpu", 1)),
                          sample="per sample, through the C++ host above the C ABI: HLA-A + HLA-B diplotype calls (64 reads per gene, DNA + cDNA, "
                                 "against that gene's full allele set: K1 x2, K2, het/hom, K5 + K4 read assignment), CYP2D6 39-template search with "
                                 "K4 tracebacks + weight_sequence + chains + find_best_chain_pair on a diploid 96-read case, result JSON text out "
                                 "(BASELINE configs[4], SURVEY 8d.5)")
        elif host_info:
            cohort = host_info
        line = dict(
            metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
            ms_per_step=ms_total / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
            dtype="u32", data="synthetic",
            config=bench_config(world, args.scale),
            best_pairs={g: (r[0][:4] if r else None) for g, r in result.items()},
            clocks=dict(sm_mhz=clocks["sm_mhz"], sm_max_mhz=clocks["sm_max_mhz"], reasons=clocks["reasons"], samples=clocks["samples"],
                        period_ms=ClockSampler.PERIOD_MS),
            e2e=dict(value=e2e_val, unit=UNIT, h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h),
                     note="per step: read set from pinned host memory on rank 0 (sp_comm_bcast_targets x2), K1 x2 + all-gather, K2 per gene + "
                          "merge, u16 distance matrices [reads x alleles] (each rank its row block) + top-k records back to pinned host memory"),
            gpu_launches=int(launches),
            multi_gpu="sp_comm_* (NCCL inside libstarphase_gpu.so): bcast_targets, score_allgather, pair_minsum_topk" if world > 1 else None,
            samples_per_s=(cohort or {}).get("samples_per_s"),
            cohort=cohort,
            panel=(dict(gcups=panel["cells"] * args.panel_steps / (panel["ms"] * 1e-3) / 1e9, ms_per_step=panel["ms"] / args.panel_steps,
                        steps=args.panel_steps, scaling="strong", reads=args.panel_reads, cells_per_step=panel["cells"],
                        k1_dna_ms=panel["k1_ms"], best_pairs=panel["best_pairs"],
                        workload="panel_1000x: %d reads (fixed) x 12,451 DNA + 19,629 cDNA alleles, alleles sharded %d ways "
                                 "(BASELINE configs[2]); same step as the main leg" % (args.panel_reads, world))
                   if panel else None),
            roofline=dict(bound="int_alu", kernel="k1_infix (DNA launches, all lane-width classes)", achieved=achieved / 1e12,
                          peak=int_peak2 / 1e12, unit="Tops/s (algorithmic INT32 lane-ops, 23/64 per cell, SURVEY 8d)",
                          frac=achieved / int_peak2,
                          peak_source="measured live: dependent-free LOP3+IMAD loop = ALU and FMA pipes together (sp_int_peak kind 2); "
                                      "MEASURED_PEAKS.json holds no integer peak",
                          peak_alu_pipe_only=int_peak / 1e12, frac_alu_pipe_only=achieved / int_peak,
                          peak_theoretical=148 * 128 * 1.965e9 / 1e12,
                          note="K1 issues 7 of its ~11 instructions per 32 cells on the ALU pipe (the binding one) and 4 "
                               "as IMAD on the FMA pipe (the algorithmic count of SURVEY 8d is 11.5), so the algorithmic count "
                               "exceeds the ALU-pipe-only peak (DESIGN.md 4.1)",
                          k1_ms=k1_avg_ms, k1_tcups=cells_dna_local / (k1_avg_ms * 1e-3) / 1e12,
                          traffic=(traffic.get("bytes_per_step") if world == 1 and args.scale == 1.0 else None),
                          traffic_source=traffic.get("source") if traffic else None,
                          traffic_unit="bytes per step (all K1 DNA launches), algorithmic bytes = %d" % hbm_bytes,
                          hbm=dict(achieved=hbm_bytes / (k1_avg_ms * 1e-3) / 1e9, peak=hbm_peak, unit="GB/s",
                                   frac=hbm_bytes / (k1_avg_ms * 1e-3) / 1e9 / hbm_peak,
                                   peak_source="MEASURED_PEAKS.json" if peaks else "fallback")),
            cpu_baseline=(dict(value=cpu["gcups"], unit=UNIT, cores=cpu["cores"], kind="port", sample=cpu["sample"]) if cpu else None),
        )
        _emit(line)
    comm.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    _claim_stdout()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
