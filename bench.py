#!/usr/bin/env python
"""
bench.py — the genotyping hot path on the synthetic cohort of BASELINE.json configs[3]: samples x 30 TREDs,
sharded by (sample, locus) over one process per GPU, no collective on the data path, final host gather.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--samples S] [--cohort C] [--impl reference]

The cohort is a list of (sample, locus) problems (tredparse_b200.simulate.problem_spec: alleles drawn from each
locus' population histogram, 1 % forced into the risk range, gender 50/50, depth ~ N(35, 5^2)).  Every rank owns
the problems the cost-sorted deal of tredparse_b200.dist.shard_by_cost gives it (a-priori cost = depth x ploidy
x template cells of the locus) and simulates exactly those — DISTINCT reads in every batch, nothing replayed.

  default       weak scaling: N x (W + K) x S samples; every rank gets ~(W + K) batches of S x 30 problems
                (W warm-up batches, K timed ones).  At N = 1, K = 20, S = 384: 8,832 samples, 264,960 problems.
  --cohort C    strong scaling of a fixed C-sample cohort (configs[3] names C = 10,000): the rank's share is cut
                into K timed batches; the warm-up repeats the first one.

A *step* is one pass of the whole hot path — Smith-Waterman of every read against its locus' template family +
classification, tallies, candidate ranges, KDE, likelihood grid, call / CI / PP / label — over one batch.

Rank 0 prints ONE JSON line:
  value        loci genotyped / s, whole job, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e          the same through the C ABI from HOST buffers: per step the batch's base codes are packed into the
               transfer format (native, inside the timed region), copied H2D, processed, the calls copied D2H;
               the call records of all ranks are gathered on rank 0 (dist.gather_records) before the clock stops
  roofline     dominant kernel = sw_family classify kernels (integer/DPX pipe, see DESIGN.md); roofline_grid /
               roofline_grid_stress = likelihood grid vs the measured HBM copy bandwidth
  cpu_baseline the reference's own CPU code (oracle/refdrive.py: BamParser.parse + IntegratedCaller.call through
               oracle/refshim.py, bound to the reference's ssw.c) on the first samples of the SAME cohort, one
               persistent process pool over all host cores, median of passes; also a call-by-call parity check

`--impl reference` times only that CPU path (rank 0 alone when launched under torchrun).

`--dump-outputs DIR` writes the call records of the last timed step (rank 0) as DIR/<field>.npy, so that two builds
can be compared output for output: the cohort is seeded, so the same arguments give the same inputs.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the source tree may be read-only: nothing is written there

METRIC = "loci genotyped/sec"
UNIT = "loci/s"
READLEN = 150
COHORT_SEED = 20240000


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--samples", type=int, default=384, help="samples per batch per GPU (x 30 loci) in the default mode")
    p.add_argument("--cohort", type=int, default=0, help="strong scaling: a fixed cohort of this many samples")
    p.add_argument("--no-grid-stress", action="store_true", help="skip the long-expansion grid measurement "
                   "(BASELINE configs[4]) reported as roofline_grid_stress")
    p.add_argument("--depth", type=int, default=3, help="host-buffer calls kept in flight by the e2e pipeline")
    p.add_argument("--streams", type=int, default=3, help="streams the device-resident steps alternate over "
                   "(the tail of one step's persistent SW kernel overlaps the head of the next step)")
    p.add_argument("--no-numa", action="store_true", help="do not bind the ranks to the cores next to their GPUs")
    p.add_argument("--transfer", default="auto", choices=("auto", "bytes", "packed4"),
                   help="e2e leg: copy the reads as ingest leaves them (one byte per base, pinned), or pack them to "
                        "4 bit/base on the host first (inside the timed region) — less PCIe traffic, more host work")
    p.add_argument("--from-bam", type=int, default=32, help="samples of the from-BAM leg (N = 1 only; 0 = skip): synthetic "
                   "whole-sample BAMs (+-10 kb windows at 30 loci) through tred.run_chunks (chunks of 8 samples, two stages "
                   "deep), GPU ingest included; the reference arm reads the first 8 of them")
    p.add_argument("--impl", default="tredsw", choices=("tredsw", "reference"))
    p.add_argument("--cpu-sample", type=int, default=0, help="samples in the CPU baseline sample (0 = auto)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the call records of the last "
                   "timed step of rank 0 as DIR/<field>.npy (float64; ci is n x 4) and DIR/problem.npy (cohort index "
                   "sample x loci + locus of every row); above 64 MB in all, a fixed seeded sample of the rows")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    return args


def distinct_loci(repo):
    """30 distinct locations among the 32 catalogue names (FXS == FXTAS, SBMA == AR coordinates)."""
    seen, names = set(), []
    for n in repo.names:
        t = repo[n]
        key = (t.chr, t.repeat_start, t.repeat_end)
        if key in seen:
            continue
        seen.add(key)
        names.append(n)
    return names


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fp:
            d = json.load(fp)
        return float(d.get("hbm_gbs", 6650.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (every 100 ms: faster polling
    contends for the driver and measurably slows the host-buffer calls of the e2e leg)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------
# cohort generation (host processes, before CUDA is touched)
# ---------------------------------------------------------------------------------------------------------
_GEN = {}


def _gen_batch(pairs):
    """Worker: simulate the (sample, locus) problems `pairs` and lay them out as one batch (flat buffers in the
    layout tredsw_genotype_batch consumes — what the native BAM ingest writes for real data)."""
    from tredparse_b200 import cohort, simulate
    from tredparse_b200.meta import TREDsRepo
    if "repo" not in _GEN:
        _GEN["repo"] = TREDsRepo()
        _GEN["names"] = distinct_loci(_GEN["repo"])
    repo, names = _GEN["repo"], _GEN["names"]
    problems = [simulate.simulate_from_spec(repo, simulate.problem_spec(repo, names, int(s), int(li), READLEN, COHORT_SEED))
                for s, li in pairs]
    b = cohort.CohortBatch(problems, family_keys=[(repo[n], READLEN) for n in names])
    return {"rbuf": b.rbuf, "roff": b.roff, "read_problem": b.read_problem, "problems": b.problems,
            "pe_lens": b.pe_lens, "max_read_len": b.max_read_len}


def build_batches(pair_chunks, workers):
    """[[(sample, locus)]] -> list of array dicts, generated by a process pool."""
    import multiprocessing as mp
    if workers <= 1 or len(pair_chunks) == 1:
        return [_gen_batch(c) for c in pair_chunks]
    # smaller tasks than batches keep all workers busy; the pieces of a batch are concatenated afterwards
    pieces, owner = [], []
    for bi, chunk in enumerate(pair_chunks):
        k = max(1, min(len(chunk), (workers * 2 + len(pair_chunks) - 1) // len(pair_chunks)))
        for part in np.array_split(np.asarray(chunk, dtype=np.int64).reshape(-1, 2), k):
            if len(part):
                pieces.append(part)
                owner.append(bi)
    with mp.get_context("fork").Pool(processes=workers) as pool:
        parts = pool.map(_gen_batch, pieces, chunksize=1)
    out = []
    for bi in range(len(pair_chunks)):
        mine = [p for p, o in zip(parts, owner) if o == bi]
        out.append(merge_parts(mine))
    return out


def merge_parts(parts):
    if len(parts) == 1:
        return parts[0]
    rbuf = np.concatenate([p["rbuf"] for p in parts])
    pe = np.concatenate([p["pe_lens"] for p in parts])
    roff, rprob, probs = [np.zeros(1, np.int64)], [], []
    rbase = pbase = pebase = 0
    for p in parts:
        roff.append(p["roff"][1:] + rbase)
        rprob.append(p["read_problem"] + pbase)
        q = p["problems"].copy()
        q["off_global"] += pebase
        q["off_target"] += pebase
        probs.append(q)
        rbase += int(p["roff"][-1]); pbase += len(p["problems"]); pebase += len(p["pe_lens"])
    return {"rbuf": rbuf, "roff": np.concatenate(roff), "read_problem": np.concatenate(rprob),
            "problems": np.concatenate(probs), "pe_lens": pe, "max_read_len": max(p["max_read_len"] for p in parts)}


def batch_from_arrays(cohort, template, arr):
    """A CohortBatch around generated arrays (the family / locus tables are those of `template`)."""
    b = object.__new__(cohort.CohortBatch)
    b.__dict__.update(template.__dict__)
    b.problems, b.rbuf, b.roff, b.read_problem, b.pe_lens = (arr["problems"], arr["rbuf"], arr["roff"],
                                                             arr["read_problem"], arr["pe_lens"])
    b.nproblems, b.nreads, b.max_read_len = len(arr["problems"]), len(arr["roff"]) - 1, int(arr["max_read_len"])
    b.objects, b._dev, b._packed, b.read_name = None, None, None, None
    return b


def _write_bam(job):
    from tredparse_b200 import simulate, bamio
    from tredparse_b200.meta import TREDsRepo
    path, sample = job
    repo = TREDsRepo()
    names = distinct_loci(repo)
    sam = bamio.AlignmentFile(os.path.join(ROOT, "tests", "golden", "t001.mini.bam"))
    refs = list(zip(sam.references, sam.lengths))
    sam.close()
    simulate.write_sample_bam(path, repo, names, refs, sample, READLEN, COHORT_SEED)
    return path


def make_bams(nsamples, workers, d):
    """Synthetic whole-sample BAMs of the first `nsamples` cohort samples, written into the directory `d`."""
    import multiprocessing as mp
    jobs = [(os.path.join(d, "s{:04d}.bam".format(s)), s) for s in range(nsamples)]
    with mp.get_context("fork").Pool(processes=max(1, min(workers, len(jobs)))) as pool:
        pool.map(_write_bam, jobs, chunksize=1)
    return [j[0] for j in jobs]


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(d, calls, problem):
    """--dump-outputs: one float64 .npy per CALL_DTYPE field plus problem.npy.  When the rows exceed DUMP_BYTES, the
    same seeded sample of rows (kept in order) is written on every run."""
    cols = {name: calls[name] for name in calls.dtype.names}
    cols["problem"] = problem
    row_bytes = 8 * sum(int(np.prod(c.shape[1:])) for c in cols.values())
    limit = (DUMP_BYTES - 1024 * len(cols)) // row_bytes            # (1 KB per file for the .npy header)
    rows = np.arange(len(calls))
    if len(rows) > limit:
        rows = np.sort(np.random.default_rng(0).choice(len(rows), limit, replace=False))
    os.makedirs(d, exist_ok=True)
    for name, c in cols.items():
        np.save(os.path.join(d, name + ".npy"), np.ascontiguousarray(c[rows], dtype=np.float64))


def _ref_run_bam(job):
    from oracle import refdrive
    return refdrive.run_bam(job)


# ---------------------------------------------------------------------------------------------------------
# the reference's CPU path (cpu_baseline and --impl reference)
# ---------------------------------------------------------------------------------------------------------
def reference_tasks(nsamples):
    """The first `nsamples` samples of the cohort x 30 loci as tasks of oracle.refdrive.genotype_problem."""
    from tredparse_b200 import simulate
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    names = distinct_loci(repo)
    tasks, keys = [], []
    for s in range(nsamples):
        for li in range(len(names)):
            pr = simulate.simulate_from_spec(repo, simulate.problem_spec(repo, names, s, li, READLEN, COHORT_SEED))
            tasks.append((names[li], pr.readlen, pr.ploidy, pr.depth, pr.read_strings(), pr.name_strings(),
                          pr.global_lens.tolist(), pr.target_lens.tolist()))
            keys.append((s, li))
    return tasks, keys, len(names)


def _ref_one_thread():
    """Pool initializer: one BLAS / OpenMP thread per worker process.  The pool already runs one process per core; with
    the libraries' default (one thread per core in EVERY process) the numpy / scipy calls of the reference
    oversubscribe the host 16-fold and the arm runs ~4x slower — and torchrun exports OMP_NUM_THREADS=1 while a plain
    `python bench.py` does not, which made the arm differ by that factor between N = 1 and N > 1 (round-1 verdict)."""
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[k] = "1"
    try:
        import threadpoolctl
        global _REF_LIMIT
        _REF_LIMIT = threadpoolctl.threadpool_limits(limits=1)
    except Exception:
        pass


def _ref_warm(_):
    from oracle import refdrive
    refdrive.reference()
    return os.getpid()


class ReferencePool:
    """One persistent process pool for the whole run (the reference forks one per run too, tred.py:528); the
    workers load the reference package once."""

    def __init__(self, cores):
        import multiprocessing as mp
        from oracle import refdrive
        if not refdrive.usable():
            raise RuntimeError("the reference package is not loadable here (oracle/_ref/ not built)")
        self.cores = cores
        # the workers bind the reference's own ssw.c (oracle/_ref/libssw_ref.so) through its ssw_wrap.py; load it in
        # this process too, so that whoever watches the loaded libraries of the arm sees it (the workers are forks)
        import ctypes
        self._libssw = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libssw_ref.so"))
        self.pool = mp.get_context("fork").Pool(processes=cores, initializer=_ref_one_thread)
        self.pool.map(_ref_warm, range(cores * 2), chunksize=1)

    def run(self, tasks):
        from oracle import refdrive
        t0 = time.perf_counter()
        res = self.pool.map(refdrive.genotype_problem, tasks, chunksize=1)
        return res, time.perf_counter() - t0

    def run_bams(self, jobs):
        t0 = time.perf_counter()
        res = self.pool.map(_ref_run_bam, jobs, chunksize=1)
        return res, time.perf_counter() - t0

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_sample_size(args, cores, nloci, passes=1):
    """Whole samples worth ~10 s of wall time per pass at the ~5 loci/s/core of the reference's Python + ssw.c
    path (fewer per pass when many passes are asked for, so that the run ends within minutes)."""
    if args.cpu_sample:
        return max(1, args.cpu_sample)
    seconds = min(10.0, 150.0 / max(1, passes))
    return max(1, min(32, int(round(seconds * 5.0 * cores / nloci))))


def ssw_c_loop_ceiling(tasks, cores, max_pairs=40000):
    """SURVEY 8(d), CPU baseline (2): the reference's own ssw.c in a plain C loop (ssw_init -> ssw_align(flag=1) ->
    destroy per pair, oracle/ref_batch.c), no Python in the loop — one process, and one process per core."""
    import multiprocessing as mp
    from oracle import sw, evidence_oracle as evo
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    queries, templates, qidx, tidx = [], [], [], []
    for name, readlen, _, _, reads, _, _, _ in tasks:
        t = repo[name]
        mu = -(-readlen // len(t.repeat))
        db = [x for _, x in evo.template_family(t.prefix, t.repeat, t.suffix, mu)]
        t0 = len(templates)
        templates += db
        for r in reads[:8]:
            q0 = len(queries)
            queries.append(r)
            qidx += [q0] * len(db)
            tidx += list(range(t0, t0 + len(db)))
        if len(qidx) >= max_pairs:
            break
    qidx, tidx = np.array(qidx, dtype=np.int32), np.array(tidx, dtype=np.int32)
    cells = float(sum(len(queries[a]) * len(templates[b]) for a, b in zip(qidx, tidx)))
    sw.ref_align_pairs(queries[:1], templates[:1], qidx[:1] * 0, tidx[:1] * 0)       # load / warm
    t0 = time.perf_counter()
    sw.ref_align_pairs(queries, templates, qidx, tidx)
    dt1 = time.perf_counter() - t0
    _SSW["job"] = (queries, templates, qidx, tidx)
    with mp.get_context("fork").Pool(processes=cores) as pool:
        pool.map(_ssw_job, range(cores))                                              # warm
        t0 = time.perf_counter()
        pool.map(_ssw_job, range(cores))
        dtn = time.perf_counter() - t0
    return {"pairs": int(len(qidx)), "us_per_alignment": 1e6 * dt1 / len(qidx), "gcups_one_core": cells / dt1 / 1e9,
            "processes": cores, "gcups_all_cores": cores * cells / dtn / 1e9}


_SSW = {}


def _ssw_job(_):
    from oracle import sw
    sw.ref_align_pairs(*_SSW["job"])
    return 0


def run_reference(args, rank):
    """--impl reference: the reference's CPU implementation of the path, rank 0 only."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    passes = args.warmup + args.steps
    tasks, keys, nloci = reference_tasks(cpu_sample_size(args, cores, 30, passes=passes))
    pool = ReferencePool(cores)
    times = []
    for it in range(passes):
        res, dt = pool.run(tasks)
        if it >= args.warmup:
            times.append(dt)
    pool.close()
    med = float(np.median(times))
    value = len(tasks) / med
    reads, cells = sum(r[4] for r in res), sum(r[5] for r in res)
    sample = "samples 0..{} of the cohort x {} loci = {} problems ({} reads) per step".format(
        len(tasks) // nloci - 1, nloci, len(tasks), reads)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * med,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/int16 (ssw.c SSE2) / f64",
        "data": "synthetic",
        "config": {"workload": "synthetic cohort x 30 TREDs (BASELINE configs[3]), same cohort as the GPU arm, "
                               "bounded sample: " + sample,
                   "readlen": READLEN, "maxinsert": 300,
                   "parallelism": "one persistent multiprocessing.Pool({}); value = problems / median step time".format(cores)},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample,
                         "loci_per_s_per_core": value / cores, "reads_per_s": reads / med,
                         "sw_gcups": cells / med / 1e9, "step_seconds": [round(t, 3) for t in times],
                         "code": "the reference's own tredparse/bam_parser.py + models.py + src/ssw_wrap.py (oracle/refshim.py) "
                                 "on its own src/ssw.c (oracle/_ref/libssw_ref.so)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------------------
# calibration of the executed-instruction count (see DESIGN.md §6)
# ---------------------------------------------------------------------------------------------------------
def kernel_fingerprint():
    """SHA-1 over the SASS (opcodes and operands, no addresses) of the Smith-Waterman classify kernels of the
    shipped library, or None when cuobjdump is not available."""
    so = os.path.join(ROOT, "tredparse_b200", "libtredsw.so")
    try:
        out = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, timeout=300).stdout
    except Exception:
        return None
    h, on, n = hashlib.sha1(), False, 0
    for ln in out.splitlines():
        t = ln.strip()
        if t.startswith("Function :"):
            on = "sw_family" in t and "classify_kernel" in t
            continue
        if on and t.startswith("/*") and ";" in t:
            h.update(t.split("*/", 1)[1].split(";")[0].strip().encode())
            n += 1
    return h.hexdigest() if n else None


def load_calibration():
    """profiles/r2_counters.json: per-kernel counters of this round's ncu capture (tools/calibrate.py) with the
    SASS fingerprint of the kernel they were measured on."""
    path = os.path.join(ROOT, "profiles", "r2_counters.json")
    if not os.path.exists(path):
        return None
    with open(path) as fp:
        return json.load(fp)


def main():
    args = parse_args()
    # stdout carries exactly ONE JSON line: libraries that print there (NCCL's version banner, ...) are sent
    # to stderr for the whole run, the line itself goes to the saved descriptor
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        _main(args)
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)
        for ln in _LINES:
            print(ln, flush=True)


_LINES = []


def emit(line):
    _LINES.append(json.dumps(line))


def _main(args):
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    from tredparse_b200 import simulate, dist as tdist
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    names = distinct_loci(repo)
    nloci = len(names)
    W, K = max(args.warmup, 3), args.steps
    # several ranks on one host: each next to its GPU (the staging buffers of the e2e leg are first-touched here)
    numa = tdist.bind_to_gpu_numa(local_rank) if world > 1 and not args.no_numa else None
    if args.transfer == "auto":
        # packing the reads to 4 bit/base halves the PCIe bytes but costs host cores: it pays with one GPU per host
        # (+10 % where PCIe is the slower side), not with 4-8 ranks sharing the cores (measured: profiles/)
        args.transfer = "packed4" if world == 1 else "bytes"

    # ---- the cohort and this rank's share of it (no communication: every rank computes the same partition) ---
    t_gen = time.perf_counter()
    strong = args.cohort > 0
    nsamples = args.cohort if strong else world * (W + K) * args.samples
    costs = simulate.problem_costs(repo, names, nsamples, READLEN, COHORT_SEED)
    owner = tdist.shard_by_cost(costs, world)
    all_counts = np.bincount(owner, minlength=world)
    mine = np.nonzero(owner == rank)[0]                      # flat index = sample * nloci + locus
    nbatches = K if strong else W + K
    chunks = [np.stack([c // nloci, c % nloci], axis=1) for c in np.array_split(mine, nbatches)]
    workers = max(1, min(16, (os.cpu_count() or 1) // max(1, min(world, 8))))
    arrays = build_batches(chunks, workers)
    t_gen = time.perf_counter() - t_gen
    bams, bam_dir = [], None
    if rank == 0 and world == 1 and args.from_bam > 0:
        t_b = time.perf_counter()
        bam_dir = tempfile.TemporaryDirectory(prefix="tredsw_bench_bams-")
        bams = make_bams(args.from_bam, workers, bam_dir.name)
        t_bams = time.perf_counter() - t_b
    # the CPU baseline's process pool is forked here, before CUDA / NCCL exist in this process (rank 0, N = 1 only)
    ref_pool, ref_pool_error = None, "not requested"
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            ref_pool = ReferencePool(os.cpu_count() or 1)
        except Exception as e:
            ref_pool_error = repr(e)

    import torch
    import torch.distributed as dist
    from tredparse_b200 import _lib, cohort

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (tredparse_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        tdist.init("nccl", device_id=torch.device("cuda", local_rank))

    template = cohort.CohortBatch([], family_keys=[(repo[n], READLEN) for n in names])
    batches = [batch_from_arrays(cohort, template, a) for a in arrays]
    # the timed batches come first in the rank's (index-sorted) share, the warm-up batches last
    timed = batches if strong else batches[:K]
    warm = [batches[0]] * W if strong else batches[K:]
    timed_idx = np.concatenate([np.asarray(c[:, 0] * nloci + c[:, 1]) for c in (chunks if strong else chunks[:K])])
    timed_counts = []                                        # of every rank (the partition is deterministic)
    for r in range(world):
        sizes = [len(c) for c in np.array_split(np.nonzero(owner == r)[0], nbatches)]
        timed_counts.append(int(sum(sizes if strong else sizes[:K])))

    stream = torch.cuda.Stream(device=local_rank)
    ctx = _lib.Context(local_rank, stream=stream.cuda_stream)
    int_peak = ctx.int_pipe_peak()
    for b in batches:
        b.to_device(local_rank)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing -------------------------------------------------------------------
    with torch.cuda.stream(stream):
        for b in warm:
            b.run_device(ctx)
    stream.synchronize()
    # stage timing and unit counters of one extra (untimed) pass over the first timed batch, for the rooflines
    ctx.enable_timing(True)
    with torch.cuda.stream(stream):
        timed[0].run_device(ctx)
    stage = ctx.timing()
    ctx.enable_timing(False)
    st = timed[0].run_host(ctx=ctx, want_stats=True)["stats"]

    # the timed steps alternate over `--streams` contexts (each with its own stream and scratch): consecutive
    # steps are independent batches of the cohort, so nothing orders them
    lanes = [(ctx, stream)]
    for _ in range(max(1, args.streams) - 1):
        s2 = torch.cuda.Stream(device=local_rank)
        lanes.append((_lib.Context(local_rank, stream=s2.cuda_stream), s2))
    for c2, s2 in lanes[1:]:
        for b in warm[:2]:
            b.run_device(c2)
        s2.synchronize()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    launches0 = sum(c.launches for c, _ in lanes)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _, s2 in lanes[1:]:
        s2.wait_event(e0)
    for i, b in enumerate(timed):
        b.run_device(lanes[i % len(lanes)][0])
    for _, s2 in lanes[1:]:
        ev = torch.cuda.Event()
        ev.record(s2)
        stream.wait_event(ev)
    e1.record(stream)
    stream.synchronize()
    barrier()
    launches = sum(c.launches for c, _ in lanes) - launches0
    ms = e0.elapsed_time(e1)
    calls_dev = np.concatenate([b.calls_from_device() for b in timed])

    # ---- end to end through the C ABI from host buffers ---------------------------------------------
    # Per step, inside the timed region: the batch's base codes (one byte per base, as ingest leaves them) and
    # pair lengths are packed into the transfer formats by native host code, copied H2D from pinned memory,
    # processed, and the calls copied D2H; `depth` calls are kept in flight (the packing and the copy of batch
    # k+1 overlap the kernels of batch k).  The call records of every rank are gathered on rank 0 at the end.
    def pin(a):
        t = torch.from_numpy(a.view(np.uint8) if a.dtype.fields else a).pin_memory()
        return t.numpy().view(a.dtype) if a.dtype.fields else t.numpy()
    for b in batches:
        for name in ("roff", "read_problem", "problems"):
            setattr(b, name, pin(getattr(b, name)))
    # pair lengths: the producer's format is int16 already (what is kept is < 1000, bam_parser.py:356-357) — pinned
    # once, like the offsets; the base codes arrive one byte per base and are packed per step
    packing = args.transfer == "packed4"
    for b in batches:
        b.pe16 = pin(b.pe_lens.astype(np.int16))
        if not packing:
            b.rbuf = pin(b.rbuf)                                   # ingest writes into caller-owned pinned buffers
    depth = max(1, args.depth)
    max_bases = max(len(b.rbuf) for b in batches)
    slots = [pin(np.zeros(((max_bases + 7) // 8) * 4, np.uint8)) if packing else None for _ in range(depth)]
    pipe = cohort.HostPipeline(local_rank, depth=depth)
    pack_threads = max(1, min(4, (os.cpu_count() or 1) // max(1, world * depth)))

    def step_e2e(ctx_slot, b):
        cx, slot = ctx_slot
        if packing:
            return b.run_host(ctx=cx, packed={"rbuf": b.pack_reads4(slot, pack_threads), "pe_lens": b.pe16})["calls"]
        return b.run_host(ctx=cx, packed={"pe_lens": b.pe16})["calls"]

    import queue
    from concurrent.futures import ThreadPoolExecutor
    free = queue.Queue()
    for cx, slot in zip(pipe.contexts, slots):
        free.put((cx, slot))

    def worker(b):
        cs = free.get()
        try:
            return step_e2e(cs, b)
        finally:
            free.put(cs)

    with ThreadPoolExecutor(max_workers=depth) as tp:
        for _ in tp.map(worker, warm + warm[:depth]):
            pass
        # the gather path once, untimed (NCCL sets up the channels of a collective on its first use)
        tdist.gather_records(np.zeros(timed_counts[rank], dtype=cohort.CALL_DTYPE), timed_idx, nsamples * nloci,
                             all_counts=timed_counts, require_all=False, return_seen=True)
        barrier()
        e2e_launch0 = pipe.launches
        t0 = time.perf_counter()
        host_calls = list(tp.map(worker, timed))
        torch.cuda.synchronize()
        local_calls = np.concatenate(host_calls)
        gathered, seen = tdist.gather_records(local_calls, timed_idx, nsamples * nloci, all_counts=timed_counts,
                                              require_all=strong, return_seen=True)
        t_e2e = time.perf_counter() - t0
    barrier()
    clocks = sampler.stop()
    e2e_launches = pipe.launches - e2e_launch0
    h2d = sum(b.h2d_bytes for b in timed) / len(timed)
    d2h = sum(b.d2h_bytes for b in timed) / len(timed)
    pipe.close()
    assert local_calls.tobytes() == calls_dev.tobytes(), "device-resident and host paths disagree"
    if rank == 0:
        assert gathered is not None and int(seen.sum()) == sum(timed_counts)
        if args.dump_outputs:
            n = timed[-1].nproblems
            dump_outputs(args.dump_outputs, calls_dev[len(calls_dev) - n:], timed_idx[len(timed_idx) - n:])

    # ---- reduce over ranks: timings MAX, unit counters SUM (no data-path collective anywhere) --------
    nprob_timed = sum(b.nproblems for b in timed)
    nreads_timed = sum(b.nreads for b in timed)
    (ms, t_e2e_ms), cnt = tdist.reduce_max_sum(
        [ms, t_e2e * 1e3], [nprob_timed, nreads_timed, launches, h2d, d2h],
        device="cuda" if world > 1 else "cpu")
    t_e2e = t_e2e_ms / 1e3
    nprob, nreads, launches, h2d_all, d2h_all = cnt

    if rank == 0:
        sec = ms / 1e3
        value = nprob / sec
        b0 = timed[0]
        hbm, hbm_src = peaks()
        sw_s = stage["sw"] / 1e3
        grid_s = max(stage["grid"], 1e-6) / 1e3
        # executed integer-pipe lane-instructions = executed DP cells (counted by the kernel) x ALU instructions per
        # cell.  The factor comes from this round's ncu capture of the SAME kernel binary (profiles/r2_counters.json
        # carries the SASS fingerprint it was measured on); when the shipped kernel differs from the profiled one
        # the line says so instead of silently reusing the number.
        cal, fp = load_calibration(), kernel_fingerprint()
        ccal = (cal or {}).get("classify") or {}
        alu_per_cell = ccal.get("alu_lane_instr_per_executed_cell")
        cal_state = "none (no profiles/r2_counters.json)"
        if alu_per_cell:
            cal_state = "current" if (fp and fp == ccal.get("sass_sha1")) else \
                ("unverified (cuobjdump unavailable)" if fp is None else "STALE: the shipped classify kernel differs from the profiled one")
        executed_cells = int(st[1]) + int(st[2])
        achieved = executed_cells * alu_per_cell / sw_s / 1e9 if alu_per_cell else None
        scale = b0.nreads / max(1.0, float(ccal.get("reads", b0.nreads)))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": len(timed),
            "warmup": W, "ms_per_step": ms / len(timed), "higher_is_better": True,
            "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "int16 (SW, DPX s16x2) / f64 (likelihood)", "data": "synthetic",
            "config": {"workload": "synthetic cohort x 30 TREDs (BASELINE configs[3]): {} samples x {} loci = {} problems, "
                                   "sharded by (sample, locus) with the cost-sorted deal of dist.shard_by_cost; {} distinct "
                                   "batches of ~{} problems timed per GPU ({} problems, {} reads in all)".format(
                                       nsamples, nloci, nsamples * nloci, len(timed), b0.nproblems, int(nprob), int(nreads)),
                       "readlen": READLEN, "maxinsert": 300, "fullsearch": False,
                       "parallelism": "{} GPU(s), one process each, no collective on the data path, final gather of the call "
                                      "records on rank 0; {} stream(s) per GPU".format(world, len(lanes)),
                       "l2": "every timed step reads a different batch ({:.0f} MB of inputs + scratch per step, L2 is 126 MB): "
                             "nothing is replayed".format((b0.rbuf.nbytes + b0.pe_lens.nbytes + 8 * b0.nproblems * 1000) / 1e6)},
            "reads_per_s": nreads / sec,
            "sw_gcups_algorithmic": int(st[0]) * (nreads / max(1, b0.nreads)) / sec / 1e9,
            "e2e": {"value": nprob / t_e2e, "unit": UNIT,
                    "h2d_bytes_per_step": int(h2d_all), "d2h_bytes_per_step": int(d2h_all),
                    "ms_per_step": 1e3 * t_e2e / len(timed), "calls_in_flight": depth,
                    "transfer": args.transfer, "numa": numa,
                    "includes": ("per step: native packing of the batch's base codes (1 byte/base as ingest leaves them -> "
                                 "4 bit/base, {} host threads), ".format(pack_threads) if packing else
                                 "per step: the batch's reads as ingest leaves them (1 byte/base, no host-side repacking), ") +
                                "H2D from pinned memory, kernels, D2H of the calls; at the end the gather of the {} call records "
                                "on rank 0.  Pair lengths are int16 from the producer (kept lengths are < 1000).".format(int(seen.sum()))},
            "gpu_launches": int(launches) + int(e2e_launches),
            "clocks": clocks,
            "roofline": {"kernel": "classify_kernel<P> (sw_family.cu), all period instantiations of one step",
                         "bound": "int", "achieved": achieved, "peak": int_peak, "unit": "G lane-instr/s",
                         "frac": achieved / int_peak if achieved else None,
                         "traffic": ccal.get("dram_bytes") * scale if ccal.get("dram_bytes") else None,
                         "calibration": cal_state,
                         "peak_source": "tredsw_int_pipe_peak (VIADDMNMX.S16x2 register loop, 64 lanes/clk/SM) measured in this run; "
                                        "achieved = executed DP cells of this run x ALU lane-instructions per executed cell "
                                        "from the ncu capture of this kernel binary (profiles/r2_counters.json)",
                         "alu_lane_instr_per_executed_cell": alu_per_cell,
                         "algorithmic_int_ops_per_s": 10.0 * int(st[0]) / sw_s,
                         "kernel_ms": stage["sw"], "share_of_step": stage["sw"] / max(stage["total"], 1e-9),
                         "executed_gcups": executed_cells / sw_s / 1e9,
                         "algorithmic_gcups": int(st[0]) / sw_s / 1e9,
                         "timing": "one batch alone on one stream (the headline value overlaps consecutive batches on {} streams)".format(len(lanes))},
            "roofline_grid": {"kernel": "grid_classify + grid_points_setup + grid_reduce_eval + grid_rows_reduce (default search)",
                              "bound": "hbm", "achieved": 8.0 * int(st[4]) / grid_s / 1e9, "peak": hbm, "unit": "GB/s",
                              "frac": 8.0 * int(st[4]) / grid_s / 1e9 / hbm, "peak_source": hbm_src,
                              "kernel_ms": stage["grid"], "points": int(st[4]), "bytes_per_point": 8,
                              "note": "a few dozen points per problem: launch latency of four kernels, not bandwidth"},
            "stage_ms": stage, "setup_s": {"simulate_and_layout": t_gen, "workers": workers},
        }
        if not args.no_grid_stress:
            # the grid kernels at the configuration their HBM roofline is quoted on (BASELINE configs[4]: 64
            # problems x 500,500 points, --fullsearch, maxinsert 1000)
            try:
                sys.path.insert(0, os.path.join(ROOT, "tools"))
                import grid_stress
                gs = grid_stress.run(problems=64, maxinsert=1000, readlen=150, reps=5, device=local_rank)
                gcal = (cal or {}).get("grid_stress") or {}
                line["roofline_grid_stress"] = {
                    "kernel": "grid_classify + grid_points_setup + grid_reduce_eval + grid_rows_reduce (row-structured, surface not materialised)",
                    "workload": "long-expansion stress (BASELINE configs[4]): 64 problems x 500,500 points, fullsearch, maxinsert 1000, 150 bp",
                    "bound": "hbm", "achieved": gs["algorithmic_GBps"], "peak": hbm, "unit": "GB/s",
                    "frac": gs["algorithmic_GBps"] / hbm, "kernel_ms": gs["grid_ms"], "points": gs["points"],
                    "bytes_per_point": 8, "traffic": gcal.get("dram_bytes"),
                    "fp64_pipe_pct": gcal.get("fp64_pipe_pct"),
                    "note": "8 algorithmic bytes per point (SURVEY 8d); traffic / FP64-pipe utilisation from the ncu capture in "
                            "profiles/ (the surface is not materialised: DRAM traffic is tables + near-region scratch)"}
            except Exception as e:
                line["roofline_grid_stress"] = {"error": str(e)}
        if not args.no_cpu_baseline and world == 1:
            try:
                if ref_pool is None:
                    raise RuntimeError(ref_pool_error)
                cores = os.cpu_count() or 1
                nsamp = cpu_sample_size(args, cores, nloci)
                tasks, keys, _ = reference_tasks(nsamp)
                pool = ref_pool
                res, dt1 = pool.run(tasks)
                res, dt2 = pool.run(tasks)
                res, dt3 = pool.run(tasks)
                med = float(np.median([dt1, dt2, dt3]))
                # the sample doubles as a parity check of the GPU calls: calls, CI, PP, label and the tallies
                agree = compared = 0
                for (s, li), r in zip(keys, res):
                    gi = s * nloci + li
                    if not seen[gi]:
                        continue
                    d = cohort.decode_call(gathered[gi])
                    compared += 1
                    agree += int(d["alleles"] == r[0] and d["CI"] == r[1] and abs(d["PP"] - r[2]) < 1e-9 and
                                 d["label"] == r[3] and (d["FDP"], d["PDP"], d["RDP"]) == (r[6], r[7], r[8]))
                reads = sum(r[4] for r in res)
                cells = sum(r[5] for r in res)
                line["cpu_baseline"] = {
                    "value": len(tasks) / med, "unit": UNIT, "cores": cores, "kind": "reference",
                    "sample": "samples 0..{} of the same cohort x {} loci = {} problems, {} reads; median of 3 passes "
                              "({:.1f} / {:.1f} / {:.1f} s) on one persistent pool".format(nsamp - 1, nloci, len(tasks), reads, dt1, dt2, dt3),
                    "loci_per_s_per_core": len(tasks) / med / cores,
                    "reads_per_s": reads / med, "sw_gcups": cells / med / 1e9,
                    "code": "the reference's own bam_parser.py + models.py + ssw_wrap.py (oracle/refshim.py) on its own ssw.c",
                    "identical_to_gpu": "{}/{} problems: alleles, CI, PP (1e-9), label, FDP/PDP/RDP".format(agree, compared),
                    "ssw_c_loop": ssw_c_loop_ceiling(tasks, cores)}
            except Exception as e:  # the GPU line must still be printed
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": repr(e)}
        if bams:
            # ---- from BAM: native ingest (host threads) + the fused device call, through the product's tred.run_chunk
            try:
                from tredparse_b200 import tred as T
                tasks_b = [("s{:04d}".format(i), p, repo, list(names), 300, False, False, True, True, "INFO")
                           for i, p in enumerate(bams)]
                for pth in bams:                                                   # both arms read from the page cache
                    for ext in ("", ".bai"):
                        with open(pth + ext, "rb") as fh:
                            while fh.read(1 << 24):
                                pass
                T.run_chunk(tasks_b[:8])                                           # warm (library, pools, arenas)
                t0 = time.perf_counter()
                got = list(T.run_chunks(tasks_b, chunk=8))
                dt = time.perf_counter() - t0
                fb = {"value": len(bams) * nloci / dt, "unit": UNIT, "samples": len(bams), "loci": nloci, "seconds": dt,
                      "chunk_samples": 8,
                      "bam_mb_per_sample": os.path.getsize(bams[0]) / 1e6, "host_threads": T.INGEST_THREADS,
                      "gpu_ingest": bool(T.GPU_INGEST),
                      "what": "tred.run_chunk on synthetic whole-sample BAMs (+-10 kb windows, ~35x, 30 loci): the host reads the "
                              "compressed BGZF blocks; inflate (one warp per block, CRC-32 checked) + record walk + read selection "
                              "+ pairing by name + depth on the GPU (csrc/bgzf_gpu.cu), then ONE fused device call for all loci of "
                              "all samples and the reference's JSON fields assembled on the host; pre-steps (gender, read length) "
                              "included; the files are in the page cache for both arms; tred.run_chunks, two stages deep",
                      "setup_write_bams_s": t_bams}
                if ref_pool is not None:
                    jobs = [("s{:04d}".format(i), p, list(names)) for i, p in enumerate(bams[:8])]
                    res_b, dt_b = ref_pool.run_bams(jobs)
                    same = total = 0
                    for mine_r, theirs in zip(got, res_b):
                        for n in names:
                            total += 1
                            keys = (".1", ".2", ".CI", ".label", ".FR", ".PR", ".RR", ".FDP", ".PDP", ".RDP", ".PEDP", ".PEG", ".PET")
                            ok = all(mine_r["tredCalls"].get(n + k) == theirs.get(n + k) for k in keys)
                            ok = ok and abs(float(mine_r["tredCalls"].get(n + ".PP", -9)) - float(theirs.get(n + ".PP", -8))) < 1e-9
                            ok = ok and abs(float(mine_r["tredCalls"].get(n + ".DP", -9)) - float(theirs.get(n + ".DP", -8))) < 1e-9
                            same += int(ok)
                    fb["reference"] = {"value": len(jobs) * nloci / dt_b, "unit": UNIT, "cores": ref_pool.cores, "seconds": dt_b,
                                       "samples": len(jobs),
                                       "what": "the reference's own tred.run (oracle/refshim.py) on the same BAM files, one sample per "
                                               "process; its pysam calls are served by the repo's pure-Python BAM reader",
                                       "identical_to_gpu": "{}/{} loci: alleles, CI, PP, label, FR/PR/RR, depths, PE summaries".format(same, total)}
                line["from_bam"] = fb
            except Exception as e:
                line["from_bam"] = {"error": repr(e)}
            bam_dir.cleanup()
        if ref_pool is not None:
            ref_pool.close()
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
