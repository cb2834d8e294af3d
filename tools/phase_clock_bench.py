#!/usr/bin/env python
"""Where the packed family kernel's time goes: per-phase clock shares of classify_kernel<true> (DESIGN.md §4.1), and
optionally the Smith-Waterman stage of this build against another build in alternating rounds.

Builds the library with -DTREDSW_PHASE_CLOCKS into a temporary directory (the tree is not written), then runs the
fused device-resident call (CohortBatch.run_device) over batches of bench.py's cohort, built with bench.py's own
functions (same seed, same 150 bp reads, ~S x 30 problems per batch).  The timing build's lane 0 adds clock64() deltas
per item and phase to global counters (no shared memory, so it keeps the production occupancy):

    setup         item fetch, family, code load
    suffix        suffix_pass (suffix potentials)
    prefix        the prefix strip
    main          the main strips
    loc_main      locate_packed, main strip
    loc_suffix    locate_packed, suffix block
    begin         begin sweep (diagonal walk or sw_sweep), the longest lane of each round
    pick          candidate picking, classification, records

Reported: shares of the summed SM clocks per phase, overall and per instance period, clocks per item, phase-2 rounds per
item, and the occupancy API's resident CTAs per SM of the packed kernel (before the cap of 8).  With --compare LIB
(the production libtredsw.so of another build) this tree's production library and LIB run the same batches in
alternating rounds; per build the median and spread of the per-batch mean "sw" (pre-filter, grouping, classify
kernels) and "total" call times from the library's CUDA events, and whether the call records are identical.  The
card's name, power limit and max SM clock are read first.

    python tools/phase_clock_bench.py [--samples 384] [--batches 4] [--rounds 7] [--compare LIB] [--out result.json]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import bench  # noqa: E402

PHASES = ["setup", "suffix", "prefix", "main", "loc_main", "loc_suffix", "begin", "pick"]
NPHASE, NPERIODS = len(PHASES) + 2, 13        # + rounds, items (sw_family.cu: PH_ROUNDS, PH_ITEMS)


def shares(v):
    tot = sum(int(v[i]) for i in range(len(PHASES)))
    out = {"clocks": tot, "items": int(v[NPHASE - 1]),
           "rounds_per_item": int(v[NPHASE - 2]) / max(1, int(v[NPHASE - 1])),
           "clocks_per_item": tot / max(1, int(v[NPHASE - 1]))}
    out["share"] = {n: int(v[i]) / max(1, tot) for i, n in enumerate(PHASES)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=384, help="samples per batch (x 30 loci)")
    ap.add_argument("--batches", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--compare", metavar="LIB", help="production libtredsw.so of another build to time against this one")
    ap.add_argument("--out")
    args = ap.parse_args()
    try:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True).stdout.strip()
    except OSError as e:
        card = "unknown ({})".format(e)
    res = {"card": card}

    from tredparse_b200 import build as B
    timing_dir = tempfile.mkdtemp(prefix="tredsw_phase_")
    timing_lib = B.build(outdir=timing_dir, defines=["TREDSW_PHASE_CLOCKS"])
    B.build()                                           # this tree's production library (no-op when up to date)

    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    names = bench.distinct_loci(repo)
    nloci = len(names)
    flat = np.arange(args.samples * args.batches * nloci)
    chunks = [np.stack([c // nloci, c % nloci], axis=1) for c in np.array_split(flat, args.batches)]
    arrays = bench.build_batches(chunks, max(1, min(16, os.cpu_count() or 1)))

    import torch
    from tredparse_b200 import _lib, cohort
    if not torch.cuda.is_available():
        raise SystemExit("phase_clock_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    template = cohort.CohortBatch([], family_keys=[(repo[n], bench.READLEN) for n in names])
    batches = [bench.batch_from_arrays(cohort, template, a) for a in arrays]
    stream = torch.cuda.Stream()

    def context(path):                                  # a context bound to the library at path
        _lib._lib, _lib.LIB_PATH = None, path
        return _lib.Context(0, stream=stream.cuda_stream)
    builds = {"this": context(B.OUT)}
    if args.compare:
        builds["compare"] = context(os.path.abspath(args.compare))
    tctx = context(timing_lib)
    tlib = tctx.lib
    tlib.tredsw_phase_clocks.restype = ctypes.c_int
    tlib.tredsw_phase_clocks.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    for b in batches:
        b.to_device(0)
    torch.cuda.synchronize()

    def run_all(ctx, timed):
        sw, tot = [], []
        ctx.enable_timing(timed)
        with torch.cuda.stream(stream):
            for b in batches:
                b.run_device(ctx)
                if timed:
                    t = ctx.timing()
                    sw.append(t["sw"])
                    tot.append(t["total"])
        ctx.enable_timing(False)
        stream.synchronize()
        return sw, tot

    def phase_clocks():
        a = np.zeros(NPERIODS * NPHASE, dtype=np.int64)
        occ = ctypes.c_int32(0)
        _lib.check(tlib.tredsw_phase_clocks(tctx.handle, _lib.ptr(a), ctypes.byref(occ)), "tredsw_phase_clocks")
        return a.reshape(NPERIODS, NPHASE), occ.value

    # phase clocks: one warm-up pass, then one counted pass over the batches
    run_all(tctx, False)
    c0, _ = phase_clocks()
    run_all(tctx, False)
    c1, occ = phase_clocks()
    d = c1 - c0
    res["ctas_per_sm_occupancy_api"] = occ
    res["phases"] = shares(d.sum(axis=0))
    res["by_period"] = {str(p): shares(d[p]) for p in range(1, NPERIODS) if d[p, NPHASE - 1] > 0}
    calls = {"timing": np.concatenate([b.calls_from_device() for b in batches])}

    for name, ctx in builds.items():                    # warm-up and records
        run_all(ctx, False)
        calls[name] = np.concatenate([b.calls_from_device() for b in batches])
    res["calls_identical"] = all(v.tobytes() == calls["this"].tobytes() for v in calls.values())
    rounds = {n: {"sw": [], "total": []} for n in builds}
    order = list(builds)
    for r in range(args.rounds):
        for name in (order if r % 2 == 0 else order[::-1]):
            sw, tot = run_all(builds[name], True)
            rounds[name]["sw"].append(statistics.mean(sw))
            rounds[name]["total"].append(statistics.mean(tot))
    for name in builds:
        res[name] = {k: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v), "rounds": v}
                     for k, v in rounds[name].items()}
    if args.compare:
        res["sw_speedup"] = res["compare"]["sw"]["median_ms"] / res["this"]["sw"]["median_ms"]
        res["total_speedup"] = res["compare"]["total"]["median_ms"] / res["this"]["total"]["median_ms"]
    res["config"] = {"samples_per_batch": args.samples, "batches": args.batches, "rounds": args.rounds,
                     "compare": args.compare, "problems_per_batch": batches[0].nproblems,
                     "reads_per_batch": batches[0].nreads, "readlen": bench.READLEN, "seed": bench.COHORT_SEED,
                     "timing": "library CUDA events per call, one stream; per round the mean over the batches",
                     "phase_clocks": "SM clock64() of lane 0 per item and phase, one pass over the batches"}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fp:
            fp.write(line + "\n")
    if not res["calls_identical"]:
        raise SystemExit("call records differ between the builds")


if __name__ == "__main__":
    main()
