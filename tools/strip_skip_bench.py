#!/usr/bin/env python
"""The fixed-point exit of the packed family kernel's main strips (DESIGN.md §4.1), or the convergence order of the
reads (§7.2), on and off in one command.

Builds batches of bench.py's cohort with bench.py's own functions (same seed, same 150 bp reads, ~S x 30 problems per
batch), then runs the fused device-resident call (CohortBatch.run_device) over them in alternating rounds with the
switch's variable (--switch skip: TREDSW_NO_STRIP_SKIP, --switch order: TREDSW_NO_CONVERGENCE_ORDER) unset and set.
Each call is timed by the library's CUDA events (stage "sw" = pre-filter, grouping and the classify kernels; "total" =
the whole call).  Reported per mode: median and spread (min, max) over rounds of the per-batch mean sw and total ms;
main strips skipped / planned per loop instantiation period, the same per lane holding a read (lane_skipped /
lane_planned) next to the per-lane bound (lane_skippable / lane_planned: what no order of the reads can beat), items that skipped nothing, and skipped phase-1 cells (from the
context's counters, one round); and whether the call records of both modes, and the per-read records of one batch,
are identical byte for byte.  The card's name and power limit are read first.

    python tools/strip_skip_bench.py [--switch skip|order] [--samples 384] [--batches 4] [--rounds 7] [--out result.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import bench  # noqa: E402

SWITCHES = {"skip": ("TREDSW_NO_STRIP_SKIP", ("skip", "no_skip")),
            "order": ("TREDSW_NO_CONVERGENCE_ORDER", ("order", "no_order"))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--switch", choices=sorted(SWITCHES), default="skip")
    ap.add_argument("--samples", type=int, default=384, help="samples per batch (x 30 loci)")
    ap.add_argument("--batches", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out")
    args = ap.parse_args()
    var, MODES = SWITCHES[args.switch]

    def set_mode(mode):
        if mode == MODES[0]:
            os.environ.pop(var, None)
        else:
            os.environ[var] = "1"
    try:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True).stdout.strip()
    except OSError as e:
        card = "unknown ({})".format(e)
    res = {"card": card}

    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    names = bench.distinct_loci(repo)
    nloci = len(names)
    nsamples = args.samples * args.batches
    flat = np.arange(nsamples * nloci)
    chunks = [np.stack([c // nloci, c % nloci], axis=1) for c in np.array_split(flat, args.batches)]
    arrays = bench.build_batches(chunks, max(1, min(16, os.cpu_count() or 1)))

    import torch
    from tredparse_b200 import _lib, cohort
    if not torch.cuda.is_available():
        raise SystemExit("strip_skip_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    template = cohort.CohortBatch([], family_keys=[(repo[n], bench.READLEN) for n in names])
    batches = [bench.batch_from_arrays(cohort, template, a) for a in arrays]
    stream = torch.cuda.Stream()
    ctx = _lib.Context(0, stream=stream.cuda_stream)
    for b in batches:
        b.to_device(0)
    torch.cuda.synchronize()

    def run_all(mode, timed):
        set_mode(mode)
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

    for mode in MODES:                                  # warm-up (module load, scratch allocation)
        run_all(mode, False)
    calls = {}
    for mode in MODES:                                  # counters and outputs of one untimed pass per mode
        s0 = ctx.strip_skip_stats()
        run_all(mode, False)
        s1 = ctx.strip_skip_stats()
        calls[mode] = np.concatenate([b.calls_from_device() for b in batches])
        per = {}
        for p, d in s1["by_period"].items():
            d0 = s0["by_period"].get(p, {})
            per[p] = {k: v - d0.get(k, 0) for k, v in d.items()}
            per[p]["skipped_share"] = per[p]["skipped"] / max(1, per[p]["planned"])
            per[p]["lane_skipped_share"] = per[p]["lane_skipped"] / max(1, per[p]["lane_planned"])
            per[p]["lane_bound_share"] = per[p]["lane_skippable"] / max(1, per[p]["lane_planned"])
        planned = sum(v["planned"] for v in per.values())
        res.setdefault("strips", {})[mode] = {
            "by_period": per, "cells_skipped": s1["cells_skipped"] - s0["cells_skipped"],
            "skipped_share": sum(v["skipped"] for v in per.values()) / max(1, planned)}
    reads = {}
    for mode in MODES:
        set_mode(mode)
        reads[mode] = batches[0].run_host(ctx=ctx, want_reads=True)["reads"]
    res["calls_identical"] = calls[MODES[0]].tobytes() == calls[MODES[1]].tobytes()
    res["reads_identical"] = reads[MODES[0]].tobytes() == reads[MODES[1]].tobytes()

    rounds = {m: {"sw": [], "total": []} for m in MODES}
    for r in range(args.rounds):
        for mode in (MODES if r % 2 == 0 else MODES[::-1]):
            sw, tot = run_all(mode, True)
            rounds[mode]["sw"].append(statistics.mean(sw))
            rounds[mode]["total"].append(statistics.mean(tot))
    set_mode(MODES[0])
    for mode in MODES:
        res[mode] = {k: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v), "rounds": v}
                     for k, v in rounds[mode].items()}
    res["sw_speedup"] = res[MODES[1]]["sw"]["median_ms"] / res[MODES[0]]["sw"]["median_ms"]
    res["total_speedup"] = res[MODES[1]]["total"]["median_ms"] / res[MODES[0]]["total"]["median_ms"]
    res["config"] = {"switch": var, "samples_per_batch": args.samples, "batches": args.batches, "rounds": args.rounds,
                     "problems_per_batch": batches[0].nproblems, "reads_per_batch": batches[0].nreads,
                     "readlen": bench.READLEN, "seed": bench.COHORT_SEED,
                     "timing": "library CUDA events per call, one stream; per round the mean over the batches"}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fp:
            fp.write(line + "\n")
    if not (res["calls_identical"] and res["reads_identical"]):
        raise SystemExit("records differ between the modes")


if __name__ == "__main__":
    main()
