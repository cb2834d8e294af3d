#!/usr/bin/env python
"""The cost of the STR profile in the scan of a BAM without an index: the synthetic whole-sample BAM of
tools/scan_bench.py (background pairs over every contig, the reads of every catalogue locus) with planted expansions
added (simulate.expansion_records: AAGGG, CAG, ATTC and AT at positions away from the catalogue, with mismapped and
IRR-IRR pairs in the unmapped tail).

Alternates, best of --reps each, on the GPU the context runs on:
  * the scan with every catalogue locus and the chrY depth regions (what tred.run does for such a file), without and
    with the IRR stage (ingest.scan_sample(..., irr=IrrParams())): wall time, host read and device time per slab; the
    evidence and depths of the two must be identical;
  * the profile-only scan (strprofile.profile): wall time, IRR records, the profile of the planted motifs.
The card's name and power limit are read in the same run.  The file is written to a temporary directory, so the
page cache is warm after the first scan (the file is read from memory: a cold-cache read is not measured).

    python tools/str_profile_bench.py [--gb 2.2] [--reps 3] [--out profiles/r3_str_profile_bench.json]
(without --out the result line is only printed)
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

PLANTS = [("AAGGG", 4, 0.31, 120), ("CAG", 6, 0.52, 90), ("ATTC", 9, 0.23, 70), ("AT", 11, 0.67, 150)]


def planted(refs):
    """expansions away from the catalogue: (motif, contig index, relative position, units) -> records"""
    from tredparse_b200 import simulate
    recs = []
    for k, (motif, t, rel, units) in enumerate(PLANTS):
        t = min(t, len(refs) - 1)
        recs += simulate.expansion_records(t, int(refs[t][1] * rel), motif, units, cov=15, seed=900 + k,
                                           tag="plant{}_".format(k), mismap_fraction=0.1,
                                           mismap_to=(0, 1000000, 2000000))
    return recs


def canonical(motif):
    """the profile's name of a motif: the smallest rotation of it and of its reverse complement"""
    rc = motif[::-1].translate(str.maketrans("ACGT", "TGCA"))
    return min(x[t:] + x[:t] for x in (motif, rc) for t in range(len(motif)))


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip().splitlines()[0]
    except Exception as e:
        return "unknown ({})".format(e)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=2.2, help="inflated size of the synthetic BAM")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import scan_bench
    from tredparse_b200 import _lib, bamio, ingest, strprofile
    from tredparse_b200.meta import TREDsRepo
    from tredparse_b200.bam_parser import BamDepth
    repo = TREDsRepo()
    res = {"card": card()}
    tmp = tempfile.mkdtemp(prefix="str_profile_bench_")
    try:
        sam = bamio.AlignmentFile(os.path.join(ROOT, "tests", "golden", "t001.mini.bam"))
        refs = list(zip(sam.references, sam.lengths))
        sam.close()
        path = os.path.join(tmp, "sample.bam")
        t = time.perf_counter()
        nrec, inflated = scan_bench.write_sample(path, a.gb, extra=planted(refs))
        os.remove(path + ".bai")
        res.update(write_s=time.perf_counter() - t, records=nrec, inflated_bytes=inflated, file_bytes=os.path.getsize(path))
        ctx = _lib.default_context(0)

        def scan(irr):
            h = ingest.BamIngest.unindexed(path)
            qs, keep = [], []
            for n in repo.names:
                q = ingest.locus_query(h, repo[n], scan_bench.READLEN, alts=repo[n].alt)
                if q is not None:
                    qs.append(q[0]); keep.append(q[1])
            yreg = [(h.tid(c), s, e) for c, s, e in BamDepth.y_regions(repo.ref)]
            t0 = time.perf_counter()
            b = ingest.scan_sample(ctx, h, qs, keep, yreg, irr=irr)
            wall = time.perf_counter() - t0
            st = b.stats()
            st["wall_s"] = wall
            out = (st, [b.evidence(i) for i in range(len(qs))], list(b.depths), b.scan_status,
                   None if b.irr is None else b.irr["stats"])
            b.close(); h.close()
            return out
        runs = {"plain": [], "profile": []}
        last = {}
        for _ in range(a.reps):
            for kind, irr in (("plain", None), ("profile", ingest.IrrParams())):
                st, ev, depths, status, irr_stats = scan(irr)
                assert status == 0
                if irr_stats:
                    st["irr"] = irr_stats
                runs[kind].append(st)
                last[kind] = (ev, depths)
        (e0, d0), (e1, d1) = last["plain"], last["profile"]
        same = d0 == d1 and all(
            np.array_equal(x.reads, y.reads) and np.array_equal(x.roff, y.roff) and x.names == y.names
            and np.array_equal(x.global_lens, y.global_lens) and np.array_equal(x.target_lens, y.target_lens)
            and x.depth == y.depth for x, y in zip(e0, e1))
        assert same, "the IRR stage changed the scan's evidence"
        for kind in runs:
            best = min(runs[kind], key=lambda s: s["wall_s"])
            res[kind] = {"runs": runs[kind], "best_wall_s": best["wall_s"],
                         "ms_host_read_per_slab": best["ms_host_read"] / best["slabs"],
                         "ms_device_per_slab": best["ms_device"] / best["slabs"],
                         "bound_by": "device" if best["ms_device"] > best["ms_host_read"] else "host read"}
        res["profile_over_plain_wall"] = res["profile"]["best_wall_s"] / res["plain"]["best_wall_s"]
        res["evidence_identical"] = same
        # the profile-only scan and what it finds at the planted sites
        times, prof = [], None
        for _ in range(a.reps):
            t0 = time.perf_counter()
            prof = strprofile.profile(path, ctx=ctx)
            times.append(time.perf_counter() - t0)
        res["profile_only"] = {"runs_s": times, "best_s": min(times), "stats": prof["stats"], "depth": prof["depth"],
                               "planted": {m: prof["profile"].get(canonical(m)) for m, _, _, _ in PLANTS}}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fp:
            fp.write(line + "\n")


if __name__ == "__main__":
    main()
