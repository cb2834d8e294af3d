#!/usr/bin/env python
"""What ``tred.py --str-profile`` costs: catalogue calls and the STR profile of one synthetic whole-sample BAM
(``scan_bench.write_sample`` with the planted expansions of ``str_profile_bench``, at least 1 GB inflated) from one
read, against calls and a separate profile scan.  Three arms, alternating, best of --reps each:
  1. ``tred.run_chunks`` without the profile (every catalogue locus with its alt regions, gender from chrY);
  2. ``tred.run_chunks(..., str_profile=True)``;
  3. arm 1 followed by ``strprofile.profile`` (what a user ran before: a second read of the file).
Each arm runs on three inputs: the file without an index (one scan either way), a pipe fed by a separate process
(``cat``; arm 3 needs the stream twice, so it starts ``cat`` twice) and an indexed copy (arm 1 reads the loci through
the indexed GPU ingest; arm 2 scans the whole file instead).  Reported per (input, arm): wall time, and per scan its
host read and device time per slab.  The calls of arms 1 and 2 must be equal and so must the profiles of arms 2 and 3.
The card's name and power limit are read in the same run.  Everything is written to a temporary directory; the file
is in the page cache after it is written (a cold-cache read is not measured).

    python tools/tred_profile_bench.py [--gb 2.2] [--reps 3] [--out profiles/r3_tred_profile_bench.json]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from str_profile_bench import PLANTS, canonical, card, planted  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=2.2, help="inflated size of the synthetic BAM (at least 1)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.gb < 1:
        ap.error("--gb: the measurement is of a whole-sample BAM of at least 1 GB")
    import scan_bench
    from tredparse_b200 import _lib, bamio, ingest, strprofile, tred as T
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    res = {"card": card()}
    scans = []
    real_scan = ingest.scan_sample

    def recorded(*args, **kw):                      # the statistics of every scan the arms run
        b = real_scan(*args, **kw)
        st = b.stats()
        scans.append({"slabs": st["slabs"], "ms_host_read_per_slab": st["ms_host_read"] / max(1, st["slabs"]),
                      "ms_device_per_slab": st["ms_device"] / max(1, st["slabs"]), "ms_total": st["ms_total"],
                      "irr": kw.get("irr") is not None})
        return b
    ingest.scan_sample = strprofile.scan_sample = recorded
    tmp = tempfile.mkdtemp(prefix="tred_profile_bench_")
    try:
        sam = bamio.AlignmentFile(os.path.join(ROOT, "tests", "golden", "t001.mini.bam"))
        refs = list(zip(sam.references, sam.lengths))
        sam.close()
        indexed = os.path.join(tmp, "indexed", "sample.bam")
        os.makedirs(os.path.dirname(indexed))
        t = time.perf_counter()
        nrec, inflated = scan_bench.write_sample(indexed, a.gb, extra=planted(refs))
        unindexed = os.path.join(tmp, "sample.bam")
        shutil.copy(indexed, unindexed)
        res.update(write_s=time.perf_counter() - t, records=nrec, inflated_bytes=inflated,
                   file_bytes=os.path.getsize(unindexed))
        _lib.default_context(0)
        task = lambda path: [("sample", path, repo, list(repo.names), 300, False, False, True, True, "INFO")]

        def source(kind):
            """(path, producer process or None) of one read of the input"""
            if kind == "pipe":
                prod = subprocess.Popen(["cat", unindexed], stdout=subprocess.PIPE)
                return "/dev/fd/{}".format(prod.stdout.fileno()), prod
            return (indexed if kind == "indexed" else unindexed), None

        def done(prod):
            if prod is not None:
                prod.stdout.close()
                prod.wait()

        def arm(kind, which):
            """-> (wall s, tredCalls, profile or None, the scans it ran)"""
            del scans[:]
            t0 = time.perf_counter()
            path, prod = source(kind)
            try:
                r = list(T.run_chunks(task(path), str_profile=(which == 2)))[0]
            finally:
                done(prod)
            prof = r.pop(T.STR_PROFILE, None)
            if which == 3:
                path, prod = source(kind)
                try:
                    prof = strprofile.profile(path, sample="sample")
                finally:
                    done(prod)
            wall = time.perf_counter() - t0
            assert "error" not in r, r.get("error")
            return wall, r["tredCalls"], prof, list(scans)

        arm("indexed", 1)                            # warm-up: context, modules, tables
        runs = {k: {w: [] for w in (1, 2, 3)} for k in ("unindexed", "pipe", "indexed")}
        first = {}
        for _ in range(a.reps):
            for kind in runs:
                for which in (1, 2, 3):
                    wall, calls, prof, sc = arm(kind, which)
                    runs[kind][which].append({"wall_s": wall, "scans": sc})
                    first.setdefault((kind, which), (calls, prof))
        checks = {}
        for kind in runs:
            c1, _ = first[kind, 1]
            c2, p2 = first[kind, 2]
            c3, p3 = first[kind, 3]
            p2 = dict(p2, bam=None)
            p3 = dict(p3, bam=None)
            checks[kind] = {"calls_equal": c1 == c2 == c3, "profiles_equal": json.dumps(p2, sort_keys=True) ==
                            json.dumps(p3, sort_keys=True)}
            assert checks[kind]["calls_equal"] and checks[kind]["profiles_equal"], (kind, checks[kind])
        ref_calls = first["indexed", 1][0]
        checks["calls_equal_across_inputs"] = all(first[k, 1][0] == ref_calls for k in runs)
        assert checks["calls_equal_across_inputs"]
        names = {1: "calls", 2: "calls_and_profile", 3: "calls_then_profile_scan"}
        for kind in runs:
            res[kind] = {}
            for which, rr in runs[kind].items():
                best = min(rr, key=lambda r: r["wall_s"])
                res[kind][names[which]] = {"best_wall_s": best["wall_s"], "scans_of_best": best["scans"],
                                           "runs_s": [r["wall_s"] for r in rr]}
            b = {w: res[kind][names[w]]["best_wall_s"] for w in (1, 2, 3)}
            res[kind]["arm2_over_arm1"] = b[2] / b[1]
            res[kind]["arm2_over_arm3"] = b[2] / b[3]
        res["checks"] = checks
        prof = first["unindexed", 2][1]
        res["planted"] = {m: prof["profile"].get(canonical(m)) for m, _, _, _ in PLANTS}
    finally:
        ingest.scan_sample = strprofile.scan_sample = real_scan
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fp:
            fp.write(line + "\n")


if __name__ == "__main__":
    main()
