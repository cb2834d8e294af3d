#!/usr/bin/env python
"""The scan of one synthetic whole-sample BAM (``scan_bench.write_sample``, at least 1 GB) read two ways in one command:
  * from the file (``BamIngest.unindexed``: pread slabs, the next slab read while the device works on this one);
  * through a pipe fed by a separate process (``cat``) and read in order (``BamIngest.stream``), the way
    ``samtools view -u x.cram | python -m tredparse_b200.tred -`` reads it.
Both scan every catalogue locus with its alt regions and the chrY regions of the gender inference; their evidence
must be equal problem by problem.  Also timed: draining the same pipe without scanning it (what the producer and the
pipe deliver on their own).  Reported per arm: wall time, GB/s compressed and inflated, host read and device time
per slab, slabs, blocks and repaired blocks; the card's name and power limit are printed with them.  Everything is
written to a temporary directory.

    python tools/stream_bench.py [--gb 2.2] [--slab-mb 0] [--reps 3] [--out result.json]
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

from scan_bench import READLEN, write_sample  # noqa: E402


def summary(st, wall):
    return {"wall_s": wall, "GBps_compressed": st["compressed_bytes"] / wall / 1e9,
            "GBps_inflated": st["inflated_bytes"] / wall / 1e9,
            "ms_host_read_per_slab": st["ms_host_read"] / max(1, st["slabs"]),
            "ms_device_per_slab": st["ms_device"] / max(1, st["slabs"]),
            "slabs": st["slabs"], "blocks": st["blocks"], "repaired_blocks": st["repaired_blocks"],
            "records": st["records"], "compressed_bytes": st["compressed_bytes"], "inflated_bytes": st["inflated_bytes"]}


def same(x, y):
    return (np.array_equal(x.reads, y.reads) and np.array_equal(x.roff, y.roff) and x.names == y.names
            and np.array_equal(x.global_lens, y.global_lens) and np.array_equal(x.target_lens, y.target_lens)
            and x.depth == y.depth and x.n_unmapped == y.n_unmapped)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=2.2, help="inflated size of the synthetic BAM")
    ap.add_argument("--slab-mb", type=float, default=0, help="compressed MiB per slab (0: the library's default)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from tredparse_b200 import ingest, _lib
    from tredparse_b200.meta import TREDsRepo
    from tredparse_b200.bam_parser import BamDepth
    repo = TREDsRepo()
    res = {}
    try:
        res["card"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                     capture_output=True, text=True).stdout.strip().splitlines()[0]
    except Exception as e:
        res["card"] = "unknown ({})".format(e)
    tmp = tempfile.mkdtemp(prefix="stream_bench_")
    try:
        path = os.path.join(tmp, "sample.bam")
        t = time.perf_counter()
        nrec, inflated = write_sample(path, a.gb)
        res.update(write_s=time.perf_counter() - t, records=nrec, inflated_bytes=inflated, file_bytes=os.path.getsize(path))
        ctx = _lib.default_context(0)
        slab = int(a.slab_mb * (1 << 20)) or None

        def scan(h):
            qs, keep = [], []
            for n in repo.names:
                q = ingest.locus_query(h, repo[n], READLEN, alts=repo[n].alt)
                qs.append(q[0]); keep.append(q[1])
            yreg = [(h.tid(c), s, e) for c, s, e in BamDepth.y_regions(repo.ref)]
            t = time.perf_counter()
            b = ingest.scan_sample(ctx, h, qs, keep, yreg, slab_bytes=slab)
            wall = time.perf_counter() - t
            assert b.scan_status == 0 and not b.status.any(), "scan failed"
            return b, summary(b.stats(), wall)

        def piped():
            """a stream handle on the read end of a pipe that `cat` writes the file into"""
            prod = subprocess.Popen(["cat", path], stdout=subprocess.PIPE)
            h = ingest.BamIngest.stream("/dev/fd/{}".format(prod.stdout.fileno()))
            return prod, h

        file_runs, pipe_runs, drain = [], [], []
        ref = None
        for rep in range(a.reps):                   # the arms alternate; the file is in the page cache after the write
            with ingest.BamIngest.unindexed(path) as uh:
                b, s = scan(uh)
            file_runs.append(s)
            if ref is None:
                ref = b
            else:
                b.close()
            prod, sh = piped()
            try:
                t = time.perf_counter()
                sh.read_length()
                b, s = scan(sh)
                s["wall_s_with_header_and_read_length"] = time.perf_counter() - t
            finally:
                sh.close()
                prod.stdout.close()
                prod.wait()
            pipe_runs.append(s)
            if rep == 0:
                bad = sum(not same(b.evidence(i), ref.evidence(i)) for i in range(ref.nproblems))
                assert bad == 0 and np.array_equal(b.depths, ref.depths), "the stream and the file scans differ"
                res["problems"], res["problems_differing"] = int(ref.nproblems), bad
            b.close()
            prod = subprocess.Popen(["cat", path], stdout=subprocess.PIPE)
            t, n = time.perf_counter(), 0
            fd = prod.stdout.fileno()
            while True:
                k = len(os.read(fd, 1 << 20))
                if not k:
                    break
                n += k
            drain.append({"wall_s": time.perf_counter() - t, "GBps": n / (time.perf_counter() - t) / 1e9})
            prod.stdout.close()
            prod.wait()
        ref.close()
        best = lambda runs: min(runs, key=lambda r: r["wall_s"])
        res["file"] = {"best": best(file_runs), "runs": file_runs}
        res["pipe"] = {"best": best(pipe_runs), "runs": pipe_runs}
        res["pipe_drain_only"] = {"best": best(drain), "runs": drain}
        for arm in ("file", "pipe"):
            bb = res[arm]["best"]
            res[arm]["bound_by"] = "device" if bb["ms_device_per_slab"] > bb["ms_host_read_per_slab"] else "host read"
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fp:
            fp.write(line + "\n")


if __name__ == "__main__":
    main()
