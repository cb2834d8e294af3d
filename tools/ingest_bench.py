#!/usr/bin/env python
"""Time the native one-pass BAM ingest (csrc/ingest.cpp) beside the Python reader that makes the reference's
three passes per locus (select_reads + PEextractor + region_depth).  Host code only.

    python tools/ingest_bench.py [bam] [tred] [--reps 5]
"""
import argparse
import logging
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("bam", nargs="?", default=os.path.join(ROOT, "tests", "golden", "t001.mini.bam"))
    ap.add_argument("tred", nargs="?", default="HD")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--all-loci", action="store_true", help="time a synthetic BAM with reads at every catalogue locus")
    a = ap.parse_args()
    from tredparse_b200 import bamio, ingest
    from tredparse_b200.bam_parser import BamParser, PEextractor, BamDepth
    from tredparse_b200.meta import TREDsRepo
    from tredparse_b200.utils import InputParams
    repo = TREDsRepo()
    t = repo[a.tred]

    def python_path():
        ip = InputParams(bam=a.bam, READLEN=150, tredName=a.tred, repo=repo, maxinsert=300, fullsearch=False,
                         gender="Unknown", depth=30, clip=False, alts=True, repeatpairs=True, log="INFO")
        bp = BamParser(ip)
        sam = bamio.AlignmentFile(a.bam)
        reads = bp.select_reads(sam)
        sam.close()
        pe = PEextractor(bp)
        d = BamDepth(a.bam, "hg38", logging.getLogger()).region_depth(t.chr, max(0, t.repeat_start - 1000), t.repeat_end + 1000)
        return len(reads), len(pe.global_lens), d

    def native_path():
        with ingest.BamIngest(a.bam) as ing:
            ev = ing.extract_locus(t, 150, alts=t.alt, want_names=True)
        return ev.nreads, len(ev.global_lens), ev.depth

    for name, fn in (("python (3 passes)", python_path), ("native (1 pass)", native_path)):
        fn()
        t0 = time.perf_counter()
        for _ in range(a.reps):
            r = fn()
        dt = (time.perf_counter() - t0) / a.reps
        print("{:18s} {:8.2f} ms / locus  ({:.1f} loci/s/core)  reads={} pairs={} depth={:.2f}".format(name, dt * 1e3, 1 / dt, *r))

    # a whole sample: every catalogue locus, dealt to host threads (tred.ingest_loci).  The test BAMs hold reads at
    # one locus only, so --all-loci first builds a BAM with the HD window of the mini fixture transplanted to
    # every distinct catalogue locus (same coverage and pair structure everywhere, like a whole-genome BAM)
    from tredparse_b200 import tred as tredmod
    log = logging.getLogger()
    names = list(repo.names)
    if a.all_loci:
        import copy
        import tempfile
        src = bamio.AlignmentFile(os.path.join(ROOT, "tests", "golden", "t001.mini.bam"))
        hd = repo["HD"]
        recs0 = [r for r in src.fetch(hd.chr, max(0, hd.repeat_start - 10500), hd.repeat_end + 10500)
                 if not r.is_unmapped and r.next_reference_id == r.reference_id]
        refs = list(zip(src.references, src.lengths))
        out, seen = [], set()
        for k, nm in enumerate(names):
            tr = repo[nm]
            if (tr.chr, tr.repeat_start) in seen or src.get_tid(tr.chr) < 0:
                continue
            seen.add((tr.chr, tr.repeat_start))
            tid, shift = src.get_tid(tr.chr), tr.repeat_start - hd.repeat_start
            for r in recs0:
                q = copy.copy(r)
                q.query_name = "{}_{}".format(r.query_name, k)
                q.reference_id = q.next_reference_id = tid
                q.reference_start = r.reference_start + shift
                q.next_reference_start = r.next_reference_start + shift
                q._ref_end = None
                if q.reference_start >= 0:
                    out.append(q)
        src.close()
        out.sort(key=lambda r: (r.reference_id, r.reference_start))
        a.bam = os.path.join(tempfile.mkdtemp(prefix="tredsw_ingest_"), "all_loci.bam")
        bamio.write_bam(a.bam, refs, out, level=6)
        print("synthetic whole-sample BAM: {} records at {} loci -> {}".format(len(out), len(seen), a.bam))
    for th in (1, 2, 4, 8):
        tredmod.ingest_loci(a.bam, repo, names, 150, True, False, log, threads=th)
        t0 = time.perf_counter()
        for _ in range(a.reps):
            ev = tredmod.ingest_loci(a.bam, repo, names, 150, True, False, log, threads=th)
        dt = (time.perf_counter() - t0) / a.reps
        print("sample of {} loci, {} thread(s): {:8.2f} ms  ({:.0f} loci/s, {} reads)".format(
            len(names), th, dt * 1e3, len(names) / dt, sum(e.nreads for e in ev.values())))


if __name__ == "__main__":
    main()
