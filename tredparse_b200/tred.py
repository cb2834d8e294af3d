"""
TRED caller entry point: parse the target regions of the input BAMs, classify full / partial / repeat
reads on the GPU, evaluate the likelihood grids on the GPU and report the most likely repeat sizes.

Keeps the reference's ``tredparse/tred.py`` surface: ``set_argparse`` (:64-103), ``read_csv``
(:401-440), ``runBam`` (:153-169), ``run`` (:180-278), ``counter_s`` (:149-150), ``to_json``
(:296-313), ``to_vcf`` (:316-374), ``main`` (:451-539) and the JSON layout (SURVEY.md Appendix C).

Differences that are the point of this build:
  * every (sample, locus) gets one evidence record (``ingest.LocusEvidence``: reads, names, pair lengths, depth),
    from the GPU ingest, the native host reader or — for a BAM without a usable index or a contig the native
    reader does not know — the Python reader (``bam_parser.extract_locus``); a locus whose window cannot be read
    gets no record and no call;
  * ``run`` / ``run_chunk`` genotype *all loci of a chunk of samples* in one fused device call
    (``genotype_evidence``) instead of looping ``runBam`` per locus (``runBam`` is still there and gives identical
    results).  If that call fails, the chunk fails: ``run_chunks(..., isolate=True)`` turns that into error records
    for its samples;
  * samples are sharded over GPUs (``--gpus``), one worker process per GPU, instead of over CPU cores
    with ``multiprocessing.Pool`` (tred.py:528-532).  No collective: workers return their dicts;
  * a BAM that can be read only once, in order (``-`` for stdin, a FIFO; e.g. ``samtools view -u x.cram | ... -``) is
    read by one GPU scan that serves its read length, gender and every locus; there is no fallback reader for it.
S3 / ``@HLI-id`` inputs are out of scope (SURVEY.md §2 row 5).
"""
import argparse
import gzip
import json
import logging
import os
import os.path as op
import shutil
import sys
import time
from datetime import datetime as dt, timedelta

import numpy as np

from . import __version__
from .utils import DefaultHelpParser, mkdir
from .bam_parser import BamDepth, BamReadLen, BamParser, BamParserResults, extract_locus, read_alignment
from .models import IntegratedCaller, mean_std, histogram
from .meta import TREDsRepo, locus_names

logging.basicConfig()
logger = logging.getLogger(__name__)

INFO = """##INFO=<ID=RPA,Number=1,Type=String,Description="Repeats per allele">
##INFO=<ID=END,Number=1,Type=Integer,Description="End position of variant">
##INFO=<ID=MOTIF,Number=1,Type=String,Description="Canonical repeat motif">
##INFO=<ID=NS,Number=1,Type=Integer,Description="Number of samples with data">
##INFO=<ID=REF,Number=1,Type=Integer,Description="Reference copy number">
##INFO=<ID=CR,Number=1,Type=Integer,Description="Disease copy number cutoff">
##INFO=<ID=IH,Number=1,Type=String,Description="Inheritance">
##INFO=<ID=RL,Number=1,Type=Integer,Description="Reference STR track length in bp">
##INFO=<ID=VT,Number=1,Type=String,Description="Variant type">
##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">
##FORMAT=<ID=GA,Number=1,Type=String,Description="Genotype with absolute copy numbers">
##FORMAT=<ID=FR,Number=1,Type=String,Description="Full spanning reads aligned to locus">
##FORMAT=<ID=PR,Number=1,Type=String,Description="Partial reads aligned to locus">
##FORMAT=<ID=RR,Number=1,Type=String,Description="Repeat-only reads aligned to locus">
##FORMAT=<ID=DP,Number=1,Type=Integer,Description="Mean read depth around locus">
##FORMAT=<ID=FDP,Number=1,Type=Integer,Description="Full spanning read depth">
##FORMAT=<ID=PDP,Number=1,Type=Integer,Description="Partial read depth">
##FORMAT=<ID=RDP,Number=1,Type=Integer,Description="Repeat read depth">
##FORMAT=<ID=PEDP,Number=1,Type=Integer,Description="Paired-end read depth">
##FORMAT=<ID=CI,Number=1,Type=String,Description="95% conf interval of estimates">
##FORMAT=<ID=PP,Number=1,Type=Float,Description="Posterior probability of disease">
##FORMAT=<ID=LABEL,Number=1,Type=String,Description="Risk assessment">
"""


def set_argparse():
    TRED_NAMES = locus_names()
    p = DefaultHelpParser(description=__doc__, prog=op.basename(__file__),
                          formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    p.add_argument("infile", nargs="?", help="Input path (BAM, list of BAMs, or csv format)")
    p.add_argument("--ref", help="Reference genome version",
                   choices=("hg38", "hg38_nochr", "hg19", "hg19_nochr"), default="hg38")
    p.add_argument("--tred", help="STR disorder, default is to run all", action="append",
                   choices=sorted(TRED_NAMES), default=None)
    p.add_argument("--haploid", help="Treat these chromosomes as haploid", action="append")
    p.add_argument("--useclippedreads", default=False, action="store_true",
                   help="Include clipped reads in inference")
    p.add_argument("--noalts", default=False, action="store_true",
                   help="Do not scan extra sites for mismapped reads, faster but less accurate")
    p.add_argument("--norepeatpairs", default=False, action="store_true",
                   help="Exclude pairs of repeat-only reads from evidence")
    p.add_argument("--log", choices=("INFO", "DEBUG"), default="INFO", help="Print debug logs, DEBUG=verbose")
    p.add_argument("--version", action="version", version="%(prog)s " + __version__)
    p.add_argument("--toy", help=argparse.SUPPRESS, action="store_true")

    g = p.add_argument_group("Performance options")
    g.add_argument("--cpus", help="Accepted for compatibility with the reference CLI (host cores are "
                   "not the compute resource here)", type=int, default=os.cpu_count())
    g.add_argument("--gpus", help="Number of GPUs to shard samples over", type=int, default=1)
    g.add_argument("--maxinsert", default=300, type=int, help="Maximum number of repeats")
    g.add_argument("--fullsearch", default=False, action="store_true", help="Full grid search")

    g = p.add_argument_group("I/O options")
    g.add_argument("--workdir", default=os.getcwd(), help="Specify work dir")
    g.add_argument("--cleanup", default=False, action="store_true", help="Cleanup the workdir after done")
    g.add_argument("--checkexists", default=False, action="store_true", help="Do not run if JSON output exists")
    g.add_argument("--no-output", default=False, action="store_true", help="Do not write JSON and VCF output")
    return p


def bam_path(bam):
    if bam == "-" or bam.startswith(("s3://", "http://", "ftp://", "https://")):
        return bam
    return op.abspath(bam)


def check_bam(bam):
    logger.debug("Working on `{}`".format(bam))
    try:
        read_alignment(bam).close()
    except (IOError, ValueError) as e:
        logger.error("Cannot retrieve file `{}` ({})".format(bam, e))
        return None
    return bam


def counter_s(c):
    return ";".join("{}|{}".format(k, int(v)) for k, v in sorted(c.items()))


def runBam(inputParams):
    """Parse one BAM at one locus and run the caller on it.  :return: BamParserResults"""
    maxinsert = inputParams.kwargs["maxinsert"]
    fullsearch = inputParams.kwargs["fullsearch"]
    bp = BamParser(inputParams)
    bp.parse()
    integratedCaller = IntegratedCaller(bp, maxinsert=maxinsert, fullsearch=fullsearch)
    integratedCaller.call(**inputParams.kwargs)
    return BamParserResults(inputParams, bp, integratedCaller)


def alt_regions(tred, ref, alts, clip):
    """The mis-mapping regions whose reads are added to a locus (bam_parser.py:215-243): none without alts or with
    clipped reads; contig names without the 'chr' prefix on a '_nochr' reference."""
    if not alts or clip:
        return []
    return [(c[3:] if "nochr" in ref else c, s, e) for (c, s, e) in tred.alt]


def locus_evidence(ing, tred, readlen, alts, clip, ref):
    """One native pass over the BAM for one locus (reads + names + pair distances + depth)."""
    return ing.extract_locus(tred, readlen, alts=alt_regions(tred, ref, alts, clip), want_names=True)


TAGNAME = {1: "FULL", 2: "PREF", 3: "POST", 4: "REPT"}


def genotype_evidence(items, maxinsert=300, fullsearch=False, clip=False, repeatpairs=True, ctx=None, device_batch=None):
    """The fused device path, whichever reader produced the evidence: ONE ``tredsw_genotype_batch_ex``
    call (Smith-Waterman + classification -> tallies -> candidate ranges -> KDE -> likelihood grid -> call / CI / PP
    / label -> sparse posteriors) over any number of (sample, locus) problems, then the reference's per-locus
    result fields (tred.py:251-275) assembled from what comes back.
    :param items: list of (tred, READLEN, gender, depth, ingest.LocusEvidence)
    :param device_batch: the ``ingest.IngestBatch`` the items came from, problem i = item i: its buffers are consumed
                         where they lie in device memory (no batch is assembled on the host, nothing is uploaded again)
    :return: list of dicts keyed like the ``<T>.xxx`` entries of tredCalls, without the prefix."""
    from . import cohort, _lib
    from .simulate import Problem
    if not items:
        return []
    ploidy_of = lambda tred, gender: 1 if (gender == "Male" and tred.is_xlinked) else tred.ploidy
    if device_batch is not None:
        keys, fam_of = {}, []
        for tred, readlen, gender, depth, ev in items:
            fam_of.append(keys.setdefault((tred.name, readlen), len(keys)))
        family_keys = [None] * len(keys)
        for (tred, readlen, gender, depth, ev), f in zip(items, fam_of):
            family_keys[f] = (tred, readlen)
        batch = cohort.CohortBatch.from_ingest(
            device_batch, np.array(fam_of, dtype=np.int32),
            np.array([ploidy_of(it[0], it[2]) for it in items], dtype=np.int32),
            np.array([it[3] for it in items], dtype=np.float64), family_keys,
            names=None if (repeatpairs or clip) else [it[4].names for it in items],
            maxinsert=maxinsert, fullsearch=fullsearch, clip=clip, repeatpairs=repeatpairs)
        out = batch.run_ingest(ctx or _lib.default_context(), want_reads=True, want_hist=True, want_post=True)
    else:
        problems = []
        for tred, readlen, gender, depth, ev in items:
            pr = Problem()
            pr.tred, pr.readlen = tred, readlen
            pr.ploidy = ploidy_of(tred, gender)
            pr.depth, pr.reads, pr.roff = depth, ev.reads, ev.roff
            pr.global_lens, pr.target_lens = ev.global_lens, ev.target_lens
            pr.alleles, pr.names = None, ev.names
            problems.append(pr)
        batch = cohort.CohortBatch(problems, maxinsert=maxinsert, fullsearch=fullsearch, clip=clip, repeatpairs=repeatpairs)
        out = batch.run_host(ctx=ctx, want_reads=True, want_hist=True, want_post=True)
    post = cohort.posteriors(out["post"], len(items))
    results, r0 = [], 0
    calls = out["calls"].tolist()                                    # (plain tuples: no numpy scalars in the loop)

    def cs(row):                                                     # "units|count;..." of one histogram row
        nz = np.flatnonzero(row).tolist()
        return ";".join(["{}|{}".format(k, v) for k, v in zip(nz, row[nz].tolist())]) if nz else ""
    for i, (tred, readlen, gender, depth, ev) in enumerate(items):
        c = cohort.decode_call(calls[i])
        if c["n_points"] < 0:
            raise RuntimeError("likelihood arena overflow")          # (run_host repeats the call; not expected)
        rows = out["reads"][r0:r0 + ev.nreads]
        r0 += ev.nreads
        names = ev.names or [""] * ev.nreads
        tags, hs = rows[:, 0].tolist(), rows[:, 1].tolist()
        text, off = ev.read_text(), ev.roff.tolist()
        details = [{"tag": TAGNAME[t], "h": hs[k], "id": names[k], "seq": text[off[k]:off[k + 1]]}
                   for k, t in enumerate(tags) if t in TAGNAME]
        hist = out["hist"][i]
        missing = c["alleles"][0] < 0
        g, t = np.asarray(ev.global_lens), np.asarray(ev.target_lens)
        results.append({
            "1": c["alleles"][0], "2": c["alleles"][1], "FR": cs(hist[0]), "PR": cs(hist[1]), "RR": cs(hist[2]),
            "DP": depth, "FDP": c["FDP"], "PDP": c["PDP"], "RDP": c["RDP"], "PEDP": len(t),
            "PEG": mean_std(g), "PET": mean_std(t), "CI": c["CI"], "PP": c["PP"], "label": c["label"],
            "details": details,
            "P_h1": "" if missing else post[i]["P_h1"], "P_h2": "" if missing else post[i]["P_h2"],
            "P_h1h2": "" if missing else post[i]["P_h1h2"], "P_PEG": histogram(g), "P_PET": histogram(t)})
    return results


INGEST_THREADS = int(os.environ.get("TREDSW_INGEST_THREADS", "0")) or min(8, os.cpu_count() or 1)


def ingest_loci(bam, repo, tredNames, READLEN, alts, clip, logger, threads=None, want_names=True):
    """Evidence of every requested locus of one BAM.
    Native ingest (csrc/ingest.cpp): one indexed pass per locus yields reads, pair distances AND depth; the loci
    are dealt to `threads` host threads, each with its own clone of the BAM handle (own file descriptor, shared
    index; ctypes releases the GIL during the pass).  When the BAM has no usable index or the native reader does not
    know the contig, ``bam_parser.extract_locus`` builds the same record with the Python BAM reader (three passes per
    locus, like the reference's pysam calls, tred.py:225-243).  A locus whose window cannot be read (truncated /
    corrupt BAM) gets no record and so no call: the reference's `except Exception: continue` (tred.py:245-249).
    :return: {tredName: ingest.LocusEvidence}"""
    ing = None
    try:
        from .ingest import BamIngest
        ing = BamIngest(bam_path(bam))
    except Exception as e:
        logger.debug("native BAM ingest unavailable for `{}` ({}); using the Python reader".format(bam, e))

    def one(handle, tred):
        xtred = repo[tred]
        try:
            if handle is not None and handle.tid(xtred.chr) >= 0:
                return tred, locus_evidence(handle, xtred, READLEN, alts, clip, repo.ref)
            return tred, extract_locus(bam, repo, tred, READLEN, alts, clip, logger)
        except Exception as e:
            logger.error("Exception on `{}` {} ({})".format(bam, tred, e))
            return tred, None

    threads = max(1, min(threads or INGEST_THREADS, len(tredNames)))
    if ing is None or threads == 1:
        done = [one(ing, tred) for tred in tredNames]
    else:
        from concurrent.futures import ThreadPoolExecutor
        handles = [ing] + [ing.clone() for _ in range(threads - 1)]

        def lane(k):
            return [one(handles[k], tred) for tred in tredNames[k::threads]]
        try:
            with ThreadPoolExecutor(max_workers=threads) as pool:
                done = [r for part in pool.map(lane, range(threads)) for r in part]
        finally:
            for h in handles[1:]:
                h.close()
    if ing is not None:
        ing.close()
    evidence = {}
    for tred, ev in done:
        if ev is not None:
            evidence[tred] = ev
            logger.debug("Inferred depth at locus {}: {}".format(tred, ev.depth))
    return evidence


GPU_INGEST = os.environ.get("TREDSW_GPU_INGEST", "1") != "0"
DEVICE_HANDOFF = os.environ.get("TREDSW_DEVICE_HANDOFF", "1") != "0"     # genotype from the ingest's device buffers


def ingest_chunk_gpu(samples, ctx=None, keep_batch=None):
    """Evidence of every (sample, locus) of a chunk through the GPU ingest (csrc/bgzf_gpu.cu): the host reads the
    compressed BGZF blocks behind the windows, the device inflates them, walks the records and applies the
    selection / pairing / depth rules — same evidence as ``ingest_loci`` locus by locus.
    :param samples: [(key, run-argument tuple, wanted TRED names, READLEN, open ingest.BamIngest)]
    :param keep_batch: a list; when every problem of the batch is good, (IngestBatch, [(key, tredName)]) is appended
                       and the batch stays open (the evidence objects are views into it): the caller genotypes from
                       its device buffers and closes it
    :return: {key: {tredName: LocusEvidence}} — loci the device path could not serve (contig missing, a block the
             decoder refused, corrupt records) are left out: the caller reads them with the host reader."""
    from . import _lib
    from .ingest import IngestBatch, locus_query
    handles, qs, so, keep, key = [], [], [], [], []
    try:
        for k, arg, wanted, READLEN, h in samples:
            samplekey, bam, repo, tredNames, maxinsert, fullsearch, clip, alts, repeatpairs, log = arg
            if h is None:
                continue
            handles.append(h)
            for t in wanted:
                xtred = repo[t]
                q = locus_query(h, xtred, READLEN, alts=alt_regions(xtred, repo.ref, alts, clip))
                if q is None:
                    continue
                qs.append(q[0]); keep.append(q[1]); so.append(len(handles) - 1); key.append((k, t))
        got = {}
        if not qs:
            return got
        ctx = ctx or _lib.default_context()
        b = IngestBatch(ctx, handles, so, qs, keep=keep)
        try:
            hold = keep_batch is not None and not b.status.any()
            for i, (k, t) in enumerate(key):
                if b.status[i]:
                    logger.debug("GPU ingest handed {} / {} back (status {})".format(k, t, int(b.status[i])))
                    continue
                got.setdefault(k, {})[t] = b.evidence(i, copy=not hold)
            if hold:
                # every problem is good: the caller may genotype straight from the batch's device buffers
                keep_batch.append((b, key))
                b = None
        finally:
            if b is not None:
                b.close()
        return got
    except Exception as e:
        logger.error("GPU ingest failed ({}); reading with the host reader".format(e))
        return {}


def ingest_sample_scan(arg, wanted, READLEN, h, with_gender, ctx=None, stream=False):
    """Evidence of every wanted locus of one sample whose BAM has no usable index, and its chrY depth when
    ``with_gender``, in ONE streaming pass over the file on the GPU (``ingest.scan_sample``).
    :param h: the sample's handle from ``ingest.BamIngest.unindexed`` or ``ingest.BamIngest.stream``
    :param stream: `h` is a stream, which can be read only once: a scan that fails raises (no partial evidence, no
                   second reader), and a header without the chrY regions gives gender ('Unknown', -1)
    :return: ({tredName: LocusEvidence}, (gender, depthY) or None) — loci the scan could not serve (contig missing,
             a corrupt or unsorted file) are left out, and so is the gender: the caller reads them with the Python
             reader (not a stream's: a locus whose contig the header lacks gets no call)."""
    from . import _lib
    from .ingest import locus_query, scan_sample
    samplekey, bam, repo, tredNames, maxinsert, fullsearch, clip, alts, repeatpairs, log = arg
    qs, keep, names = [], [], []
    for t in wanted:
        xtred = repo[t]
        q = locus_query(h, xtred, READLEN, alts=alt_regions(xtred, repo.ref, alts, clip))
        if q is None:
            continue
        qs.append(q[0]); keep.append(q[1]); names.append(t)
    yreg = []
    if with_gender:
        rows = BamDepth.y_regions(repo.ref)
        tids = [h.tid(c) for c, s, e in rows]
        if rows and min(tids) >= 0:
            yreg = [(t, s, e) for t, (c, s, e) in zip(tids, rows)]
    got, gender = {}, (("Unknown", -1) if stream and with_gender and not yreg else None)
    if not qs and not yreg:
        return got, gender
    try:
        with scan_sample(ctx or _lib.default_context(), h, qs, keep, yreg) as b:
            if stream and b.scan_status:
                raise IOError("the GPU scan of `{}` failed (status {}): {}".format(bam, b.scan_status, _lib.last_error()))
            for i, t in enumerate(names):
                if b.status[i]:
                    logger.debug("GPU scan handed {} / {} back (status {})".format(samplekey, t, int(b.status[i])))
                    continue
                got[t] = b.evidence(i)
            if yreg and not b.scan_status:
                ydepth = float(np.median(b.depths))
                gender = ("Male" if ydepth > 1 else "Female", ydepth)
    except Exception as e:
        if stream:
            raise
        logger.error("GPU scan of `{}` failed ({}); reading with the Python reader".format(bam, e))
        return {}, None
    return got, gender


OPEN_STREAMS = {}       # stream path -> ingest.BamIngest whose header was read early (the sample key of `-`)


def stream_presteps(bam):
    """(handle, pre-steps) of a stream sample: its handle (``ingest.BamIngest.stream``) and the read length from the
    records the handle reads ahead; gender comes later, from the chrY regions of the sample's one scan."""
    from .ingest import BamIngest
    from . import _lib
    if not GPU_INGEST:
        raise IOError("`{}` is a stream: only the GPU scan reads it (TREDSW_GPU_INGEST=0)".format(bam))
    h = OPEN_STREAMS.pop(bam, None) or BamIngest.stream(bam)
    READLEN = 150
    try:
        READLEN = h.read_length()[0]
    except _lib.TredswError:
        pass                    # no records (the scan finds none either) or a damaged stream (the scan reports it)
    logger.debug("Read length: {}bp".format(READLEN))
    return h, {"inferredGender": "Unknown", "depthY": -1, "readLen": READLEN}


def infer_gender(bam, repo, tredNames, logger, ing=None):
    """Gender from the chrY depth (tred.py:195-211) — only when an X-linked locus is requested; 'Unknown' / -1 when
    the lookup fails.  -> (gender, depthY)"""
    gender, ydepth = "Unknown", -1
    if any(repo[tred].is_xlinked for tred in tredNames):
        try:
            ydepth = BamDepth(bam, repo.ref, logger, ing=ing).get_Y_depth()
            gender = "Male" if ydepth > 1 else "Female"
        except Exception:
            pass
        logger.debug("Inferred gender: {} (depthY={})".format(gender, ydepth))
    return gender, ydepth


def presteps(bam, repo, tredNames, logger, ing=None, with_gender=True):
    """The per-sample pre-steps of tred.run (tred.py:195-223): gender (``infer_gender``; 'Unknown' / -1 without
    ``with_gender``) and the read length (150 when it cannot be read).  They decide ploidy (bam_parser.py:58-61) and
    the number of templates (:73), so they gate parity on real BAMs."""
    gender, ydepth = infer_gender(bam, repo, tredNames, logger, ing=ing) if with_gender else ("Unknown", -1)
    READLEN = 150
    try:
        READLEN = BamReadLen(bam, logger, ing=ing).readlen
    except Exception:
        pass
    logger.debug("Read length: {}bp".format(READLEN))
    return {"inferredGender": gender, "depthY": ydepth, "readLen": READLEN}


def run(arg):
    """Run the TRED caller on a list of TREDs for one sample.  :return: dict of calls"""
    return run_chunk([arg])[0]


def prepare_chunk(args, only=None, ctx=None):
    """First half of ``run_chunk``: per-sample pre-steps and the evidence of every (sample, locus) — the GPU ingest,
    the host reader for what it hands back.  Touches no state of the genotyping context, so the next chunk can be
    prepared (on ``ctx``, a context of its own) while the previous one is genotyped.
    :return: an opaque state for ``finish_chunk``"""
    out, items, where, todo = [], [], [], []
    for si, arg in enumerate(args):
        samplekey, bam, repo, tredNames, maxinsert, fullsearch, clip, alts, repeatpairs, log = arg
        tredCalls = {"inferredGender": "Unknown", "depthY": -1}
        out.append({"samplekey": samplekey, "bam": bam, "tredCalls": tredCalls, "_fields": {}, "_names": list(tredNames)})
    # per sample: one native handle (validity check, pre-steps, GPU ingest), the pre-steps (gender looks at every
    # requested locus); the samples are dealt to host threads
    # a BAM without a usable index is scanned once on the GPU (unless the GPU ingest is off): its gender comes from
    # that scan, so its pre-steps here read only the read length.  So is a stream, which nothing else may read: a
    # stream that cannot be scanned makes its sample an error
    def pre(si):
        samplekey, bam, repo, tredNames = args[si][:4]
        from .ingest import BamIngest, is_stream
        if is_stream(bam):
            try:
                return stream_presteps(bam) + ("stream",)
            except Exception as e:
                return e
        ing = None
        try:
            ing = BamIngest(bam_path(bam))
        except Exception as e:
            logger.debug("native BAM ingest unavailable for `{}` ({})".format(bam, e))
            if check_bam(bam) is None:
                return None
            if GPU_INGEST:
                try:
                    uh = BamIngest.unindexed(bam_path(bam))
                    return uh, presteps(bam, repo, tredNames, logger, ing=uh, with_gender=False), True
                except Exception as e2:
                    logger.debug("GPU scan unavailable for `{}` ({})".format(bam, e2))
        return ing, presteps(bam, repo, tredNames, logger, ing=ing), False
    if len(args) > 1 and INGEST_THREADS > 1:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=min(INGEST_THREADS, len(args))) as pool:
            pres = list(pool.map(pre, range(len(args))))
    else:
        pres = [pre(si) for si in range(len(args))]
    wanted_of, handle_of, unindexed, streams, failed = {}, {}, set(), set(), set()

    def fail(si, e):
        logger.error("Sample `{}`: {}".format(args[si][0], e))
        failed.add(si)
        out[si].update({"tredCalls": {}, "error": repr(e), "_names": []})
    for si, ps in enumerate(pres):
        if ps is None:
            continue
        if isinstance(ps, Exception):
            fail(si, ps)
            continue
        todo.append(si)
        handle_of[si] = ps[0]
        if ps[2]:
            unindexed.add(si)
        if ps[2] == "stream":
            streams.add(si)
        out[si]["tredCalls"].update(ps[1])
        tredNames = args[si][3]
        wanted_of[si] = [t for t in tredNames if only is None or t in only[si]]
        out[si]["_names"] = wanted_of[si]
    # evidence: the GPU ingest for every (sample, locus) of the chunk in one pass, one GPU scan per sample without an
    # index; the host reader for what they hand back (corrupt blocks, unsorted files, unknown contig) or when they are
    # switched off (TREDSW_GPU_INGEST=0)
    kept = []
    try:
        got = ingest_chunk_gpu([(si, args[si], wanted_of[si], out[si]["tredCalls"]["readLen"],
                                 None if si in unindexed else handle_of[si]) for si in todo],
                               ctx=ctx, keep_batch=kept if DEVICE_HANDOFF else None) if GPU_INGEST else {}
        for si in sorted(unindexed):
            samplekey, bam, repo, tredNames = args[si][:4]
            with_gender = any(repo[t].is_xlinked for t in tredNames)
            try:
                got[si], gender = ingest_sample_scan(args[si], wanted_of[si], out[si]["tredCalls"]["readLen"],
                                                     handle_of[si], with_gender, ctx=ctx, stream=si in streams)
            except Exception as e:
                if si not in streams:
                    raise
                fail(si, e)
                continue
            if gender is None and with_gender:
                gender = infer_gender(bam, repo, tredNames, logger)
            if gender is not None:
                logger.debug("Inferred gender: {} (depthY={})".format(*gender))
                out[si]["tredCalls"].update({"inferredGender": gender[0], "depthY": gender[1]})
    finally:
        for h in handle_of.values():
            if h is not None:
                h.close()
    for si in todo:
        if si in failed:
            continue
        samplekey, bam, repo, tredNames, maxinsert, fullsearch, clip, alts, repeatpairs, log = args[si]
        gender, READLEN = out[si]["tredCalls"]["inferredGender"], out[si]["tredCalls"]["readLen"]
        wanted = wanted_of[si]
        evidence = got.get(si, {})
        rest = [t for t in wanted if t not in evidence]
        if rest and si not in streams:              # (a stream's bytes are gone: its missing loci get no call)
            evidence.update(ingest_loci(bam, repo, rest, READLEN, alts, clip, logger, want_names=True))
        for t in wanted:
            if t in evidence:
                items.append((repo[t], READLEN, gender, evidence[t].depth, evidence[t]))
                where.append((si, t))
    # the fused call can run on the ingest's device buffers when the items are exactly the problems of the batch
    device_batch = None
    if kept:
        b, key = kept[0]
        if key == where:
            device_batch = b
        else:                                   # (some locus came from the host reader: assemble the batch on the host)
            items = [(it[0], it[1], it[2], it[3], _own_evidence(it[4])) for it in items]
            b.close()
    return args, out, items, where, device_batch


def _own_evidence(ev):
    """a LocusEvidence whose arrays no longer point into an IngestBatch"""
    for name in ("reads", "global_lens", "target_lens"):
        setattr(ev, name, np.array(getattr(ev, name)))
    return ev


def finish_chunk(state, ctx=None):
    """Second half of ``run_chunk``: ONE fused device call for the loci of all the samples of the chunk, then the
    reference's per-locus JSON fields.
    :return: list of {"samplekey", "bam", "tredCalls"}"""
    args, out, items, where, device_batch = state
    if not args:
        return []
    _, _, _, _, maxinsert, fullsearch, clip, _, repeatpairs, _ = args[0]
    # all the loci in one call: on the ingest's own device buffers when the whole chunk came from the GPU ingest,
    # else from a batch assembled on the host
    try:
        res = genotype_evidence(items, maxinsert=maxinsert, fullsearch=fullsearch, clip=clip, repeatpairs=repeatpairs,
                                ctx=ctx, device_batch=device_batch)
    finally:
        if device_batch is not None:
            device_batch.close()
    for (si, t), r in zip(where, res):
        out[si]["_fields"][t] = r
    for o in out:
        fields = o.pop("_fields")
        for tred in o.pop("_names"):
            for k, v in fields.get(tred, {}).items():
                o["tredCalls"][tred + "." + k] = v
    return out


def run_chunk(args, only=None):
    """Several samples at once: per-sample pre-steps, then the evidence of every (sample, locus) of the chunk in one
    pass of the GPU ingest, then the loci of ALL the samples through ONE fused device call.  Same results as ``run``
    sample by sample.
    :param args: list of ``run`` argument tuples (same maxinsert / fullsearch / clip / repeatpairs for all)
    :param only: optional list, per sample, of the TRED names to process (a rank's share of a sharded cohort);
                 the other requested names of that sample are left out of its tredCalls
    :return: list of {"samplekey", "bam", "tredCalls"}"""
    return finish_chunk(prepare_chunk(args, only))


def run_chunks(args, only=None, chunk=None, isolate=False):
    """``run_chunk`` over a long list of samples, ``chunk`` samples at a time, two stages deep: a helper thread
    prepares chunk k + 1 (file reads and the GPU ingest, on a context and stream of its own; the C calls release the
    GIL) while this thread genotypes chunk k and assembles its JSON fields.  Yields the per-sample results in order.
    isolate: a chunk that raises yields {"samplekey", "bam", "tredCalls": {}, "error"} for its samples instead of
    ending the run."""
    from concurrent.futures import ThreadPoolExecutor
    from . import _lib
    chunk = chunk or CHUNK_SAMPLES
    spans = [(c0, min(len(args), c0 + chunk)) for c0 in range(0, len(args), chunk)]
    if not spans:
        return
    ictx = None
    if GPU_INGEST and len(spans) > 1:
        try:
            ictx = _lib.Context(_lib.default_context().device)
        except Exception:
            ictx = None

    def prep(k):
        a, b = spans[k]
        return prepare_chunk(args[a:b], None if only is None else only[a:b], ctx=ictx)
    try:
        with ThreadPoolExecutor(max_workers=1) as pool:
            fut = pool.submit(prep, 0)
            for k in range(len(spans)):
                try:
                    state, err = fut.result(), None
                except Exception as e:
                    if not isolate:
                        raise
                    state, err = None, e
                if k + 1 < len(spans):
                    fut = pool.submit(prep, k + 1)
                if err is None:
                    try:
                        results = finish_chunk(state)
                    except Exception as e:
                        if not isolate:
                            raise
                        err = e
                if err is not None:
                    a, b = spans[k]
                    results = [{"samplekey": x[0], "bam": x[1], "tredCalls": {}, "error": repr(err)} for x in args[a:b]]
                for r in results:
                    yield r
    finally:
        if ictx is not None:
            ictx.close()


def vcfstanza(sampleid, bam, tredCalls, ref):
    m = "##fileformat=VCFv4.1\n"
    now = dt.now()
    m += "##fileDate={}{:02d}{:02d}\n".format(now.year, now.month, now.day)
    m += "##source={} {}\n".format(__file__, bam)
    m += "##reference={}\n".format(ref)
    m += "##inferredGender={} depthY={}\n".format(tredCalls["inferredGender"], tredCalls["depthY"])
    m += "##readLen={}bp\n".format(tredCalls["readLen"])
    m += INFO
    header = "CHROM POS ID REF ALT QUAL FILTER INFO FORMAT\n".split() + [sampleid]
    m += "#" + "\t".join(header)
    return m


def to_json(results, ref, repo, treds=("HD",), store=None):
    sampleid = results["samplekey"]
    calls = results["tredCalls"]
    if not calls:
        logger.debug("No calls are found for {} `{}`".format(sampleid, results["bam"]))
        return
    jsonfile = ".".join((sampleid, "json"))
    js = json.dumps(results, sort_keys=True, indent=4, separators=(",", ": "))
    print(js)
    with open(jsonfile, "w") as fw:
        print(js, file=fw)


def to_vcf(results, ref, repo, treds=("HD",), store=None):
    registry = {tred: repo.get_info(tred) for tred in treds}
    sampleid, bam, calls = results["samplekey"], results["bam"], results["tredCalls"]
    if not calls:
        return
    vcffile = ".".join((sampleid, "tred.vcf.gz"))
    contents = []
    for tred in treds:
        if tred + ".1" not in calls:
            continue
        a, b = calls[tred + ".1"], calls[tred + ".2"]
        chr, start, ref_copy, repeat, info = registry[tred]
        alleles = set([a, b])
        rpa = sorted(alleles - set([ref_copy]))
        alt = ",".join(x * repeat for x in rpa) if (rpa and rpa[0] != -1) else "."
        if rpa:
            info += ";RPA={}".format(",".join(str(x) for x in rpa))
            if ref_copy in alleles:
                gt = "0/1"
            elif len(rpa) == 1:
                gt = "1/1"
            else:
                gt = "1/2"
        else:
            gt = "0/0"
        gb = "{}/{}".format(a, b)
        fields = "{}:{}:{}:{}:{}:{}:{}:{}:{}:{}:{}:{:.4g}:{}".format(
            gt, gb, calls[tred + ".FR"], calls[tred + ".PR"], calls[tred + ".RR"], calls[tred + ".DP"],
            calls[tred + ".FDP"], calls[tred + ".PDP"], calls[tred + ".RDP"], calls[tred + ".PEDP"],
            calls[tred + ".CI"], calls[tred + ".PP"], calls[tred + ".label"])
        m = "\t".join(str(x) for x in (chr, start, tred, ref_copy * repeat, alt, ".", ".", info,
                                       "GT:GB:FR:PR:RR:DP:FDP:PDP:RDP:PEDP:CI:PP:LABEL", fields))
        contents.append((chr, start, m))
    with gzip.open(vcffile, "wt") as fw:
        print(vcfstanza(sampleid, bam, calls, ref), file=fw)
        contents.sort()
        for chr, start, m in contents:
            print(m, file=fw)
    logger.debug("VCF file written to `{}`".format(vcffile))


def read_csv(csvfile, args):
    if csvfile == "-":
        # one sample on stdin: its key is the SM of the header's first @RG line (the header is read here and the
        # handle kept for the run)
        from .ingest import BamIngest
        h = OPEN_STREAMS["-"] = BamIngest.stream("-")
        return [(h.read_group_sample() or "stdin", "-", None)]
    if csvfile[0] == "@":
        raise ValueError("@HLI-id inputs are not supported by this build")
    if csvfile.endswith(".bam") or csvfile.endswith(".cram"):
        bam = bam_path(csvfile)
        samplekey = op.basename(bam).rsplit(".", 1)[0]
        return [(samplekey, bam, None)]
    with open(csvfile) as fp:
        rows = [r.strip() for r in fp if r.strip()]
    header = rows[0]
    contents = []
    if header.endswith(".bam") and header.count(",") == 0:
        for row in rows:
            bam = bam_path(row)
            contents.append((op.basename(bam).rsplit(".", 1)[0], bam, None))
        return contents
    for row in rows:
        atoms = row.split(",")
        samplekey, bam = atoms[:2]
        tred = atoms[2] if len(atoms) == 3 else None
        bam = bam_path(bam)
        if bam.endswith(".bam"):
            contents.append((samplekey, bam, tred))
    return contents


def write_vcf_json(results, ref, repo, treds, store):
    try:
        to_vcf(results, ref, repo, treds=treds, store=store)
        to_json(results, ref, repo, treds=treds, store=store)
    except Exception as e:
        print("Error writing: {} ({})".format(results.get("samplekey"), e), file=sys.stderr)


CHUNK_SAMPLES = int(os.environ.get("TREDSW_CHUNK_SAMPLES", "16"))     # samples per fused device call


def locus_costs(repo, task_args, readlen=150):
    """A-priori cost of every (sample, locus) problem of a task list, flat in task order: the forward cells of the
    locus' template family (all a scheduler knows before reading the BAMs).  -> (costs, [(sample index, tred)])"""
    costs, keys = [], []
    for si, ta in enumerate(task_args):
        for t in ta[3]:
            tr = repo[t]
            P, flank = len(tr.repeat), len(tr.prefix) + len(tr.suffix)
            mu = -(-readlen // P)
            costs.append(2.0 * readlen * sum(flank + P * u for u in range(1, mu + 1)))
            keys.append((si, t))
    return np.array(costs), keys


def _worker(rank, ngpus, task_args, queue):
    """One process per GPU.  The (sample, locus) problems are dealt by cost (dist.shard_by_cost: every rank computes
    the same partition, no communication); a rank ingests only the windows of its own problems and sends back, per
    chunk of samples, the per-locus fields it produced.  The parent merges them into the per-sample JSON."""
    try:
        os.environ["TREDSW_DEVICE"] = str(rank)
        from .dist import shard_by_cost
        costs, keys = locus_costs(task_args[0][2], task_args)
        owner = shard_by_cost(costs, ngpus)
        mine = {}
        for (si, t), o in zip(keys, owner):
            if o == rank:
                mine.setdefault(si, []).append(t)
        order = sorted(mine)
        got = run_chunks([task_args[i] for i in order], only=[mine[i] for i in order], isolate=True)
        for i, r in zip(order, got):                                # (a failed chunk must not hang the parent)
            queue.put(("part", i, r, len(mine[i])))
    finally:
        queue.put(("done", rank, None, 0))


def main(args):
    p = set_argparse()
    args = p.parse_args(args)
    loglevel = getattr(logging, args.log.upper(), "INFO")
    logger.setLevel(loglevel)
    logger.debug("Commandline Arguments:{}".format(vars(args)))

    start = time.time()
    workdir = args.workdir
    cwd = os.getcwd()
    if workdir != cwd:
        mkdir(workdir, logger=logger)
    infile = args.infile
    if not infile:
        sys.exit(not p.print_help())
    # ranks scan their own loci of every sample, and a stream can be read only once
    multi_gpu_stream = "--gpus {} with a stream input: a stream can be read only once, by one GPU".format(args.gpus)
    if args.gpus > 1 and infile == "-":
        p.error(multi_gpu_stream)
    samples = read_csv(infile, args)
    from .ingest import is_stream
    if args.gpus > 1 and any(is_stream(bam) for _, bam, _ in samples):
        p.error(multi_gpu_stream)
    logger.debug("Total samples: {}".format(len(samples)))

    task_args = []
    sites = op.join(os.getcwd(), "sites")
    os.chdir(workdir)
    ref = args.ref
    repo = TREDsRepo(ref=ref, toy=args.toy, sites=sites)
    repo.set_ploidy(args.haploid)
    treds = args.tred or repo.names
    if args.toy:
        treds = ["HD"]
    for samplekey, bam, tred in samples:
        jsonfile = ".".join((samplekey, "json"))
        if args.checkexists and op.exists(jsonfile):
            logger.debug("File `{}` exists. Skipped computation.".format(jsonfile))
            if bam in OPEN_STREAMS:
                OPEN_STREAMS.pop(bam).close()
            continue
        _treds = [tred] if tred else treds
        task_args.append((samplekey, bam, repo, _treds, args.maxinsert, args.fullsearch,
                          args.useclippedreads, (not args.noalts), (not args.norepeatpairs), args.log))
    if not task_args:
        logger.debug("All jobs already completed.")
        os.chdir(cwd)
        return

    def emit(results):
        if not args.no_output:
            write_vcf_json(results, ref, repo, treds, None)

    ngpus = max(1, args.gpus)
    if ngpus == 1:
        # chunks of samples: one fused device call per chunk (all loci of all its samples)
        for results in run_chunks(task_args):
            emit(results)
    else:
        import multiprocessing as mp
        import queue as pyqueue
        ctx = mp.get_context("spawn")
        queue = ctx.Queue()
        procs = [ctx.Process(target=_worker, args=(r, ngpus, task_args, queue)) for r in range(ngpus)]
        for pr in procs:
            pr.start()
        merged = [None] * len(task_args)
        got = [0] * len(task_args)
        need = [len(ta[3]) for ta in task_args]
        done, nxt = 0, 0
        while done < ngpus:
            try:
                kind, i, res, n = queue.get(timeout=30)
            except pyqueue.Empty:
                # a worker that died without its sentinel (segfault, OOM kill) must not hang the run
                dead = [pr for pr in procs if not pr.is_alive() and pr.exitcode not in (0, None)]
                if dead:
                    raise RuntimeError("worker process(es) died: exit codes {}".format([pr.exitcode for pr in dead]))
                continue
            if kind == "done":
                done += 1
                continue
            if merged[i] is None:
                merged[i] = {"samplekey": res["samplekey"], "bam": res["bam"], "tredCalls": {}}
            merged[i]["tredCalls"].update(res["tredCalls"])
            if "error" in res:
                logger.error("Sample `{}`: {}".format(res["samplekey"], res["error"]))
            got[i] += n
            while nxt < len(task_args) and got[nxt] >= need[nxt]:          # emit in input order, like Pool.imap
                emit(merged[nxt])
                merged[nxt] = None
                nxt += 1
        for pr in procs:
            pr.join()
        while nxt < len(task_args):                                         # (samples no rank owned a locus of)
            if merged[nxt] is not None:
                emit(merged[nxt])
            nxt += 1

    print("Elapsed time={}".format(timedelta(seconds=time.time() - start)), file=sys.stderr)
    os.chdir(cwd)
    if args.cleanup:
        shutil.rmtree(workdir)


if __name__ == "__main__":
    main(sys.argv[1:])
