"""
Evidence extraction from a BAM — host side of the hot path.

Keeps the reference's ``tredparse/bam_parser.py`` interface: ``BamParser(inputParams).parse()`` with
``counts / details / rept / ploidy / READLEN / depth / repeatSize`` (:35-287), ``BamParserResults``
(:290-313), ``PEextractor`` (:316-369), ``BamReadLen`` (:372-391), ``BamDepth`` (:394-429),
``read_alignment`` (:432-436), ``rc`` (:448-450).  ``extract_locus`` packs what ``select_reads``,
``PEextractor`` and ``BamDepth`` read for one locus into the ``ingest.LocusEvidence`` the native reader produces.

What runs where:
  host   BAM window fetches (own BGZF/BAI reader instead of pysam), read selection rules
         (:206-243), tallies (:259-287);
  GPU    all reads x all templates Smith-Waterman, post-filter, classification and per-read arg-max
         (:123-182 over src/ssw_wrap.py over src/ssw.c) in ONE ``tredsw_classify_reads`` call per locus
         (or per whole cohort shard through ``classify_problems``).
"""
import logging
import os
import math
from collections import defaultdict

import numpy as np

from . import bamio, ssw, _lib
from .utils import datafile  # noqa: F401  (API parity)

SPAN = 1000
FLANKMATCH = 9
DNAPE_ELONGATE = SPAN * 10

_COMPLEMENT = str.maketrans("ATCGatcgNnXx", "TAGCtagcNnXx")


def rc(s):
    return s.translate(_COMPLEMENT)[::-1]


def read_alignment(samfile):
    """Open a BAM (``tag`` kept for API parity; CRAM is not supported by the built-in reader)."""
    if samfile.endswith(".cram"):
        raise ValueError("CRAM input is not supported by the built-in reader")
    return bamio.AlignmentFile(samfile, "rb")


def test_fetch(samfile, chr, start, end, logger):
    try:
        samfile.fetch(chr, start, end)
        return True
    except ValueError:
        logger.error("No reads extracted for region {}:{}-{}".format(chr, start, end))
        return False


test_fetch.__test__ = False  # not a pytest test


def tally(details, counts):
    for x in details:
        counts[x["tag"]][x["h"]] += 1


def new_counts():
    """counts dict of the reference: PREF and POST share ONE histogram (bam_parser.py:77, quirk Q12)."""
    shared = defaultdict(int)
    counts = {"PREF": shared, "POST": shared}
    for tag in ("FULL", "REPT", "HANG"):
        counts[tag] = defaultdict(int)
    return counts


class BamParser:
    """Find TRED repeats from an aligned-reads BAM file.  :inputParams: InputParams object"""

    def __init__(self, inputParams):
        self.inputParams = inputParams
        self.logger = logging.getLogger("BamParser")
        self.logger.setLevel(inputParams.getLogLevel())
        self.bam = inputParams.bam
        self.gender = inputParams.gender
        self.depth = inputParams.depth
        self.READLEN = inputParams.READLEN
        self.clip = inputParams.clip
        self.alts = inputParams.alts
        self.repeatpairs = inputParams.repeatpairs
        self.ref = inputParams.ref
        self.tred = inputParams.tred
        self.repeatSize = len(self.tred.repeat)
        self.chr = self.tred.chr
        if self.gender == "Male" and self.tred.is_xlinked:
            self.ploidy = 1
        else:
            self.ploidy = self.tred.ploidy
        self.repeat = self.tred.repeat
        self.alt = self.tred.alt
        self.startRepeat, self.endRepeat = self.tred.repeat_start, self.tred.repeat_end
        self.referenceLen = self.tred.repeat_end - self.tred.repeat_start + 1
        self.fullPrefix, self.fullSuffix = self.tred.prefix, self.tred.suffix
        self.period = len(self.repeat)
        self.max_units = int(math.ceil(self.READLEN * 1. / self.period))
        self.counts = new_counts()
        self.details = []
        self.rept = 0

    def _buildDB(self):
        """The locus' template family as the record the CUDA kernel consumes (instead of the
        reference's list of 2*max_units Aligner objects, bam_parser.py:84-100)."""
        return ssw.make_family(self.fullPrefix, self.repeat, self.fullSuffix, self.max_units, self.clip)

    def select_reads(self, samfile, pad=SPAN):
        """The reads the reference hands to Smith-Waterman, in its order (bam_parser.py:194-243)."""
        WINDOW_START = max(0, self.startRepeat - pad)
        WINDOW_END = self.endRepeat + pad
        READ_START = max(0, self.startRepeat - self.READLEN)
        READ_END = self.endRepeat + self.READLEN
        chr, start, end = self.chr, WINDOW_START, WINDOW_END
        selected = []
        n_unmapped = 0
        if test_fetch(samfile, chr, start, end, self.logger):
            for read in samfile.fetch(chr, start, end):
                if read.is_unmapped:
                    n_unmapped += 1
                else:
                    if read.reference_start < READ_START:
                        continue
                    if read.reference_start > READ_END:
                        continue
                selected.append(read)
            if self.alts:
                for c, s, e in self.alt:
                    if self.clip:
                        continue
                    try:
                        if "nochr" in self.ref:
                            c = c[3:]
                        for read in samfile.fetch(c, s, e):
                            rid = read.next_reference_id
                            if rid == -1:
                                continue
                            if samfile.getrname(rid) != chr:
                                continue
                            rstart = read.next_reference_start
                            if rstart < WINDOW_START or rstart > WINDOW_END:
                                continue
                            selected.append(read)
                    except Exception as ex:
                        self.logger.debug("Fetch failed for region {}:{}-{} ({})".format(c, s, e, ex))
                        continue
        self.logger.debug("A total of {} unmapped reads in {}:{}-{}".format(n_unmapped, chr, start, end))
        self.n_unmapped = n_unmapped
        return selected

    def absorb(self, names, seqs, results):
        """Turn per-read kernel results (tag, h, ...) into counts / details (bam_parser.py:172-182,
        248-257)."""
        for rid, seq, row in zip(names, seqs, results):
            tag = _lib.TAG_NAMES.get(int(row[0]))
            if tag is None:
                continue
            h = int(row[1])
            self.counts["HANG"][h] += 1
            if tag == "HANG":
                continue
            self.details.append({"tag": tag, "h": h, "id": rid, "seq": seq})
        if not (self.repeatpairs or self.clip):
            self.remove_pairs_of_rept()
        self.tally_counts()
        self.rept = sum(self.counts["REPT"].values()) if self.counts["REPT"] else 0

    def parse(self, pad=SPAN):
        samfile = read_alignment(self.bam)
        reads = self.select_reads(samfile, pad=pad)
        samfile.close()
        seqs = [r.query_sequence for r in reads]
        names = [r.query_name for r in reads]
        if seqs:
            fam = self._buildDB()
            out = ssw.classify_reads(seqs, np.zeros(len(seqs), dtype=np.int32), fam)
        else:
            out = np.zeros((0, 8), dtype=np.int32)
        self.sw_results = out
        self.absorb(names, seqs, out)

    def tally_counts(self):
        tally(self.details, self.counts)
        for tag in ("FULL", "PREF", "REPT"):
            countMap = self.counts[tag]
            total = sum(countMap.values())
            s = " ".join("{}:{}".format(k, v) for (k, v) in sorted(countMap.items()))
            self.logger.debug("Counts [{}] (total={}) => {}".format(tag, total, s))

    def remove_pairs_of_rept(self):
        """Drop read names that occur more than once as REPT (bam_parser.py:270-287)."""
        rept_counts = defaultdict(int)
        for x in self.details:
            if x["tag"] == "REPT":
                rept_counts[x["id"]] += 1
        remove_ids = set(rid for rid, count in rept_counts.items() if count > 1)
        self.details = [x for x in self.details if x["id"] not in remove_ids]
        self.logger.debug("Tagging pairs of REPT to remove: {} pairs".format(len(remove_ids)))


class BamParserResults:
    """All results of one (sample, locus) problem: counts from BamParser, calls from the caller."""

    def __init__(self, inputParams, bamParser, caller):
        self.inputParams = inputParams
        self.tred = bamParser.tred
        self.counts = bamParser.counts
        self.details = bamParser.details
        self.FDP = sum(bamParser.counts["FULL"].values())
        self.PDP = sum(bamParser.counts["PREF"].values())
        self.RDP = bamParser.rept
        for k in ("PEDP", "PEG", "PET", "CI", "PP", "label", "alleles", "P_h1", "P_h2", "P_h1h2",
                  "P_PEG", "P_PET"):
            setattr(self, k, getattr(caller, k))


class PEextractor:
    """Distances of read pairs around / spanning the repeat (bam_parser.py:316-369)."""

    def __init__(self, bp):
        samfile = read_alignment(bp.bam)
        chr = bp.chr
        start, end = bp.startRepeat, bp.endRepeat
        self.ref = bp.referenceLen
        pstart = max(start - DNAPE_ELONGATE, 0)
        pend = end + DNAPE_ELONGATE
        cache = {}
        if test_fetch(samfile, chr, pstart, pend, bp.logger):
            cache = defaultdict(list)
            for x in samfile.fetch(chr, pstart, pend):
                if not x.is_paired or x.is_unmapped or x.is_duplicate:
                    continue
                cache[x.query_name].append(x)
        samfile.close()
        self.global_lens, self.target_lens = [], []
        tstart = start - FLANKMATCH
        tend = end + FLANKMATCH
        for name, reads in cache.items():
            if len(reads) < 2:
                continue
            a, b = reads[:2]
            if not ((not a.is_reverse) and b.is_reverse):
                continue
            tlen = self.get_target_length(a, b)
            if tlen >= SPAN:
                continue
            if a.reference_start < tstart and b.reference_end > tend:
                self.target_lens.append(tlen)
            else:
                self.global_lens.append(tlen)
        self.MINPE = end - start + 2 * FLANKMATCH + 2

    @staticmethod
    def get_target_length(a, b):
        start, end = a.reference_start, b.reference_end
        if a.query_alignment_start > 0:
            start -= a.query_alignment_start
        if b.query_alignment_end < b.query_length:
            end += b.query_length - b.query_alignment_end
        return end - start


class BamReadLen:
    """Read length of a BAM: longest of the first ~100 reads (bam_parser.py:372-391)."""

    def __init__(self, bamfile, logger, ing=None):
        """ing: an open ``ingest.BamIngest`` on the same file to use instead of opening another one"""
        self.bamfile = bamfile
        self.logger = logger
        self.ing = ing

    @property
    def readlen(self, firstN=100):
        try:                                   # native reader (csrc/ingest.cpp); needs the .bai next to the BAM
            from .ingest import BamIngest
            if self.ing is not None:
                rmax, rmin = self.ing.read_length(firstN)
            else:
                with BamIngest(os.path.abspath(self.bamfile)) as ing:
                    rmax, rmin = ing.read_length(firstN)
            if rmin != rmax:
                self.logger.debug("Read length: min={}bp max={}bp".format(rmin, rmax))
            return rmax
        except (IOError, OSError, _lib.TredswError):
            pass
        sam = read_alignment(self.bamfile)
        rls = []
        for read in sam.fetch():
            rls.append(read.query_length)
            if len(rls) > firstN:
                break
        sam.close()
        rmin, rmax = min(rls), max(rls)
        if rmin != rmax:
            self.logger.debug("Read length: min={}bp max={}bp".format(rmin, rmax))
        return rmax


class BamDepth:
    """Average depth of a region, for the repeat-only read model and for gender inference
    (bam_parser.py:394-429)."""

    def __init__(self, bamfile, ref, logger, ing=None):
        """ing: an open ``ingest.BamIngest`` on the same file to use instead of opening another one"""
        self.bamfile = bamfile
        self.logger = logger
        self.ref = ref
        self.ing = ing

    def region_depth(self, chr, start, end, verbose=False):
        sam = read_alignment(self.bamfile)
        try:
            depth = bamio.region_depth(sam, chr, start, end)
        finally:
            sam.close()
        if verbose:
            self.logger.debug("Depth of region {}:{}-{}: {}".format(chr, start, end, depth))
        return depth

    # rows of the chrY table that "still have mapped reads" in females and are skipped (bam_parser.py:417-418)
    Y_SKIP_ROWS = (1, 4, 6, 7, 10, 11, 13, 16, 18, 19)

    @classmethod
    def y_regions(cls, ref, N=5):
        """The first N usable unique chrY regions of the reference build: [(contig, start, end)]"""
        build = ref.split("_")[0]
        regions = []
        with open(datafile("chrY.tsv")) as fp:
            next(fp)
            for line in fp:
                b, row, c, start, end, _gc = line.split()
                if b != build or int(row) in cls.Y_SKIP_ROWS:
                    continue
                regions.append((c, int(start), int(end)))
                if len(regions) >= N:
                    break
        return regions

    def get_Y_depth(self, N=5):
        """Median depth over the first N usable unique chrY regions (bam_parser.py:413-429).  Raises when the
        BAM has no such contig — the caller then keeps gender 'Unknown' like the reference (tred.py:203-211)."""
        regions = self.y_regions(self.ref, N)
        depths = []
        ing, own = self.ing, False
        if ing is None:
            try:
                from .ingest import BamIngest
                ing, own = BamIngest(os.path.abspath(self.bamfile)), True
            except Exception:
                ing = None
        try:
            for c, start, end in regions:
                depths.append(ing.region_depth(c, start, end) if ing is not None else self.region_depth(c, start, end))
        finally:
            if own:
                ing.close()
        self.logger.debug("Y depths (first {} regions): {}".format(N, np.array(depths)))
        return float(np.median(depths))


def extract_locus(bam, repo, tredName, readlen, alts, clip, logger):
    """``ingest.BamIngest.extract_locus(..., want_names=True)`` made of this module's readers, for a BAM the native
    reader cannot serve (no usable index, contig unknown to it): the reads ``BamParser.select_reads`` keeps,
    ``PEextractor``'s pair lengths and ``BamDepth.region_depth`` of the +-SPAN window.  A depth lookup that raises
    gives depth 30, like the reference (tred.py:236-240); a failure to read the reads propagates.
    :return: ingest.LocusEvidence"""
    from .ingest import LocusEvidence
    from .utils import InputParams
    bp = BamParser(InputParams(bam=bam, READLEN=readlen, repo=repo, tredName=tredName, clip=clip, alts=alts))
    sam = read_alignment(bam)
    try:
        reads = bp.select_reads(sam)
    finally:
        sam.close()
    pe = PEextractor(bp)
    ev = LocusEvidence()
    ev.reads, ev.roff = ssw.flatten([r.query_sequence for r in reads])
    ev.names = [r.query_name for r in reads]
    ev.global_lens = np.array(pe.global_lens, dtype=np.int32)
    ev.target_lens = np.array(pe.target_lens, dtype=np.int32)
    ev.n_unmapped = bp.n_unmapped
    try:
        ev.depth = BamDepth(bam, repo.ref, logger).region_depth(bp.chr, max(0, bp.startRepeat - SPAN), bp.endRepeat + SPAN)
    except Exception as e:
        logger.error("Exception on `{}` {} ({}). Set depth={}".format(bam, tredName, e, 30))
        ev.depth = 30
    return ev
