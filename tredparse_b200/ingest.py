"""
Native BAM ingest (``tredsw_bam_*`` in ``include/tredsw.h``, ``csrc/ingest.cpp``): one indexed pass per locus
instead of the reference's three pysam passes — read selection (``tredparse/bam_parser.py:194-243``),
``PEextractor`` (``:316-369``) and ``BamDepth.region_depth`` (``:404-411``) — straight into flat buffers in the
layout ``cohort.CohortBatch`` / ``tredsw_genotype_batch`` consume.  Host code only: no GPU is needed here.

    with BamIngest("sample.bam") as bam:
        ev = bam.extract_locus(repo["HD"], readlen=150)          # reads (codes), pair lengths, depth
        problem = bam.problem(repo["HD"], readlen=150)           # ready for cohort.CohortBatch([...])

A BAM without a usable index is read on the GPU in one pass per sample: ``scan_sample(ctx, BamIngest.unindexed(path),
...)``.  So is a BAM that can be read only once, in order (a pipe, a FIFO, stdin as ``-``): ``scan_sample(ctx,
BamIngest.stream(path), ...)``.
"""
import os
import stat
import ctypes

import numpy as np

from . import _lib
from .meta import TREDsRepo  # noqa: F401  (documentation cross-reference)

SPAN = 1000
FLANKMATCH = 9
DNAPE_ELONGATE = SPAN * 10


class LocusQuery(ctypes.Structure):
    """tredsw_locus_query (include/tredsw.h)"""
    _fields_ = [(n, ctypes.c_int32) for n in ("tid", "repeat_start", "repeat_end", "readlen", "pad", "pe_window",
                                              "flankmatch", "span", "n_alts", "reserved_")] + [("alts", ctypes.c_void_p)]


class LocusSummary(ctypes.Structure):
    """tredsw_locus_summary (include/tredsw.h)"""
    _fields_ = [("nreads", ctypes.c_int32), ("n_unmapped", ctypes.c_int32), ("n_global", ctypes.c_int32),
                ("n_target", ctypes.c_int32), ("nbases", ctypes.c_int64), ("name_bytes", ctypes.c_int64),
                ("depth", ctypes.c_double), ("overflow", ctypes.c_int32), ("reserved_", ctypes.c_int32)]


def _bind(lib):
    if getattr(lib, "_ingest_bound", False):
        return
    lib.tredsw_bam_open.restype = ctypes.c_void_p
    lib.tredsw_bam_open.argtypes = [ctypes.c_char_p, ctypes.c_char_p]
    lib.tredsw_bam_open_unindexed.restype = ctypes.c_void_p
    lib.tredsw_bam_open_unindexed.argtypes = [ctypes.c_char_p]
    lib.tredsw_bam_open_stream.restype = ctypes.c_void_p
    lib.tredsw_bam_open_stream.argtypes = [ctypes.c_char_p]
    lib.tredsw_bam_header_text.restype = ctypes.c_int64
    lib.tredsw_bam_header_text.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int64]
    lib.tredsw_bam_inflate_stats.restype = None
    lib.tredsw_bam_inflate_stats.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]
    lib.tredsw_inflate_raw.restype = ctypes.c_int
    lib.tredsw_inflate_raw.argtypes = [ctypes.c_char_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64]
    lib.tredsw_bam_clone.restype = ctypes.c_void_p
    lib.tredsw_bam_clone.argtypes = [ctypes.c_void_p]
    lib.tredsw_bam_close.restype = None
    lib.tredsw_bam_close.argtypes = [ctypes.c_void_p]
    lib.tredsw_bam_nref.restype = ctypes.c_int32
    lib.tredsw_bam_nref.argtypes = [ctypes.c_void_p]
    lib.tredsw_bam_ref.restype = ctypes.c_int64
    lib.tredsw_bam_ref.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_char_p, ctypes.c_int64]
    lib.tredsw_bam_tid.restype = ctypes.c_int32
    lib.tredsw_bam_tid.argtypes = [ctypes.c_void_p, ctypes.c_char_p]
    lib.tredsw_bam_header_signature.restype = ctypes.c_uint64
    lib.tredsw_bam_header_signature.argtypes = [ctypes.c_void_p]
    lib.tredsw_bam_extract_locus.restype = ctypes.c_int
    lib.tredsw_bam_extract_locus.argtypes = [ctypes.c_void_p, ctypes.POINTER(LocusQuery), ctypes.c_void_p,
                                             ctypes.c_int64, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p,
                                             ctypes.c_int32, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p,
                                             ctypes.c_int64, ctypes.POINTER(LocusSummary)]
    lib.tredsw_bam_region_depth.restype = ctypes.c_int
    lib.tredsw_bam_region_depth.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_int64,
                                            ctypes.POINTER(ctypes.c_double)]
    lib.tredsw_bam_read_length.restype = ctypes.c_int
    lib.tredsw_bam_read_length.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32),
                                           ctypes.POINTER(ctypes.c_int32)]
    lib._ingest_bound = True


def is_stream(path):
    """True when `path` can be read only once, in order: ``-`` (stdin), a FIFO, a character device or a socket."""
    if path == "-":
        return True
    try:
        mode = os.stat(path).st_mode
    except OSError:
        return False
    return stat.S_ISFIFO(mode) or stat.S_ISCHR(mode) or stat.S_ISSOCK(mode)


class LocusEvidence:
    """What one locus of one BAM contributes to the hot path."""
    __slots__ = ("reads", "roff", "names", "global_lens", "target_lens", "depth", "n_unmapped")

    @property
    def nreads(self):
        return len(self.roff) - 1

    _TO_BASES = bytes.maketrans(bytes(range(5)), b"ACGTN")

    def read_string(self, i):
        return self.reads[self.roff[i]:self.roff[i + 1]].tobytes().translate(self._TO_BASES).decode("ascii")

    def read_text(self):
        """all reads as one string of bases (read i = text[roff[i]:roff[i + 1]])"""
        return self.reads.tobytes().translate(self._TO_BASES).decode("ascii")

    def read_strings(self):
        text = self.read_text()
        off = self.roff.tolist()
        return [text[off[i]:off[i + 1]] for i in range(self.nreads)]


class BamIngest:
    def __init__(self, path, index=None):
        self.lib = _lib.load()
        _bind(self.lib)
        self.path = path
        self.handle = self.lib.tredsw_bam_open(path.encode(), index.encode() if index else None)
        if not self.handle:
            raise IOError("tredsw_bam_open({}): {}".format(path, _lib.last_error()))
        self._caps = dict(reads=512, bases=512 * 256, pairs=8192, names=512 * 48)

    @classmethod
    def unindexed(cls, path):
        """A handle on a BAM without a usable index: header, contig ids and read length only (``scan_sample`` reads
        its evidence in one pass over the file; ``extract_locus`` and ``region_depth`` refuse it)."""
        return cls._open_header_only(path, "tredsw_bam_open_unindexed")

    @classmethod
    def stream(cls, path):
        """A handle on a BAM that is read strictly in order, once (``is_stream``; ``-`` is stdin): header, contig ids and
        read length, then ONE ``scan_sample``.  ``clone``, ``extract_locus`` and ``region_depth`` refuse it."""
        return cls._open_header_only(path, "tredsw_bam_open_stream")

    @classmethod
    def _open_header_only(cls, path, opener):
        self = object.__new__(cls)
        self.lib = _lib.load()
        _bind(self.lib)
        self.path = path
        self.handle = getattr(self.lib, opener)(path.encode())
        if not self.handle:
            raise IOError("{}({}): {}".format(opener, path, _lib.last_error()))
        self._caps = dict(reads=512, bases=512 * 256, pairs=8192, names=512 * 48)
        return self

    def references(self):
        """[(contig, length)] of the binary reference dictionary, in tid order (the @SQ text of the header may be absent)"""
        out, buf = [], ctypes.create_string_buffer(8192)                # (the header reader takes names up to 4 KiB)
        for t in range(int(self.lib.tredsw_bam_nref(self.handle))):
            n = int(self.lib.tredsw_bam_ref(self.handle, t, buf, len(buf)))
            out.append((buf.value.decode("latin-1"), n))
        return out

    def header_text(self):
        """the SAM header text (@HD, @SQ, @RG, ... lines)"""
        n = int(self.lib.tredsw_bam_header_text(self.handle, None, 0))
        buf = ctypes.create_string_buffer(n + 1)
        self.lib.tredsw_bam_header_text(self.handle, buf, n + 1)
        return buf.value.decode("utf-8", "replace")

    def read_group_sample(self):
        """the SM field of the header's first @RG line; None when there is none"""
        for line in self.header_text().splitlines():
            if line.startswith("@RG"):
                for field in line.split("\t")[1:]:
                    if field.startswith("SM:"):
                        return field[3:]
                return None
        return None

    def inflate_stats(self):
        """(blocks inflated by the library's own decoder, blocks that fell back to zlib) for this handle."""
        a, b = ctypes.c_int64(), ctypes.c_int64()
        self.lib.tredsw_bam_inflate_stats(self.handle, ctypes.byref(a), ctypes.byref(b))
        return int(a.value), int(b.value)

    def clone(self):
        """An independent handle on the same BAM for another host thread (shares the parsed index)."""
        other = object.__new__(BamIngest)
        other.lib, other.path = self.lib, self.path
        other.handle = self.lib.tredsw_bam_clone(self.handle)
        if not other.handle:
            raise IOError("tredsw_bam_clone({}): {}".format(self.path, _lib.last_error()))
        other._caps = dict(self._caps)
        return other

    def close(self):
        if getattr(self, "handle", None):
            self.lib.tredsw_bam_close(self.handle)
            self.handle = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    _TIDS = {}          # header signature -> {contig: tid}: the samples of a cohort share one reference dictionary

    @property
    def signature(self):
        sig = getattr(self, "_signature", None)
        if sig is None:
            sig = self._signature = int(self.lib.tredsw_bam_header_signature(self.handle))
        return sig

    def tid(self, contig):
        tids = BamIngest._TIDS.setdefault(self.signature, {})
        t = tids.get(contig)
        if t is None:
            t = tids[contig] = int(self.lib.tredsw_bam_tid(self.handle, contig.encode()))
        return t

    def region_depth(self, contig, start, end):
        """``BamDepth.region_depth`` (bam_parser.py:404-411) on the native reader."""
        tid = self.tid(contig)
        if tid < 0:
            raise ValueError("invalid contig `{}`".format(contig))
        d = ctypes.c_double()
        _lib.check(self.lib.tredsw_bam_region_depth(self.handle, tid, int(start), int(end), ctypes.byref(d)),
                   "tredsw_bam_region_depth")
        return float(d.value)

    def read_length(self, firstN=100):
        """``BamReadLen.readlen`` (bam_parser.py:372-391) -> (max, min) over the first firstN + 1 records."""
        mx, mn = ctypes.c_int32(), ctypes.c_int32()
        _lib.check(self.lib.tredsw_bam_read_length(self.handle, int(firstN), ctypes.byref(mx), ctypes.byref(mn)),
                   "tredsw_bam_read_length")
        return int(mx.value), int(mn.value)

    def extract_locus(self, tred, readlen, alts=(), want_names=False, pad=SPAN):
        """alts: iterable of (contig, start, end) mis-mapping regions (``TREDsRepo.get_alts``)."""
        tid = self.tid(tred.chr)
        if tid < 0:
            raise ValueError("invalid contig `{}`".format(tred.chr))
        alt_rows = []
        for (c, s, e) in alts:
            t = self.tid(c)
            if t >= 0:
                alt_rows.append((t, int(s), int(e)))
        alt_arr = np.ascontiguousarray(np.array(alt_rows, dtype=np.int32).reshape(-1, 3))
        q = LocusQuery(tid=tid, repeat_start=tred.repeat_start, repeat_end=tred.repeat_end, readlen=readlen, pad=pad,
                       pe_window=DNAPE_ELONGATE, flankmatch=FLANKMATCH, span=SPAN, n_alts=len(alt_rows),
                       alts=alt_arr.ctypes.data if len(alt_rows) else None)
        summ = LocusSummary()
        while True:
            c = self._caps
            rbuf = np.empty(c["bases"], dtype=np.int8)
            roff = np.zeros(c["reads"] + 1, dtype=np.int64)
            gl = np.empty(c["pairs"], dtype=np.int32)
            tl = np.empty(c["pairs"], dtype=np.int32)
            names = np.empty(c["names"], dtype=np.uint8) if want_names else None
            rc = self.lib.tredsw_bam_extract_locus(
                self.handle, ctypes.byref(q), rbuf.ctypes.data, len(rbuf), roff.ctypes.data, c["reads"],
                gl.ctypes.data, len(gl), tl.ctypes.data, len(tl), names.ctypes.data if want_names else None,
                len(names) if want_names else 0, ctypes.byref(summ))
            _lib.check(rc, "tredsw_bam_extract_locus")
            if not summ.overflow:
                break
            c["reads"] = max(c["reads"], 2 * summ.nreads)
            c["bases"] = max(c["bases"], 2 * int(summ.nbases))
            c["pairs"] = max(c["pairs"], 2 * max(summ.n_global, summ.n_target))
            c["names"] = max(c["names"], 2 * int(summ.name_bytes))
        ev = LocusEvidence()
        ev.reads = rbuf[:summ.nbases].copy()
        ev.roff = roff[:summ.nreads + 1].copy()
        ev.global_lens = gl[:summ.n_global].copy()
        ev.target_lens = tl[:summ.n_target].copy()
        ev.depth = float(summ.depth)
        ev.n_unmapped = int(summ.n_unmapped)
        ev.names = (bytes(names[:summ.name_bytes]).decode("latin-1").split("\0")[:-1] if want_names else None)
        return ev

    def problem(self, tred, readlen, gender="Unknown", alts=(), depth=None):
        """A (sample, locus) problem for ``cohort.CohortBatch`` straight from the BAM."""
        from .simulate import Problem
        ev = self.extract_locus(tred, readlen, alts=alts)
        pr = Problem()
        pr.tred, pr.readlen = tred, readlen
        pr.ploidy = 1 if (gender == "Male" and tred.is_xlinked) else tred.ploidy
        pr.depth = ev.depth if depth is None else depth
        pr.reads, pr.roff = ev.reads, ev.roff
        pr.global_lens, pr.target_lens = ev.global_lens, ev.target_lens
        pr.alleles, pr.names = None, None
        return pr


# ---------------------------------------------------------------------------------------------------------
# Batched ingest on the GPU (csrc/bgzf_gpu.cu): compressed BGZF blocks in, flat cohort buffers out
# ---------------------------------------------------------------------------------------------------------
INGEST_NO_NAMES, INGEST_NO_CRC = 1, 2


class ProblemSpan(ctypes.Structure):
    """tredsw_problem_span (include/tredsw.h)"""
    _fields_ = [(n, ctypes.c_int64) for n in ("read0", "base0", "name0", "off_global", "off_target")]


SUMMARY_DTYPE = np.dtype([("nreads", "<i4"), ("n_unmapped", "<i4"), ("n_global", "<i4"), ("n_target", "<i4"),
                          ("nbases", "<i8"), ("name_bytes", "<i8"), ("depth", "<f8"), ("overflow", "<i4"), ("reserved_", "<i4")])
SPAN_DTYPE = np.dtype([(n, "<i8") for n in ("read0", "base0", "name0", "off_global", "off_target")])
assert SUMMARY_DTYPE.itemsize == ctypes.sizeof(LocusSummary) and SPAN_DTYPE.itemsize == ctypes.sizeof(ProblemSpan)


class IngestView(ctypes.Structure):
    """tredsw_ingest_view (include/tredsw.h)"""
    _fields_ = [("nproblems", ctypes.c_int32), ("nreads", ctypes.c_int32), ("nbases", ctypes.c_int64),
                ("name_bytes", ctypes.c_int64), ("n_pe_lens", ctypes.c_int64),
                ("d_rbuf", ctypes.c_void_p), ("d_roff", ctypes.c_void_p), ("d_read_problem", ctypes.c_void_p),
                ("d_pe_lens", ctypes.c_void_p),
                ("h_rbuf", ctypes.c_void_p), ("h_roff", ctypes.c_void_p), ("h_pe_lens", ctypes.c_void_p),
                ("h_names", ctypes.c_void_p),
                ("summaries", ctypes.POINTER(LocusSummary)), ("spans", ctypes.POINTER(ProblemSpan)),
                ("status", ctypes.POINTER(ctypes.c_int32)),
                ("n_blocks", ctypes.c_int64), ("n_records", ctypes.c_int64), ("comp_bytes", ctypes.c_int64),
                ("inflated_bytes", ctypes.c_int64), ("ms_host_stage", ctypes.c_double), ("ms_total", ctypes.c_double),
                ("ms_marks", ctypes.c_double * 4)]


class IrrParams(ctypes.Structure):
    """tredsw_irr_params (include/tredsw.h): what makes a read an in-repeat read (IRR)"""
    _fields_ = [(n, ctypes.c_int32) for n in ("min_period", "max_period", "purity_num", "purity_den", "min_read_len")]

    def __init__(self, min_period=2, max_period=20, purity_num=9, purity_den=10, min_read_len=50):
        super().__init__(min_period, max_period, purity_num, purity_den, min_read_len)

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


IRR_STATS = ("records_considered", "irr_records", "depth_bases", "max_l_seq", "anchors_without_mq", "unparsed_aux")


class IrrView(ctypes.Structure):
    """tredsw_irr_view (include/tredsw.h)"""
    _fields_ = [("n_entries", ctypes.c_int64), ("entries", ctypes.c_void_p), ("names", ctypes.c_void_p),
                ("name_bytes", ctypes.c_int64)] + [(n, ctypes.c_int64) for n in IRR_STATS]
IRR_ENTRY_DTYPE = np.dtype([("tid", "<i4"), ("pos", "<i4"), ("next_tid", "<i4"), ("next_pos", "<i4"), ("flag", "<i4"),
                            ("mapq", "<i4"), ("mq", "<i4"), ("period", "<i4"), ("motif", "<u8"), ("name_off", "<i8"),
                            ("name_len", "<i4"), ("mate", "<i4")])


def irr_classify_host(codes, params=None):
    """The IRR classifier body run on the host (test hook): codes 0..3 = A C G T, anything else N -> (period, motif);
    period 0: not an IRR."""
    lib = _lib.load()
    _bind_batch(lib)
    a = np.ascontiguousarray(np.asarray(codes, dtype=np.int8))
    per, mot = ctypes.c_int32(), ctypes.c_uint64()
    _lib.check(lib.tredsw_irr_classify_host(a.ctypes.data if len(a) else None, len(a), ctypes.byref(params or IrrParams()),
                                            ctypes.byref(per), ctypes.byref(mot)), "tredsw_irr_classify_host")
    return int(per.value), int(mot.value)


def _bind_batch(lib):
    if getattr(lib, "_ingest_batch_bound", False):
        return
    lib.tredsw_ingest_batch_run.restype = ctypes.c_int
    lib.tredsw_ingest_batch_run.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p,
                                            ctypes.POINTER(LocusQuery), ctypes.c_int32, ctypes.c_uint32,
                                            ctypes.POINTER(ctypes.c_void_p)]
    lib.tredsw_ingest_batch_emulate.restype = ctypes.c_int
    lib.tredsw_ingest_batch_emulate.argtypes = lib.tredsw_ingest_batch_run.argtypes[1:]
    lib.tredsw_ingest_batch_view.restype = ctypes.c_int
    lib.tredsw_ingest_batch_view.argtypes = [ctypes.c_void_p, ctypes.POINTER(IngestView)]
    lib.tredsw_ingest_batch_free.restype = None
    lib.tredsw_ingest_batch_free.argtypes = [ctypes.c_void_p]
    lib.tredsw_ingest_scan_run.restype = ctypes.c_int
    lib.tredsw_ingest_scan_run.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(LocusQuery), ctypes.c_int32,
                                           ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_int64,
                                           ctypes.c_uint32, ctypes.POINTER(ctypes.c_void_p)]
    lib.tredsw_ingest_scan_emulate.restype = ctypes.c_int
    lib.tredsw_ingest_scan_emulate.argtypes = lib.tredsw_ingest_scan_run.argtypes[1:]
    lib.tredsw_ingest_scan_stats.restype = ctypes.c_int
    lib.tredsw_ingest_scan_stats.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    lib.tredsw_inflate_raw_device_code.restype = ctypes.c_int
    lib.tredsw_inflate_raw_device_code.argtypes = [ctypes.c_char_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64]
    lib.tredsw_ingest_scan_run_ex.restype = ctypes.c_int
    lib.tredsw_ingest_scan_run_ex.argtypes = (lib.tredsw_ingest_scan_run.argtypes[:-1] + [ctypes.POINTER(IrrParams)]
                                              + lib.tredsw_ingest_scan_run.argtypes[-1:])
    lib.tredsw_ingest_scan_emulate_ex.restype = ctypes.c_int
    lib.tredsw_ingest_scan_emulate_ex.argtypes = lib.tredsw_ingest_scan_run_ex.argtypes[1:]
    lib.tredsw_ingest_scan_irr.restype = ctypes.c_int
    lib.tredsw_ingest_scan_irr.argtypes = [ctypes.c_void_p, ctypes.POINTER(IrrView)]
    lib.tredsw_irr_classify_host.restype = ctypes.c_int
    lib.tredsw_irr_classify_host.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(IrrParams),
                                             ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_uint64)]
    lib._ingest_batch_bound = True


_QUERIES = {}           # (header signature, locus, readlen, pad, alts) -> (LocusQuery, keep-alive array)


def locus_query(handle, tred, readlen, alts=(), pad=SPAN):
    """(LocusQuery, keep-alive array) of one locus on one open BAM; None when the contig is unknown.  Queries depend
    on the BAM only through its reference dictionary, so they are built once per dictionary."""
    key = (handle.signature, tred.chr, tred.repeat_start, tred.repeat_end, readlen, pad, tuple(alts))
    hit = _QUERIES.get(key)
    if hit is not None:
        return hit if hit else None
    tid = handle.tid(tred.chr)
    if tid < 0:
        _QUERIES[key] = ()
        return None
    rows = [(t, int(s), int(e)) for (t, s, e) in ((handle.tid(c), s, e) for (c, s, e) in alts) if t >= 0]
    arr = np.ascontiguousarray(np.array(rows, dtype=np.int32).reshape(-1, 3))
    q = LocusQuery(tid=tid, repeat_start=tred.repeat_start, repeat_end=tred.repeat_end, readlen=readlen, pad=pad,
                   pe_window=DNAPE_ELONGATE, flankmatch=FLANKMATCH, span=SPAN, n_alts=len(rows),
                   alts=arr.ctypes.data if len(rows) else None)
    if len(_QUERIES) > 100000:
        _QUERIES.clear()
    _QUERIES[key] = (q, arr)
    return q, arr


class IngestBatch:
    """The evidence of many (sample, locus) problems extracted on the GPU in one pass.

        batch = IngestBatch(ctx, handles, sample_of, queries)      # handles: [BamIngest], queries: [LocusQuery]
        batch.status[i] == 0        problem i is good; otherwise read it with BamIngest.extract_locus
        batch.evidence(i)           LocusEvidence (host copies), identical to BamIngest.extract_locus
        batch.view.d_rbuf ...       device buffers in the tredsw_cohort layout (valid until close())

    ``ctx=None`` runs the serial host emulation of the device code — test infrastructure only."""

    def __init__(self, ctx, handles, sample_of, queries, keep=(), want_names=True, check_crc=True):
        self.lib = _lib.load()
        _bind(self.lib)
        _bind_batch(self.lib)
        n = len(queries)
        self._keep = (list(keep), list(handles))
        hs = (ctypes.c_void_p * max(1, len(handles)))(*[h.handle for h in handles])
        so = np.ascontiguousarray(np.asarray(sample_of, dtype=np.int32))
        qs = (LocusQuery * max(1, n))(*queries)
        flags = (0 if want_names else INGEST_NO_NAMES) | (0 if check_crc else INGEST_NO_CRC)
        out = ctypes.c_void_p()
        if ctx is None:
            rc = self.lib.tredsw_ingest_batch_emulate(hs, so.ctypes.data, qs, n, flags, ctypes.byref(out))
        else:
            rc = self.lib.tredsw_ingest_batch_run(ctx.handle, hs, so.ctypes.data, qs, n, flags, ctypes.byref(out))
        _lib.check(rc, "tredsw_ingest_batch_run")
        self._attach(out, n, want_names)

    def _attach(self, out, n, want_names):
        """take over the tredsw_ingest_batch `out` of n problems"""
        self.handle = out
        self.view = IngestView()
        _lib.check(self.lib.tredsw_ingest_batch_view(self.handle, ctypes.byref(self.view)), "tredsw_ingest_batch_view")
        v = self.view
        self.nproblems, self.nreads = int(v.nproblems), int(v.nreads)
        self.status = np.ctypeslib.as_array(v.status, shape=(max(1, n),))[:n].copy() if n else np.zeros(0, np.int32)
        self.summaries = [v.summaries[i] for i in range(n)]
        self.spans = [v.spans[i] for i in range(n)]
        raw = lambda ptr, dt: (np.ctypeslib.as_array(ctypes.cast(ptr, ctypes.POINTER(ctypes.c_uint8)),
                                                      shape=(n * dt.itemsize,)).view(dt).copy() if n else np.zeros(0, dt))
        self.summary_table = raw(v.summaries, SUMMARY_DTYPE)      # the same records as numpy tables
        self.span_table = raw(v.spans, SPAN_DTYPE)
        as_np = lambda ptr, ct, m: (np.ctypeslib.as_array(ctypes.cast(ptr, ctypes.POINTER(ct)), shape=(m,)) if m and ptr
                                    else np.zeros(0, dtype=ct))
        self.h_rbuf = as_np(v.h_rbuf, ctypes.c_int8, int(v.nbases))
        self.h_roff = as_np(v.h_roff, ctypes.c_int64, self.nreads + 1)
        self.h_pe_lens = as_np(v.h_pe_lens, ctypes.c_int32, int(v.n_pe_lens))
        self.h_names = ctypes.string_at(v.h_names, int(v.name_bytes)) if v.h_names and v.name_bytes else b""
        self.want_names = want_names

    def evidence(self, i, copy=True):
        """copy=False: views into the batch's page-locked buffers (valid until close())"""
        s, sp = self.summaries[i], self.spans[i]
        ev = LocusEvidence()
        r0, b0 = int(sp.read0), int(sp.base0)
        own = (lambda a: a.copy()) if copy else (lambda a: a)
        ev.reads = own(self.h_rbuf[b0:b0 + int(s.nbases)])
        ev.roff = (self.h_roff[r0:r0 + s.nreads + 1] - b0).astype(np.int64)
        ev.global_lens = own(self.h_pe_lens[int(sp.off_global):int(sp.off_global) + s.n_global])
        ev.target_lens = own(self.h_pe_lens[int(sp.off_target):int(sp.off_target) + s.n_target])
        ev.depth = float(s.depth)
        ev.n_unmapped = int(s.n_unmapped)
        if self.want_names:
            raw = self.h_names[int(sp.name0):int(sp.name0) + int(s.name_bytes)]
            ev.names = raw.decode("latin-1").split("\0")[:-1]
        else:
            ev.names = None
        return ev

    def stats(self):
        v = self.view
        return {"blocks": int(v.n_blocks), "records": int(v.n_records), "compressed_bytes": int(v.comp_bytes),
                "inflated_bytes": int(v.inflated_bytes), "ms_host_stage": float(v.ms_host_stage),
                "ms_total": float(v.ms_total), "ms_marks": [float(x) for x in v.ms_marks]}

    def close(self):
        if getattr(self, "handle", None):
            self.lib.tredsw_ingest_batch_free(self.handle)
            self.handle = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


SCAN_NSTATS = 10


class ScanBatch(IngestBatch):
    """The evidence of one sample read in ONE pass over a BAM without an index (``tredsw_ingest_scan_run``): an
    ``IngestBatch`` (``.status``, ``.evidence(i)``, the device buffers), plus ``.depths`` (the depth of every
    requested region) and the scan's statistics.  Build it with ``scan_sample``."""

    def __init__(self, ctx, handle, queries, keep=(), depth_regions=(), slab_bytes=None, want_names=True, check_crc=True,
                 irr=None):
        self.lib = _lib.load()
        _bind(self.lib)
        _bind_batch(self.lib)
        n = len(queries)
        self._keep = (list(keep), [handle])
        qs = (LocusQuery * max(1, n))(*queries)
        dr = np.ascontiguousarray(np.array(depth_regions, dtype=np.int32).reshape(-1, 3))
        depths = np.zeros(max(1, len(dr)), dtype=np.float64)
        flags = (0 if want_names else INGEST_NO_NAMES) | (0 if check_crc else INGEST_NO_CRC)
        out = ctypes.c_void_p()
        args = (handle.handle, qs, n, dr.ctypes.data if len(dr) else None, len(dr), depths.ctypes.data,
                int(slab_bytes or 0), flags)
        irr_arg = None if irr is None else ctypes.byref(irr)
        if ctx is None:
            rc = self.lib.tredsw_ingest_scan_emulate_ex(*args, irr_arg, ctypes.byref(out))
        else:
            rc = self.lib.tredsw_ingest_scan_run_ex(ctx.handle, *args, irr_arg, ctypes.byref(out))
        _lib.check(rc, "tredsw_ingest_scan_run")
        self._attach(out, n, want_names)
        self.irr = self._irr() if irr is not None else None
        self.depths = depths[:len(dr)]
        st = np.zeros(SCAN_NSTATS, dtype=np.int64)
        _lib.check(self.lib.tredsw_ingest_scan_stats(self.handle, st.ctypes.data), "tredsw_ingest_scan_stats")
        self.scan_status = int(st[9])
        self._scan = dict(zip(("slabs", "blocks", "records", "repaired_blocks", "compressed_bytes", "inflated_bytes"),
                              (int(x) for x in st[:6])))
        self._scan.update(ms_host_read=st[6] * 1e-3, ms_device=st[7] * 1e-3, ms_total=st[8] * 1e-3)

    def stats(self):
        return dict(self._scan)

    def _irr(self):
        """the STR profile's records: dict(entries = numpy array of IRR_ENTRY_DTYPE in file order, names = their query
        names, stats = the counters of tredsw_irr_view)"""
        v = IrrView()
        _lib.check(self.lib.tredsw_ingest_scan_irr(self.handle, ctypes.byref(v)), "tredsw_ingest_scan_irr")
        n = int(v.n_entries)
        raw = ctypes.string_at(v.entries, n * IRR_ENTRY_DTYPE.itemsize) if n else b""
        ent = np.frombuffer(raw, dtype=IRR_ENTRY_DTYPE).copy()
        text = ctypes.string_at(v.names, int(v.name_bytes)) if v.name_bytes else b""
        names = [text[o:o + k].decode("latin-1") for o, k in zip(ent["name_off"].tolist(), ent["name_len"].tolist())]
        return {"entries": ent, "names": names, "stats": {k: int(getattr(v, k)) for k in IRR_STATS}}


def scan_sample(ctx, handle, queries, keep, depth_regions, slab_bytes=None, irr=None):
    """Every locus of one sample (``queries``: ``LocusQuery`` records, alt regions included) and the depth of
    ``depth_regions`` ((tid, start, end) rows) in one streaming pass over a BAM opened with ``BamIngest.unindexed`` or
    ``BamIngest.stream`` (a stream can be scanned once).
    ``slab_bytes``: compressed bytes read per step (None: 128 MiB).  ``irr``: an ``IrrParams`` to find the in-repeat
    reads of the whole file in the same pass (``ScanBatch.irr``; ``strprofile`` builds the STR profile from them).
    ``ctx=None`` runs the serial host emulation of the device code — test infrastructure only.  -> ScanBatch"""
    return ScanBatch(ctx, handle, queries, keep=keep, depth_regions=depth_regions, slab_bytes=slab_bytes, irr=irr)
