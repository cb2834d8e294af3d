"""
ctypes binding of ``libtredsw.so`` (C ABI declared in ``include/tredsw.h``).

This is the *only* compute back end of the package: there is no CPU path.  If the shared library has
not been built (``python -c "import __graft_entry__ as g; g.build()"`` or
``python -m tredparse_b200.build``), or no CUDA device is usable, the first call raises
:class:`TredswError`.
"""
import ctypes
import os
import threading

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libtredsw.so")

DEVICE_PTRS, SCORE2, NO_BEGIN, CIGAR, FORCE_WORD = 1, 2, 4, 8, 16
DEVICE_INPUTS = 64      # tredsw_genotype_batch: bulk evidence in device memory, problems + outputs on the host

TAG_NAMES = {0: None, 1: "FULL", 2: "PREF", 3: "POST", 4: "REPT", 5: "HANG"}

EXPORTS = [
    # libssw.so drop-in
    "ssw_init", "init_destroy", "ssw_align", "align_destroy", "cigar_int_to_op", "cigar_int_to_len",
    # batched API
    "tredsw_version", "tredsw_device_count", "tredsw_last_error", "tredsw_create", "tredsw_destroy",
    "tredsw_synchronize", "tredsw_sm_count", "tredsw_launch_count", "tredsw_strip_skip_stats", "tredsw_enable_timing",
    "tredsw_get_timing", "tredsw_get_timeline", "tredsw_int_pipe_peak", "tredsw_align_pairs", "tredsw_classify_reads",
    "tredsw_likelihood_grid", "tredsw_pe_kde", "tredsw_genotype_batch", "tredsw_genotype_batch_ex", "tredsw_pack_reads4", "tredsw_narrow_i16",
    # native BAM ingest
    "tredsw_bam_open", "tredsw_bam_close", "tredsw_bam_nref", "tredsw_bam_tid", "tredsw_bam_extract_locus",
    "tredsw_bam_region_depth", "tredsw_bam_read_length", "tredsw_bam_clone", "tredsw_bam_inflate_stats", "tredsw_inflate_raw",
    "tredsw_bam_header_signature", "tredsw_bam_ref",
    # BAM ingest on the GPU (batched); *_emulate / *_device_code run the device code on the host for the CPU tests
    "tredsw_ingest_batch_run", "tredsw_ingest_batch_view", "tredsw_ingest_batch_free", "tredsw_ingest_batch_emulate",
    "tredsw_inflate_raw_device_code",
    # BAMs without an index: one streaming pass per sample
    "tredsw_bam_open_unindexed", "tredsw_ingest_scan_run", "tredsw_ingest_scan_emulate", "tredsw_ingest_scan_stats",
    "tredsw_bam_open_stream", "tredsw_bam_header_text",
    # the STR profile of a scan (in-repeat reads)
    "tredsw_ingest_scan_run_ex", "tredsw_ingest_scan_emulate_ex", "tredsw_ingest_scan_irr", "tredsw_irr_classify_host",
    # the reference tract scan (alt regions of discovered loci); *_emulate runs the device code on the host
    "tredsw_ref_tracts", "tredsw_ref_tracts_emulate", "tredsw_ref_tracts_view", "tredsw_ref_tracts_free",
    "tredsw_ref_tracts_ex", "tredsw_ref_tracts_emulate_ex",
]


class TredswError(RuntimeError):
    pass


class Family(ctypes.Structure):
    """tredsw_family (include/tredsw.h)"""
    _fields_ = [("prefix", ctypes.c_int8 * 32), ("suffix", ctypes.c_int8 * 32),
                ("repeat", ctypes.c_int8 * 32), ("prefix_len", ctypes.c_int32),
                ("suffix_len", ctypes.c_int32), ("period", ctypes.c_int32),
                ("max_units", ctypes.c_int32), ("clip", ctypes.c_int32),
                ("reserved", ctypes.c_int32 * 3)]


class GridProblem(ctypes.Structure):
    """tredsw_grid_problem (include/tredsw.h)"""
    _fields_ = [(n, ctypes.c_int32) for n in (
        "period", "readlen", "ploidy", "n_rept", "max_partial", "run_pe", "pe_ref", "pe_minpe",
        "n_span", "n_part", "n_target", "n_h1", "n_h2", "expansion", "recessive", "cutoff_risk")] + \
        [(n, ctypes.c_double) for n in ("half_depth", "stutter_a", "stutter_w2", "stutter_c3", "stutter_c4")] + \
        [(n, ctypes.c_int64) for n in ("off_span", "off_part", "off_target", "off_h1", "off_h2",
                                       "off_pdf", "off_step", "off_surface", "off_ph1", "off_ph2")]


class GridResult(ctypes.Structure):
    """tredsw_grid_result (include/tredsw.h)"""
    _fields_ = [("max_ml", ctypes.c_double), ("sum_all", ctypes.c_double), ("sum_path", ctypes.c_double),
                ("arg_i1", ctypes.c_int32), ("arg_i2", ctypes.c_int32), ("n_points", ctypes.c_int32),
                ("pad", ctypes.c_int32), ("sum_uniq", ctypes.c_double)]


GRID_PROBLEM_DTYPE = np.dtype(
    [(n, "<i4") for n in ("period", "readlen", "ploidy", "n_rept", "max_partial", "run_pe", "pe_ref",
                          "pe_minpe", "n_span", "n_part", "n_target", "n_h1", "n_h2", "expansion",
                          "recessive", "cutoff_risk")] +
    [(n, "<f8") for n in ("half_depth", "stutter_a", "stutter_w2", "stutter_c3", "stutter_c4")] +
    [(n, "<i8") for n in ("off_span", "off_part", "off_target", "off_h1", "off_h2", "off_pdf",
                          "off_step", "off_surface", "off_ph1", "off_ph2")])
GRID_RESULT_DTYPE = np.dtype([("max_ml", "<f8"), ("sum_all", "<f8"), ("sum_path", "<f8"),
                              ("arg_i1", "<i4"), ("arg_i2", "<i4"), ("n_points", "<i4"), ("pad", "<i4"),
                              ("sum_uniq", "<f8")])
POSTERIOR_DTYPE = np.dtype([("problem", "<i4"), ("kind", "<i4"), ("a", "<i4"), ("b", "<i4"), ("p", "<f8")])
POST_H1, POST_H2, POST_JOINT, POST_JOINT_TOTAL = 1, 2, 3, 4
FAMILY_DTYPE = np.dtype([("prefix", "i1", 32), ("suffix", "i1", 32), ("repeat", "i1", 32),
                         ("prefix_len", "<i4"), ("suffix_len", "<i4"), ("period", "<i4"),
                         ("max_units", "<i4"), ("clip", "<i4"), ("reserved", "<i4", 3)])
FAI_ENTRY_DTYPE = np.dtype([("length", "<i8"), ("offset", "<i8"), ("line_bases", "<i4"), ("line_width", "<i4")])
MOTIF_DTYPE = np.dtype([("period", "<i4"), ("reserved", "<i4"), ("code", "<u8")])
TRACT_DTYPE = np.dtype([("start", "<i8"), ("length", "<i8"), ("code", "<u8"), ("contig", "<i4"), ("period", "<i4")])


class TractParams(ctypes.Structure):
    """tredsw_tract_params (include/tredsw.h)"""
    _fields_ = [("min_units", ctypes.c_int32), ("min_len", ctypes.c_int32), ("step_bytes", ctypes.c_int64)]


class TractChain(ctypes.Structure):
    """tredsw_tract_chain (include/tredsw.h)"""
    _fields_ = [("max_interrupt", ctypes.c_int32), ("purity_num", ctypes.c_int32), ("purity_den", ctypes.c_int32),
                ("reserved_", ctypes.c_int32)]


class TractsView(ctypes.Structure):
    """tredsw_tracts_view (include/tredsw.h)"""
    _fields_ = [("n_tracts", ctypes.c_int64), ("tracts", ctypes.c_void_p), ("steps", ctypes.c_int64),
                ("bytes", ctypes.c_int64), ("bases", ctypes.c_int64), ("invalid_bases", ctypes.c_int64),
                ("step_read_ms", ctypes.POINTER(ctypes.c_double)), ("step_device_ms", ctypes.POINTER(ctypes.c_double)),
                ("ms_total", ctypes.c_double), ("comp_bytes", ctypes.c_int64), ("blocks", ctypes.c_int64),
                ("segments", ctypes.POINTER(ctypes.c_int32))]


assert GRID_PROBLEM_DTYPE.itemsize == ctypes.sizeof(GridProblem)
assert GRID_RESULT_DTYPE.itemsize == ctypes.sizeof(GridResult)
assert FAMILY_DTYPE.itemsize == ctypes.sizeof(Family)

_lib = None
_lock = threading.Lock()

_vp = ctypes.c_void_p


def load():
    """Load libtredsw.so (no GPU needed for loading) and declare prototypes."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise TredswError(
                "{} is missing: build it with `python -m tredparse_b200.build` (needs nvcc). "
                "tredparse_b200 has no CPU fallback.".format(LIB_PATH))
        lib = ctypes.CDLL(LIB_PATH)
        lib.tredsw_version.restype = ctypes.c_int
        lib.tredsw_device_count.restype = ctypes.c_int
        lib.tredsw_last_error.restype = ctypes.c_char_p
        lib.tredsw_create.restype = _vp
        lib.tredsw_create.argtypes = [ctypes.c_int, _vp]
        lib.tredsw_destroy.restype = None
        lib.tredsw_destroy.argtypes = [_vp]
        lib.tredsw_synchronize.argtypes = [_vp]
        lib.tredsw_sm_count.argtypes = [_vp]
        lib.tredsw_launch_count.restype = ctypes.c_int64
        lib.tredsw_launch_count.argtypes = [_vp]
        lib.tredsw_strip_skip_stats.restype = ctypes.c_int
        lib.tredsw_strip_skip_stats.argtypes = [_vp, _vp]
        lib.tredsw_enable_timing.argtypes = [_vp, ctypes.c_int]
        lib.tredsw_get_timing.argtypes = [_vp, _vp]
        lib.tredsw_get_timeline.argtypes = [_vp, _vp]
        lib.tredsw_int_pipe_peak.argtypes = [_vp, _vp]
        lib.tredsw_align_pairs.restype = ctypes.c_int
        lib.tredsw_align_pairs.argtypes = [_vp, _vp, _vp, ctypes.c_int32, _vp, _vp, ctypes.c_int32, _vp,
                                           _vp, ctypes.c_int64, _vp, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_uint32, _vp, _vp, ctypes.c_int32]
        lib.tredsw_classify_reads.restype = ctypes.c_int
        lib.tredsw_classify_reads.argtypes = [_vp, _vp, _vp, ctypes.c_int32, _vp, _vp, ctypes.c_int32,
                                              _vp, ctypes.c_int, ctypes.c_int, ctypes.c_uint32, _vp, _vp]
        lib.tredsw_likelihood_grid.restype = ctypes.c_int
        lib.tredsw_likelihood_grid.argtypes = [_vp, _vp, ctypes.c_int32, _vp, ctypes.c_int64, _vp,
                                               ctypes.c_int64, _vp, ctypes.c_int64, _vp, ctypes.c_int64,
                                               _vp, ctypes.c_uint32]
        lib.tredsw_pe_kde.restype = ctypes.c_int
        lib.tredsw_pe_kde.argtypes = [_vp, _vp, _vp, ctypes.c_int32, _vp, ctypes.c_uint32]
        lib.tredsw_pack_reads4.restype = ctypes.c_int
        lib.tredsw_pack_reads4.argtypes = [_vp, ctypes.c_int64, _vp, ctypes.c_int]
        lib.tredsw_narrow_i16.restype = ctypes.c_int
        lib.tredsw_narrow_i16.argtypes = [_vp, ctypes.c_int64, _vp, ctypes.c_int]
        for f in (lib.tredsw_ref_tracts, lib.tredsw_ref_tracts_emulate):
            f.restype = ctypes.c_int
            f.argtypes = [_vp, ctypes.c_char_p, _vp, ctypes.c_int32, _vp, ctypes.c_int32,
                          ctypes.POINTER(TractParams), ctypes.POINTER(_vp)]
        for f in (lib.tredsw_ref_tracts_ex, lib.tredsw_ref_tracts_emulate_ex):
            f.restype = ctypes.c_int
            f.argtypes = [_vp, ctypes.c_char_p, _vp, ctypes.c_int32, _vp, ctypes.c_int32,
                          ctypes.POINTER(TractParams), ctypes.POINTER(TractChain), ctypes.POINTER(_vp)]
        lib.tredsw_ref_tracts_view.restype = ctypes.c_int
        lib.tredsw_ref_tracts_view.argtypes = [_vp, ctypes.POINTER(TractsView)]
        lib.tredsw_ref_tracts_free.restype = None
        lib.tredsw_ref_tracts_free.argtypes = [_vp]
        _lib = lib
        return lib


def last_error():
    return load().tredsw_last_error().decode("utf-8", "replace")


def check(rc, what):
    if rc != 0:
        raise TredswError("{} failed (code {}): {}".format(what, rc, last_error()))


def ref_tracts(path, contigs, motifs, min_units, min_len, step_bytes=0, ctx=None, emulate=False, max_interrupt=0,
               purity_num=9, purity_den=10):
    """Every tract of `motifs` in the FASTA at `path`, plain text or BGZF (tredsw_ref_tracts, DESIGN §4.5).  contigs:
    FAI_ENTRY_DTYPE rows in FASTA order; motifs: (period, canonical code) pairs.  -> (TRACT_DTYPE array by (contig,
    start, period), stats dict; its comp_bytes and blocks are 0 for a text file, and its segments the int32 array of
    each tract's chain segments).  ``max_interrupt`` >= 1 joins pure tracts across interruptions of up to that many
    bases when the chain has purity purity_num / purity_den (tredsw_ref_tracts_ex, DESIGN §4.5.1); 0 is the pure rule.
    ``ctx``: a Context (default the process's); ``emulate`` runs the serial host emulation of the device code
    instead — test infrastructure only.  Raises TredswError (no device, I/O, an index that does not fit the file,
    chain parameters out of range)."""
    lib = load()
    cs = np.ascontiguousarray(contigs, dtype=FAI_ENTRY_DTYPE)
    ms = np.zeros(len(motifs), dtype=MOTIF_DTYPE)
    for i, (k, code) in enumerate(motifs):
        ms[i]["period"], ms[i]["code"] = k, code
    prm = TractParams(int(min_units), int(min_len), int(step_bytes))
    chain = TractChain(int(max_interrupt), int(purity_num), int(purity_den), 0)
    res = ctypes.c_void_p()
    if emulate:
        rc = lib.tredsw_ref_tracts_emulate_ex(None, path.encode(), ptr(cs), len(cs), ptr(ms), len(ms),
                                              ctypes.byref(prm), ctypes.byref(chain), ctypes.byref(res))
    else:
        handle = (ctx or default_context()).handle
        rc = lib.tredsw_ref_tracts_ex(handle, path.encode(), ptr(cs), len(cs), ptr(ms), len(ms), ctypes.byref(prm),
                                      ctypes.byref(chain), ctypes.byref(res))
    check(rc, "tredsw_ref_tracts")
    try:
        v = TractsView()
        check(lib.tredsw_ref_tracts_view(res, ctypes.byref(v)), "tredsw_ref_tracts_view")
        n = int(v.n_tracts)
        tracts = np.zeros(n, dtype=TRACT_DTYPE)
        segments = np.zeros(n, dtype=np.int32)
        if n:
            ctypes.memmove(tracts.ctypes.data, v.tracts, n * TRACT_DTYPE.itemsize)
            ctypes.memmove(segments.ctypes.data, v.segments, n * 4)
        stats = {"steps": int(v.steps), "bytes": int(v.bytes), "bases": int(v.bases),
                 "invalid_bases": int(v.invalid_bases), "tracts": n, "ms_total": float(v.ms_total),
                 "step_read_ms": [float(v.step_read_ms[i]) for i in range(v.steps)],
                 "step_device_ms": [float(v.step_device_ms[i]) for i in range(v.steps)],
                 "comp_bytes": int(v.comp_bytes), "blocks": int(v.blocks), "segments": segments}
    finally:
        lib.tredsw_ref_tracts_free(res)
    return tracts, stats


def ptr(a):
    """host numpy array -> void*  |  int (device pointer) -> void*  |  None"""
    if a is None:
        return None
    if isinstance(a, (int, np.integer)):
        return ctypes.c_void_p(int(a))
    assert a.flags["C_CONTIGUOUS"]
    return ctypes.c_void_p(a.ctypes.data)


class Context:
    """One tredsw context: a device, a stream and grow-only staging buffers.  Not thread-safe across
    threads by design of the workload (one host thread / process per GPU)."""

    def __init__(self, device=0, stream=None):
        lib = load()
        if lib.tredsw_device_count() <= 0:
            raise TredswError("no CUDA device visible: tredparse_b200 computes on the GPU only "
                              "(there is no CPU fallback)")
        self.lib = lib
        self.device = device
        self.handle = lib.tredsw_create(device, ctypes.c_void_p(stream) if stream else None)
        if not self.handle:
            raise TredswError("tredsw_create({}) failed: {}".format(device, last_error()))

    def close(self):
        if getattr(self, "handle", None):
            self.lib.tredsw_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def sm_count(self):
        return self.lib.tredsw_sm_count(self.handle)

    def synchronize(self):
        check(self.lib.tredsw_synchronize(self.handle), "tredsw_synchronize")

    @property
    def launches(self):
        return int(self.lib.tredsw_launch_count(self.handle))

    def strip_skip_stats(self):
        """Main strips of the packed family kernel skipped at the fixed point of their boundary column, summed over
        this context's calls so far: dict(cells_skipped, by_period={p: dict(planned, skipped, items, items_no_skip,
        lane_planned, lane_skipped, lane_skippable)}) for the loop instantiation periods p that ran
        (tredsw_strip_skip_stats).  The lane_ counters sum over the lanes holding a read: planned strips, strips their
        warp skipped, and strips the lane could skip on its own — lane_skippable / lane_planned bounds
        lane_skipped / lane_planned whatever the order of the reads."""
        a = np.zeros(85, dtype=np.int64)
        check(self.lib.tredsw_strip_skip_stats(self.handle, ptr(a)), "tredsw_strip_skip_stats")
        per = a[1:49].reshape(12, 4)
        lanes = a[49:85].reshape(12, 3)
        return {"cells_skipped": int(a[0]),
                "by_period": {p + 1: dict(zip(("planned", "skipped", "items", "items_no_skip", "lane_planned",
                                               "lane_skipped", "lane_skippable"), map(int, (*per[p], *lanes[p]))))
                              for p in range(12) if per[p, 2]}}

    def enable_timing(self, on=True):
        check(self.lib.tredsw_enable_timing(self.handle, int(on)), "tredsw_enable_timing")

    def timing(self):
        """Device ms of the last call's stages: dict(sw, grid, kde, total)."""
        ms = (ctypes.c_float * 4)()
        check(self.lib.tredsw_get_timing(self.handle, ms), "tredsw_get_timing")
        return {"sw": ms[0], "grid": ms[1], "kde": ms[2], "total": ms[3]}

    def timeline(self):
        """Device timestamps (ms since a process-wide reference) of the last timed call: dict of marks."""
        ms = (ctypes.c_float * 10)()
        check(self.lib.tredsw_get_timeline(self.handle, ms), "tredsw_get_timeline")
        names = ("sw0", "sw1", "grid0", "grid1", "kde0", "kde1", "inputs", "final", "start", "copied")
        return {n: ms[i] for i, n in enumerate(names)}

    def int_pipe_peak(self):
        """Measured packed-DPX instruction throughput, giga lane-instructions / s."""
        v = ctypes.c_double(0)
        check(self.lib.tredsw_int_pipe_peak(self.handle, ctypes.byref(v)), "tredsw_int_pipe_peak")
        return v.value


_default = {}


def default_context(device=None):
    """Process-wide context per device (device defaults to $TREDSW_DEVICE, $LOCAL_RANK or 0)."""
    if device is None:
        device = int(os.environ.get("TREDSW_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    with _lock:
        ctx = _default.get(device)
    if ctx is None:
        ctx = Context(device)
        with _lock:
            _default[device] = ctx
    return ctx
