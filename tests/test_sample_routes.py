"""The reader of each sample of ``tred.prepare_chunk``, input kind by input kind, through the host emulation of the
device code (``_lib.default_context`` returns None).  One case per route, with the readers each route may touch
counted: the chunk's GPU ingest batch (``ingest.IngestBatch``), the GPU scan (``ingest.scan_sample``), the host reader
(``tred.ingest_loci``; the Python reader ``extract_locus`` below it), the gender from the chrY depth
(``tred.infer_gender``) and the validity check (``tred.check_bam``).

  input                          GPU ingest  profile  route
  stream (a FIFO)                on          any      stream: one scan; a scan that fails is an error record
  stream                         off         any      none: an error record
  indexed BAM                    on          no       indexed: the chunk's one ingest batch
  indexed BAM                    on          yes      scan on an unindexed handle (that open fails: indexed)
  indexed BAM                    off         any      indexed, read by the host reader
  BAM without an index           on          any      scan (the unindexed open fails: host)
  BAM without an index           off         any      host
  not a BAM (check_bam fails)    any         any      none: gender Unknown / -1, no loci, no error

Every route's evidence equals the host reader's on the indexed original, byte for byte."""
import contextlib
import logging
import os
import shutil
import threading

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
NAMES = ["HD", "FXS"]                   # FXS is X-linked: the gender is inferred
READLEN = 125                           # (not the 150 a failed read-length lookup gives)
READERS = ("IngestBatch", "scan_sample", "irr", "ingest_loci", "infer_gender", "check_bam", "extract_locus")


def _write(path, with_y=True):
    """a male sample: reads at HD and FXS, ~15x over the chrY regions of the gender inference (a header without chrY
    when not `with_y`)"""
    from tredparse_b200 import bamio, simulate
    from tredparse_b200.bam_parser import BamDepth
    from tredparse_b200.meta import TREDsRepo
    sam = bamio.AlignmentFile(os.path.join(GOLDEN, "t001.mini.bam"))
    lengths = dict(zip(sam.references, sam.lengths))
    sam.close()
    refs = [(c, lengths[c]) for c in ("chr4", "chrX") + (("chrY",) if with_y else ())]
    tid = {c: i for i, (c, _) in enumerate(refs)}
    repo, rng = TREDsRepo(), np.random.default_rng(3)
    recs = []
    for li, name in enumerate(NAMES):
        t = repo[name]
        recs += simulate.locus_records(t, tid[t.chr], (20, 31), READLEN, 6.0, seed=li, tag="l{}_".format(li),
                                       flank=1000)
    if with_y:
        for c, a, b in BamDepth.y_regions("hg38"):
            for k, p in enumerate(sorted(rng.integers(a, b - 100, 15 * (b - a) // 100).tolist())):
                seq = "".join("ACGT"[x] for x in rng.integers(0, 4, 100))
                recs.append(bamio.AlignedSegment("y{}_{}".format(a, k), 0, tid[c], p, 60, [(0, 100)], -1, -1, 0, seq))
    bamio.write_bam(path, refs, simulate.coordinate_sort(recs))
    return path


@pytest.fixture(scope="module")
def bams(tmp_path_factory):
    """{"male", "noy": indexed BAMs; "male_noindex": a copy without its index; "junk": a file that is no BAM}"""
    d = tmp_path_factory.mktemp("sample_routes")
    out = {"male": _write(str(d / "male.bam")), "noy": _write(str(d / "noy.bam"), with_y=False)}
    os.makedirs(str(d / "noindex"))
    out["male_noindex"] = str(d / "noindex" / "male.bam")
    shutil.copy(out["male"], out["male_noindex"])
    out["junk"] = str(d / "junk.bam")
    with open(out["junk"], "wb") as fp:
        fp.write(b"not a BAM file\n" * 100)
    return out


def _read(path):
    with open(path, "rb") as fp:
        return fp.read()


@contextlib.contextmanager
def _fifo(path, data):
    """a named pipe at `path` that a thread writes `data` into once a reader opens it"""
    os.mkfifo(path)

    def feed():
        fd = os.open(path, os.O_WRONLY)
        try:
            view, i = memoryview(data), 0
            while i < len(data):
                i += os.write(fd, view[i:i + (1 << 16)])
        except BrokenPipeError:
            pass
        finally:
            os.close(fd)
    t = threading.Thread(target=feed, daemon=True)
    t.start()
    try:
        yield path
    finally:
        if t.is_alive():                            # (never opened: let the writer's open return)
            os.close(os.open(path, os.O_RDONLY | os.O_NONBLOCK))
        t.join(timeout=60)
        os.unlink(path)


def _record(ev):
    return (ev.reads.tobytes(), ev.roff.tobytes(), tuple(ev.names), np.asarray(ev.global_lens).tobytes(),
            np.asarray(ev.target_lens).tobytes(), ev.depth)


@pytest.fixture(scope="module")
def host(bams):
    """(alts) -> {tredName: evidence record} of the host reader on the indexed original"""
    from tredparse_b200 import tred as T
    from tredparse_b200.meta import TREDsRepo
    memo = {}

    def get(alts):
        if alts not in memo:
            evs = T.ingest_loci(bams["male"], TREDsRepo(), NAMES, READLEN, alts, False, logging.getLogger())
            memo[alts] = {t: _record(ev) for t, ev in evs.items()}
        return memo[alts]
    return get


@pytest.fixture
def emulated(monkeypatch):
    """no device: the GPU ingest and the scan run their host emulation (a None context)"""
    from tredparse_b200 import _lib
    monkeypatch.setattr(_lib, "default_context", lambda device=None: None)


@pytest.fixture
def readers(monkeypatch):
    """the calls of every reader a route may touch, counted: {name: calls}; "irr" counts the scans that also find
    in-repeat reads"""
    from tredparse_b200 import tred as T, ingest, bam_parser
    n = dict.fromkeys(READERS, 0)

    def counted(name, real):
        def f(*a, **k):
            n[name] += 1
            if name == "scan_sample" and k.get("irr") is not None:
                n["irr"] += 1
            return real(*a, **k)
        return f
    for mod, name in ((ingest, "IngestBatch"), (ingest, "scan_sample"), (T, "ingest_loci"), (T, "infer_gender"),
                      (T, "check_bam"), (T, "extract_locus"), (bam_parser, "extract_locus")):
        monkeypatch.setattr(mod, name, counted(name, getattr(mod, name)))
    return n


def _calls(**k):
    """the reader counts `readers` must show: k, and 0 for every other reader"""
    return dict(dict.fromkeys(READERS, 0), **k)


def _tasks(paths, names=NAMES, alts=True):
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    return [("s{}".format(i), p, repo, list(names), 300, False, False, alts, True, "INFO") for i, p in enumerate(paths)]


def _prepare(tasks, **kw):
    """prepare_chunk -> (out records, {(sample index, tredName): (readlen, gender, depth, evidence record)}, whether the
    fused call would run on the ingest batch's device buffers)"""
    from tredparse_b200 import tred as T
    _, out, items, where, device_batch = T.prepare_chunk(tasks, **kw)
    ev = {k: (it[1], it[2], it[3], _record(it[4])) for k, it in zip(where, items)}
    if device_batch is not None:
        device_batch.close()
    return out, ev, device_batch is not None


def _assert_evidence(ev, si, want, gender):
    """sample si's items: every locus, with the pre-step fields, and evidence equal to `want`"""
    got = {t: e for (s, t), e in ev.items() if s == si}
    assert sorted(got) == sorted(want)
    for t, (readlen, g, depth, rec) in got.items():
        assert readlen == READLEN and g == gender and depth == rec[-1]
        assert rec == want[t], t


def _assert_male(calls):
    assert calls["inferredGender"] == "Male" and calls["depthY"] > 1 and calls["readLen"] == READLEN


def test_stream_route_reads_each_stream_once_and_nothing_else(bams, host, emulated, readers, tmp_path):
    """streams: the read length from the handle, gender from the scan's chrY regions (Unknown / -1 when the header has
    none), the loci from the same scan (DM1, whose contig the header lacks, gets no call); a stream whose scan fails is
    an error record; no other reader opens them"""
    from tredparse_b200 import tred as T
    data = _read(bams["male"])
    with _fifo(str(tmp_path / "a.bam"), data) as a, _fifo(str(tmp_path / "b.bam"), _read(bams["noy"])) as b, \
            _fifo(str(tmp_path / "c.bam"), data[:len(data) * 2 // 3]) as c:
        tasks = _tasks([a, b, c])
        tasks[1] = _tasks([b], names=NAMES + ["DM1"])[0]
        out, ev, _ = _prepare(tasks, str_profile=[False, False, True])
    assert readers == _calls(scan_sample=3, irr=1)
    _assert_male(out[0]["tredCalls"])
    assert out[1]["tredCalls"] == {"inferredGender": "Unknown", "depthY": -1, "readLen": READLEN}
    _assert_evidence(ev, 0, host(True), "Male")
    _assert_evidence(ev, 1, host(True), "Unknown")
    assert out[2]["tredCalls"] == {} and "status" in out[2]["error"] and not any(s == 2 for s, _ in ev)
    assert all("error" not in o and T.STR_PROFILE not in o for o in out[:2])


def test_stream_without_the_gpu_ingest_is_an_error_record(bams, emulated, readers, tmp_path, monkeypatch):
    from tredparse_b200 import tred as T
    monkeypatch.setattr(T, "GPU_INGEST", False)
    with _fifo(str(tmp_path / "a.bam"), _read(bams["male"])) as a:
        out, ev, _ = _prepare(_tasks([a, bams["male"]]))
    assert readers == _calls(ingest_loci=1, infer_gender=1)           # (the file in the same chunk)
    assert out[0]["tredCalls"] == {} and "TREDSW_GPU_INGEST=0" in out[0]["error"] and not any(s == 0 for s, _ in ev)
    assert "error" not in out[1] and len(ev) == len(NAMES)


def test_indexed_route_one_ingest_batch_for_the_chunk(bams, host, emulated, readers):
    """indexed BAMs: native pre-steps (gender only with an X-linked locus), every locus of every sample from ONE
    ingest batch, whose device buffers the fused call uses"""
    tasks = _tasks([bams["male"]]) + _tasks([bams["male"]], names=["HD"])
    out, ev, handoff = _prepare(tasks)
    assert readers == _calls(IngestBatch=1, infer_gender=2)
    assert handoff
    _assert_male(out[0]["tredCalls"])
    assert out[1]["tredCalls"] == {"inferredGender": "Unknown", "depthY": -1, "readLen": READLEN}
    _assert_evidence(ev, 0, host(True), "Male")
    _assert_evidence(ev, 1, {"HD": host(True)["HD"]}, "Unknown")


def test_indexed_route_with_a_profile_is_one_scan(bams, host, emulated, readers):
    from tredparse_b200 import tred as T
    out, ev, handoff = _prepare(_tasks([bams["male"]]), str_profile=True)
    assert readers == _calls(scan_sample=1, irr=1)
    assert not handoff and out[0][T.STR_PROFILE]["sample"] == "s0"
    _assert_male(out[0]["tredCalls"])
    _assert_evidence(ev, 0, host(True), "Male")


def test_indexed_route_with_a_profile_and_no_unindexed_handle(bams, host, emulated, readers, monkeypatch, caplog):
    """the unindexed open fails: an error says the sample gets no profile, and the indexed route serves its calls"""
    from tredparse_b200 import tred as T, ingest

    def refused(cls, path):
        raise IOError("refused")
    monkeypatch.setattr(ingest.BamIngest, "unindexed", classmethod(refused))
    with caplog.at_level(logging.ERROR, logger="tredparse_b200.tred"):
        out, ev, handoff = _prepare(_tasks([bams["male"]]), str_profile=True)
    assert readers == _calls(IngestBatch=1, infer_gender=1)
    assert handoff and T.STR_PROFILE not in out[0] and "error" not in out[0]
    assert any("`s0`" in r.getMessage() and "no STR profile" in r.getMessage() for r in caplog.records)
    _assert_male(out[0]["tredCalls"])
    _assert_evidence(ev, 0, host(True), "Male")


def test_indexed_route_with_a_profile_whose_scan_raises(bams, host, emulated, readers, monkeypatch, caplog):
    """a scan that raises gives no evidence, no gender and no profile: gender from infer_gender, every locus from the
    host reader"""
    from tredparse_b200 import tred as T, ingest

    def broken(*a, **k):
        raise RuntimeError("broken scan")
    monkeypatch.setattr(ingest, "scan_sample", broken)
    with caplog.at_level(logging.ERROR, logger="tredparse_b200.tred"):
        out, ev, handoff = _prepare(_tasks([bams["male"]]), str_profile=True)
    assert readers == _calls(ingest_loci=1, infer_gender=1)
    assert not handoff and T.STR_PROFILE not in out[0] and "error" not in out[0]
    assert any("`s0`" in r.getMessage() and "no STR profile" in r.getMessage() for r in caplog.records)
    _assert_male(out[0]["tredCalls"])
    _assert_evidence(ev, 0, host(True), "Male")


@pytest.mark.parametrize("profile", [False, True])
def test_indexed_route_without_the_gpu_ingest(bams, host, emulated, readers, monkeypatch, profile):
    from tredparse_b200 import tred as T
    monkeypatch.setattr(T, "GPU_INGEST", False)
    out, ev, handoff = _prepare(_tasks([bams["male"]]), str_profile=profile)
    assert readers == _calls(ingest_loci=1, infer_gender=1)
    assert not handoff and T.STR_PROFILE not in out[0]
    _assert_male(out[0]["tredCalls"])
    _assert_evidence(ev, 0, host(True), "Male")


@pytest.mark.parametrize("profile", [False, True])
def test_unindexed_file_scan_route(bams, host, emulated, readers, profile):
    """a BAM without an index: checked, then one scan serves the loci and gender (and the profile when wanted)"""
    from tredparse_b200 import tred as T
    out, ev, handoff = _prepare(_tasks([bams["male_noindex"]]), str_profile=profile)
    assert readers == _calls(check_bam=1, scan_sample=1, irr=int(profile))
    assert not handoff and (T.STR_PROFILE in out[0]) == profile
    _assert_male(out[0]["tredCalls"])
    _assert_evidence(ev, 0, host(True), "Male")


@pytest.mark.parametrize("why", ["gpu_ingest_off", "unindexed_open_fails"])
def test_unindexed_file_host_route(bams, host, emulated, readers, monkeypatch, why):
    """a BAM without an index that the GPU scan cannot take: the Python readers serve pre-steps and loci"""
    from tredparse_b200 import tred as T, ingest
    if why == "gpu_ingest_off":
        monkeypatch.setattr(T, "GPU_INGEST", False)
    else:
        def refused(cls, path):
            raise IOError("refused")
        monkeypatch.setattr(ingest.BamIngest, "unindexed", classmethod(refused))
    out, ev, handoff = _prepare(_tasks([bams["male_noindex"]], alts=False), str_profile=True)
    assert readers == _calls(check_bam=1, ingest_loci=1, infer_gender=1, extract_locus=len(NAMES))
    assert not handoff and T.STR_PROFILE not in out[0] and "error" not in out[0]
    _assert_male(out[0]["tredCalls"])
    _assert_evidence(ev, 0, host(False), "Male")


@pytest.mark.parametrize("gpu_ingest", [True, False])
def test_file_check_bam_refuses_has_no_route_and_no_error(bams, emulated, readers, monkeypatch, gpu_ingest):
    from tredparse_b200 import tred as T
    monkeypatch.setattr(T, "GPU_INGEST", gpu_ingest)
    out, ev, handoff = _prepare(_tasks([bams["junk"]]), str_profile=True)
    assert readers == _calls(check_bam=1)
    assert out[0]["tredCalls"] == {"inferredGender": "Unknown", "depthY": -1} and "error" not in out[0]
    assert ev == {} and not handoff and T.STR_PROFILE not in out[0]
