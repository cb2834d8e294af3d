"""A BAM read strictly in order, once (tredsw_bam_open_stream: a pipe, a FIFO, stdin as `-`): the handle parses the header
and the first records from the bytes it has read, and the scan (tredsw_ingest_scan_run, csrc/bgzf_gpu.cu run_scan) reads
the rest with read() slab by slab.

The streams here are real pipes and FIFOs written by a thread in irregular pieces (1, 7 and 4093 bytes and random sizes),
so that read() returns short counts.  Every case compares the stream's scan with the scan of the same file
(tredsw_bam_open_unindexed) and with the host reader on the indexed file, field for field.  CPU tests run the device
code serially on the host (tredsw_ingest_scan_emulate); the `gpu` tests run the kernels and the CLI."""
import contextlib
import gzip
import json
import os
import random
import struct
import subprocess
import sys
import threading

import numpy as np
import pytest

from test_ingest_scan import (MINIS, ROOT, SLAB_TINY, _fooling_quality, _queries, _records, _rewrite, _same, _sample,
                              ctypes_depth, ybams)  # noqa: F401  (ybams: the chrY fixture BAMs)


@pytest.fixture(scope="module")
def repo():
    from tredparse_b200.meta import TREDsRepo
    return TREDsRepo()


def _write_irregularly(fd, data, seed):
    """write `data` to fd in pieces of 1, 7, 4093 and random sizes; close fd"""
    rng = random.Random(seed)
    view = memoryview(data)
    i = 0
    try:
        while i < len(data):
            n = rng.choice([1, 7, 4093, rng.randrange(1, 1 << 17)])
            i += os.write(fd, view[i:i + n])
    except BrokenPipeError:
        pass                                # the reader stopped early (a failed scan): the rest is not wanted
    finally:
        os.close(fd)


@contextlib.contextmanager
def piped(data, seed=0):
    """a path that reads `data` through a pipe fed by a thread (the read end as /dev/fd/N: a FIFO to stat)"""
    r, w = os.pipe()
    t = threading.Thread(target=_write_irregularly, args=(w, bytes(data), seed), daemon=True)
    t.start()
    try:
        yield "/dev/fd/{}".format(r)
    finally:
        os.close(r)                        # (a writer still blocked gets EPIPE)
        t.join(timeout=60)


@contextlib.contextmanager
def fifo(path, data, seed=0):
    """a named pipe at `path` that a thread writes `data` into once a reader opens it"""
    os.mkfifo(path)

    def feed():
        try:
            fd = os.open(path, os.O_WRONLY)
        except OSError:
            return
        _write_irregularly(fd, bytes(data), seed)
    t = threading.Thread(target=feed, daemon=True)
    t.start()
    try:
        yield path
    finally:
        if t.is_alive():                   # nobody opened it: a reader that opens and closes it releases the writer
            try:
                os.close(os.open(path, os.O_RDONLY | os.O_NONBLOCK))
            except OSError:
                pass
        t.join(timeout=60)
        os.unlink(path)


def _read(path):
    with open(path, "rb") as fp:
        return fp.read()


def _readlen(h, first_n=100):
    """(max, min) read length, or the error (a file without records has none)"""
    from tredparse_b200 import _lib
    try:
        return h.read_length(first_n)
    except _lib.TredswError as e:
        return str(e)


def _stream_check(ctx, indexed, repo, names, readlen=150, slab_bytes=None, depth_regions=(), seed=0):
    """stream the bytes of `indexed` through a pipe and scan them: every locus and depth region equals the scan of the
    same file and the host reader on `indexed`; the read length equals the file handle's.  -> (stats, reads in total)"""
    from tredparse_b200 import ingest
    ref, un = ingest.BamIngest(indexed), ingest.BamIngest.unindexed(indexed)
    try:
        with piped(_read(indexed), seed) as path:
            with ingest.BamIngest.stream(path) as st:
                assert st.signature == un.signature and st.tid("chr4") == un.tid("chr4")
                assert _readlen(st) == _readlen(un) and _readlen(st, 7) == _readlen(un, 7)
                qs, keep, key = _queries(st, repo, names, readlen)
                with ingest.scan_sample(ctx, st, qs, keep, depth_regions, slab_bytes=slab_bytes) as b, \
                        ingest.scan_sample(ctx, un, qs, keep, depth_regions, slab_bytes=slab_bytes) as f:
                    assert b.scan_status == 0 and f.scan_status == 0 and not b.status.any()
                    total = 0
                    for i, n in enumerate(key):
                        ev = b.evidence(i)
                        assert _same(ev, f.evidence(i)), (indexed, n, readlen, slab_bytes)
                        assert _same(ev, ref.extract_locus(repo[n], readlen, alts=repo[n].alt, want_names=True))
                        total += ev.nreads
                    for (c, s, e), d, d_file in zip(depth_regions, b.depths, f.depths):
                        assert d == d_file == ctypes_depth(ref, c, s, e), ((c, s, e), d, d_file)
                    sb, sf = b.stats(), f.stats()
                    for k in ("blocks", "records", "repaired_blocks", "compressed_bytes", "inflated_bytes"):
                        assert sb[k] == sf[k], (k, sb, sf)
                    return sb, total
    finally:
        ref.close()
        un.close()


def _level0(tmp_path, src):
    """a copy of `src` made of stored DEFLATE blocks (what `samtools view -u` writes), with its index"""
    refs, recs = _records(src)
    from tredparse_b200 import bamio
    dst = str(tmp_path / ("u_" + os.path.basename(src)))
    bamio.write_bam(dst, refs, recs, level=0)
    return dst


def _blocks(data):
    """(compressed end, inflated end) of every BGZF block of a file"""
    out, off, u = [], 0, 0
    while off < len(data):
        bsize = struct.unpack_from("<H", data, off + 16)[0] + 1
        u += struct.unpack_from("<I", data, off + bsize - 4)[0]
        off += bsize
        out.append((off, u))
    return out


def _record_starts(data):
    """inflated offsets of every record start of a BAM (and the end of the last record)"""
    raw = gzip.decompress(bytes(data))
    l_text = struct.unpack_from("<i", raw, 4)[0]
    o = 8 + l_text
    n_ref = struct.unpack_from("<i", raw, o)[0]
    o += 4
    for _ in range(n_ref):
        o += 8 + struct.unpack_from("<i", raw, o)[0]
    starts = set()
    while o < len(raw):
        starts.add(o)
        o += 4 + struct.unpack_from("<i", raw, o)[0]
    starts.add(o)
    return starts


# ---- the cases, run through the emulation (ctx None) and on the GPU (ctx a context) -----------------------------------
def _fixtures_case(ctx, repo, tmp_path):
    for k, src in enumerate(MINIS):
        _, recs = _records(src)
        for readlen in (150, 101):
            for slab in (None, SLAB_TINY):
                st, total = _stream_check(ctx, src, repo, repo.names, readlen, slab, seed=k)
                assert total > 50 and st["records"] == len(recs)
                assert st["slabs"] == 1 if slab is None else st["slabs"] >= 3
        st, total = _stream_check(ctx, _level0(tmp_path, src), repo, repo.names, 150, SLAB_TINY, seed=k)
        assert total > 50 and st["records"] == len(recs) and st["slabs"] > 10


def _synthetic_case(ctx, repo, tmp_path, names):
    for readlen in (150, 251):
        src = _sample(str(tmp_path / "s{}.bam".format(readlen)), repo, names, 3, 11, readlen)
        st, total = _stream_check(ctx, src, repo, names, readlen, SLAB_TINY, seed=readlen)
        assert total > 200 and st["slabs"] > 2
    st, total = _stream_check(ctx, _level0(tmp_path, src), repo, names, 251, SLAB_TINY, seed=3)
    assert total > 200 and st["slabs"] > 10


def _adversarial_case(ctx, repo, tmp_path):
    from tredparse_b200 import bamio
    refs, recs = _records(MINIS[0])
    fooled = [r for r in recs]
    for r in fooled:
        r._qual = _fooling_quality(r)
    st, total = _stream_check(ctx, _rewrite(str(tmp_path / "fooled.bam"), refs, fooled), repo, repo.names, 150, SLAB_TINY)
    assert st["repaired_blocks"] > 0 and total > 50
    refs, recs = _records(MINIS[0])
    hd = repo["HD"]
    tid = [n for n, _ in refs].index(hd.chr)
    big = bamio.AlignedSegment("big", 0, tid, hd.repeat_start - 100, 60, [(0, 60000)], -1, -1, 0, "ACGT" * 15000)
    import bisect
    at = bisect.bisect_right([(r.reference_id if r.reference_id >= 0 else 1 << 30, r.reference_start) for r in recs],
                             (tid, big.reference_start))
    src = _rewrite(str(tmp_path / "big.bam"), refs, recs[:at] + [big] + recs[at:])
    for slab in (None, SLAB_TINY):
        st, total = _stream_check(ctx, src, repo, ["HD", "DM1"], 150, slab)
        assert st["records"] == len(recs) + 1
    st, total = _stream_check(ctx, _rewrite(str(tmp_path / "header_only.bam"), refs, []), repo, ["HD", "FXS"], 150)
    assert st["records"] == 0 and total == 0


def _depth_case(ctx, repo, tmp_path, ybams):
    """the chrY depths, depthY and gender of a stream equal the file handle's"""
    from tredparse_b200 import ingest
    from tredparse_b200.bam_parser import BamDepth
    with ingest.BamIngest(MINIS[0]) as h:
        t4, tx, ty = h.tid("chr4"), h.tid("chrX"), h.tid("chrY")
    regions = [(t4, 3074000, 3076000), (t4, 0, 10), (tx, 147911000, 147913000), (ty, 2784557, 2791188)]
    _stream_check(ctx, MINIS[0], repo, ["HD"], 150, SLAB_TINY, regions)
    for name, want in (("m", "Male"), ("f", "Female")):
        src = ybams[name]
        with ingest.BamIngest.unindexed(src) as un:
            rows = [(un.tid(c), s, e) for c, s, e in BamDepth.y_regions("hg38")]
            with ingest.scan_sample(ctx, un, [], [], rows) as f:
                want_depths = f.depths.copy()
        with piped(_read(src)) as path, ingest.BamIngest.stream(path) as st:
            with ingest.scan_sample(ctx, st, [], [], rows, slab_bytes=SLAB_TINY) as b:
                assert b.scan_status == 0 and np.array_equal(b.depths, want_depths)
                ydepth = float(np.median(b.depths))
        assert ("Male" if ydepth > 1 else "Female") == want


def _status_case(ctx, repo, tmp_path):
    """a stream cut inside a BGZF block: status 1; cut between blocks inside a record: 3; unsorted: 4.  Never evidence."""
    from tredparse_b200 import ingest
    refs, recs = _records(MINIS[0])
    big = _rewrite(str(tmp_path / "cut.bam"), refs, recs, index=False)
    data = _read(big)
    blocks = _blocks(data)
    starts = _record_starts(data)
    mid_record = [c for c, u in blocks[2:-2] if u not in starts]
    assert mid_record
    k = len(recs) // 2
    swapped = recs[:k] + [recs[k + 1], recs[k]] + recs[k + 2:]
    cases = [("mid-block", data[:blocks[len(blocks) // 2][0] + 100], {1}),
             ("mid-record", data[:mid_record[len(mid_record) // 2]], {3}),
             ("unsorted", _read(_rewrite(str(tmp_path / "unsorted.bam"), refs, swapped, index=False)), {4})]
    for name, blob, want in cases:
        with piped(blob) as path, ingest.BamIngest.stream(path) as st:
            qs, keep, key = _queries(st, repo, repo.names, 150)
            with ingest.scan_sample(ctx, st, qs, keep, [(st.tid("chrY"), 2784557, 2791188)], slab_bytes=SLAB_TINY) as b:
                got = set(b.status.tolist())
                assert len(got) == 1 and got == want and b.scan_status in got, (name, b.status)
                assert np.isnan(b.depths).all() and b.nreads == 0


# ---- CPU: the device code, executed serially on the host --------------------------------------------------------------
def test_stream_handle_serves_the_header_once_and_refuses_the_rest(repo):
    from tredparse_b200 import ingest, _lib
    with piped(_read(MINIS[0]), 5) as path:
        with ingest.BamIngest.stream(path) as st, ingest.BamIngest.unindexed(MINIS[0]) as un:
            assert ingest.is_stream(path) and not ingest.is_stream(MINIS[0]) and ingest.is_stream("-")
            assert st.header_text() == un.header_text() and st.signature == un.signature
            assert st.read_length() == un.read_length()
            with pytest.raises(IOError, match="stream"):
                st.clone()
            with pytest.raises(_lib.TredswError, match="stream"):
                st.extract_locus(repo["HD"], 150)
            with pytest.raises(_lib.TredswError, match="stream"):
                st.region_depth("chr4", 1000, 2000)
            q, keep = ingest.locus_query(st, repo["HD"], 150)
            with pytest.raises(_lib.TredswError, match="stream"):
                ingest.IngestBatch(None, [st], [0], [q], keep=[keep])
            with ingest.scan_sample(None, st, [q], [keep], []) as b:
                assert b.scan_status == 0 and b.evidence(0).nreads > 50
            with pytest.raises(_lib.TredswError, match="already consumed"):
                ingest.scan_sample(None, st, [q], [keep], [])
            with pytest.raises(_lib.TredswError, match="already consumed"):
                st.read_length()
    with pytest.raises(IOError):
        with piped(b"not a BAM at all") as path:
            ingest.BamIngest.stream(path)


def test_stream_read_group_sample(tmp_path):
    from tredparse_b200 import bamio, ingest
    refs, recs = _records(MINIS[0])
    text = "@HD\tVN:1.4\tSO:coordinate\n@RG\tID:a\tPL:ILLUMINA\tSM:NA12878\n@RG\tID:b\tSM:other\n"
    src = str(tmp_path / "rg.bam")
    bamio.write_bam(src, refs, recs[:100], header_text=text, index=False)
    with piped(_read(src)) as path, ingest.BamIngest.stream(path) as st:
        assert st.read_group_sample() == "NA12878"
    with piped(_read(MINIS[0])) as path, ingest.BamIngest.stream(path) as st:
        assert st.read_group_sample() is None


def test_emulated_stream_scan_equals_the_file_scan_on_the_fixtures(repo, tmp_path):
    _fixtures_case(None, repo, tmp_path)


def test_emulated_stream_scan_on_synthetic_whole_sample_bams(repo, tmp_path):
    _synthetic_case(None, repo, tmp_path, ["HD", "DM1", "FXS", "SCA10"])


def test_emulated_stream_scan_on_adversarial_layouts(repo, tmp_path):
    _adversarial_case(None, repo, tmp_path)


def test_emulated_stream_scan_depth_regions_and_gender(repo, tmp_path, ybams):
    _depth_case(None, repo, tmp_path, ybams)


def test_emulated_stream_scan_reports_cut_and_unsorted_streams(repo, tmp_path):
    _status_case(None, repo, tmp_path)


def _cli(args, cwd, **kw):
    env = dict(os.environ, PYTHONPATH=ROOT)
    return subprocess.run([sys.executable, "-m", "tredparse_b200.tred"] + args, cwd=cwd, env=env, capture_output=True,
                          timeout=900, **kw)


def test_cli_refuses_several_gpus_for_a_stream_before_reading_it(tmp_path):
    """`-` with --gpus 2: the error comes before anything is read (stdin stays open and empty: a read would block)"""
    r, w = os.pipe()
    try:
        res = _cli(["-", "--workdir", str(tmp_path), "--gpus", "2", "--tred", "HD"], str(tmp_path), stdin=r)
    finally:
        os.close(r)
        os.close(w)
    assert res.returncode != 0 and b"read only once" in res.stderr, res.stderr[-2000:]
    csv = tmp_path / "samples.csv"
    with fifo(str(tmp_path / "s.bam"), _read(MINIS[0])) as path:
        csv.write_text("s1,{}\n".format(path))
        res = _cli([str(csv), "--workdir", str(tmp_path), "--gpus", "2", "--tred", "HD"], str(tmp_path))
    assert res.returncode != 0 and b"read only once" in res.stderr, res.stderr[-2000:]


# ---- GPU -----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    from tredparse_b200 import _lib
    return _lib.default_context(0)


@pytest.mark.gpu
def test_gpu_stream_scan_equals_the_file_scan_on_the_fixtures(repo, tmp_path, ctx):
    _fixtures_case(ctx, repo, tmp_path)


@pytest.mark.gpu
def test_gpu_stream_scan_on_synthetic_whole_sample_bams(repo, tmp_path, ctx):
    _synthetic_case(ctx, repo, tmp_path, [n for n in repo.names][:12])


@pytest.mark.gpu
def test_gpu_stream_scan_on_adversarial_layouts(repo, tmp_path, ctx):
    _adversarial_case(ctx, repo, tmp_path)


@pytest.mark.gpu
def test_gpu_stream_scan_depth_regions_and_gender(repo, tmp_path, ctx, ybams):
    _depth_case(ctx, repo, tmp_path, ybams)


@pytest.mark.gpu
def test_gpu_stream_scan_reports_cut_and_unsorted_streams(repo, tmp_path, ctx):
    _status_case(ctx, repo, tmp_path)


@pytest.mark.gpu
def test_run_chunks_on_stream_samples_equals_the_indexed_run_without_other_readers(repo, tmp_path, monkeypatch):
    """tred.run_chunks on FIFOs carrying both mini BAMs and a synthetic whole-sample BAM, every catalogue locus with alt
    regions: the same tredCalls (gender, depthY, readLen included) as on the indexed files, one scan per sample, and
    neither the Python reader nor check_bam nor an indexed open touches a stream; a cut stream is a sample error"""
    from tredparse_b200 import tred as T, bam_parser, ingest
    names = list(repo.names)
    synth = _sample(str(tmp_path / "synth.bam"), repo, names, 1, 41, 150)
    indexed = MINIS + [synth]
    tasks = lambda paths: [("s{}".format(i), p, repo, list(names), 300, False, False, True, True, "INFO")
                           for i, p in enumerate(paths)]
    want = [r["tredCalls"] for r in T.run_chunks(tasks(indexed))]

    def forbidden(*a, **k):
        raise AssertionError("a stream was read by something else than its one scan")
    for mod, name in ((bam_parser, "extract_locus"), (T, "extract_locus"), (bam_parser, "read_alignment"),
                      (T, "read_alignment"), (T, "check_bam"), (T, "ingest_loci"), (T, "infer_gender")):
        monkeypatch.setattr(mod, name, forbidden)
    monkeypatch.setattr(bam_parser.BamDepth, "region_depth", forbidden)
    monkeypatch.setattr(ingest.BamIngest, "__init__", forbidden)
    scans = []
    real = ingest.scan_sample

    def counted(*a, **k):
        b = real(*a, **k)
        scans.append(b.stats())
        return b
    monkeypatch.setattr(ingest, "scan_sample", counted)
    with contextlib.ExitStack() as es:
        paths = [es.enter_context(fifo(str(tmp_path / "f{}.bam".format(i)), _read(p), i)) for i, p in enumerate(indexed)]
        got = [r for r in T.run_chunks(tasks(paths))]
    assert len(scans) == 3 and all(s["records"] > 6000 for s in scans)
    assert len(got) == len(want) == 3
    for a, b in zip(got, want):
        assert "error" not in a and len(a["tredCalls"]) > 20 * len(names) and a["tredCalls"] == b
    # a stream cut inside a block: that sample is an error, the others of the chunk are called
    data = _read(MINIS[1])
    with fifo(str(tmp_path / "cut.bam"), data[:len(data) // 2]) as cut, fifo(str(tmp_path / "ok.bam"), _read(MINIS[0])) as ok:
        got = list(T.run_chunks(tasks([cut, ok])))
    assert got[0]["tredCalls"] == {} and "status" in got[0]["error"]
    assert got[1]["tredCalls"] == want[0] and "error" not in got[1]


def _calls_without_key(js):
    d = dict(js)
    d.pop("samplekey"); d.pop("bam")
    return d


@pytest.mark.gpu
def test_cli_on_stdin_equals_the_run_on_the_file(tmp_path):
    """`cat t001.mini.bam | python -m tredparse_b200.tred - --tred HD --tred DM1`: the JSON of the file-path run, apart
    from samplekey (`stdin`: the fixture has no @RG line) and bam (`-`); --checkexists skips it the second time"""
    wf, ws = tmp_path / "file", tmp_path / "stdin"
    res = _cli([MINIS[0], "--workdir", str(wf), "--tred", "HD", "--tred", "DM1"], str(tmp_path))
    assert res.returncode == 0, res.stderr[-3000:]
    want = json.loads((wf / "t001.mini.json").read_text())
    res = _cli(["-", "--workdir", str(ws), "--tred", "HD", "--tred", "DM1"], str(tmp_path), input=_read(MINIS[0]))
    assert res.returncode == 0, res.stderr[-3000:]
    got = json.loads((ws / "stdin.json").read_text())
    assert got["samplekey"] == "stdin" and got["bam"] == "-"
    assert _calls_without_key(got) == _calls_without_key(want)
    for k in ("HD.1", "HD.2", "HD.FR", "HD.PR", "HD.RR", "HD.CI", "HD.PP"):
        assert got["tredCalls"][k] == want["tredCalls"][k]
    with gzip.open(str(ws / "stdin.tred.vcf.gz"), "rt") as a, gzip.open(str(wf / "t001.mini.tred.vcf.gz"), "rt") as b:
        body = lambda fp: [l for l in fp.read().splitlines() if not l.startswith("##")][1:]
        assert body(a) == body(b)
    os.remove(str(ws / "stdin.tred.vcf.gz"))
    res = _cli(["-", "--workdir", str(ws), "--tred", "HD", "--checkexists"], str(tmp_path), input=_read(MINIS[0]))
    assert res.returncode == 0 and not (ws / "stdin.tred.vcf.gz").exists(), res.stderr[-3000:]


@pytest.mark.gpu
def test_cli_on_a_fifo_listed_in_a_csv(tmp_path):
    wf, ws = tmp_path / "file", tmp_path / "fifo"
    res = _cli([MINIS[1], "--workdir", str(wf), "--tred", "DM1", "--tred", "HD"], str(tmp_path))
    assert res.returncode == 0, res.stderr[-3000:]
    want = json.loads((wf / "t002.mini.json").read_text())
    with fifo(str(tmp_path / "t002.bam"), _read(MINIS[1]), 9) as path:
        csv = tmp_path / "samples.csv"
        csv.write_text("t002x,{}\n".format(path))
        res = _cli([str(csv), "--workdir", str(ws), "--tred", "DM1", "--tred", "HD"], str(tmp_path))
    assert res.returncode == 0, res.stderr[-3000:]
    got = json.loads((ws / "t002x.json").read_text())
    assert got["bam"] == os.path.abspath(path) and _calls_without_key(got) == _calls_without_key(want)
