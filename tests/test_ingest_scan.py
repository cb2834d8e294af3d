"""The scan of a BAM without an index (tredsw_ingest_scan_run, csrc/bgzf_gpu.cu run_scan): one streaming pass per sample
finds the record boundaries without an index, keeps the records of every locus window, alt region and depth region, and
hands them to the selection / pairing steps of the indexed GPU ingest.

Every problem is checked against the host reader on an indexed copy of the same file (BamIngest.extract_locus with
names).  CPU tests run the device code serially on the host (tredsw_ingest_scan_emulate: test infrastructure); the
`gpu` tests run the kernels."""
import logging
import os
import shutil
import struct
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
MINIS = [os.path.join(GOLDEN, "t001.mini.bam"), os.path.join(GOLDEN, "t002.mini.bam")]
SLAB_TINY = 65536          # the smallest slab: one or two BGZF blocks, so records straddle block AND slab boundaries


@pytest.fixture(scope="module")
def repo():
    from tredparse_b200.meta import TREDsRepo
    return TREDsRepo()


def _same(ev, ref):
    """(as in test_ingest_gpu.py) the evidence of one locus, field for field"""
    return (np.array_equal(ev.reads, ref.reads) and np.array_equal(ev.roff, ref.roff)
            and np.array_equal(ev.global_lens, ref.global_lens) and np.array_equal(ev.target_lens, ref.target_lens)
            and ev.depth == ref.depth and ev.n_unmapped == ref.n_unmapped and ev.names == ref.names)


def _unindexed(tmp_path, src):
    dst = str(tmp_path / ("noindex_" + os.path.basename(src)))
    shutil.copy(src, dst)
    return dst


def _queries(h, repo, names, readlen):
    from tredparse_b200 import ingest
    qs, keep, key = [], [], []
    for n in names:
        q = ingest.locus_query(h, repo[n], readlen, alts=repo[n].alt)
        if q is not None:
            qs.append(q[0]); keep.append(q[1]); key.append(n)
    return qs, keep, key


def _scan_check(ctx, indexed, unindexed, repo, names, readlen=150, slab_bytes=None, depth_regions=()):
    """scan `unindexed`; every locus (alt regions included) and every depth region equals the host reader on
    `indexed`.  -> (scan statistics, reads in total)"""
    from tredparse_b200 import ingest
    ref, un = ingest.BamIngest(indexed), ingest.BamIngest.unindexed(unindexed)
    try:
        qs, keep, key = _queries(un, repo, names, readlen)
        with ingest.scan_sample(ctx, un, qs, keep, depth_regions, slab_bytes=slab_bytes) as b:
            assert b.scan_status == 0 and b.nproblems == len(key) and not b.status.any()
            total = 0
            for i, n in enumerate(key):
                want = ref.extract_locus(repo[n], readlen, alts=repo[n].alt, want_names=True)
                assert _same(b.evidence(i), want), (unindexed, n, readlen, slab_bytes)
                total += want.nreads
            for (c, s, e), d in zip(depth_regions, b.depths):
                d_ref = ctypes_depth(ref, c, s, e)
                assert d == d_ref, ((c, s, e), d, d_ref)
            return b.stats(), total
    finally:
        ref.close()
        un.close()


def ctypes_depth(handle, tid, start, end):
    import ctypes
    from tredparse_b200 import _lib
    d = ctypes.c_double()
    _lib.check(handle.lib.tredsw_bam_region_depth(handle.handle, tid, start, end, ctypes.byref(d)), "region_depth")
    return d.value


def _records(path):
    from tredparse_b200 import bamio
    sam = bamio.AlignmentFile(path)
    refs = list(zip(sam.references, sam.lengths))
    recs = list(sam.fetch())
    sam.close()
    return refs, recs


def _rewrite(dst, refs, recs, index=True):
    from tredparse_b200 import bamio
    bamio.write_bam(dst, refs, recs, index=index)
    return dst


def _fooling_quality(rec):
    """a quality string that starts with a record header whose block_size points exactly at the next record: a
    candidate search that meets it before the block's true first record picks it, and the chain it starts looks
    right.  (write_bam writes no aux fields: the quality string ends the record.)"""
    n = len(rec.query_sequence)
    fake = struct.pack("<iiiBBHHHiiii", n - 4, 0, 0, 1, 0, 0, 0, 0, 0, -1, -1, 0) + b"\0"
    return fake + b"I" * (n - len(fake))


def _sample(path, repo, names, sample, seed, readlen):
    from tredparse_b200 import simulate
    refs, _ = _records(MINIS[0])
    simulate.write_sample_bam(path, repo, names, refs, sample, readlen, seed)
    return path


@pytest.fixture(scope="module")
def ybams(tmp_path_factory):
    """(as in test_ingest.py) BAMs with uniform 15x / 0.2x coverage of the chrY regions of the gender inference"""
    from tredparse_b200 import bamio
    from tredparse_b200.bam_parser import BamDepth
    from tredparse_b200.utils import datafile
    d = tmp_path_factory.mktemp("ybams")
    rng = np.random.default_rng(7)
    regions = []
    with open(datafile("chrY.tsv")) as fp:
        next(fp)
        for line in fp:
            b, row, c, s, e, _ = line.split()
            if b == "hg38":
                regions.append((int(row), int(s), int(e)))
    out = {}
    for name, ydepth in (("m", 15), ("f", 0.2)):
        recs = []
        for row, s, e in regions[:12]:
            dd = ydepth if row not in BamDepth.Y_SKIP_ROWS else 40
            n = int(dd * (e - s + 1) / 100)
            for k, pos in enumerate(sorted(rng.integers(s, e - 100, size=n))):
                recs.append(bamio.AlignedSegment("y{}_{}".format(row, k), 0, 1, int(pos), 60, [(0, 100)], -1, -1, 0,
                                                 "ACGT" * 25))
        recs.sort(key=lambda r: r.reference_start)
        out[name] = _rewrite(str(d / (name + ".bam")), [("chr4", 190214555), ("chrY", 57227415)], recs)
    return out


# ---- the cases, run through the emulation (ctx None) and on the GPU (ctx a context) -----------------------------------
def _fixtures_case(ctx, repo, tmp_path):
    for src in MINIS:
        un = _unindexed(tmp_path, src)
        _, recs = _records(src)
        for readlen in (150, 101):
            for slab in (None, SLAB_TINY):
                st, total = _scan_check(ctx, src, un, repo, repo.names, readlen, slab)
                assert total > 50 and st["records"] == len(recs) and st["repaired_blocks"] == 0
                assert st["slabs"] == 1 if slab is None else st["slabs"] >= 3
                assert st["compressed_bytes"] + 28 >= os.path.getsize(src) - 65536


def _synthetic_case(ctx, repo, tmp_path, names):
    for readlen in (150, 251):
        src = _sample(str(tmp_path / "s{}.bam".format(readlen)), repo, names, 3, 11, readlen)
        st, total = _scan_check(ctx, src, _unindexed(tmp_path, src), repo, names, readlen, SLAB_TINY)
        assert total > 200 and st["slabs"] > 2 and st["repaired_blocks"] == 0


def _adversarial_case(ctx, repo, tmp_path):
    from tredparse_b200 import bamio
    refs, recs = _records(MINIS[0])
    # (1) record headers inside quality strings fool the candidate search: the chain from the known first record
    #     repairs those blocks
    for r in recs:
        r._qual = _fooling_quality(r)
    src = _rewrite(str(tmp_path / "fooled.bam"), refs, recs)
    st, total = _scan_check(ctx, src, _unindexed(tmp_path, src), repo, repo.names, 150, SLAB_TINY)
    assert st["repaired_blocks"] > 0 and total > 50
    # (2) a record longer than a BGZF block: at least one block holds no record start
    hd = repo["HD"]
    tid = [n for n, _ in refs].index(hd.chr)
    big = bamio.AlignedSegment("big", 0, tid, hd.repeat_start - 100, 60, [(0, 60000)], -1, -1, 0, "ACGT" * 15000)
    keys = [(r.reference_id if r.reference_id >= 0 else 1 << 30, r.reference_start) for r in recs]
    import bisect
    at = bisect.bisect_right(keys, (tid, big.reference_start))
    src = _rewrite(str(tmp_path / "big.bam"), refs, recs[:at] + [big] + recs[at:])
    for slab in (None, SLAB_TINY):
        st, total = _scan_check(ctx, src, _unindexed(tmp_path, src), repo, ["HD", "DM1"], 150, slab)
        assert st["records"] == len(recs) + 1
    with __import__("tredparse_b200.ingest", fromlist=["x"]).BamIngest(src) as h:
        assert "big" in h.extract_locus(hd, 150, want_names=True).names
    # (3) a file with only a header: no records, empty evidence; (4) one with only the EOF block is not a BAM
    src = _rewrite(str(tmp_path / "header_only.bam"), refs, [])
    st, total = _scan_check(ctx, src, _unindexed(tmp_path, src), repo, ["HD", "FXS"], 150)
    assert st["records"] == 0 and total == 0
    eof = str(tmp_path / "eof_only.bam")
    with open(src, "rb") as fp:
        data = fp.read()
    with open(eof, "wb") as fp:
        fp.write(data[-28:])
    from tredparse_b200 import ingest
    with pytest.raises(IOError):
        ingest.BamIngest.unindexed(eof)


def _depth_case(ctx, repo, tmp_path, ybams):
    """depth_out = tredsw_bam_region_depth on the indexed copy; gender and depthY as the chrY set-up gives them"""
    from tredparse_b200 import ingest
    from tredparse_b200.bam_parser import BamDepth
    log = logging.getLogger()
    with ingest.BamIngest(MINIS[0]) as h:
        t4, tx, ty = h.tid("chr4"), h.tid("chrX"), h.tid("chrY")
    regions = [(t4, 3074000, 3076000), (t4, 0, 10), (tx, 147911000, 147913000), (ty, 2784557, 2791188), (t4, 3074500, 3074500)]
    _scan_check(ctx, MINIS[0], _unindexed(tmp_path, MINIS[0]), repo, ["HD"], 150, SLAB_TINY, regions)
    for name, want in (("m", "Male"), ("f", "Female")):
        src = ybams[name]
        with ingest.BamIngest.unindexed(_unindexed(tmp_path, src)) as un:
            rows = [(un.tid(c), s, e) for c, s, e in BamDepth.y_regions("hg38")]
            with ingest.scan_sample(ctx, un, [], [], rows) as b:
                assert b.scan_status == 0 and b.stats()["records"] > 1000
                ydepth = float(np.median(b.depths))
        assert ydepth == BamDepth(src, "hg38", log).get_Y_depth()
        assert ("Male" if ydepth > 1 else "Female") == want


def _status_case(ctx, repo, tmp_path):
    """an unsorted file: status 4 for every problem; a flipped byte inside a block: 2; a truncated file: a status,
    never partial evidence"""
    from tredparse_b200 import ingest
    refs, recs = _records(MINIS[0])
    k = len(recs) // 2
    swapped = recs[:k] + [recs[k + 1], recs[k]] + recs[k + 2:]
    assert (swapped[k].reference_id, swapped[k].reference_start) > (swapped[k + 1].reference_id, swapped[k + 1].reference_start)
    cases = {"unsorted": (_rewrite(str(tmp_path / "unsorted.bam"), refs, swapped, index=False), {4})}
    data = bytearray(open(MINIS[0], "rb").read())
    flip = bytearray(data)
    flip[len(flip) // 2] ^= 0x55
    for name, blob, want in (("flip", flip, {2}), ("truncated", data[:len(data) // 2], {1, 3})):
        p = str(tmp_path / (name + ".bam"))
        with open(p, "wb") as fp:
            fp.write(bytes(blob))
        cases[name] = (p, want)
    for name, (path, want) in cases.items():
        with ingest.BamIngest.unindexed(path) as un:
            qs, keep, key = _queries(un, repo, repo.names, 150)
            with ingest.scan_sample(ctx, un, qs, keep, [(un.tid("chrY"), 2784557, 2791188)], slab_bytes=SLAB_TINY) as b:
                got = set(b.status.tolist())
                assert len(got) == 1 and got <= want and b.scan_status in got, (name, b.status)
                assert np.isnan(b.depths).all() and b.nreads == 0


# ---- CPU: the device code, executed serially on the host --------------------------------------------------------------
def test_unindexed_handle_serves_the_header_and_refuses_indexed_queries(repo, tmp_path):
    from tredparse_b200 import ingest, _lib
    import logging as lg
    un_path = _unindexed(tmp_path, MINIS[0])
    with pytest.raises(IOError):
        ingest.BamIngest(un_path)                                  # the indexed open still wants a .bai
    with ingest.BamIngest(MINIS[0]) as ref, ingest.BamIngest.unindexed(un_path) as un:
        assert un.signature == ref.signature and un.tid("chr4") == ref.tid("chr4") >= 0
        assert un.read_length() == ref.read_length()
        from tredparse_b200.bam_parser import BamReadLen
        assert BamReadLen(un_path, lg.getLogger(), ing=un).readlen == ref.read_length()[0]
        with pytest.raises(_lib.TredswError, match="code -?3|no index"):
            un.extract_locus(repo["HD"], 150)
        with pytest.raises(_lib.TredswError, match="no index"):
            un.region_depth("chr4", 1000, 2000)
        q, keep = ingest.locus_query(un, repo["HD"], 150)
        with pytest.raises(_lib.TredswError, match="no index"):
            ingest.IngestBatch(None, [un], [0], [q], keep=[keep])


def test_emulated_scan_equals_the_indexed_reader_on_the_fixtures(repo, tmp_path):
    _fixtures_case(None, repo, tmp_path)


def test_emulated_scan_on_synthetic_whole_sample_bams(repo, tmp_path):
    _synthetic_case(None, repo, tmp_path, ["HD", "DM1", "FXS", "SCA10"])


def test_emulated_scan_on_adversarial_layouts(repo, tmp_path):
    _adversarial_case(None, repo, tmp_path)


def test_emulated_scan_depth_regions_and_gender(repo, tmp_path, ybams):
    _depth_case(None, repo, tmp_path, ybams)


def test_emulated_scan_reports_unsorted_corrupt_and_truncated_files(repo, tmp_path):
    _status_case(None, repo, tmp_path)


_SCAN_FUZZ = r"""
import os, sys, random
sys.path.insert(0, {root!r})
from tredparse_b200 import ingest, _lib
from tredparse_b200.meta import TREDsRepo
repo = TREDsRepo()
good = open({bam!r}, "rb").read()
rng = random.Random(13)
ok = flagged = refused = 0
for trial in range(80):
    bad = bytearray(good)
    how = trial % 3
    if how == 0:                                           # bytes anywhere in the file: headers, payloads, footers
        for _ in range(rng.randrange(1, 6)):
            p = rng.randrange(len(bad)); bad[p] = rng.randrange(256)
    elif how == 1:                                         # truncated file
        bad = bad[:rng.randrange(100, len(bad))]
    else:                                                  # BGZF framing fields (XLEN, BSIZE, ISIZE) of some block
        off = 0
        for _ in range(rng.randrange(0, 25)):
            nxt = off + int.from_bytes(bad[off + 16:off + 18], "little") + 1
            if nxt + 28 >= len(bad): break
            off = nxt
        p = off + rng.choice([10, 11, 16, 17]); bad[p] = rng.randrange(256)
    p2 = os.path.join({tmp!r}, "bad.bam")
    open(p2, "wb").write(bytes(bad))
    try:
        h = ingest.BamIngest.unindexed(p2)
    except Exception:
        refused += 1
        continue
    try:
        qs = [ingest.locus_query(h, repo[n], 150, alts=repo[n].alt) for n in ("HD", "SCA17")]
        qs = [q for q in qs if q is not None]
        with ingest.scan_sample(None, h, [q[0] for q in qs], [q[1] for q in qs], [], slab_bytes=rng.choice([0, 65536])) as b:
            for i in range(len(qs)):
                if b.status[i]:
                    flagged += 1
                else:
                    ev = b.evidence(i); assert ev.nreads == len(ev.roff) - 1 and ev.roff[-1] == len(ev.reads)
                    ok += 1
    except _lib.TredswError:
        refused += 1
    finally:
        h.close()
print("survived", ok, flagged, refused)
"""


def test_damaged_files_do_not_take_the_scan_down(tmp_path):
    """the damage cases of the indexed ingest's test, through the scan: every outcome is a result, a per-problem
    flag or a TredswError — never a crash"""
    code = _SCAN_FUZZ.format(root=ROOT, bam=MINIS[0], tmp=str(tmp_path))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-500:], r.stderr[-2000:])
    assert "survived" in r.stdout


# ---- GPU -----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    from tredparse_b200 import _lib
    return _lib.default_context(0)


@pytest.mark.gpu
def test_gpu_scan_equals_the_indexed_reader_on_the_fixtures(repo, tmp_path, ctx):
    _fixtures_case(ctx, repo, tmp_path)


@pytest.mark.gpu
def test_gpu_scan_on_synthetic_whole_sample_bams(repo, tmp_path, ctx):
    _synthetic_case(ctx, repo, tmp_path, [n for n in repo.names][:12])


@pytest.mark.gpu
def test_gpu_scan_on_adversarial_layouts(repo, tmp_path, ctx):
    _adversarial_case(ctx, repo, tmp_path)


@pytest.mark.gpu
def test_gpu_scan_depth_regions_and_gender(repo, tmp_path, ctx, ybams):
    _depth_case(ctx, repo, tmp_path, ybams)


@pytest.mark.gpu
def test_gpu_scan_reports_unsorted_corrupt_and_truncated_files(repo, tmp_path, ctx):
    _status_case(ctx, repo, tmp_path)


@pytest.mark.gpu
def test_run_chunks_on_unindexed_bams_equals_the_indexed_run_without_the_python_reader(repo, tmp_path, monkeypatch):
    """tred.run_chunks on unindexed copies of both mini BAMs and of a synthetic whole-sample BAM, every catalogue locus
    with alt regions: the same tredCalls (gender, depthY, readLen included) as on the indexed files, one scan per
    sample, and the Python reader is never used"""
    from tredparse_b200 import tred as T, bam_parser, ingest
    names = list(repo.names)
    synth = _sample(str(tmp_path / "synth.bam"), repo, names, 1, 41, 150)
    indexed = MINIS + [synth]
    tasks = lambda paths: [("s{}".format(i), p, repo, list(names), 300, False, False, True, True, "INFO")
                           for i, p in enumerate(paths)]
    want = [r["tredCalls"] for r in T.run_chunks(tasks(indexed))]

    def no_python_reader(*a, **k):
        raise AssertionError("the Python reader was used on an unindexed BAM the GPU scan can serve")
    monkeypatch.setattr(bam_parser, "extract_locus", no_python_reader)
    monkeypatch.setattr(T, "extract_locus", no_python_reader)
    monkeypatch.setattr(bam_parser.BamDepth, "region_depth", no_python_reader)
    scans = []
    real = ingest.scan_sample

    def counted(*a, **k):
        b = real(*a, **k)
        scans.append(b.stats())
        return b
    monkeypatch.setattr(ingest, "scan_sample", counted)
    got = [r["tredCalls"] for r in T.run_chunks(tasks([_unindexed(tmp_path, p) for p in indexed]))]
    assert len(scans) == 3 and all(s["records"] > 6000 for s in scans)
    assert len(got) == len(want) == 3
    for a, b in zip(got, want):
        assert len(a) > 20 * len(names) and a == b
