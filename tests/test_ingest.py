"""Native BAM ingest (csrc/ingest.cpp, host code) against the Python host path that mirrors the reference —
BamParser.select_reads (bam_parser.py:194-243), PEextractor (:316-369), BamDepth.region_depth (:404-411) —
on the committed mini BAMs.  No GPU needed."""
import logging
import os

import numpy as np
import pytest

from tredparse_b200 import bamio, bam_parser, ingest, ssw
from tredparse_b200.bam_parser import BamParser, PEextractor, BamDepth
from tredparse_b200.meta import TREDsRepo
from tredparse_b200.utils import InputParams

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
CASES = [("t001", "HD"), ("t002", "DM1")]
BAMS = [(s, t, os.path.join(GOLDEN, s + ".mini.bam")) for s, t in CASES]
EMPTY = ("t001", "DM1", os.path.join(GOLDEN, "t001.mini.bam"))      # chr19: no reads in the chr4 mini BAM


@pytest.fixture(scope="module")
def repo():
    return TREDsRepo()


def _python_path(bam, tredname, repo, alts):
    ip = InputParams(bam=bam, READLEN=150, tredName=tredname, repo=repo, maxinsert=300, fullsearch=False,
                     gender="Unknown", depth=30, clip=False, alts=alts, repeatpairs=True, log="INFO")
    bp = BamParser(ip)
    sam = bamio.AlignmentFile(bam)
    reads = bp.select_reads(sam)
    sam.close()
    pe = PEextractor(bp)
    t = repo[tredname]
    depth = BamDepth(bam, "hg38", logging.getLogger()).region_depth(t.chr, max(0, t.repeat_start - 1000), t.repeat_end + 1000)
    return bp, reads, pe, depth


@pytest.mark.parametrize("sample,tredname,bam", BAMS + [EMPTY], ids=[b[0] for b in BAMS] + ["t001-DM1"])
@pytest.mark.parametrize("alts", [False, True])
def test_extract_locus_equals_python_host_path(sample, tredname, bam, alts, repo):
    bp, reads, pe, depth = _python_path(bam, tredname, repo, alts)
    with ingest.BamIngest(bam) as ing:
        ev = ing.extract_locus(repo[tredname], 150, alts=bp.alt if alts else (), want_names=True)
    empty = (sample, tredname, bam) == EMPTY
    assert ev.nreads == len(reads) and (empty or len(reads) > 50)
    assert ev.names == [r.query_name for r in reads]
    assert ev.read_strings() == ["".join(c if c in "ACGT" else "N" for c in r.query_sequence.upper()) for r in reads]
    assert np.array_equal(ev.reads, np.concatenate([ssw.encode(r.query_sequence) for r in reads] or [np.zeros(0, np.int8)]))
    assert list(ev.global_lens) == list(pe.global_lens) and (empty or len(pe.global_lens) > 1000)
    assert list(ev.target_lens) == list(pe.target_lens) and (empty or len(pe.target_lens) >= 5)
    assert ev.depth == depth
    if not alts:
        assert ev.n_unmapped == sum(1 for r in reads if r.is_unmapped)
    # the same record built from the Python reader (BAMs without a usable index, contigs the native reader lacks)
    _assert_same_record(bam_parser.extract_locus(bam, repo, tredname, 150, alts, False, logging.getLogger()), ev)


def _assert_same_record(a, b):
    """two ingest.LocusEvidence field for field, array dtypes included"""
    for f in ingest.LocusEvidence.__slots__:
        x, y = getattr(a, f), getattr(b, f)
        if isinstance(y, np.ndarray):
            assert isinstance(x, np.ndarray) and x.dtype == y.dtype and np.array_equal(x, y), f
        else:
            assert type(x) is type(y) and x == y, f


def test_missing_locus_and_errors(repo):
    with ingest.BamIngest(os.path.join(GOLDEN, "t001.mini.bam")) as ing:
        ev = ing.extract_locus(repo["DM1"], 150)             # chr19: no reads in the chr4 mini BAM
        assert ev.nreads == 0 and len(ev.global_lens) == 0 and ev.depth == 0.0
        assert ing.tid("chr4") >= 0 and ing.tid("nope") == -1
        tiny = ingest.BamIngest(os.path.join(GOLDEN, "t001.mini.bam"))
        tiny._caps = dict(reads=1, bases=8, pairs=1, names=4)      # forces the overflow / retry path
        ev2 = tiny.extract_locus(repo["HD"], 150, want_names=True)
        ev1 = ing.extract_locus(repo["HD"], 150, want_names=True)
        assert np.array_equal(ev1.reads, ev2.reads) and ev1.names == ev2.names
        assert list(ev1.global_lens) == list(ev2.global_lens)
    with pytest.raises(IOError):
        ingest.BamIngest("/nonexistent.bam")


def test_problem_feeds_the_cohort_packer(repo):
    from tredparse_b200 import cohort
    with ingest.BamIngest(os.path.join(GOLDEN, "t001.mini.bam")) as a, \
            ingest.BamIngest(os.path.join(GOLDEN, "t002.mini.bam")) as b:
        probs = [a.problem(repo["HD"], 150), b.problem(repo["DM1"], 150)]
    batch = cohort.CohortBatch(probs)
    assert batch.nproblems == 2 and batch.nreads == probs[0].nreads + probs[1].nreads
    assert 25 < probs[0].depth < 35 and 40 < probs[1].depth < 55


# ---- pre-steps: depth of arbitrary regions, read length, gender (bam_parser.py:372-429, tred.py:201-223) --------
@pytest.mark.parametrize("sample,tredname,bam", BAMS[:2], ids=[b[0] for b in BAMS[:2]])
def test_region_depth_and_read_length_equal_python_reader(sample, tredname, bam, repo):
    t = repo[tredname]
    sam = bamio.AlignmentFile(bam)
    rls = []
    for r in sam.fetch():                                   # BamReadLen.readlen: first 101 records
        rls.append(r.query_length)
        if len(rls) > 100:
            break
    with ingest.BamIngest(bam) as ing:
        for (s, e) in [(t.repeat_start - 1000, t.repeat_end + 1000), (t.repeat_start - 50, t.repeat_start + 50),
                       (t.repeat_start - 9000, t.repeat_start - 8000), (1, 1000)]:
            s = max(0, s)
            assert ing.region_depth(t.chr, s, e) == bamio.region_depth(sam, t.chr, s, e)
        assert ing.read_length(100) == (max(rls), min(rls))
        with pytest.raises(ValueError):
            ing.region_depth("chrNope", 1, 100)
    sam.close()
    from tredparse_b200.bam_parser import BamReadLen
    assert BamReadLen(bam, logging.getLogger()).readlen == max(rls)


def _ybam(path, ydepth, rng):
    """A BAM with uniform `ydepth`x coverage of the chrY regions the gender inference looks at."""
    from tredparse_b200.utils import datafile
    regions = []
    with open(datafile("chrY.tsv")) as fp:
        next(fp)
        for line in fp:
            b, row, c, s, e, _ = line.split()
            if b == "hg38":
                regions.append((int(row), int(s), int(e)))
    recs = []
    for row, s, e in regions[:12]:
        d = ydepth if row not in BamDepth.Y_SKIP_ROWS else 40        # the skipped rows are covered in everybody
        n = int(d * (e - s + 1) / 100)
        for k, pos in enumerate(sorted(rng.integers(s, e - 100, size=n))):
            recs.append(bamio.AlignedSegment("y{}_{}".format(row, k), 0, 1, int(pos), 60, [(0, 100)], -1, -1, 0,
                                             "ACGT" * 25))
    recs.sort(key=lambda r: r.reference_start)
    bamio.write_bam(path, [("chr4", 190214555), ("chrY", 57227415)], recs)


def test_gender_inference_from_chrY_depth(tmp_path):
    from tredparse_b200 import tred as tredmod
    repo = TREDsRepo()
    rng = np.random.default_rng(7)
    log = logging.getLogger()
    male, female = str(tmp_path / "m.bam"), str(tmp_path / "f.bam")
    _ybam(male, 15, rng)
    _ybam(female, 0.2, rng)
    ym, yf = BamDepth(male, "hg38", log).get_Y_depth(), BamDepth(female, "hg38", log).get_Y_depth()
    assert 12 < ym < 18 and yf < 1                           # tred.py:205-208: Male iff depthY > 1
    # the native reader and the Python reader agree region by region
    sam = bamio.AlignmentFile(male)
    with ingest.BamIngest(male) as ing:
        assert ing.region_depth("chrY", 2784557, 2791188) == bamio.region_depth(sam, "chrY", 2784557, 2791188) > 10
    sam.close()
    # no chrY contig -> the lookup raises and the caller keeps "Unknown" (tred.py:209-210)
    noy = str(tmp_path / "noy.bam")
    bamio.write_bam(noy, [("chr4", 190214555)],
                    [bamio.AlignedSegment("r0", 0, 0, 1000, 60, [(0, 100)], -1, -1, 0, "ACGT" * 25)])
    with pytest.raises(Exception):
        BamDepth(noy, "hg38", log).get_Y_depth()
    assert tredmod.presteps(noy, repo, ["FXS"], log) == {"inferredGender": "Unknown", "depthY": -1, "readLen": 100}
    # a BAM whose header lists chrY but holds no reads there reads as depth 0 -> Female, like the reference
    assert BamDepth(os.path.join(GOLDEN, "t001.mini.bam"), "hg38", log).get_Y_depth() == 0.0
    # through tred.run: gender and depthY are reported, readLen detected (tred.py:195-223)
    for bam, want in ((male, "Male"), (female, "Female")):
        pre = tredmod.presteps(bam, repo, ["FXS"], log)
        assert pre["inferredGender"] == want and pre["readLen"] == 100 and pre["depthY"] == (ym if want == "Male" else yf)
    pre = tredmod.presteps(male, repo, ["HD"], log)            # no X-linked locus requested: gender not inferred
    assert pre["inferredGender"] == "Unknown" and pre["depthY"] == -1


# ---- loci dealt to host threads (tred.ingest_loci) ------------------------------------------------------------
def _evidence_equal(a, b):
    return (np.array_equal(a.reads, b.reads) and np.array_equal(a.roff, b.roff) and a.names == b.names and
            np.array_equal(a.global_lens, b.global_lens) and np.array_equal(a.target_lens, b.target_lens) and
            a.depth == b.depth)


@pytest.mark.parametrize("sample,tredname,bam", BAMS, ids=[b[0] for b in BAMS])
def test_threaded_ingest_records_equal_serial(sample, tredname, bam, repo):
    from tredparse_b200 import tred as tredmod
    log = logging.getLogger()
    names = list(repo.names)
    ev1 = tredmod.ingest_loci(bam, repo, names, 150, True, False, log, threads=1)
    ev4 = tredmod.ingest_loci(bam, repo, names, 150, True, False, log, threads=4)
    assert set(ev1) == set(ev4) == set(names)
    assert all(_evidence_equal(ev1[k], ev4[k]) for k in ev1)
    assert ev1[tredname].nreads > 50 and ev1[tredname].depth > 5
    # clones are independent handles that share the index
    with ingest.BamIngest(bam) as ing:
        c = ing.clone()
        a = ing.extract_locus(repo[tredname], 150, want_names=True)
        b = c.extract_locus(repo[tredname], 150, want_names=True)
        c.close()
        assert _evidence_equal(a, b)
        assert _evidence_equal(a, ing.extract_locus(repo[tredname], 150, want_names=True))   # the parent still works


def test_run_wiring_without_the_gpu(monkeypatch, repo):
    """tred.run up to the kernels: pre-steps, threaded ingest, one item per locus with the locus depth
    (tred.py:195-249); the fused device stage (tred.genotype_evidence) is replaced by a recorder."""
    from tredparse_b200 import tred as tredmod
    seen = {}

    def fake_genotype_evidence(items, **kw):
        seen["items"], seen["kw"] = items, kw
        return [{} for _ in items]
    monkeypatch.setattr(tredmod, "genotype_evidence", fake_genotype_evidence)
    bam = os.path.join(GOLDEN, "t001.mini.bam")
    names = ["HD", "DM1", "FXS"]
    out = tredmod.run(("t001", bam, repo, names, 300, False, False, True, True, "INFO"))
    assert out["samplekey"] == "t001" and out["bam"] == bam
    calls = out["tredCalls"]
    assert calls["readLen"] == 150 and calls["inferredGender"] == "Female" and calls["depthY"] == 0.0
    assert not any(k.startswith("HD.") for k in calls)                   # the recorder returned no fields
    items = seen["items"]                                                # (tred, READLEN, gender, depth, evidence)
    assert [it[0].name for it in items] == names
    assert all(it[1] == 150 and it[2] == "Female" for it in items)
    hd, dm1 = items[0], items[1]
    assert hd[3] == hd[4].depth > 5 and hd[4].nreads > 50
    assert dm1[4].nreads == 0 and dm1[3] == 0.0                          # chr19: nothing in the chr4 mini BAM
    assert seen["kw"]["maxinsert"] == 300 and seen["kw"]["fullsearch"] is False
    assert seen["kw"]["clip"] is False and seen["kw"]["repeatpairs"] is True


def _unindexed_copy(tmp_path, sample):
    import shutil
    path = str(tmp_path / (sample + ".noindex.bam"))
    shutil.copy(os.path.join(GOLDEN, sample + ".mini.bam"), path)
    return path


def test_unindexed_bam_gets_the_native_evidence_records(monkeypatch, tmp_path, repo):
    """A BAM without a .bai: the native reader cannot open it, the Python reader builds every locus' record, and the
    records equal the native reader's on the indexed file — one genotyping batch, whichever reader served a locus."""
    from tredparse_b200 import tred as tredmod
    monkeypatch.setattr(tredmod, "GPU_INGEST", False)
    bam = os.path.join(GOLDEN, "t001.mini.bam")
    copy = _unindexed_copy(tmp_path, "t001")
    with pytest.raises(IOError):
        ingest.BamIngest(copy)
    # every catalogue locus without the alt regions (each alt region is a scan of the whole unindexed file), and HD
    # with them
    for names, alts in ((list(repo.names), False), (["HD"], True)):
        args, out, items, where, device_batch = tredmod.prepare_chunk(
            [("t001", copy, repo, names, 300, False, False, alts, True, "INFO")])
        assert device_batch is None and where == [(0, t) for t in names]
        gender = "Female" if len(names) > 1 else "Unknown"              # (gender only with an X-linked locus)
        assert out[0]["tredCalls"]["inferredGender"] == gender and out[0]["tredCalls"]["readLen"] == 150
        native = tredmod.ingest_loci(bam, repo, names, 150, alts, False, logging.getLogger())
        for t, (tred, readlen, g, depth, ev) in zip(names, items):
            assert tred is repo[t] and readlen == 150 and g == gender and depth == ev.depth
            _assert_same_record(ev, native[t])
        assert items[names.index("HD")][4].nreads > 50


def test_a_failing_genotyping_call_fails_its_chunk(monkeypatch, repo):
    """No second route: when the fused call raises, run_chunk raises and run_chunks(isolate=True) reports the chunk's
    samples as errors; the BAM is not read again."""
    from tredparse_b200 import tred as tredmod
    monkeypatch.setattr(tredmod, "GPU_INGEST", False)
    reads, calls = [], []
    ingest_loci = tredmod.ingest_loci

    def counted_ingest_loci(bam, *a, **k):
        reads.append(os.path.basename(bam))
        return ingest_loci(bam, *a, **k)

    def failing_genotype_evidence(items, **kw):
        calls.append(len(items))
        if len(calls) == 1:
            raise RuntimeError("fused call failed")
        return [{"1": 5} for _ in items]
    monkeypatch.setattr(tredmod, "ingest_loci", counted_ingest_loci)
    monkeypatch.setattr(tredmod, "genotype_evidence", failing_genotype_evidence)
    tasks = [(s, os.path.join(GOLDEN, s + ".mini.bam"), repo, [t], 300, False, False, True, True, "INFO")
             for s, t in CASES]
    got = list(tredmod.run_chunks(tasks, chunk=1, isolate=True))
    assert [r["samplekey"] for r in got] == ["t001", "t002"]
    assert got[0]["tredCalls"] == {} and "fused call failed" in got[0]["error"]
    assert "error" not in got[1] and got[1]["tredCalls"]["DM1.1"] == 5
    assert reads == ["t001.mini.bam", "t002.mini.bam"] and calls == [1, 1]
    del reads[:], calls[:]
    with pytest.raises(RuntimeError, match="fused call failed"):
        tredmod.run_chunk(tasks[:1])
    assert reads == ["t001.mini.bam"] and calls == [1]


# ---- corrupt input must not take the process down ---------------------------------------------------------------
_FUZZ = r"""
import os, sys, zlib, random
sys.path.insert(0, {root!r})
from tredparse_b200 import bamio, ingest
from tredparse_b200.meta import TREDsRepo
repo = TREDsRepo()
src = bamio.AlignmentFile({bam!r})
hd = repo["HD"]
recs = [r for r in src.fetch(hd.chr, hd.repeat_start - 3000, hd.repeat_end + 3000)]
refs = list(zip(src.references, src.lengths))
src.close()
path = os.path.join({tmp!r}, "stored.bam")
bamio.write_bam(path, refs, recs, level=0)                 # stored blocks: content bytes sit in the file as they are
good = open(path, "rb").read()
with ingest.BamIngest(path) as ing:
    base = ing.extract_locus(hd, 150, want_names=True)
assert base.nreads > 50
blocks, off = [], 0
while off < len(good):
    xlen = int.from_bytes(good[off + 10:off + 12], "little")
    bsize = int.from_bytes(good[off + 16:off + 18], "little") + 1
    blocks.append((off, xlen, bsize))
    off += bsize
rng = random.Random(3)
ok = failed = 0
for trial in range(150):
    bad = bytearray(good)
    off, xlen, bsize = blocks[rng.randrange(1, len(blocks) - 1)]      # not the header block, not the EOF block
    lo, hi = off + 12 + xlen, off + bsize - 8
    for _ in range(rng.randrange(1, 5)):
        p = rng.randrange(lo, hi)
        bad[p] = rng.randrange(256) if rng.random() < 0.5 else (bad[p] ^ (1 << rng.randrange(8)))
    try:                                                   # keep the block's CRC valid where it still inflates:
        data = zlib.decompress(bytes(bad[lo:hi]), -15)     # the damage must reach the record parser
        bad[off + bsize - 8:off + bsize - 4] = (zlib.crc32(data) & 0xffffffff).to_bytes(4, "little")
    except zlib.error:
        pass
    p2 = os.path.join({tmp!r}, "bad.bam")
    open(p2, "wb").write(bytes(bad))
    open(p2 + ".bai", "wb").write(open(path + ".bai", "rb").read())
    try:
        with ingest.BamIngest(p2) as ing:
            ev = ing.extract_locus(hd, 150, alts=hd.alt, want_names=True)
            ing.region_depth(hd.chr, hd.repeat_start - 1000, hd.repeat_end + 1000)
            ing.read_length(100)
        ok += 1
    except Exception:
        failed += 1
print("survived", ok, failed)
"""


def test_corrupt_bam_records_do_not_crash_the_reader(tmp_path):
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = _FUZZ.format(root=root, bam=os.path.join(GOLDEN, "t001.mini.bam"), tmp=str(tmp_path))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "survived" in r.stdout


def _damaged_copies(tmp_path):
    """The fixture truncated to half its size, and with one byte flipped in the middle of a compressed block."""
    import shutil
    src = os.path.join(GOLDEN, "t001.mini.bam")
    data = open(src, "rb").read()
    out = []
    for name, blob in (("truncated.bam", data[:len(data) // 2]),
                       ("flipped.bam", data[:len(data) // 2] + bytes([data[len(data) // 2] ^ 0x5A]) + data[len(data) // 2 + 1:])):
        p = str(tmp_path / name)
        with open(p, "wb") as fw:
            fw.write(blob)
        shutil.copy(src + ".bai", p + ".bai")
        out.append(p)
    return out


def test_truncated_or_corrupt_bam_is_an_error_not_partial_evidence(tmp_path):
    """A BGZF stream that ends early or fails its CRC must surface as an error from every native entry point — never
    as 'fewer reads' (pysam raises on such files; a silent partial result would become a plausible wrong genotype)."""
    from tredparse_b200 import ingest, _lib
    from tredparse_b200.meta import TREDsRepo
    hd = TREDsRepo()["HD"]
    with ingest.BamIngest(os.path.join(GOLDEN, "t001.mini.bam")) as good:
        ev = good.extract_locus(hd, 150, alts=())
        assert ev.nreads == 68 and abs(ev.depth - 29.3) < 0.1
    for path in _damaged_copies(tmp_path):
        with ingest.BamIngest(path) as ing:
            with pytest.raises(_lib.TredswError):
                ing.extract_locus(hd, 150, alts=())
            with pytest.raises(_lib.TredswError):
                ing.region_depth(hd.chr, hd.repeat_start - 1000, hd.repeat_end + 1000)


@pytest.mark.gpu
def test_run_reports_no_call_for_a_damaged_bam(tmp_path):
    """tred.run on a damaged BAM: the locus is skipped with an error logged (the reference's `except: continue`,
    tred.py:245-249), no genotype is invented."""
    from tredparse_b200 import tred as T
    from tredparse_b200.meta import TREDsRepo
    for path in _damaged_copies(tmp_path):
        try:
            res = T.run(("x", path, TREDsRepo(), ["HD"], 300, False, False, True, True, "INFO"))
        except Exception:
            continue                                     # raising is fine too
        assert "HD.1" not in res["tredCalls"] or res["tredCalls"]["HD.1"] == -1
