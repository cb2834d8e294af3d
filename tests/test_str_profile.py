"""The STR profile of a scan (DESIGN §4.5): in-repeat reads (IRRs) found by the scan's IRR stage
(tredsw_ingest_scan_run_ex), joined, anchored and merged by tredparse_b200.strprofile, compared across a cohort by
strprofile.outliers — everything against oracle/irr_oracle.py, the definitions in plain Python over bamio records.

CPU tests run the device code serially on the host (tredsw_ingest_scan_emulate_ex, tredsw_irr_classify_host: test
infrastructure); the `gpu` tests run the kernels."""
import contextlib
import json
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
SLAB_TINY = 65536
FAR = "AAGGG"                 # the expansion planted away from the catalogue


def _refs():
    from tredparse_b200 import bamio
    sam = bamio.AlignmentFile(os.path.join(GOLDEN, "t001.mini.bam"))
    refs = list(zip(sam.references, sam.lengths))
    sam.close()
    return refs


def _tid(refs, name):
    return [n for n, _ in refs].index(name)


def _background(refs, seed, n=300, readlen=150):
    """proper pairs scattered over the first contigs (depth, and records that are not IRRs)"""
    from tredparse_b200 import simulate
    rng = np.random.default_rng(seed)
    recs = []
    for k in range(n):
        t = int(rng.integers(0, 3))
        p = int(rng.integers(1000, refs[t][1] - 1000))
        recs += simulate.expansion_records(t, p, "AC", 0, readlen=readlen, cov=2, flank=400, seed=seed * 1000 + k,
                                           tag="bg{}_{}_".format(seed, k))
    return recs


def _whole_sample(path, seed=1, mq_tags=True, far_units=200, readlen=150):
    """catalogue loci (simulate.locus_records), a CAG expansion at HD, an AAGGG expansion away from the catalogue with
    mismapped IRRs, background pairs"""
    from tredparse_b200 import bamio, simulate
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    refs = _refs()
    recs = _background(refs, seed, readlen=readlen)
    for li, name in enumerate(("HD", "DM1", "FXS")):
        t = repo[name]
        if t.chr in [n for n, _ in refs]:
            recs += simulate.locus_records(t, _tid(refs, t.chr), (15, 60), readlen, 5.0, seed=seed + li, tag="l{}".format(li),
                                           flank=1000)
    hd = repo["HD"]
    recs += simulate.expansion_records(_tid(refs, hd.chr), hd.repeat_start + 5000, "CAG", 120, readlen=readlen, cov=8,
                                       seed=seed + 10, tag="hd", mq_tags=mq_tags)
    far = (1, refs[1][1] // 2)
    recs += simulate.expansion_records(far[0], far[1], FAR, far_units, readlen=readlen, cov=10, seed=seed + 20, tag="far",
                                       mq_tags=mq_tags, mismap_fraction=0.3, mismap_to=(2, 1000, refs[2][1] - 1000))
    bamio.write_bam(path, refs, simulate.coordinate_sort(recs), index=False, aux=True)
    return path


def _with_decoys(path, src):
    """secondary / supplementary / duplicate / QC-fail copies of IRR records, single-end IRRs, corrupt aux areas"""
    from tredparse_b200 import bamio, simulate
    from oracle import irr_oracle
    sam = bamio.AlignmentFile(src)
    refs = list(zip(sam.references, sam.lengths))
    recs = list(sam.fetch())
    sam.close()
    irr = [r for r in recs if irr_oracle.classify(r.query_sequence)[0]]
    extra = []
    bad_aux = [b"MQ", b"XZZabc", b"XYq\x01", b"MQf\x00\x00\x80?", b"MQc\xfb", b"XBBc\x03\x00\x00\x00abc" + b"MQi\x39\x00\x00\x00",
               b"XBBq\x01\x00\x00\x00a", b"MQI\xff\xff\xff\xff", b"RGZgrp\x00MQs\x28\x00"]
    for k, r in enumerate(irr[:60]):
        c = bamio.AlignedSegment(r.query_name, r.flag | (0x100, 0x800, 0x400, 0x200)[k % 4], r.reference_id,
                                 r.reference_start, r.mapping_quality, r.cigartuples, r.next_reference_id,
                                 r.next_reference_start, 0, r.query_sequence, aux=r.aux)
        extra.append(c)
    for k, r in enumerate(irr[60:60 + len(bad_aux)]):
        r.aux = bad_aux[k]
    for k, r in enumerate(irr[80:100]):                        # single-end reads: no 0x1, no segment flags
        extra.append(bamio.AlignedSegment("se{}".format(k), r.flag & 0x14, r.reference_id, r.reference_start,
                                          r.mapping_quality, r.cigartuples, -1, -1, 0, r.query_sequence, aux=r.aux))
    bamio.write_bam(path, refs, simulate.coordinate_sort(recs + extra), index=False, aux=True)
    return path


@pytest.fixture(scope="module")
def bams(tmp_path_factory):
    d = tmp_path_factory.mktemp("strprofile")
    out = {"sample": _whole_sample(str(d / "sample.bam")),
           "no_mq": _whole_sample(str(d / "no_mq.bam"), seed=2, mq_tags=False),
           "short": _whole_sample(str(d / "short.bam"), seed=3, readlen=100)}
    out["decoys"] = _with_decoys(str(d / "decoys.bam"), out["sample"])
    return out


def _entry_keys(irr):
    """the IRR entries of a scan as a sorted list of per-record tuples"""
    e = irr["entries"]
    return sorted((n, int(x["tid"]), int(x["pos"]), int(x["next_tid"]), int(x["next_pos"]), int(x["flag"]),
                   int(x["mapq"]), int(x["mq"]), int(x["period"]), int(x["motif"])) for n, x in zip(irr["names"], e))


def _oracle_keys(entries):
    return sorted((e["name"], e["tid"], e["pos"], e["next_tid"], e["next_pos"], e["flag"], e["mapq"], e["mq"],
                   e["period"], e["motif"]) for e in entries)


def _scan_irr(ctx, path, slab_bytes=None, params=None):
    from tredparse_b200 import ingest
    h = ingest.BamIngest.unindexed(path)
    try:
        with ingest.scan_sample(ctx, h, [], [], [], slab_bytes=slab_bytes, irr=params or ingest.IrrParams()) as b:
            assert b.scan_status == 0
            return b.irr
    finally:
        h.close()


# ---------------------------------------------------------------------------------------------------------------
# the classifier
# ---------------------------------------------------------------------------------------------------------------
def _crafted(rng):
    """sequences (code lists) around every rule of the classifier"""
    out = []
    rand = lambda n: rng.integers(0, 4, n).tolist()
    for k in range(2, 22):                                  # every period 2..20, and 21 (rejected)
        for _ in range(40):
            m = rand(k)
            L = int(rng.integers(50, 200))
            s = (m * (L // k + 1))[:L]
            for i in rng.choice(L, int(rng.integers(0, L // 8)), replace=False):
                s[i] = int(rng.integers(0, 5))
            out.append(s)
    for b in range(5):                                      # homopolymers, with noise
        for _ in range(20):
            s = [b] * int(rng.integers(50, 160))
            for i in rng.choice(len(s), int(rng.integers(0, 10)), replace=False):
                s[i] = int(rng.integers(0, 4))
            out.append(s)
    for _ in range(3000):                                   # AT / ATAT near the threshold (reduced to AT)
        L = int(rng.integers(50, 160))
        s = ([0, 3] * L)[:L]
        for i in rng.choice(L, int(rng.integers(L // 25, L // 6)), replace=False):
            s[i] = int(rng.integers(0, 5))
        out.append(s)
    for _ in range(500):                                    # N runs and an all-N phase
        k = int(rng.integers(2, 9))
        m = rand(k)
        L = int(rng.integers(60, 150))
        s = (m * (L // k + 1))[:L]
        a, run = int(rng.integers(0, L - 10)), int(rng.integers(1, 12))
        for i in range(a, min(L, a + run)):
            s[i] = 4
        if rng.random() < 0.5:
            ph = int(rng.integers(0, k))
            for i in range(ph, L, k):
                s[i] = 4
        out.append(s)
        out.append([3 - c if c < 4 else 4 for c in reversed(s)])       # its reverse complement
    for _ in range(200):                                    # lengths below and at min_read_len
        out.append(([1, 2, 2] * 30)[:int(rng.integers(40, 52))])
    return out


def _exact_threshold(s, num=9, den=10, kmin=2, kmax=20):
    for k in range(kmin, kmax + 1):
        n = len(s) - k
        m = sum(1 for i in range(n) if s[i] < 4 and s[i] == s[i + k])
        if m * den == num * n:
            return True
    return False


def test_classifier_equals_oracle():
    from tredparse_b200 import ingest
    from oracle import irr_oracle
    rng = np.random.default_rng(7)
    seqs = _crafted(rng)
    while len(seqs) < 100000:
        seqs.append(rng.integers(0, 4, int(rng.integers(50, 180))).tolist())
    at_threshold = sum(_exact_threshold(s) for s in seqs[:12000])
    assert at_threshold >= 20, at_threshold             # the crafted set does hit m * den == num * (L - k)
    kinds = set()
    for s in seqs:
        got = ingest.irr_classify_host(s)
        want = irr_oracle.classify(s)
        assert got == want, (s, got, want)
        kinds.add(got[0])
    assert kinds >= set(range(2, 21)) | {0}, kinds
    # ATAT-like reads are reported as AT, homopolymers and period-21 reads are not IRRs
    assert ingest.irr_classify_host([0, 3, 0, 3] * 20) == (2, 0b0011)
    assert ingest.irr_classify_host([2] * 100) == (0, 0)
    # other parameters
    p = ingest.IrrParams(min_period=3, max_period=12, purity_num=4, purity_den=5, min_read_len=30)
    for s in seqs[:20000]:
        assert ingest.irr_classify_host(s, p) == irr_oracle.classify(s, 3, 12, 4, 5, 30)


def test_out_of_range_parameters():
    import ctypes
    from tredparse_b200 import _lib, ingest
    bad = [dict(min_period=1), dict(min_period=5, max_period=4), dict(max_period=21, min_read_len=50),
           dict(purity_num=0), dict(purity_num=11, purity_den=10), dict(purity_num=900, purity_den=1001),
           dict(max_period=20, min_read_len=39)]
    lib = _lib.load()
    ingest._bind_batch(lib)
    for kw in bad:
        p = ingest.IrrParams(**kw)
        per, mot = ctypes.c_int32(), ctypes.c_uint64()
        codes = np.zeros(100, np.int8)
        assert lib.tredsw_irr_classify_host(codes.ctypes.data, 100, ctypes.byref(p), ctypes.byref(per),
                                            ctypes.byref(mot)) == -2, kw
        h = ingest.BamIngest.unindexed(os.path.join(GOLDEN, "t001.mini.bam"))
        out = ctypes.c_void_p()
        assert lib.tredsw_ingest_scan_emulate_ex(h.handle, None, 0, None, 0, None, 0, 0, ctypes.byref(p),
                                                 ctypes.byref(out)) == -2, kw
        assert not out.value
        h.close()


# ---------------------------------------------------------------------------------------------------------------
# the scan's IRR stage (host emulation of the device code) and the profile
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["sample", "no_mq", "short", "decoys"])
@pytest.mark.parametrize("slab", [None, SLAB_TINY])
def test_scan_entries_and_profile_equal_oracle(bams, which, slab):
    from tredparse_b200 import strprofile
    from oracle import irr_oracle
    path = bams[which]
    want = irr_oracle.scan(path)
    irr = _scan_irr(None, path, slab_bytes=slab)
    assert _entry_keys(irr) == _oracle_keys(want["entries"])
    for k in ("records_considered", "irr_records", "depth_bases", "max_l_seq", "unparsed_aux"):
        assert irr["stats"][k] == want["stats"][k], k
    got = strprofile.profile(path, emulate=True, slab_bytes=slab)
    ref = irr_oracle.profile(path, sample=got["sample"])
    assert got == ref
    assert got["profile"][FAR]["anchored_irr_count"] > 3 and got["profile"][FAR]["paired_irr_count"] > 3
    if which == "no_mq":
        assert got["stats"]["anchors_without_mq"] == got["stats"]["anchored_irrs"] > 0
    if which == "decoys":
        assert got["stats"]["unparsed_aux"] >= 4


def test_profile_parameters_equal_oracle(bams):
    from tredparse_b200 import strprofile
    from oracle import irr_oracle
    kw = dict(min_period=3, max_period=6, purity_num=17, purity_den=20, min_read_len=60)
    got = strprofile.profile(bams["decoys"], emulate=True, min_anchor_mapq=61, merge_distance=50, **kw)
    ref = irr_oracle.profile(bams["decoys"], kw, min_anchor_mapq=61, merge_distance=50, sample=got["sample"])
    assert got == ref and got["stats"]["anchors_below_mapq"] > 0


def test_irr_stage_leaves_the_scan_unchanged(bams):
    """with irr set, the evidence, depths and statistics of a scan with queries equal the same scan without it"""
    from tredparse_b200 import ingest
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    runs = []
    for irr in (None, ingest.IrrParams()):
        h = ingest.BamIngest.unindexed(bams["sample"])
        qs, keep = [], []
        for n in ("HD", "DM1", "FXS", "SCA1"):
            q = ingest.locus_query(h, repo[n], 150, alts=repo[n].alt)
            if q is not None:
                qs.append(q[0]); keep.append(q[1])
        dr = [(0, 1000, 90000), (1, 0, 5000)]
        with ingest.scan_sample(None, h, qs, keep, dr, slab_bytes=SLAB_TINY, irr=irr) as b:
            ev = [b.evidence(i) for i in range(len(qs))]
            st = {k: v for k, v in b.stats().items() if not k.startswith("ms_")}
            runs.append((ev, list(b.depths), st, b.status.tolist(), b.scan_status, b.irr))
        h.close()
    (e0, d0, s0, p0, c0, i0), (e1, d1, s1, p1, c1, i1) = runs
    assert i0 is None and i1["stats"]["irr_records"] > 0
    assert d0 == d1 and s0 == s1 and p0 == p1 and c0 == c1 == 0
    for x, y in zip(e0, e1):
        assert (np.array_equal(x.reads, y.reads) and np.array_equal(x.roff, y.roff) and x.names == y.names
                and np.array_equal(x.global_lens, y.global_lens) and np.array_equal(x.target_lens, y.target_lens)
                and x.depth == y.depth and x.n_unmapped == y.n_unmapped)


def test_profile_of_a_corrupt_file_raises(tmp_path, bams):
    from tredparse_b200 import strprofile
    data = bytearray(open(bams["sample"], "rb").read())
    bad = tmp_path / "truncated.bam"
    bad.write_bytes(bytes(data[:len(data) * 2 // 3]))
    with pytest.raises(IOError):
        strprofile.profile(str(bad), emulate=True)


def test_join_anchor_and_merge_rules_by_hand(tmp_path):
    """a small BAM whose profile is written out by hand: pairs, anchors, the MQ rule, merging, decoys"""
    from tredparse_b200 import bamio, simulate, strprofile
    from oracle import irr_oracle
    AS = bamio.AlignedSegment
    at, aag = "AT" * 50, ("AAG" * 34)[:100]
    rnd = "".join("ACGT"[int(x)] for x in np.random.default_rng(3).integers(0, 4, 100))
    mq = lambda v: b"MQC" + bytes([v])
    M = [(0, 100)]
    recs = []

    def anchored(name, tid, pos, aux):            # an unmapped IRR at its mapped mate's position, and the mate
        recs.append(AS(name, 0x1 | 0x4 | 0x40, tid, pos, 0, [], tid, pos, 0, at, aux=aux))
        recs.append(AS(name, 0x1 | 0x8 | 0x80, tid, pos, 60, M, tid, pos, 0, rnd))
    anchored("A", 0, 1000, mq(60))
    anchored("B", 0, 1400, mq(55))                 # 400 bp from A: the same region
    anchored("C", 0, 1450, mq(10))                 # MQ below 50: not an anchor
    anchored("D", 0, 2000, b"")                    # no MQ: counted, and in anchors_without_mq; 600 bp from B: a new region
    anchored("I", 1, 300, mq(60))
    recs.append(AS("A", 0x1 | 0x4 | 0x40 | 0x100, 0, 1000, 0, [], 0, 1000, 0, at, aux=mq(60)))      # secondary: ignored
    for name, s1, s2 in (("E", at, at), ("F", at, aag), ("G", at, rnd)):   # unmapped tail: paired, two motifs, mate unmapped
        recs.append(AS(name, 0x1 | 0x4 | 0x8 | 0x40, -1, -1, 0, [], -1, -1, 0, s1))
        recs.append(AS(name, 0x1 | 0x4 | 0x8 | 0x80, -1, -1, 0, [], -1, -1, 0, s2))
    path = str(tmp_path / "hand.bam")
    # a header without @SQ lines: contigs and lengths come from the binary reference dictionary
    bamio.write_bam(path, [("c1", 100000), ("c2", 50000)], simulate.coordinate_sort(recs), index=False, aux=True,
                    header_text="@HD\tVN:1.4\tSO:coordinate\n")
    want = {"AT": {"anchored_irr_count": 4, "paired_irr_count": 1,
                   "regions": [{"contig": "c1", "start": 1000, "end": 1401, "count": 2},
                               {"contig": "c1", "start": 2000, "end": 2001, "count": 1},
                               {"contig": "c2", "start": 300, "end": 301, "count": 1}]}}
    for prof in (strprofile.profile(path, emulate=True), irr_oracle.profile(path, sample="hand")):
        st = prof["stats"]
        assert prof["profile"] == want
        assert (st["irr_records"], st["anchored_irrs"], st["paired_irrs"], st["irr_pairs_motif_mismatch"],
                st["anchors_below_mapq"], st["anchors_without_mq"]) == (10, 4, 1, 1, 1, 1)
        assert prof["depth"] == 5 * 100 / 150000 and prof["read_length"] == 100


def test_cli_refuses_sample_keys_that_repeat(tmp_path):
    """two inputs with one sample key would write one profile over the other: refused before anything is read"""
    for d in ("a", "b"):
        os.makedirs(str(tmp_path / d))
        open(str(tmp_path / d / "x.bam"), "wb").close()
    r = subprocess.run([sys.executable, "-m", "tredparse_b200.strprofile", "profile", str(tmp_path / "a" / "x.bam"),
                        str(tmp_path / "b" / "x.bam"), "--workdir", str(tmp_path / "w")],
                       env=dict(os.environ, PYTHONPATH=ROOT), cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 2 and "repeat" in r.stderr and not os.path.exists(str(tmp_path / "w"))


def test_outlier_rows_by_hand():
    """three profiles at depth 40 (a normalised count is the count): region merging across samples, z, the sort"""
    from tredparse_b200 import strprofile
    from oracle import irr_oracle

    def prof(name, regions, paired=0):
        return {"sample": name, "depth": 40.0, "params": {"merge_distance": 500},
                "profile": {"AT": {"anchored_irr_count": sum(r[3] for r in regions), "paired_irr_count": paired,
                                   "regions": [dict(zip(("contig", "start", "end", "count"), r)) for r in regions]}}}
    profs = [prof("a", [("c1", 100, 200, 10)]), prof("b", [("c1", 600, 700, 2)]), prof("c", [("c1", 5000, 5001, 1)])]
    # [100, 700): a 10, b 2, c 0 -> z_a = (10 - 1) / max(1, 1) = 9; [5000, 5001): c 1 -> z_c = 1; paired: all 0 -> z 0
    want = [("c1", 100, 700, "a", 9.0, [10.0, 2.0, 0.0]), ("c1", 5000, 5001, "c", 1.0, [0.0, 0.0, 1.0]),
            ("-", None, None, "a", 0.0, [0.0, 0.0, 0.0])]
    for rows in (strprofile.outliers(profs), irr_oracle.outliers(profs)):
        assert [(r["contig"], r["start"], r["end"], r["top_sample"], r["z"], [r["counts"][s] for s in "abc"])
                for r in rows] == want


# ---------------------------------------------------------------------------------------------------------------
# the cohort
# ---------------------------------------------------------------------------------------------------------------
COHORT_REFS = [("c1", 30000), ("c2", 20000), ("c3", 12000)]     # small contigs: a depth of about 10x


def _cohort_sample(path, s, planted):
    from tredparse_b200 import bamio, simulate
    refs = COHORT_REFS
    recs = _background(refs, 100 + s, n=300)
    rng = np.random.default_rng(s)
    # every sample: a CAG site and an ATTC site of varying length; the planted one: an AAGGG expansion of 400 bp
    if planted:
        recs += simulate.expansion_records(1, 10000, FAR, 80, cov=8, seed=500 + s, tag="far{}_".format(s))
    recs += simulate.expansion_records(0, 15000, "CAG", int(rng.integers(40, 70)), cov=8, seed=600 + s, tag="cag{}_".format(s))
    recs += simulate.expansion_records(2, 6000, "ATTC", int(rng.integers(35, 60)), cov=8, seed=700 + s, tag="attc{}_".format(s))
    bamio.write_bam(path, refs, simulate.coordinate_sort(recs), index=False, aux=True)
    return path


@pytest.fixture(scope="module")
def cohort(tmp_path_factory):
    d = tmp_path_factory.mktemp("cohort")
    return [_cohort_sample(str(d / "s{}.bam".format(s)), s, planted=(s == 4)) for s in range(6)]


def _same_rows(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert {k: x[k] for k in ("contig", "start", "end", "motif", "top_sample")} == \
               {k: y[k] for k in ("contig", "start", "end", "motif", "top_sample")}
        assert x["z"] == pytest.approx(y["z"], rel=1e-12, abs=1e-12)
        assert x["counts"] == pytest.approx(y["counts"], rel=1e-12, abs=1e-12)


def test_outliers_rank_the_planted_expansion_first(cohort):
    from tredparse_b200 import strprofile
    from oracle import irr_oracle
    profs = [strprofile.profile(p, emulate=True) for p in cohort]
    for p, path in zip(profs, cohort):
        assert p == irr_oracle.profile(path, sample=p["sample"])
    rows = strprofile.outliers(profs)
    _same_rows(rows, irr_oracle.outliers(profs))
    top = rows[0]
    assert top["top_sample"] == "s4" and top["motif"] == FAR and top["contig"] == "c2"
    assert top["start"] - 500 <= 10000 < top["end"] + 500 and top["z"] > 3
    with pytest.raises(ValueError):
        strprofile.outliers(profs[:1])


# ---------------------------------------------------------------------------------------------------------------
# on the GPU
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("slab", [None, SLAB_TINY])
def test_gpu_entries_equal_emulation_and_oracle(bams, slab):
    from tredparse_b200 import _lib, strprofile
    from oracle import irr_oracle
    ctx = _lib.default_context(0)
    for which, path in sorted(bams.items()):
        dev, emu = _scan_irr(ctx, path, slab_bytes=slab), _scan_irr(None, path, slab_bytes=slab)
        assert np.array_equal(dev["entries"], emu["entries"]) and dev["names"] == emu["names"], which
        assert dev["stats"] == emu["stats"], which
        got = strprofile.profile(path, ctx=ctx, slab_bytes=slab)
        assert got == irr_oracle.profile(path, sample=got["sample"]), which


@contextlib.contextmanager
def _piped(path):
    r, w = os.pipe()
    data = open(path, "rb").read()

    def feed():
        try:
            for i in range(0, len(data), 40000):
                os.write(w, data[i:i + 40000])
        except BrokenPipeError:
            pass
        finally:
            os.close(w)
    t = threading.Thread(target=feed, daemon=True)
    t.start()
    try:
        yield "/dev/fd/{}".format(r)
    finally:
        os.close(r)
        t.join(timeout=60)


@pytest.mark.gpu
def test_gpu_pipe_gives_the_file_profile(bams):
    from tredparse_b200 import _lib, strprofile
    ctx = _lib.default_context(0)
    want = strprofile.profile(bams["decoys"], ctx=ctx, sample="x")
    with _piped(bams["decoys"]) as p:
        got = strprofile.profile(p, ctx=ctx, sample="x", slab_bytes=SLAB_TINY)
    got["bam"] = want["bam"]
    assert got == want


@pytest.mark.gpu
def test_gpu_cli_writes_profiles_and_table(cohort, tmp_path):
    from tredparse_b200 import strprofile
    from oracle import irr_oracle
    env = dict(os.environ, PYTHONPATH=ROOT)
    work = tmp_path / "w"
    subprocess.run([sys.executable, "-m", "tredparse_b200.strprofile", "profile", *cohort, "--workdir", str(work),
                    "--slab-bytes", str(SLAB_TINY)], check=True, env=env, cwd=ROOT)
    files = [str(work / "s{}.str_profile.json".format(s)) for s in range(6)]
    profs = []
    for f, path in zip(files, cohort):
        with open(f) as fp:
            p = json.load(fp)
        assert p == json.loads(json.dumps(irr_oracle.profile(path, sample=os.path.basename(f).split(".")[0])))
        profs.append(p)
    tsv = tmp_path / "out.tsv"
    subprocess.run([sys.executable, "-m", "tredparse_b200.strprofile", "outliers", *files, "--tsv", str(tsv)],
                   check=True, env=env, cwd=ROOT)
    lines = tsv.read_text().splitlines()
    assert lines[0].split("\t") == ["contig", "start", "end", "motif", "top_sample", "z"] + ["s{}".format(s) for s in range(6)]
    rows = irr_oracle.outliers(profs)
    assert len(lines) == len(rows) + 1
    first = lines[1].split("\t")
    assert first[3] == FAR and first[4] == "s4" and first[:3] == [rows[0]["contig"], str(rows[0]["start"]), str(rows[0]["end"])]
