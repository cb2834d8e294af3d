"""Host-side logic of the path that needs no GPU: BAM/BAI reader, locus catalogue, model tables, template
families, synthetic problems, cohort packing, candidate ranges, CI / sparsify / label, JSON + VCF writers."""
import gzip
import json
import os

import numpy as np
import pytest

from tredparse_b200 import bamio, cohort, models, simulate, ssw, tred as T
from tredparse_b200.meta import TREDsRepo

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def repo():
    return TREDsRepo()


# ---- catalogue / tables --------------------------------------------------------------------------------
def test_catalogue(repo):
    assert len(repo.names) == 32
    locs = {(repo[n].chr, repo[n].repeat_start, repo[n].repeat_end) for n in repo.names}
    assert len(locs) == 30                                   # FXS == FXTAS, SBMA == AR coordinates
    hd = repo["HD"]
    assert (hd.chr, hd.repeat_start, hd.repeat_end) == ("chr4", 3074877, 3074933)
    assert hd.repeat == "CAG" and len(hd.prefix) == 18 and len(hd.suffix) == 18 and hd.ref_copy == 19
    assert all(len(repo[n].prefix) == 18 and len(repo[n].suffix) == 18 for n in repo.names)
    assert sorted({len(repo[n].repeat) for n in repo.names}) == [3, 4, 5, 6, 12]
    assert sum("N" in repo[n].repeat for n in repo.names) == 8      # GCN / NGC motifs need code 4


def test_model_tables():
    step, noise = models.StepModel(), models.NoiseModel()
    for p in range(1, 7):
        v = np.asarray(step.step_size_by_period[p])
        assert v.shape == (37,) and abs(v.sum() - 1) < 1e-6 or v[18] == 0
    assert np.array_equal(step.step_size_by_period[12], step.step_size_by_period[6])   # models.py:59-60
    w = noise.weights
    assert [round(x, 4) for x in w] == [-7.3673, -0.8652, 0.0824, -1.0402, 4.1705]
    assert 0 < noise.predict([3, 20, .68, 1.0]) < 1


def test_tables_equal_the_reference_files(repo):
    """The columns of the reference's TREDs.meta.csv and its step / stutter models, stored in golden/ref_tables.json."""
    with open(os.path.join(GOLDEN, "ref_tables.json")) as fp:
        ref = json.load(fp)
    assert sorted(ref["catalogue"]) == sorted(repo.names)
    for n in repo.names:
        row = ref["catalogue"][n]
        assert repo[n].repeat == row["repeat"] and repo[n].prefix == row["prefix"] and repo[n].suffix == row["suffix"]
        assert "{}:{}-{}".format(repo[n].chr, repo[n].repeat_start, repo[n].repeat_end) == \
            "{}:{}-{}".format(row["chr"], row["repeat_start"], row["repeat_end"])
    ours = models.StepModel().step_size_by_period
    for p, v in ref["step_size_by_period"].items():
        assert np.array_equal(np.asarray(ours[int(p)]), np.array(v))
    assert list(models.NoiseModel().weights) == ref["stutter_weights"]


# ---- BAM / BAI -----------------------------------------------------------------------------------------
def test_bam_fetch_indexed_equals_linear_scan(repo):
    sam = bamio.AlignmentFile(os.path.join(GOLDEN, "t001.mini.bam"))
    hd = repo["HD"]
    a, b = hd.repeat_start - 150, hd.repeat_end + 150
    idx = [(r.query_name, r.flag, r.reference_start) for r in sam.fetch(hd.chr, a, b)]
    tid = sam.get_tid(hd.chr)
    lin = [(r.query_name, r.flag, r.reference_start) for r in sam.fetch()
           if r.reference_id == tid and r.reference_start < b and
           ((r.reference_end or r.reference_start + 1) if not r.is_unmapped else r.reference_start + 1) > a]
    # (placed-but-unmapped mates are returned by a region fetch, like htslib does: bam_parser.py:206-214 wants them)
    assert idx and idx == lin
    assert all(len(r.query_sequence) == 150 for r in sam.fetch(hd.chr, a, b))
    d = bamio.region_depth(sam, hd.chr, hd.repeat_start - 1000, hd.repeat_end + 1000)
    assert 25 < d < 35                                      # t001 is a ~29x genome (SURVEY 8c)


def test_bam_write_read_roundtrip(tmp_path):
    src = bamio.AlignmentFile(os.path.join(GOLDEN, "t002.mini.bam"))
    recs = list(src.fetch())[:500]
    dst = str(tmp_path / "x.bam")
    bamio.write_bam(dst, list(zip(src.references, src.lengths)), recs)
    back = list(bamio.AlignmentFile(dst).fetch())
    assert len(back) == len(recs)
    for x, y in zip(recs, back):
        assert (x.query_name, x.flag, x.reference_id, x.reference_start, x.query_sequence, x.cigartuples) == \
               (y.query_name, y.flag, y.reference_id, y.reference_start, y.query_sequence, y.cigartuples)


# ---- templates / encoding ------------------------------------------------------------------------------
def test_family_descriptor_and_encoding(repo):
    t = repo["OPMD"]                                         # GCN motif: N must encode to 4
    fam = ssw.make_family(t.prefix, t.repeat, t.suffix, 50)
    assert fam["prefix_len"][0] == 18 and fam["suffix_len"][0] == 18 and fam["period"][0] == 3
    assert fam["max_units"][0] == 50 and 4 in fam["repeat"][0][:3]
    assert list(ssw.encode("ACGTNacgtX")) == [0, 1, 2, 3, 4, 0, 1, 2, 3, 4]
    m = ssw.score_matrix(1, 5)
    assert m.shape == (5, 5) and m[0, 0] == 1 and m[0, 1] == -5 and (m[4] == 0).all() and (m[:, 4] == 0).all()


# ---- synthetic problems / cohort packing ---------------------------------------------------------------
def test_simulation_is_seeded_and_shaped(repo):
    a = simulate.simulate_problem(repo["HD"], (15, 41), seed=5)
    b = simulate.simulate_problem(repo["HD"], (15, 41), seed=5)
    c = simulate.simulate_problem(repo["HD"], (15, 41), seed=6)
    assert np.array_equal(a.reads, b.reads) and np.array_equal(a.roff, b.roff)
    assert not np.array_equal(a.reads, c.reads)
    assert a.ploidy == 2 and a.readlen == 150 and set(np.diff(a.roff)) == {150}
    assert len(a.global_lens) == 2500 and a.reads.min() >= 0 and a.reads.max() <= 4
    h = simulate.simulate_problem(repo["FXS"], (30,), seed=1)
    assert h.ploidy == 1
    long_ = simulate.simulate_problem(repo["DM1"], (5, 1000), seed=2)        # full expansion (config 3 / 5)
    assert long_.nreads > a.nreads                                            # in-repeat reads are kept


def test_sample_bam_with_reads_longer_than_the_shortest_fragment(repo, tmp_path):
    """Fragments are drawn from [200, 999] bp.  For longer reads, a fragment shorter than the read has no full-length
    proper pair, so write_sample_bam drops it: every record is `<L>M` on the reference and read 2 never starts before
    read 1 (a short fragment used to give read 2 a negative haplotype index, which numpy wraps silently, or an
    IndexError).  The 150 bp sample the tred.run fixture is made of keeps its records."""
    from conftest import golden_module
    g = golden_module("make_oracle_bam_fixture")
    with open(os.path.join(GOLDEN, "oracle_sample_bam.json")) as fp:
        gold = json.load(fp)
    path = str(tmp_path / "s150.bam")
    g.write_sample(path, repo)
    assert g.records_sha1(path) == gold["records_sha1"]
    sam = bamio.AlignmentFile(os.path.join(GOLDEN, "t001.mini.bam"))
    refs = list(zip(sam.references, sam.lengths))
    sam.close()
    for L in (230, 251, 300):
        path = str(tmp_path / "s{}.bam".format(L))
        truth = simulate.write_sample_bam(path, repo, g.NAMES, refs, g.SAMPLE, readlen=L, flank=g.FLANK)
        assert sorted(truth) == sorted(g.NAMES)
        pairs = {}
        for r in bamio.AlignmentFile(path).fetch():
            assert len(r.query_sequence) == L and r.cigartuples == [(0, L)] and r.reference_start >= 0
            pairs.setdefault(r.query_name, {})[1 if r.flag & 0x40 else 2] = r
        assert len(pairs) > 1000
        for name, p in pairs.items():
            assert sorted(p) == [1, 2], name
            assert p[2].reference_start >= p[1].reference_start, name
            assert (p[1].next_reference_start, p[2].next_reference_start) == (p[2].reference_start, p[1].reference_start)


def test_cohort_packing_offsets(repo):
    probs = simulate.simulate_cohort(repo, ["HD", "DM1", "FRDA", "HD"], 2, readlen=150)
    batch = cohort.CohortBatch(probs)
    assert batch.nproblems == len(probs) == 8
    assert batch.nreads == sum(p.nreads for p in probs) == len(batch.roff) - 1
    assert batch.roff[0] == 0 and batch.roff[-1] == len(batch.rbuf) and (np.diff(batch.roff) == 150).all()
    assert np.array_equal(np.bincount(batch.read_problem, minlength=8), [p.nreads for p in probs])
    assert len(batch.families) == 3                                           # HD appears twice: one family
    P = batch.problems
    assert (P["off_target"] == P["off_global"] + P["n_global"]).all()
    assert P["off_global"][0] == 0 and P["off_target"][-1] + P["n_target"][-1] == len(batch.pe_lens)
    L = batch.loci[P["family"][0]]
    assert L["pe_minpe"] == L["pe_ref"] - 1 + 20                               # bam_parser.py:361


def test_packed_transfer_formats_roundtrip(repo):
    """pack_inputs(): two base codes per byte (base i in bits 4*(i&1) of byte i>>1), int16 pair lengths."""
    probs = simulate.simulate_cohort(repo, ["HD", "OPMD"], 1, readlen=150)
    batch = cohort.CohortBatch(probs).pack_inputs()
    pk, pe = batch._packed["rbuf"], batch._packed["pe_lens"]
    assert pk.dtype == np.uint8 and len(pk) % 4 == 0 and len(pk) >= (len(batch.rbuf) + 1) // 2
    un = np.empty(2 * len(pk), dtype=np.int8)
    un[0::2], un[1::2] = pk & 15, pk >> 4
    assert np.array_equal(un[:len(batch.rbuf)], batch.rbuf)
    assert pe.dtype == np.int16 and np.array_equal(pe.astype(np.int32), batch.pe_lens)
    assert pk.nbytes + pe.nbytes < 0.52 * (batch.rbuf.nbytes + batch.pe_lens.nbytes)


# ---- likelihood host logic -----------------------------------------------------------------------------
def test_candidate_ranges_follow_models_py():
    # models.py:239-257 — base = sorted(spanning keys U {max partial}); extended keeps duplicates (Q9)
    h1, h2 = models.candidate_ranges({45: 4, 150: 1}, {60: 1, 123: 2}, 0, 3, 132, 123, True, 300, False)[:2]
    assert list(h1) == [45, 123, 150]
    run_pe_h2 = models.candidate_ranges({45: 4}, {60: 1, 123: 2, 126: 2}, 0, 3, 132, 123, True, 300, False)
    assert list(run_pe_h2[1])[:2] == [45, 126] and list(run_pe_h2[1])[-1] == 900
    full = models.candidate_ranges({45: 4}, {60: 1}, 0, 3, 132, 123, False, 300, True)
    assert list(full[0]) == list(range(3, 901, 3)) == list(full[1])


def test_ci_sparsify_label(repo):
    P = {30: .01, 45: .5, 48: .46, 123: .03}
    lo, hi = models.calc_CI(P)
    assert (lo, hi) == (30, 123) or (lo, hi) == (45, 123)
    sp = models.sparsify({45: 1.0, 48: 1e-6, 51: 0.5}, 3)
    assert set(sp) == {"15", "17"} and abs(sp["15"] - 1 / 1.500001) < 1e-9        # dropped BEFORE normalising
    hd = repo["HD"]
    assert models.calc_label(hd, [15, 41]) == "risk" and models.calc_label(hd, [15, 20]) == "ok"
    assert models.calc_label(hd, [15, 37]) == "prerisk"
    assert models.mean_std([]) == "" and models.mean_std([300, 400]).endswith("bp")


# ---- writers -------------------------------------------------------------------------------------------
def test_json_and_vcf_writers(tmp_path, repo, capsys):
    calls = {"inferredGender": "Unknown", "depthY": 0.0, "readLen": 150,
             "HD.1": 15, "HD.2": 41, "HD.FR": "15|4", "HD.PR": "6|1", "HD.RR": "", "HD.DP": 29.3, "HD.FDP": 4,
             "HD.PDP": 1, "HD.RDP": 0, "HD.PEDP": 13, "HD.PEG": "346+/-78bp", "HD.PET": "301+/-53bp",
             "HD.CI": "15-15|40-42", "HD.PP": 0.99999, "HD.label": "risk", "HD.details": [],
             "HD.P_h1": {"15": 1.0}, "HD.P_h2": {"41": 1.0}, "HD.P_h1h2": {"15,41": 1.0}, "HD.P_PEG": "", "HD.P_PET": ""}
    res = {"samplekey": "s1", "bam": "s1.bam", "tredCalls": calls}
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        T.to_json(res, "hg38", repo, treds=["HD"])
        T.to_vcf(res, "hg38", repo, treds=["HD"])
    finally:
        os.chdir(cwd)
    text = open(tmp_path / "s1.json").read()
    assert text.rstrip("\n") == json.dumps(res, sort_keys=True, indent=4, separators=(",", ": "))   # tred.py:296-310
    assert capsys.readouterr().out.strip() == text.strip()
    vcf = gzip.open(tmp_path / "s1.tred.vcf.gz", "rt").read().splitlines()
    assert vcf[0] == "##fileformat=VCFv4.1" and vcf[-1].startswith("chr4\t3074877\tHD\t" + "CAG" * 19)
    f = vcf[-1].split("\t")
    assert f[8] == "GT:GB:FR:PR:RR:DP:FDP:PDP:RDP:PEDP:CI:PP:LABEL" and f[9].startswith("1/2:15/41:15|4:6|1::29.3:4:1:0:13:")
    assert T.counter_s({15: 4, 6: 1}) == "6|1;15|4"


def test_run_chunks_keeps_order_prefetches_and_isolates_failures(monkeypatch):
    """tred.run_chunks: chunk k + 1 is prepared while chunk k is finished, results come back in input order, and with
    isolate=True a chunk that raises yields error records for its samples instead of ending the run."""
    import threading
    from tredparse_b200 import tred as T
    log, lock = [], threading.Lock()

    def fake_prepare(args, only=None, ctx=None):
        with lock:
            log.append(("prep", args[0][0]))
        if args[0][0] == "s4":
            raise RuntimeError("boom")
        return list(args)

    def fake_finish(state, ctx=None):
        with lock:
            log.append(("fin", state[0][0]))
        return [{"samplekey": a[0], "bam": a[1], "tredCalls": {"x": 1}} for a in state]
    monkeypatch.setattr(T, "prepare_chunk", fake_prepare)
    monkeypatch.setattr(T, "finish_chunk", fake_finish)
    monkeypatch.setattr(T, "GPU_INGEST", False)
    args = [("s{}".format(i), "b{}".format(i)) for i in range(7)]
    got = list(T.run_chunks(args, chunk=2, isolate=True))
    assert [r["samplekey"] for r in got] == ["s{}".format(i) for i in range(7)]
    assert "error" in got[4] and "error" in got[5] and "boom" in got[4]["error"] and got[4]["tredCalls"] == {}
    assert all("error" not in got[i] for i in (0, 1, 2, 3, 6))
    # chunk 1 (s2) is prepared before chunk 0 (s0) is finished: two stages deep
    assert log.index(("prep", "s2")) < log.index(("fin", "s2")) and ("fin", "s4") not in log
    with pytest.raises(RuntimeError):
        list(T.run_chunks(args, chunk=2))
