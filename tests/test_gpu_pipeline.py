"""End-to-end parity on the reference's fixtures: tredparse_b200.tred.run (BamParser / IntegratedCaller
API, GPU kernels) vs. the CPU oracle of the same loop and the values the reference pins in its README.
Needs a GPU: run with -m gpu."""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
CASES = [("t001", "HD"), ("t002", "DM1")]


def _models():
    md = json.load(open(os.path.join(os.path.dirname(GOLDEN), "..", "tredparse_b200", "data", "models.json")))
    step = {int(k): np.array(v) for k, v in md["step_size_by_period"].items()}
    for i in range(6, 18):
        step[i] = step[6]
    return step, md["stutter_weights"]


def _close(a, b, rtol=1e-9):
    if isinstance(a, dict):
        assert set(a) == set(b)
        for k in a:
            _close(a[k], b[k], rtol)
    elif isinstance(a, float) or isinstance(b, float):
        assert abs(a - b) <= rtol * max(abs(a), abs(b)) + 1e-15, (a, b)
    else:
        assert a == b, (a, b)


@pytest.mark.parametrize("sample,tredname", CASES)
def test_run_matches_oracle_and_readme(sample, tredname):
    from tredparse_b200 import tred as T, bamio
    from tredparse_b200.meta import TREDsRepo
    from oracle import genotype_oracle, evidence_oracle as evo
    repo = TREDsRepo()
    bam = os.path.join(GOLDEN, sample + ".mini.bam")
    res = T.run((sample, bam, repo, [tredname], 300, False, False, True, True, "INFO"))
    calls = res["tredCalls"]
    step, w = _models()
    sam = bamio.AlignmentFile(bam)
    exp, ev, lk = genotype_oracle.genotype_locus(sam, repo[tredname], evo.read_length(sam), step, w)
    assert calls["readLen"] == 150 and calls["inferredGender"] == "Unknown"
    for k, v in exp.items():
        _close(calls[tredname + "." + k], v)
    # what the reference itself pins (README.md:77-86)
    if sample == "t001":
        assert (calls["HD.1"], calls["HD.2"]) == (15, 41)
        assert calls["HD.FR"] == "15|4" and calls["HD.RR"] == "" and calls["HD.PR"].endswith("|1;21|1;24|2;29|1;34|1;41|1")
        assert round(calls["HD.PP"], 6) == 1 and calls["HD.label"] == "risk"
    else:
        assert calls["DM1.1"] == 5 and calls["DM1.FR"] == "5|24" and calls["DM1.RR"] == "49|3;50|8"
        assert calls["DM1.PR"].endswith("|1;39|1;40|1;42|1;43|1;46|2")
    json.dumps(res, sort_keys=True, indent=4, separators=(",", ": "))   # serialisable, reference layout


def test_runBam_equals_batched_run():
    from tredparse_b200 import tred as T
    from tredparse_b200.meta import TREDsRepo
    from tredparse_b200.utils import InputParams
    from tredparse_b200.bam_parser import BamDepth
    import logging
    repo = TREDsRepo()
    bam = os.path.join(GOLDEN, "t001.mini.bam")
    res = T.run(("t001", bam, repo, ["HD"], 300, False, False, True, True, "INFO"))["tredCalls"]
    depth = BamDepth(bam, "hg38", logging.getLogger()).region_depth("chr4", 3074877 - 1000, 3074933 + 1000)
    ip = InputParams(bam=bam, READLEN=150, tredName="HD", repo=repo, maxinsert=300, fullsearch=False,
                     gender="Unknown", depth=depth, clip=False, alts=True, repeatpairs=True, log="INFO")
    r = T.runBam(ip)
    assert r.alleles == [res["HD.1"], res["HD.2"]] and r.CI == res["HD.CI"] and abs(r.PP - res["HD.PP"]) < 1e-12
    _close(r.P_h1, res["HD.P_h1"], 1e-12); _close(r.P_h1h2, res["HD.P_h1h2"], 1e-12)      # (per-stage vs fused path: summation order)
    assert r.label == res["HD.label"]
    assert T.counter_s(r.counts["PREF"]) == res["HD.PR"]


def test_all_catalogue_loci_on_both_fixtures():
    """BASELINE config 2: every catalogue TRED on t001 + t002 — loci without reads come out 'missing'
    (alleles -1/-1, PP -1, CI ''), exactly like the reference (models.py:244-245,406-412)."""
    from tredparse_b200 import tred as T
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    for sample, hit in CASES:
        bam = os.path.join(GOLDEN, sample + ".mini.bam")
        calls = T.run((sample, bam, repo, repo.names, 300, False, False, True, True, "INFO"))["tredCalls"]
        for name in repo.names:
            if name == hit:
                assert calls[name + ".label"] in ("ok", "prerisk", "risk") and calls[name + ".1"] > 0
            else:
                assert (calls[name + ".1"], calls[name + ".2"]) == (-1, -1)
                assert calls[name + ".PP"] == -1 and calls[name + ".CI"] == "" and calls[name + ".label"] == "missing"


def test_unindexed_bams_equal_the_indexed_run_and_the_oracle(tmp_path):
    """BAMs without a .bai: the Python reader builds the evidence records and the same fused call genotypes them.
    The calls equal those of the indexed files (floats at the bar of test_runBam_equals_batched_run) and the CPU
    oracle's at 1e-9.  Every catalogue locus without the alt regions (each alt region is a scan of the whole
    unindexed file), and the locus with reads with them."""
    import shutil
    from tredparse_b200 import tred as T, bamio
    from tredparse_b200.meta import TREDsRepo
    from oracle import genotype_oracle, evidence_oracle as evo
    repo = TREDsRepo()
    step, w = _models()
    for sample, hit in CASES:
        bam = os.path.join(GOLDEN, sample + ".mini.bam")
        copy = str(tmp_path / (sample + ".noindex.bam"))
        shutil.copy(bam, copy)
        sam = bamio.AlignmentFile(bam)
        for names, alts in ((list(repo.names), False), ([hit], True)):
            indexed, unindexed = [T.run((sample, path, repo, names, 300, False, False, alts, True, "INFO"))["tredCalls"]
                                  for path in (bam, copy)]
            _close(unindexed, indexed, 1e-12)
            assert unindexed[hit + ".1"] > 0
            for name in names:
                exp = genotype_oracle.genotype_locus(sam, repo[name], evo.read_length(sam), step, w, alts=alts)[0]
                for k, v in exp.items():
                    _close(unindexed[name + "." + k], v)
        sam.close()


def test_cli_main_writes_reference_layout_json(tmp_path):
    from tredparse_b200 import tred as T
    csv = tmp_path / "samples.csv"
    csv.write_text("#SampleKey,BAM,TRED\nt001,{0}/t001.mini.bam,HD\nt002,{0}/t002.mini.bam,DM1\n".format(GOLDEN))
    cwd = os.getcwd()
    try:
        T.main([str(csv), "--workdir", str(tmp_path / "work")])
    finally:
        os.chdir(cwd)
    d = json.load(open(tmp_path / "work" / "t001.json"))
    assert set(d) == {"samplekey", "bam", "tredCalls"}
    assert d["tredCalls"]["HD.1"] == 15 and d["tredCalls"]["HD.2"] == 41
    keys = {k.split(".", 1)[1] for k in d["tredCalls"] if k.startswith("HD.")}
    assert keys == {"1", "2", "FR", "PR", "RR", "DP", "FDP", "PDP", "RDP", "PEDP", "PEG", "PET", "CI", "PP",
                    "label", "details", "P_h1", "P_h2", "P_h1h2", "P_PEG", "P_PET"}
    assert os.path.exists(tmp_path / "work" / "t002.tred.vcf.gz")


def test_cohort_pipeline_from_native_ingest_equals_run():
    """BAM -> native one-pass ingest (csrc/ingest.cpp) -> all-device cohort pipeline == tred.run's calls
    (GPU ingest -> fused call on its device buffers), and the README's 15|41."""
    from tredparse_b200 import tred as T, cohort, ingest
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    probs, want = [], []
    for sample, name in CASES:
        bam = os.path.join(GOLDEN, sample + ".mini.bam")
        calls = T.run((sample, bam, repo, [name], 300, False, False, True, True, "INFO"))["tredCalls"]
        want.append((calls[name + ".1"], calls[name + ".2"], calls[name + ".CI"], calls[name + ".PP"],
                     calls[name + ".label"], calls[name + ".FDP"], calls[name + ".PDP"], calls[name + ".RDP"]))
        with ingest.BamIngest(bam) as ing:
            probs.append(ing.problem(repo[name], 150, alts=repo[name].alt))
    out = cohort.CohortBatch(probs).run_host(packed=True)["calls"]
    for c, w in zip(out, want):
        d = cohort.decode_call(c)
        assert (d["alleles"][0], d["alleles"][1], d["CI"], d["label"], d["FDP"], d["PDP"], d["RDP"]) == \
               (w[0], w[1], w[2], w[4], w[5], w[6], w[7])
        assert abs(d["PP"] - w[3]) < 1e-9
    assert cohort.decode_call(out[0])["alleles"] == [15, 41]
