"""The CPU oracle against golden vectors produced by the REFERENCE ITSELF (tests/golden/ref_*.json, made by
tests/golden/make_ref_fixtures.py from the reference's own Python sources through oracle/refshim.py), and the
shim's transform.  No GPU needed."""
import gzip
import json
import logging
import os

import numpy as np
import pytest

from oracle import refshim, genotype_oracle, evidence_oracle as evo, likelihood_oracle as lko
from tredparse_b200 import bamio, simulate
from tredparse_b200.meta import TREDsRepo
from conftest import golden_module

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = [("t001", "HD"), ("t002", "DM1")]


def _models():
    md = json.load(open(os.path.join(ROOT, "tredparse_b200", "data", "models.json")))
    step = {int(k): np.array(v) for k, v in md["step_size_by_period"].items()}
    for i in range(6, 18):
        step[i] = step[6]
    return step, md["stutter_weights"]


def close(a, b, rtol=1e-9, path=""):
    if isinstance(b, dict):
        assert isinstance(a, dict) and set(a) == set(b), path
        for k in b:
            close(a[k], b[k], rtol, path + "/" + str(k))
    elif isinstance(b, list):
        assert len(a) == len(b), path
        for i, (x, y) in enumerate(zip(a, b)):
            close(x, y, rtol, "{}[{}]".format(path, i))
    elif isinstance(b, float) or isinstance(a, float):
        assert abs(a - b) <= rtol * max(abs(a), abs(b)) + 1e-15, (path, a, b)
    else:
        assert a == b, (path, a, b)


def load_problems():
    with gzip.open(os.path.join(GOLDEN, "ref_problems.json.gz"), "rt") as fp:
        return json.load(fp)["problems"]


def materialise(repo, spec):
    g = golden_module("make_ref_fixtures")
    pr, reads, names = g.materialise(repo, spec)
    return pr, reads, names, g.sha1_reads(reads, names, pr)


# ---------------------------------------------------------------------------------------------------------
# the transform
# ---------------------------------------------------------------------------------------------------------
def test_py2_division_semantics():
    d = refshim._py2div
    assert d(7, 2) == 3 and isinstance(d(7, 2), int) and d(-7, 2) == -4
    assert d(7, 2.0) == 3.5 and d(7.0, 2) == 3.5
    assert d(np.int64(9), 2) == 4 and d(np.int64(150), np.int64(4)) == 37
    assert np.array_equal(d(np.array([3, 4, 5]), 2), np.array([1, 2, 2]))
    assert np.allclose(d(np.array([3., 4.]), 2), np.array([1.5, 2.]))
    assert refshim._py2range(3) == [0, 1, 2] and refshim._py2range(1, 7, 3) + [9] == [1, 4, 9]


def test_text_rules():
    src = ("print >> sys.stderr, units, target\n"
           "if 1:\n"
           "    print >> fw, js\n"
           "print >> sys.stderr\n"
           "print js\n"
           "if 1:\n"
           "    print >> sys.stderr, \"Elapsed time={}\"\\\n            .format(x)\n"
           "for i in xrange(3): fp.next()\n"
           "for k, v in d.iteritems(): pass\n"
           "_c = string.maketrans('AT', 'TA')\n")
    out = refshim.py3_source(src)
    assert "print(units, target, file=sys.stderr)" in out and "    print(js, file=fw)" in out
    assert "print(file=sys.stderr)" in out and "\nprint(js)\n" in out
    assert 'print("Elapsed time={}" .format(x), file=sys.stderr)' in out
    assert "range(3): next(fp)" in out and "d.items()" in out and "str.maketrans" in out
    assert out.count("\n") == src.count("\n")           # line numbers survive
    compile(out, "x", "exec")


def test_product_tables_equal_the_reference_catalogue():
    """Our loci.tsv / alts.tsv / models.json carry what the reference's TREDsRepo / StepModel / NoiseModel load
    (stored in golden/ref_tables.json; the order of the names is that of the reference's own tred.run)."""
    with open(os.path.join(GOLDEN, "ref_tables.json")) as fp:
        ref = json.load(fp)
    ours = TREDsRepo()
    assert ref["treds"] == json.load(open(os.path.join(GOLDEN, "ref_tred_t001.json")))["treds"]
    assert list(ours.names) == ref["treds"]
    for n in ref["treds"]:
        a, b = ref["catalogue"][n], ours[n]
        for f in ("repeat", "chr", "repeat_start", "repeat_end", "ref_copy", "prefix", "suffix", "cutoff_prerisk",
                  "cutoff_risk", "inheritance", "is_xlinked", "is_recessive", "is_expansion", "ploidy"):
            assert a[f] == getattr(b, f), (n, f)
        assert [tuple(x) for x in a["alt"]] == [tuple(x) for x in b.alt], n
    step, w = _models()
    assert ref["stutter_weights"] == w
    for k, v in ref["step_size_by_period"].items():
        assert np.array_equal(np.array(v), step[int(k)])


# ---------------------------------------------------------------------------------------------------------
# oracle == reference
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sample,tredname", CASES)
def test_oracle_pipeline_equals_reference_tred_run(sample, tredname):
    repo = TREDsRepo()
    step, w = _models()
    sam = bamio.AlignmentFile(os.path.join(GOLDEN, sample + ".mini.bam"))
    exp, ev, lk = genotype_oracle.genotype_locus(sam, repo[tredname], evo.read_length(sam), step, w)
    gold = json.load(open(os.path.join(GOLDEN, "ref_tred_{}.json".format(sample))))["tredCalls"]
    assert gold["readLen"] == evo.read_length(sam)
    for k, v in exp.items():
        close(v, gold[tredname + "." + k], 1e-12, k)


@pytest.mark.parametrize("key", ["t001.useclippedreads", "t001.norepeatpairs", "t001.noalts", "t001.fullsearch60",
                                 "t002.useclippedreads", "t002.norepeatpairs", "t002.noalts", "t002.fullsearch60"])
def test_oracle_pipeline_equals_reference_under_flags(key):
    doc = json.load(open(os.path.join(GOLDEN, "ref_tred_flags.json")))[key]
    repo = TREDsRepo()
    step, w = _models()
    sample, tredname = key.split(".")[0], doc["tred"]
    sam = bamio.AlignmentFile(os.path.join(GOLDEN, sample + ".mini.bam"))
    exp, ev, lk = genotype_oracle.genotype_locus(sam, repo[tredname], evo.read_length(sam), step, w, **doc["kwargs"])
    for k, v in exp.items():
        close(v, doc["tredCalls"][tredname + "." + k], 1e-12, k)


class _PE:
    def __init__(self, pr, tred):
        self.global_lens, self.target_lens = [int(x) for x in pr.global_lens], [int(x) for x in pr.target_lens]
        self.ref = tred.repeat_end - tred.repeat_start + 1
        self.MINPE = tred.repeat_end - tred.repeat_start + 2 * 9 + 2


def oracle_problem(repo, doc, step, w):
    """Evidence + likelihood oracle on one synthetic problem -> the fields ref_problems stores."""
    spec = doc["spec"]
    pr, reads, names, digest = materialise(repo, spec)
    assert digest == doc["sha1"], "the simulator no longer reproduces the fixture's reads"
    tred = repo[spec["tred"]]
    gender = "Male" if (pr.ploidy == 1 and tred.is_xlinked) else "Unknown"
    ev = evo.EvidenceOracle(tred, pr.readlen, gender=gender, depth=pr.depth, clip=spec.get("clip", False),
                            repeatpairs=spec.get("repeatpairs", True))
    ev.parse_reads(reads, names)
    counts = {"FULL": dict(ev.counts["FULL"]), "PREF": dict(ev.counts["PREF"])}
    lk = lko.LikelihoodOracle(tred, ev.period, pr.readlen, counts, ev.rept, ev.ploidy, pr.depth, _PE(pr, tred), step, w)
    lk.call()
    return {"FR": genotype_oracle.counter_s(ev.counts["FULL"]), "PR": genotype_oracle.counter_s(ev.counts["PREF"]),
            "RR": genotype_oracle.counter_s(ev.counts["REPT"]), "rept": ev.rept,
            "hang": sum(ev.counts["HANG"].values()),
            "details": [[d["tag"], int(d["h"]), d["id"]] for d in ev.details],
            "alleles": [int(x) for x in lk.alleles], "lik": float(lk.lik), "PP": float(lk.PP), "CI": lk.CI,
            "label": lk.label, "n_points": len(lk.surface), "PEDP": lk.PEDP,
            "P_h1": lk.P_h1 or {}, "P_h2": lk.P_h2 or {}, "P_h1h2": lk.P_h1h2 or {}}


def test_oracle_equals_reference_on_synthetic_problems():
    """Every 4th problem of ref_problems (cohort, config-3 sweep, clip / norepeatpairs, 250 bp) plus all the
    flag cases: the oracle's evidence, call, CI, PP, lik and sparse posteriors equal the reference's."""
    repo = TREDsRepo()
    step, w = _models()
    docs = load_problems()
    pick = [d for i, d in enumerate(docs) if i % 4 == 0 or d["spec"]["group"] in ("clip", "norepeatpairs", "listed")]
    assert len(pick) >= 60
    for d in pick:
        got = oracle_problem(repo, d, step, w)
        close(got, d["ref"], 1e-12, "{}{}".format(d["spec"]["tred"], d["spec"]["alleles"]))


# ---------------------------------------------------------------------------------------------------------
# region_depth and README.md:80
# ---------------------------------------------------------------------------------------------------------
def test_depth_semantics_and_the_readme_dm1_call():
    """README.md:80 prints t002/DM1 = 5|62.  The reference's own code (v0.7.8), run here on its own
    tests/t002.bam, gives 5|66 under pysam's default pileup reading and 5|66 / 5|67 under every other candidate
    reading (oracle/pysam_stub.py); 62 needs a depth of ~75x, 1.6 times what the fixture holds under any
    reading (43.6 .. 50.1).  The README line is therefore not reproducible from the reference at this commit,
    and the second allele is pinned to the reference's code instead (ref_tred_t002.json)."""
    doc = json.load(open(os.path.join(GOLDEN, "ref_depth_dm1.json")))
    assert {m: v["alleles"][1] for m, v in doc["modes"].items()} == \
        {"all": 66, "truncate": 67, "nofilter": 66, "nodel": 66, "overlap": 67}
    assert all(43 < v["DP"] < 51 for v in doc["modes"].values())
    need = [d["depth"] for d in doc["sweep"] if d["alleles"][1] == 62]
    assert need and min(need) >= 70
    h2 = [d["alleles"][1] for d in doc["sweep"]]
    assert h2[0] > h2[-1] and h2[0] == 80 and h2[-1] == 59           # monotone trend: deeper -> shorter
    # the product's depth equals the reference's under pysam's default reading
    sam = bamio.AlignmentFile(os.path.join(GOLDEN, "t002.mini.bam"))
    t = TREDsRepo()["DM1"]
    assert bamio.region_depth(sam, t.chr, t.repeat_start - 1000, t.repeat_end + 1000) == pytest.approx(doc["modes"]["all"]["DP"], rel=1e-15)
    gold = json.load(open(os.path.join(GOLDEN, "ref_tred_t002.json")))["tredCalls"]
    assert (gold["DM1.1"], gold["DM1.2"]) == (5, 66) and gold["DM1.DP"] == doc["modes"]["all"]["DP"]
