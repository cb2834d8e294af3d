"""The CUDA path against golden vectors produced by the REFERENCE ITSELF (tests/golden/ref_*.json — outputs of
the reference's own BamParser / IntegratedCaller / tred.run, see tests/golden/make_ref_fixtures.py).  Needs a GPU:
run with -m gpu."""
import gzip
import json
import os

import numpy as np
import pytest

from conftest import golden_module

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
CASES = [("t001", "HD"), ("t002", "DM1")]
RTOL = 1e-9          # north_star: log-likelihood surface within 1e-9 relative in FP64


def close(a, b, rtol=RTOL, path=""):
    if isinstance(b, dict):
        assert isinstance(a, dict) and set(a) == set(b), (path, sorted(set(a) ^ set(b))[:6])
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


# ---------------------------------------------------------------------------------------------------------
# tred.run == the reference's tred.run, key by key
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sample,tredname", CASES)
def test_tred_run_equals_reference_over_the_whole_catalogue(sample, tredname):
    """BASELINE configs[1]: every catalogue TRED on the fixture BAM — every key the reference writes (calls, CI,
    PP, label, evidence strings, depth, PE summaries, details, sparse posteriors, gender / readLen)."""
    from tredparse_b200 import tred as T
    from tredparse_b200.meta import TREDsRepo
    gold = json.load(open(os.path.join(GOLDEN, "ref_tred_{}.json".format(sample))))
    repo = TREDsRepo()
    assert list(repo.names) == gold["treds"]
    bam = os.path.join(GOLDEN, sample + ".mini.bam")
    calls = T.run((sample, bam, repo, list(repo.names), 300, False, False, True, True, "INFO"))["tredCalls"]
    close(json.loads(json.dumps(calls)), gold["tredCalls"])
    assert calls[tredname + ".label"] == "risk"


@pytest.mark.parametrize("key", ["t001.useclippedreads", "t001.norepeatpairs", "t001.noalts", "t001.fullsearch60",
                                 "t002.useclippedreads", "t002.norepeatpairs", "t002.noalts", "t002.fullsearch60"])
def test_tred_run_equals_reference_under_flags(key):
    from tredparse_b200 import tred as T
    from tredparse_b200.meta import TREDsRepo
    doc = json.load(open(os.path.join(GOLDEN, "ref_tred_flags.json")))[key]
    kw = dict(clip=False, alts=True, repeatpairs=True, maxinsert=300, fullsearch=False)
    kw.update(doc["kwargs"])
    sample, name = key.split(".")[0], doc["tred"]
    bam = os.path.join(GOLDEN, sample + ".mini.bam")
    calls = T.run((sample, bam, TREDsRepo(), [name], kw["maxinsert"], kw["fullsearch"], kw["clip"], kw["alts"],
                   kw["repeatpairs"], "INFO"))["tredCalls"]
    close(json.loads(json.dumps(calls)), doc["tredCalls"])


# ---------------------------------------------------------------------------------------------------------
# synthetic problems: the all-device cohort pipeline == the reference's BamParser.parse + IntegratedCaller.call
# ---------------------------------------------------------------------------------------------------------
def _load_problems():
    with gzip.open(os.path.join(GOLDEN, "ref_problems.json.gz"), "rt") as fp:
        return json.load(fp)["problems"]


def _counter_s(row):
    return ";".join("{}|{}".format(k, int(v)) for k, v in enumerate(row) if v)


def _check_against_reference(docs, problems, out, extra=None):
    from tredparse_b200 import cohort
    for i, (d, pr) in enumerate(zip(docs, problems)):
        ref = d["ref"]
        tag = "{} {} {}".format(d["spec"]["group"], d["spec"]["tred"], d["spec"]["alleles"])
        c = cohort.decode_call(out["calls"][i])
        FR, PR, RR = (_counter_s(out["hist"][i][k]) for k in range(3))
        assert (FR, PR, RR) == (ref["FR"], ref["PR"], ref["RR"]), tag
        assert c["RDP"] == ref["rept"], tag
        assert c["alleles"] == ref["alleles"], tag
        assert c["CI"] == ref["CI"] and c["label"] == ref["label"], tag
        assert c["n_points"] == ref["n_points"], tag
        assert abs(c["PP"] - ref["PP"]) <= 1e-9, tag
        assert abs(c["lik"] - ref["lik"]) <= RTOL * abs(ref["lik"]), tag
        if extra is not None:
            extra(i, d, pr, c)


def _materialise(docs):
    from tredparse_b200.meta import TREDsRepo
    g = golden_module("make_ref_fixtures")
    repo = TREDsRepo()
    problems = []
    for d in docs:
        pr, reads, names = g.materialise(repo, d["spec"])
        assert g.sha1_reads(reads, names, pr) == d["sha1"], "the simulator no longer reproduces the fixture's reads"
        if d["spec"].get("ragged"):
            from tredparse_b200.ssw import encode
            codes = [encode(s) for s in reads]
            pr.reads = np.concatenate(codes)
            pr.roff = np.concatenate([[0], np.cumsum([len(c) for c in codes])]).astype(np.int64)
        problems.append(pr)
    return problems


TAGNAME = {1: "FULL", 2: "PREF", 3: "POST", 4: "REPT"}


@pytest.mark.parametrize("group", ["cohort", "sweep", "listed", "readlen250", "clip", "norepeatpairs"])
def test_cohort_pipeline_equals_reference_on_synthetic_problems(group):
    """BASELINE configs[2] / configs[3] / configs[4]-style problems: the cohort shard of 4 samples x 30 loci, the
    paper's "20/h" sweep (h = 5..300) at HD, the listed HD / DM1 / FXS pairs incl. full expansions, 250-bp reads,
    and the non-default flags --useclippedreads (ragged read lengths) / --norepeatpairs on the device pipeline:
    evidence strings, per-read details, call, CI, PP, lik, label and the sparse posteriors P_h1 / P_h2 / P_h1h2
    equal the reference's BamParser.parse + IntegratedCaller.call."""
    from tredparse_b200 import cohort
    docs = [d for d in _load_problems() if d["spec"]["group"] == group]
    assert docs
    for readlen in sorted({d["spec"]["readlen"] for d in docs}):
        sub = [d for d in docs if d["spec"]["readlen"] == readlen]
        problems = _materialise(sub)
        batch = cohort.CohortBatch(problems, clip=(group == "clip"), repeatpairs=(group != "norepeatpairs"))
        out = batch.run_host(want_hist=True, want_reads=True, packed=True, want_post=True)
        post = cohort.posteriors(out["post"], len(problems))
        r0 = [0]

        def extra(i, d, pr, c):
            rows = out["reads"][r0[0]:r0[0] + pr.nreads]
            r0[0] += pr.nreads
            names = pr.name_strings()
            details = [[TAGNAME[int(t)], int(h), names[k]] for k, (t, h) in enumerate(rows[:, :2]) if int(t) in TAGNAME]
            assert details == d["ref"]["details"], d["spec"]
            hang = int(np.sum(rows[:, 0] == 5))
            kept = len(details) + hang + int(np.sum(rows[:, 0] == 6))
            assert kept == d["ref"]["hang"], d["spec"]          # counts["HANG"] counts every classified read
            for name in ("P_h1", "P_h2", "P_h1h2"):
                close(post[i][name], d["ref"][name], RTOL, "{} {}".format(d["spec"], name))
        _check_against_reference(sub, problems, out, extra)
        if group == "norepeatpairs":
            assert any(int(np.sum(out["reads"][:, 0] == 6)) > 0 for _ in [0]), "no REPT pair was removed: the case is vacuous"


# ---------------------------------------------------------------------------------------------------------
# from BAM: native ingest + fused device call == the reference's tred.run on the same file
# ---------------------------------------------------------------------------------------------------------
def test_run_chunk_equals_run_sample_by_sample():
    """Several samples through ONE fused device call give what each gives alone."""
    from tredparse_b200 import tred as T
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    args = [(s, os.path.join(GOLDEN, s + ".mini.bam"), repo, ["HD", "DM1", "FXS", "SCA17"], 300, False, False, True, True, "INFO")
            for s in ("t001", "t002")]
    both = T.run_chunk(args)
    for a, got in zip(args, both):
        alone = T.run(a)
        close(json.loads(json.dumps(got)), json.loads(json.dumps(alone)), 1e-12)


def test_tred_run_on_a_synthetic_sample_bam_equals_the_reference(tmp_path):
    """A simulated whole-sample BAM (reads placed around several loci, expansions included): the product's
    tred.run (native ingest -> fused device pipeline) against the stored calls of the CPU oracle on the same file
    (golden/oracle_sample_bam.json; the oracle is held to the reference's own outputs by test_reference_pinned.py)
    and, where the reference package can be loaded, against the reference's own tred.run."""
    from oracle import refdrive
    from tredparse_b200 import tred as T
    from tredparse_b200.meta import TREDsRepo
    g = golden_module("make_oracle_bam_fixture")
    with open(os.path.join(GOLDEN, "oracle_sample_bam.json")) as fp:
        gold = json.load(fp)
    repo = TREDsRepo()
    names = gold["names"]
    path = str(tmp_path / "s.bam")
    truth = g.write_sample(path, repo)
    assert g.records_sha1(path) == gold["records_sha1"], "the simulator no longer writes the fixture's reads"
    assert json.loads(json.dumps(truth)) == gold["truth"]
    mine = json.loads(json.dumps(T.run(("s", path, repo, names, 300, False, False, True, True, "INFO"))["tredCalls"]))
    for k, v in gold["presteps"].items():
        close(mine[k], v, path=k)
    for n in names:
        for k, v in gold["calls"][n].items():
            close(mine[n + "." + k], v, path=n + "." + k)
    assert any(mine[n + ".1"] > 0 for n in names)
    if refdrive.usable():
        theirs = refdrive.run_bam(("s", path, names))
        close(mine, json.loads(json.dumps(theirs, default=float)))
