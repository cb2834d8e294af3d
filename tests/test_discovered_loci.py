"""Discovered loci (DESIGN §4.5): reference access (tredparse_b200.fasta), the locus behind an outlier region
(strprofile.locus_for, against oracle/locus_oracle.py and cases worked out by hand), the sites JSON the genotyper
reads, the `loci` CLI; on the GPU, the fused genotyping call on discovered-locus families of periods 2, 5, 13 and 20
against the CPU oracle, and the whole workflow profile -> outliers -> loci -> tred.py --tred on a synthetic cohort."""
import gzip
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENV = dict(os.environ, PYTHONPATH=ROOT)


def _fasta(tmp_path, contigs, name="ref.fa", width=60, fai=False):
    from tredparse_b200 import simulate
    from tredparse_b200.fasta import Fasta
    return Fasta(simulate.write_fasta(str(tmp_path / name), contigs, width=width, fai=fai))


def _row(contig, start, end, motif, z=9.0):
    return {"contig": contig, "start": start, "end": end, "motif": motif, "top_sample": "s", "z": z, "counts": {}}


def _canonical(unit):
    from oracle.locus_oracle import revcomp
    k = len(unit)
    return min(m[i:] + m[:i] for m in (unit, revcomp(unit)) for i in range(k))


# ---------------------------------------------------------------------------------------------------------------
# reference access
# ---------------------------------------------------------------------------------------------------------------
def test_hand_written_fai_equals_the_index_built_in_memory(tmp_path):
    from tredparse_b200.fasta import Fasta
    p = tmp_path / "x.fa"
    p.write_bytes(b">a desc\nACGTA\nCG\n>b\nAC\n>empty\n")
    fai = {"a": (7, 8, 5, 6), "b": (2, 20, 2, 3), "empty": (0, 30, 0, 0)}
    assert Fasta(str(p)).index == fai
    (tmp_path / "x.fa.fai").write_text("a\t7\t8\t5\t6\nb\t2\t20\t2\t3\nempty\t0\t30\t0\t0\n")
    fa = Fasta(str(p))
    assert fa.index == fai and fa.lengths() == {"a": 7, "b": 2, "empty": 0}
    assert fa.fetch("a", 0, 7) == "ACGTACG" and fa.fetch("a", 4, 6) == "AC" and fa.fetch("b", -3, 9) == "AC"
    assert fa.fetch("empty", 0, 5) == ""


@pytest.mark.parametrize("width", [60, 61, 1])
def test_fetch_at_line_widths_lowercase_and_n_runs(tmp_path, width):
    from tredparse_b200.fasta import Fasta
    rng = np.random.default_rng(width)
    contigs = {}
    for i, L in enumerate((1000, 1037, 7, 61 * 3)):               # short last lines, a last line of full width
        s = list(rng.choice(list("ACGT"), L))
        if L > 100:
            s[200:260] = "N" * 60
        contigs["c{}".format(i)] = "".join(s)
    lower = {n: s[:L // 2].lower() + s[L // 2:] for n, s in contigs.items() for L in [len(s)]}
    with_fai = _fasta(tmp_path, lower, "a.fa", width, fai=True)
    built = _fasta(tmp_path, lower, "b.fa", width, fai=False)
    assert not os.path.exists(str(tmp_path / "b.fa.fai"))        # nothing written next to the file
    assert built.index == with_fai.index
    assert built.lengths() == {n: len(s) for n, s in contigs.items()}
    for n, s in contigs.items():
        assert built.fetch(n, 0, len(s)) == s
        for _ in range(50):
            a = int(rng.integers(0, len(s)))
            b = int(rng.integers(a, len(s) + 1))
            assert built.fetch(n, a, b) == with_fai.fetch(n, a, b) == s[a:b]


def test_missing_contig_gzip_and_ragged_lines(tmp_path):
    from tredparse_b200.fasta import Fasta
    fa = _fasta(tmp_path, {"c1": "ACGT" * 30})
    assert "c2" not in fa and "c1" in fa
    with pytest.raises(KeyError, match="c2"):
        fa.fetch("c2", 0, 10)
    gz = tmp_path / "ref.fa.gz"
    with gzip.open(str(gz), "wb") as fp:
        fp.write(b">c1\nACGT\n")
    with pytest.raises(ValueError, match="compressed"):
        Fasta(str(gz))
    bad = tmp_path / "ragged.fa"
    bad.write_text(">c1\nACGT\nAC\nACGT\n")
    with pytest.raises(ValueError, match="unequal width"):
        Fasta(str(bad))


# ---------------------------------------------------------------------------------------------------------------
# the locus behind an outlier row
# ---------------------------------------------------------------------------------------------------------------
def _random_unit(rng, k):
    while True:
        u = "".join(rng.choice(list("ACGT"), k))
        if all(u != u[d:] + u[:d] for d in range(1, k)):        # primitive: not a repeat of a shorter unit
            return u


def test_locus_for_equals_the_oracle_on_random_references(tmp_path):
    from tredparse_b200 import simulate, strprofile
    from oracle import locus_oracle
    rng = np.random.default_rng(11)
    lengths = [("c{}".format(i), int(rng.integers(1500, 6000))) for i in range(6)]
    sites, rows = [], []
    for i, (c, L) in enumerate(lengths):
        for j in range(2):
            k = int(rng.integers(2, 21))
            u = _random_unit(rng, k)
            copies = int(rng.integers(1, 12))
            pos = int(rng.integers(0, L - k * copies)) if j else int(rng.integers(0, 30))     # some near a contig end
            sites.append((c, pos, u, copies))
    contigs = simulate.planted_reference(lengths, sites, seed=5)
    # short accidental runs: two copies of every unit at random places, and a homopolymer run
    for c, pos, u, _ in sites:
        s = contigs[c]
        p = int(rng.integers(0, len(s) - 2 * len(u)))
        contigs[c] = s[:p] + (u * 2) + s[p + 2 * len(u):]
    fa = _fasta(tmp_path, contigs)
    outcome = set()
    for c, pos, u, copies in sites:
        for _ in range(4):
            a = pos + int(rng.integers(-900, 300))
            b = a + int(rng.integers(1, 600))
            motif = _canonical(u) if rng.random() < 0.8 else _canonical(_random_unit(rng, len(u)))
            rows.append(_row(c, max(0, a), max(1, b), motif))
    rows.append(_row("-", None, None, "AT"))
    rows.append(_row("nope", 10, 20, "AT"))
    for row in rows:
        for window, mru in ((1000, 3), (50, 2), (300, 5)):
            want = locus_oracle.locus(row, contigs, 150, window, mru)
            try:
                got = strprofile.locus_for(row, fa, 150, window, mru)
            except strprofile.Skip as e:
                got = str(e)
            if isinstance(want, str):
                assert got == want, (row, window, mru, got)
            else:
                assert got[0] == want[0] and {k: got[1][k] for k in want[1]} == want[1], (row, got, want)
            outcome.add(got if isinstance(got, str) else "locus")
    assert outcome >= {"locus", "no reference tract", "flank outside contig", "no position", "contig not in FASTA"}, outcome


def _hand_ref(tmp_path, body, L=400):
    """a contig of L C's with `body` {0-based position: bases} written over it (no unit of the tests runs by chance)"""
    s = ["C"] * L
    for p, b in body.items():
        s[p:p + len(b)] = list(b)
    return _fasta(tmp_path, {"c1": "".join(s)}, "hand{}.fa".format(abs(hash(tuple(body.items()))) % 10 ** 8)), "".join(s)


def test_locus_rules_by_hand(tmp_path):
    from tredparse_b200 import strprofile
    from oracle import locus_oracle
    lf = strprofile.locus_for

    def both(fa, seq, row, **kw):
        try:
            got = lf(row, fa, 150, **kw)
        except strprofile.Skip as e:
            got = str(e)
        want = locus_oracle.locus(row, {"c1": seq}, 150, kw.get("window", 1000), kw.get("min_ref_units", 3))
        assert (got if isinstance(got, str) else got[0]) == (want if isinstance(want, str) else want[0])
        return got

    # reverse-complement orientation, repeat = the rotation at the tract's first base: TTGGG = rc(CCCAA), a rotation
    # of the canonical AACCC's reverse complement; GGGTT reads on the reference at the tract's first base
    fa, seq = _hand_ref(tmp_path, {100: "GGGTT" * 6 + "A"})
    name, row = both(fa, seq, _row("c1", 150, 160, "AACCC"))
    assert name == "c1_101_GGGTT" and row["repeat"] == "GGGTT" and row["repeat_location"] == "c1:101-130"
    assert row["prefix"] == seq[82:100] and row["suffix"] == seq[130:148]
    assert row["cutoff_risk"] == row["cutoff_prerisk"] == 30 and row["inheritance"] == "AD"
    assert row["mutation_nature"] == "increase"
    # two runs of 4 copies at 50 and 250: the one whose centre is closer to the region's centre; equidistant: leftmost
    fa, seq = _hand_ref(tmp_path, {50: "TG" * 4, 250: "GT" * 4})
    assert both(fa, seq, _row("c1", 240, 260, "AC"))[0] == "c1_251_GT"
    assert both(fa, seq, _row("c1", 40, 60, "AC"))[0] == "c1_51_TG"
    assert both(fa, seq, _row("c1", 50 + 4 + 100 - 10, 50 + 4 + 100 + 10, "AC"))[0] == "c1_51_TG"    # centre 154
    # a longer run beats a closer one
    fa, seq = _hand_ref(tmp_path, {50: "TG" * 5, 250: "GT" * 4})
    assert both(fa, seq, _row("c1", 240, 260, "AC"))[0] == "c1_51_TG"
    # a tract one base from either end of the contig: its flank is not on the contig
    fa, seq = _hand_ref(tmp_path, {1: "GGT" * 5, 400 - 16: "GGT" * 5})
    assert both(fa, seq, _row("c1", 0, 10, "ACC", ), window=20) == "flank outside contig"
    assert both(fa, seq, _row("c1", 390, 400, "ACC"), window=20) == "flank outside contig"
    # an N in a flank; fewer than min_ref_units copies
    fa, seq = _hand_ref(tmp_path, {100: "GGT" * 5, 90: "N"})
    assert both(fa, seq, _row("c1", 100, 110, "ACC")) == "N in flank"
    fa, seq = _hand_ref(tmp_path, {100: "GGT" * 2})
    assert both(fa, seq, _row("c1", 100, 110, "ACC")) == "no reference tract"
    assert both(fa, seq, _row("c1", 100, 110, "ACC"), min_ref_units=2)[0] == "c1_101_GGT"
    # a motif-only row, a contig the FASTA lacks
    assert both(fa, seq, _row("-", None, None, "ACC")) == "no position"
    assert both(fa, seq, _row("chrZ", 1, 5, "ACC")) == "contig not in FASTA"


def test_two_regions_of_one_expansion_give_one_locus(tmp_path):
    from tredparse_b200 import strprofile
    fa, seq = _hand_ref(tmp_path, {150: "GGGTT" * 12}, L=2000)
    rows = [_row("c1", 0, 120, "AACCC", z=12.0), _row("c1", 800, 900, "AACCC", z=8.0),
            _row("c1", 1500, 1600, "AACCC", z=2.0), _row("-", None, None, "AACCC", z=5.0)]
    sites, skipped = strprofile.discover_loci(rows, fa, 150)
    assert list(sites) == ["c1_151_GGGTT"] and [why for _, why in skipped] == ["no position"]
    sites, skipped = strprofile.discover_loci(rows, fa, 150, min_z=10)
    assert list(sites) == ["c1_151_GGGTT"] and skipped == []


def test_sites_json_loads_through_the_repo(tmp_path):
    from tredparse_b200 import meta, strprofile
    fa, seq = _hand_ref(tmp_path, {100: "GGGTT" * 6 + "A", 300: "TTGCA" * 3})
    sites, _ = strprofile.discover_loci([_row("c1", 90, 140, "AACCC"), _row("c1", 290, 310, "AATGC")], fa, 151)
    d = tmp_path / "sites"
    d.mkdir()
    (d / "discovered.json").write_text(json.dumps(sites))
    empty = tmp_path / "empty"
    empty.mkdir()
    base, repo = meta.TREDsRepo(sites=str(empty)), meta.TREDsRepo(sites=str(d))
    assert repo.names == base.names + ["c1_101_GGGTT", "c1_301_TTGCA"] == meta.locus_names(str(d))
    for n in base.names:
        a, b = base[n], repo[n]
        assert (str(a), a.cutoff_risk, a.cutoff_prerisk, a.ref_copy, a.inheritance) == \
               (str(b), b.cutoff_risk, b.cutoff_prerisk, b.ref_copy, b.inheritance)
    t = repo["c1_101_GGGTT"]
    assert (t.chr, t.repeat_start, t.repeat_end, t.ref_copy, t.repeat) == ("c1", 101, 130, 6, "GGGTT")
    assert (t.prefix, t.suffix) == (seq[82:100], seq[130:148])
    assert t.cutoff_prerisk == t.cutoff_risk == 31 and t.is_expansion and not t.is_recessive and not t.is_xlinked
    assert repo["c1_301_TTGCA"].ref_copy == 3
    # a sites file for hg19 holds the hg19 field only; the repo reads it with --ref hg19, the CLI lists its names
    hg19, _ = strprofile.discover_loci([_row("c1", 90, 140, "AACCC")], fa, 150, ref="hg19")
    assert "repeat_location.hg19" in hg19["c1_101_GGGTT"] and "repeat_location" not in hg19["c1_101_GGGTT"]
    d19 = tmp_path / "s19"
    d19.mkdir()
    (d19 / "x.json").write_text(json.dumps(hg19))
    assert meta.TREDsRepo(ref="hg19", sites=str(d19))["c1_101_GGGTT"].repeat_start == 101
    assert meta.TREDsRepo(ref="hg19_nochr", sites=str(d19))["c1_101_GGGTT"].chr == "c1"


def test_tred_cli_offers_the_discovered_names(tmp_path, monkeypatch):
    from tredparse_b200 import tred
    d = tmp_path / "sites"
    d.mkdir()
    (d / "x.json").write_text(json.dumps({"c9_5_AT": {"repeat_location.hg19": "c9:5-20"}}))
    monkeypatch.chdir(str(tmp_path))
    a = tred.set_argparse().parse_args(["x.bam", "--tred", "c9_5_AT", "--ref", "hg19"])
    assert a.tred == ["c9_5_AT"]


def test_step_model_covers_every_profile_period():
    from tredparse_b200 import models
    step = models.StepModel().step_size_by_period
    for p in range(1, 21):
        assert len(step[p]) == 37
    for p in range(7, 21):
        assert np.array_equal(step[p], step[6])


def test_loci_cli(tmp_path):
    from tredparse_b200 import strprofile
    fa, seq = _hand_ref(tmp_path, {100: "GGGTT" * 6 + "A", 300: "GGT" * 2})
    os.rename(fa.path, str(tmp_path / "ref.fa"))
    rows = [_row("c1", 90, 140, "AACCC", z=7.5), _row("c1", 120, 130, "AACCC", z=4.0),
            _row("c1", 290, 310, "ACC", z=6.0), _row("c9", 10, 20, "AT", z=5.0), _row("-", None, None, "AT", z=3.5),
            _row("c1", 10, 20, "AC", z=2.9)]
    for r in rows:
        r["counts"] = {"a": 1.0, "b": 0.0}
    tsv = tmp_path / "out.tsv"
    with open(str(tsv), "w") as fp:
        strprofile.write_tsv(rows, ["a", "b"], fp)
    with open(str(tsv)) as fp:
        assert [{k: r[k] for k in ("contig", "start", "end", "motif", "z")} for r in strprofile.read_tsv(fp)] == \
               [{k: r[k] for k in ("contig", "start", "end", "motif", "z")} for r in rows]
    profs = []
    for i, rl in enumerate((100, 151)):
        p = tmp_path / "s{}.str_profile.json".format(i)
        p.write_text(json.dumps({"sample": "s{}".format(i), "read_length": rl}))
        profs.append(str(p))

    def run(*extra):
        return subprocess.run([sys.executable, "-m", "tredparse_b200.strprofile", "loci", str(tsv), "--fasta",
                               str(tmp_path / "ref.fa"), "--profiles", *profs, *extra], cwd=str(tmp_path), env=ENV,
                              capture_output=True, text=True)
    r = run()
    assert r.returncode == 0, r.stderr
    assert r.stdout.split() == ["c1_101_GGGTT"]
    err = r.stderr.splitlines()
    assert "skipped c1:290-310 ACC (z 6.0000): no reference tract" in err
    assert "skipped c9:10-20 AT (z 5.0000): contig not in FASTA" in err
    assert "skipped - AT (z 3.5000): no position" in err
    assert "1 rows below --min-z 3.0" in err and not any("c1:10-20" in e for e in err)
    with open(str(tmp_path / "sites" / "discovered.json")) as fp:
        got = json.load(fp)
    assert got["c1_101_GGGTT"]["cutoff_risk"] == 31                # the longest read among the profiles: 151 bp
    r = run("--min-z", "7", "--min-ref-units", "2", "--out", str(tmp_path / "o.json"), "--ref", "hg19")
    assert r.returncode == 0 and r.stdout.split() == ["c1_101_GGGTT"] and "skipped" not in r.stderr
    with open(str(tmp_path / "o.json")) as fp:
        assert json.load(fp)["c1_101_GGGTT"]["repeat_location.hg19"] == "c1:101-130"
    with gzip.open(str(tmp_path / "ref.fa.gz"), "wb") as fp:
        fp.write(b">c1\nACGT\n")
    r = subprocess.run([sys.executable, "-m", "tredparse_b200.strprofile", "loci", str(tsv), "--fasta",
                        str(tmp_path / "ref.fa.gz"), "--profiles", *profs], cwd=str(tmp_path), env=ENV,
                       capture_output=True, text=True)
    assert r.returncode == 2 and "compressed" in r.stderr


# ---------------------------------------------------------------------------------------------------------------
# on the GPU: the fused call on discovered-locus families
# ---------------------------------------------------------------------------------------------------------------
PARITY_UNITS = {2: "TC", 5: "GGGTT", 13: "TTCAGCATGACCA", 20: "GATCCAGTTAGCCTGAAAGT"}


def _discovered_repo(tmp_path, readlen):
    """{period: meta.TRED} of loci built by locus_for from a reference with one planted tract per period"""
    from tredparse_b200 import meta, simulate, strprofile
    sites = [("c1", 1000 + 1500 * i, u, max(3, 40 // len(u))) for i, u in enumerate(PARITY_UNITS.values())]
    contigs = simulate.planted_reference([("c1", 8000)], sites, seed=17)
    fa = _fasta(tmp_path, contigs, "par{}.fa".format(readlen))
    out = {}
    for c, pos, u, n in sites:
        name, row = strprofile.locus_for(_row(c, pos - 300, pos + 200, _canonical(u)), fa, readlen)
        assert row["repeat"] == u
        out[len(u)] = meta.TRED(name, row)
    return out


def _step20():
    md = json.load(open(os.path.join(ROOT, "tredparse_b200", "data", "models.json")))
    step = {int(k): np.array(v) for k, v in md["step_size_by_period"].items()}
    for i in range(6, 21):
        step[i] = step[6]
    return step, md["stutter_weights"]


@pytest.mark.gpu
@pytest.mark.parametrize("L", [150, 250])
def test_gpu_fused_call_on_discovered_families_equals_the_oracle(tmp_path, L):
    """Per read (tag, h), tallies, alleles, CI, label, PP, likelihood and posteriors of problems at discovered loci of
    periods 2 and 5 (packed phase 1) and 13 and 20 (generic phase 1) == the CPU oracle's; per-read records of the
    family kernel == the oracle's arg-max, through the phase-1 path the period selects."""
    from test_gpu_cohort import _expected_reads, _oracle_call
    from test_gpu_read_lengths import _Fam, _Set, _check_calls, _pool, _reads
    from tredparse_b200 import cohort, simulate
    loci = _discovered_repo(tmp_path, L)
    problems = []
    for i, (k, t) in enumerate(sorted(loci.items())):
        mu = -(-L // k)
        for j, al in enumerate([(max(1, mu // 4), max(2, mu // 2)), (max(1, mu // 3), mu + 40 // k + 8), (max(2, mu // 2),)]):
            problems.append(simulate.simulate_problem(t, al, readlen=L, cov_per_hap=10, seed=7000 * L + 10 * i + j))
    step, w = _step20()

    def oracle(pr):
        exp = _expected_reads(pr)
        lk, counts, rept = _oracle_call(pr, [(a, b) for a, b in exp if a not in (0, 5)], step, w)
        return exp, lk, counts, rept
    with _pool() as ex:
        expected = list(ex.map(oracle, problems))
    out = cohort.CohortBatch(problems).run_host(want_reads=True, want_hist=True, want_stats=True, want_post=True)
    assert out["stats"][5] == 0
    _check_calls(problems, out, expected)
    assert any(e[3] for e in expected) and any(e[1].label == "risk" for e in expected)
    rng = np.random.default_rng(L)
    for k, t in sorted(loci.items()):
        fam = _Fam(t.prefix, t.repeat, t.suffix, L)
        s = _Set([fam], [_reads(fam, rng, 48, L)])
        s.check(s.classify("packed" if k <= 12 else "generic"))


# ---------------------------------------------------------------------------------------------------------------
# on the GPU: profile -> outliers -> loci -> tred.py --tred, on a synthetic cohort
# ---------------------------------------------------------------------------------------------------------------
E2E_SITES = [("c1", 12000, "GGGAA", 10, "AAGGG"), ("c2", 9000, "TGCTTACCGTCAA", 4, None)]    # (.., canonical motif)
E2E_REFS = [("c1", 24000), ("c2", 18000)]
NORMAL = {0: ((8, 12), (3, 5)), 1: ((10, 10), (4, 6)), 2: ((6, 11), (2, 4))}
EXPANDED, EXP_UNITS = 3, 200


def _e2e_cohort(d):
    """four samples on the planted reference (c1, c2) plus chr4 with HD: samples 0-2 carry short alleles at both
    sites, sample 3 a 200-unit expansion at each; samples 0 and 3 indexed, 1 and 2 not"""
    from tredparse_b200 import bamio, simulate
    from tredparse_b200.meta import TREDsRepo
    contigs = simulate.planted_reference(E2E_REFS, [s[:4] for s in E2E_SITES], seed=23)
    simulate.write_fasta(str(d / "ref.fa"), contigs, width=70)
    hd = TREDsRepo()["HD"]
    refs = E2E_REFS + [("chr4", hd.repeat_end + 20000)]
    bams = []
    for s in range(4):
        recs = []
        for si, (c, pos, u, n, _) in enumerate(E2E_SITES):
            al = (NORMAL[0][si][0], EXP_UNITS) if s == EXPANDED else NORMAL[s][si]
            recs += simulate.reference_records(contigs[c], si, pos, pos + len(u) * n, u, al, cov_per_hap=15,
                                               flank=1500, seed=100 * s + si, tag="s{}x{}".format(s, si))
        recs += simulate.locus_records(hd, 2, (17, 20), 150, 10.0, seed=40 + s, tag="s{}hd".format(s), flank=1000)
        path = str(d / "s{}.bam".format(s))
        bamio.write_bam(path, refs, simulate.coordinate_sort(recs), index=s in (0, 3), aux=True)
        bams.append(path)
    return bams


@pytest.mark.gpu
def test_gpu_discovered_loci_end_to_end(tmp_path, monkeypatch, capsys):
    from tredparse_b200 import strprofile, tred
    bams = _e2e_cohort(tmp_path)
    work = tmp_path / "w"
    assert strprofile.main(["profile", *bams, "--workdir", str(work)]) == 0
    profs = [str(work / "s{}.str_profile.json".format(s)) for s in range(4)]
    assert strprofile.main(["outliers", *profs, "--tsv", str(tmp_path / "out.tsv")]) == 0
    run = tmp_path / "run"
    run.mkdir()
    monkeypatch.chdir(str(run))
    capsys.readouterr()
    assert strprofile.main(["loci", str(tmp_path / "out.tsv"), "--fasta", str(tmp_path / "ref.fa"),
                            "--profiles", *profs]) == 0
    names = capsys.readouterr().out.split()
    want = ["{}_{}_{}".format(c, pos + 1, u) for c, pos, u, _, _ in E2E_SITES]
    assert sorted(names) == sorted(want), names
    with open("sites/discovered.json") as fp:
        sites = json.load(fp)
    for (c, pos, u, n, canon), name in zip(E2E_SITES, want):
        row = sites[name]
        assert row["repeat"] == u and row["repeat_location"] == "{}:{}-{}".format(c, pos + 1, pos + len(u) * n)
        assert row["motif"] == (canon or _canonical(u)) and row["cutoff_risk"] == -(-150 // len(u))
    assert _canonical(E2E_SITES[1][2]) not in {E2E_SITES[1][2][i:] + E2E_SITES[1][2][:i] for i in range(13)}
    csv = tmp_path / "samples.csv"
    csv.write_text("".join("s{},{}\n".format(s, b) for s, b in enumerate(bams)))
    args = [str(csv), "--workdir", str(tmp_path / "calls")] + [x for n in want for x in ("--tred", n)] + \
           ["--tred", "HD"]
    tred.main(args)
    calls = {}
    for s in range(4):
        with open(str(tmp_path / "calls" / "s{}.json".format(s))) as fp:
            calls[s] = json.load(fp)["tredCalls"]
    for si, name in enumerate(want):
        cut = sites[name]["cutoff_risk"]
        for s in range(4):
            c = calls[s]
            if s == EXPANDED:
                assert c[name + ".2"] >= cut and c[name + ".label"] == "risk" and c[name + ".PP"] > 0.9, (name, c)
            else:
                assert (c[name + ".1"], c[name + ".2"]) == NORMAL[s][si], (name, s, c[name + ".1"], c[name + ".2"])
    # the catalogue locus in the same run == a run without sites/
    bare = tmp_path / "bare"
    bare.mkdir()
    monkeypatch.chdir(str(bare))
    tred.main([str(csv), "--workdir", str(tmp_path / "calls0"), "--tred", "HD"])
    for s in range(4):
        with open(str(tmp_path / "calls0" / "s{}.json".format(s))) as fp:
            c0 = json.load(fp)["tredCalls"]
        assert {k: v for k, v in calls[s].items() if not k.startswith(tuple(want))} == c0
        assert (c0["HD.1"], c0["HD.2"]) == (17, 20)
