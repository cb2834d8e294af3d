"""Alt regions of discovered loci (DESIGN §4.5): the reference tract scan (tredsw_ref_tracts, its serial host emulation
and oracle/tract_oracle.py), the region rule of strprofile.alt_regions_for, the alts field of a sites row through
meta / tred.alt_regions, and `loci --alts`; on the GPU, the kernels against the emulation and the oracle, and the
workflow on a cohort whose expanded sample has most of its in-repeat reads mismapped onto decoy tracts."""
import json
import logging
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENV = dict(os.environ, PYTHONPATH=ROOT)

# planted units: periods 2, 3, 5, 12, 13 and 20
UNITS = ["AC", "CAG", "AAGGG", "ACGTTGCAAGCT", "TGCTTACCGTCAA", "GATCCAGTTAGCCTGAAAGT"]
# requested motifs: the units plus the root-period cases, which must give nothing
MOTIFS = UNITS + ["ATAT", "CAGCAG"]


def _rc(s):
    return s.translate(str.maketrans("ACGTacgt", "TGCAtgca"))[::-1]


def _random_contigs(seed, n=4, length=6000):
    """contigs of random bases with lowercase stretches, N runs, IUPAC codes and planted tracts (every rotation on
    both strands, some lowercase, some cut by an N or an IUPAC code, some at a contig's first or last base, two
    overlapping stretches of one period, (AT)n and (CAG)n), plus contigs shorter than 2k"""
    rng = np.random.default_rng(seed)
    out = {}
    for ci in range(n):
        s = list(rng.choice(list("ACGT"), length))
        pos = 50
        while pos < length - 400:
            u = UNITS[int(rng.integers(len(UNITS)))]
            r = int(rng.integers(len(u)))
            u = u[r:] + u[:r]
            if rng.random() < 0.5:
                u = _rc(u)
            t = u * int(rng.integers(2, max(3, 120 // len(u)) + 2))
            if rng.random() < 0.2:
                t = t.lower()
            t = list(t)
            x = rng.random()
            if x < 0.1:
                t[int(rng.integers(len(t)))] = "N"
            elif x < 0.2:
                t[int(rng.integers(len(t)))] = "RYKMSWBDHV"[int(rng.integers(10))]
            s[pos:pos + len(t)] = t
            pos += len(t) + int(rng.integers(0, 300))
        s[pos:pos + 60] = list("AT" * 30)
        s[pos + 100:pos + 100 + 60] = list("CAG" * 20)
        s[pos + 200:pos + 260] = list("AAGGG" * 8 + "AAGAGAAGAGAAGAG" + "AGAAG" * 1)   # two stretches of period 5
        for a in (0, 1):                                  # lowercase stretch and N run in random sequence
            b = int(rng.integers(0, length - 200))
            s[b:b + 150] = [c.lower() for c in s[b:b + 150]] if a else ["N"] * 150
        if ci == 0:
            s[:44] = list("ACGTTGCAAGCT" * 3 + "ACGTTGCA")            # at the first base
            s[-61:] = list("N" + "GATCCAGTTAGCCTGAAAGT" * 3)          # at the last base
        out["ctg{}".format(ci)] = "".join(s)
    out["short"] = "ACACACACACACACACACACACACACACACAC"[:int(rng.integers(3, 40))]
    out["tiny"] = "A"
    out["empty"] = ""
    return out


def _write(path, contigs, width, crlf=False):
    nl = "\r\n" if crlf else "\n"
    with open(path, "w", newline="") as fp:
        for name, seq in contigs.items():
            fp.write(">{} some description{}".format(name, nl))
            for i in range(0, len(seq), width):
                fp.write(seq[i:i + width] + nl)
    return path


def _as_tuples(res):
    t = res["tracts"]
    return [tuple(int(x) for x in r) for r in zip(t["contig"], t["start"], t["length"], t["period"], t["code"])]


# ---------------------------------------------------------------------------------------------------------------
# the tract rule: emulation of the device code == oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("width,crlf", [(1, False), (60, False), (61, False), (80, False), (60, True)])
def test_emulation_equals_the_oracle(tmp_path, width, crlf):
    from oracle import tract_oracle
    from tredparse_b200.fasta import Fasta
    contigs = _random_contigs(width + 1000 * crlf)
    fa = Fasta(_write(str(tmp_path / "r.fa"), contigs, width, crlf))
    want = tract_oracle.tracts(contigs, MOTIFS, 3, 30)
    got = fa.tracts(MOTIFS, emulate=True)
    assert _as_tuples(got) == want
    assert {t[3] for t in want} == {len(u) for u in UNITS} and len(want) > 40
    assert any(t[0] == 0 and t[1] == 0 for t in want) and any(t[0] == 0 and t[1] + t[2] == len(contigs["ctg0"]) for t in want)
    st = got["stats"]
    assert st["steps"] == 1 and st["bases"] == sum(map(len, contigs.values())) and st["tracts"] == len(want)
    assert st["invalid_bases"] == sum(1 for s in contigs.values() for c in s if c not in "ACGTacgt")
    # fewer copies / bases
    assert _as_tuples(fa.tracts(MOTIFS, min_units=5, min_len=0, emulate=True)) == tract_oracle.tracts(contigs, MOTIFS, 5, 0)
    assert _as_tuples(fa.tracts(UNITS[:2], min_units=2, min_len=10, emulate=True)) == \
        tract_oracle.tracts(contigs, UNITS[:2], 2, 10)


def test_root_period_cases_and_overlapping_stretches(tmp_path):
    from oracle import tract_oracle
    from tredparse_b200.fasta import Fasta, canonical_code
    contigs = {"a": "GT" + "AT" * 30 + "GG" + "CAG" * 20 + "T" + "AAGGG" * 8 + "AAGAGAAGAGAAGAGAAGAG" + "C" * 3}
    fa = Fasta(_write(str(tmp_path / "r.fa"), contigs, 60))
    assert _as_tuples(fa.tracts(["ATAT", "CAGCAG"], emulate=True)) == []
    assert _as_tuples(fa.tracts(["AT", "CAG"], emulate=True)) == [(0, 1, 60, 2, canonical_code("AT")),
                                                                  (0, 63, 60, 3, canonical_code("CAG"))]
    # AAGGG x 8 at 125, then AAGAG x 4: the period-5 stretches [125, 168) and [164, 185) overlap by four bases
    got = _as_tuples(fa.tracts(["AAGGG", "AAGAG"], min_len=20, emulate=True))
    assert got == tract_oracle.tracts(contigs, ["AAGGG", "AAGAG"], 3, 20)
    assert [(s, n) for _, s, n, _, _ in got] == [(125, 40), (164, 20)]


def test_steps_under_a_small_budget(tmp_path):
    from oracle import tract_oracle
    from tredparse_b200.fasta import Fasta
    contigs = _random_contigs(7, n=6, length=3000)
    contigs["big"] = _random_contigs(8, n=1, length=9000)["ctg0"]
    fa = Fasta(_write(str(tmp_path / "r.fa"), contigs, 60))
    got = fa.tracts(MOTIFS, step_bytes=4000, emulate=True)
    assert _as_tuples(got) == tract_oracle.tracts(contigs, MOTIFS, 3, 30)
    st = got["stats"]
    assert st["steps"] >= 6 and len(st["step_read_ms"]) == len(st["step_device_ms"]) == st["steps"]
    # the text from each contig's first base to its last: the file less its headers and final line breaks
    assert st["bytes"] == os.path.getsize(fa.path) - sum(len(">{} some description\n".format(n)) + (len(c) > 0)
                                                         for n, c in contigs.items())


def test_an_index_that_does_not_fit_the_file_is_an_io_error(tmp_path):
    from tredparse_b200 import _lib
    from tredparse_b200.fasta import Fasta
    contigs = {"a": "AC" * 200, "b": "CAG" * 100}
    path = _write(str(tmp_path / "r.fa"), contigs, 60)
    idx = Fasta(path).index
    with open(path + ".fai", "w") as fp:                 # line width one byte short: a base position hits '\n'
        for n, (L, off, lb, lw) in idx.items():
            fp.write("{}\t{}\t{}\t{}\t{}\n".format(n, L, off, lb, lw - 1))
    with pytest.raises(_lib.TredswError, match=r"code -4\).*index does not fit"):
        Fasta(path).tracts(["AC"], emulate=True)
    with open(path + ".fai", "w") as fp:                 # longer than the file
        fp.write("a\t400\t3\t60\t61\nb\t100000\t{}\t60\t61\n".format(idx["b"][1]))
    with pytest.raises(_lib.TredswError, match=r"code -4\).*shorter than its index"):
        Fasta(path).tracts(["AC"], emulate=True)
    with pytest.raises(_lib.TredswError, match=r"code -2\)"):
        _lib.ref_tracts(path, np.zeros(0, _lib.FAI_ENTRY_DTYPE), [(21, 0)], 3, 30, emulate=True)


# ---------------------------------------------------------------------------------------------------------------
# the region rule, by hand
# ---------------------------------------------------------------------------------------------------------------
def _tracts(rows, names=("c1", "c2", "c3")):
    from tredparse_b200 import _lib
    from tredparse_b200.fasta import canonical_code
    t = np.zeros(len(rows), dtype=_lib.TRACT_DTYPE)
    for i, (c, s, n, m) in enumerate(rows):
        t[i] = (s, n, canonical_code(m), c, len(m))
    return {"contigs": list(names), "tracts": t}


def test_alt_regions_by_hand():
    from oracle import tract_oracle
    from tredparse_b200.strprofile import alt_regions_for
    row = {"motif": "AAGGG", "repeat_location": "c1:5001-5050", "repeat_location.hg19": "c2:101-150"}
    rows = [(0, 3951, 50, "AAGGG"),       # ends at 4001 > 5001 - 1 - 1000: the locus' own window
            (0, 3800, 50, "AAGGG"),       # ends at 3850: an alt region
            (0, 5000, 50, "AAGGG"),       # the locus' own tract
            (0, 6049, 40, "CCCTT"),       # starts at 6049 < 5050 + 1000: own window (reverse strand: same motif)
            (0, 6050, 40, "CCCTT"),
            (0, 6239, 30, "AAGGG"),       # gap 149 = read length - 1: merged
            (0, 6419, 30, "AAGGG"),       # gap 150: a region of its own
            (0, 6450, 60, "AGC"),         # another motif
            (1, 10, 45, "AAGGG"), (2, 10, 45, "GGAAG")]
    tr = _tracts(sorted(rows, key=lambda r: (r[0], r[1])))
    want = "c1:3800-3850|c1:6050-6269|c1:6419-6449|c2:10-55|c3:10-55"
    assert alt_regions_for(row, tr, 150) == want
    own = ("c1", 5001, 5050)
    assert tract_oracle.alt_regions([(c, s, n, len(m), tract_oracle.code(tract_oracle.canonical(m)))
                                     for c, s, n, m in sorted(rows, key=lambda r: (r[0], r[1]))],
                                    ["c1", "c2", "c3"], own, "AAGGG", 150) == want
    # the cap: longest tract first (50 at c1:3800, 45 at c2 and c3, 40 in c1:6050-6269), ties by contig order
    assert alt_regions_for(row, tr, 150, max_alts=1) == "c1:3800-3850"
    assert alt_regions_for(row, tr, 150, max_alts=2) == "c1:3800-3850|c2:10-55"
    assert alt_regions_for(row, tr, 150, max_alts=4) == "c1:3800-3850|c1:6050-6269|c2:10-55|c3:10-55"
    # ties on one contig: by start
    tie = _tracts([(1, 10, 45, "AAGGG"), (1, 500, 45, "AAGGG"), (1, 900, 45, "AAGGG")])
    assert alt_regions_for(row, tie, 150, max_alts=2) == "c2:10-55|c2:500-545"
    # hg19 coordinates: the own window is on c2
    assert alt_regions_for(row, tr, 150, ref="hg19") == "c1:3800-4001|c1:5000-5050|c1:6049-6269|c1:6419-6449|c3:10-55"
    assert alt_regions_for(dict(row, motif="ACGTT"), tr, 150) == ""


def test_alts_field_and_sites_rows(tmp_path, monkeypatch):
    from tredparse_b200 import meta, tred
    assert meta.alts_field("hg38") == "alts" and meta.alts_field("hg19") == "alts.hg19"
    assert meta.alts_field("hg19_nochr") == "alts.hg19"
    base = {"title": "t", "gene_name": "", "id": "x", "motif": "AAGGG", "repeat": "AAGGG", "prefix": "A" * 18,
            "suffix": "C" * 18, "inheritance": "AD", "mutation_nature": "increase", "cutoff_prerisk": 30,
            "cutoff_risk": 30, "repeat_location": "c1:5001-5050", "repeat_location.hg19": "chr1:5001-5050"}
    rows = {"with": dict(base, alts="c3:10-55|1:7-9", **{"alts.hg19": "chr2:1-2"}), "empty": dict(base, alts=""),
            "without": dict(base)}
    (tmp_path / "sites").mkdir()
    (tmp_path / "sites" / "d.json").write_text(json.dumps(rows))
    monkeypatch.chdir(str(tmp_path))
    repo = meta.TREDsRepo()
    assert repo["with"].alt == [("c3", 10, 55), ("1", 7, 9)]
    assert repo["empty"].alt == [] and repo["without"].alt == []
    assert meta.TREDsRepo(ref="hg19")["with"].alt == [("chr2", 1, 2)]
    cat = meta.TREDsRepo.get_alts("hg38")
    assert repo["HD"].alt == cat["HD"] and len(cat["HD"]) == 88
    assert tred.alt_regions(repo["with"], "hg38_nochr", True, False) == [("c3", 10, 55), ("1", 7, 9)]
    t = meta.TREDsRepo(ref="hg19_nochr")["with"]
    t.alt = [("chr1", 5, 9), ("1", 7, 9)]
    assert tred.alt_regions(t, "hg19_nochr", True, False) == [("1", 5, 9), ("1", 7, 9)]
    assert tred.alt_regions(t, "hg19", True, False) == t.alt and tred.alt_regions(t, "hg19", False, False) == []
    hd = meta.TREDsRepo(ref="hg19_nochr")["HD"]
    assert tred.alt_regions(hd, "hg19_nochr", True, False) == [(c[3:], s, e) for c, s, e in hd.alt]


def test_reference_records_defaults_are_unchanged():
    from tredparse_b200 import simulate
    contigs = simulate.planted_reference([("c1", 6000)], [("c1", 3000, "AAGGG", 10)], seed=3)
    a = simulate.reference_records(contigs["c1"], 0, 3000, 3050, "AAGGG", (10, 80), seed=5)
    b = simulate.reference_records(contigs["c1"], 0, 3000, 3050, "AAGGG", (10, 80), seed=5, mismap_to=())
    def key(r):
        return tuple(getattr(r, f) for f in type(r).__slots__)
    assert [key(r) for r in a] == [key(r) for r in b]
    c = simulate.reference_records(contigs["c1"], 0, 3000, 3050, "AAGGG", (10, 80), seed=5, mismap_fraction=1.0,
                                   mismap_to=[(1, 100, 200), (1, 900, 950)])
    irr = [r for r in a if r.flag & 4 and r.reference_id == 0]
    moved = [r for r in c if r.reference_id == 1]
    assert irr and len(moved) == len(irr)
    assert all(r.mapping_quality == 0 and (100 <= r.reference_start < 200 or 900 <= r.reference_start < 950) and
               r.next_reference_id == 0 and not r.flag & 4 for r in moved)


# ---------------------------------------------------------------------------------------------------------------
# loci --alts
# ---------------------------------------------------------------------------------------------------------------
def _loci_inputs(tmp_path):
    from tredparse_b200 import simulate, strprofile
    contigs = simulate.planted_reference([("c1", 4000), ("c2", 3000)], [("c1", 1000, "GGGAA", 10),
                                                                      ("c2", 500, "TTCCC", 20)], seed=4)
    simulate.write_fasta(str(tmp_path / "ref.fa"), contigs)
    row = {"contig": "c1", "start": 990, "end": 1040, "motif": "AAGGG", "top_sample": "a", "z": 9.0,
           "counts": {"a": 1.0, "b": 0.0}}
    with open(str(tmp_path / "out.tsv"), "w") as fp:
        strprofile.write_tsv([row], ["a", "b"], fp)
    (tmp_path / "a.str_profile.json").write_text(json.dumps({"sample": "a", "read_length": 150}))


def _loci(tmp_path, *extra, env=ENV):
    return subprocess.run([sys.executable, "-m", "tredparse_b200.strprofile", "loci", str(tmp_path / "out.tsv"),
                           "--fasta", str(tmp_path / "ref.fa"), "--profiles", str(tmp_path / "a.str_profile.json"),
                           *extra], cwd=str(tmp_path), env=env, capture_output=True, text=True)


def test_loci_without_alts_writes_no_field_and_without_a_device_fails_cleanly(tmp_path):
    _loci_inputs(tmp_path)
    r = _loci(tmp_path)
    assert r.returncode == 0, r.stderr
    with open(str(tmp_path / "sites" / "discovered.json")) as fp:
        sites = json.load(fp)
    assert list(sites) == ["c1_1001_GGGAA"] and not any(k.startswith("alts") for k in sites["c1_1001_GGGAA"])
    os.remove(str(tmp_path / "sites" / "discovered.json"))
    r = _loci(tmp_path, "--alts", "--out", str(tmp_path / "o.json"), env=dict(ENV, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 1 and "no CUDA device" in r.stderr and r.stdout == ""
    assert not os.path.exists(str(tmp_path / "o.json"))


@pytest.mark.gpu
def test_gpu_loci_alts(tmp_path):
    _loci_inputs(tmp_path)
    r = _loci(tmp_path, "--alts", "--ref", "hg19")
    assert r.returncode == 0, r.stderr
    assert r.stdout.split() == ["c1_1001_GGGAA"] and "c1_1001_GGGAA: 1 alt regions" in r.stderr.splitlines()
    with open(str(tmp_path / "sites" / "discovered.json")) as fp:
        row = json.load(fp)["c1_1001_GGGAA"]
    assert row["alts.hg19"] == "c2:500-600" and "alts" not in row


# ---------------------------------------------------------------------------------------------------------------
# on the GPU: the kernels
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("width,crlf", [(1, False), (61, False), (80, False), (60, True)])
def test_gpu_kernels_equal_the_emulation_and_the_oracle(tmp_path, width, crlf):
    from oracle import tract_oracle
    from tredparse_b200.fasta import Fasta
    contigs = _random_contigs(width + 1000 * crlf)
    fa = Fasta(_write(str(tmp_path / "r.fa"), contigs, width, crlf))
    want = tract_oracle.tracts(contigs, MOTIFS, 3, 30)
    for step in (0, 2000):
        dev, emu = fa.tracts(MOTIFS, step_bytes=step), fa.tracts(MOTIFS, step_bytes=step, emulate=True)
        assert _as_tuples(dev) == _as_tuples(emu) == want
        assert {k: dev["stats"][k] for k in ("steps", "bytes", "bases", "invalid_bases", "tracts")} == \
               {k: emu["stats"][k] for k in ("steps", "bytes", "bases", "invalid_bases", "tracts")}


def _big_fasta(path, seed, sizes, width=60):
    """a seeded reference of random bases with lowercase stretches, N runs and planted tracts of UNITS"""
    rng = np.random.default_rng(seed)
    lut = np.frombuffer(b"ACGT", np.uint8)
    with open(path, "wb") as fp:
        for ci, L in enumerate(sizes):
            s = lut[rng.integers(0, 4, L)]
            for _ in range(L // 200000):
                a = int(rng.integers(0, L - 5000))
                s[a:a + int(rng.integers(100, 5000))] += 32              # lowercase
            for _ in range(L // 1000000):
                a = int(rng.integers(0, L - 20000))
                s[a:a + int(rng.integers(10, 20000))] = ord("N")
            for _ in range(L // 20000):
                u = UNITS[int(rng.integers(len(UNITS)))]
                t = np.frombuffer((u * int(rng.integers(2, 30))).encode(), np.uint8)
                a = int(rng.integers(0, L - len(t)))
                s[a:a + len(t)] = t
            fp.write(">chr{}\n".format(ci + 1).encode())
            n = (L + width - 1) // width
            body = np.full(n * (width + 1), ord("\n"), np.uint8).reshape(n, width + 1)
            pad = np.full(n * width, ord("\n"), np.uint8)
            pad[:L] = s
            body[:, :width] = pad.reshape(n, width)
            fp.write(body.tobytes()[:L + n])
    return path


@pytest.mark.gpu
def test_gpu_kernels_equal_the_emulation_on_100_mbp(tmp_path):
    from tredparse_b200.fasta import Fasta
    fa = Fasta(_big_fasta(str(tmp_path / "big.fa"), 11, [41000000, 30000000, 20000000, 9000000, 777]))
    # 16 MiB steps: the three largest contigs (41.7, 30.5 and 20.3 MB of text) are steps of their own, the last two
    # contigs (9.2 MB and 790 bytes) share one
    dev = fa.tracts(MOTIFS, step_bytes=16 << 20)
    emu = fa.tracts(MOTIFS, step_bytes=16 << 20, emulate=True)
    assert np.array_equal(dev["tracts"], emu["tracts"]) and dev["stats"]["tracts"] > 4000
    assert {k: dev["stats"][k] for k in ("steps", "bytes", "bases", "invalid_bases", "tracts")} == \
           {k: emu["stats"][k] for k in ("steps", "bytes", "bases", "invalid_bases", "tracts")}
    assert dev["stats"]["bases"] == 100000777 and dev["stats"]["steps"] == 4 and dev["stats"]["invalid_bases"] > 0


# ---------------------------------------------------------------------------------------------------------------
# on the GPU: profile -> outliers -> loci --alts -> tred.py --tred, in-repeat reads mismapped onto decoys
# ---------------------------------------------------------------------------------------------------------------
SITES = [("c1", 12000, "GGGAA", 10, "AAGGG"), ("c2", 9000, "TGCTTACCGTCAA", 4, None)]
DECOYS = [("c3", 2000, "GGGAA", 30), ("c3", 6000, "TTCCC", 20), ("c3", 10000, "TGCTTACCGTCAA", 10)]
REFS = [("c1", 24000), ("c2", 18000), ("c3", 14000)]
NORMAL = {0: ((8, 12), (3, 5)), 1: ((10, 10), (4, 6)), 2: ((6, 11), (2, 4))}
EXPANDED, EXP_UNITS, MISMAP = 3, 200, 0.7


def _cohort(d):
    """four samples on the planted reference plus chr4 with HD: samples 0-2 carry short alleles at both sites, sample 3
    a 200-unit expansion at each with 70 % of its in-repeat reads mismapped onto the decoys of the site's motif;
    samples 0 and 3 indexed, 1 and 2 not"""
    from tredparse_b200 import bamio, simulate
    from tredparse_b200.meta import TREDsRepo
    contigs = simulate.planted_reference(REFS, [s[:4] for s in SITES] + DECOYS, seed=23)
    simulate.write_fasta(str(d / "ref.fa"), contigs, width=70)
    hd = TREDsRepo()["HD"]
    refs = REFS + [("chr4", hd.repeat_end + 20000)]
    bams = []
    for s in range(4):
        recs = []
        for si, (c, pos, u, n, canon) in enumerate(SITES):
            al = (NORMAL[0][si][0], EXP_UNITS) if s == EXPANDED else NORMAL[s][si]
            decoys = [(2, p, p + len(du) * dn) for _, p, du, dn in DECOYS if _canon(du) == _canon(u)]
            recs += simulate.reference_records(contigs[c], si, pos, pos + len(u) * n, u, al, cov_per_hap=15,
                                               flank=1500, seed=100 * s + si, tag="s{}x{}".format(s, si),
                                               mismap_fraction=MISMAP if s == EXPANDED else 0.0, mismap_to=decoys)
        recs += simulate.locus_records(hd, 2, (17, 20), 150, 10.0, seed=40 + s, tag="s{}hd".format(s), flank=1000)
        path = str(d / "s{}.bam".format(s))
        bamio.write_bam(path, refs, simulate.coordinate_sort(recs), index=s in (0, 3), aux=True)
        bams.append(path)
    return bams


def _canon(u):
    from oracle.tract_oracle import canonical
    return canonical(u)


def _calls(csv, workdir, names, *extra):
    from tredparse_b200 import tred
    tred.main([str(csv), "--workdir", str(workdir)] + [x for n in names for x in ("--tred", n)] + list(extra))
    out = {}
    for s in range(4):
        with open(str(workdir / "s{}.json".format(s))) as fp:
            out[s] = json.load(fp)["tredCalls"]
    return out


@pytest.mark.gpu
def test_gpu_alt_regions_rescue_mismapped_in_repeat_reads(tmp_path, monkeypatch, capsys):
    from test_ingest import _assert_same_record as assert_same_record
    from tredparse_b200 import bam_parser, ingest, meta, strprofile
    bams = _cohort(tmp_path)
    work = tmp_path / "w"
    assert strprofile.main(["profile", *bams, "--workdir", str(work)]) == 0
    profs = [str(work / "s{}.str_profile.json".format(s)) for s in range(4)]
    assert strprofile.main(["outliers", *profs, "--tsv", str(tmp_path / "out.tsv")]) == 0
    run = tmp_path / "run"
    run.mkdir()
    monkeypatch.chdir(str(run))
    capsys.readouterr()
    assert strprofile.main(["loci", str(tmp_path / "out.tsv"), "--fasta", str(tmp_path / "ref.fa"),
                            "--profiles", *profs, "--alts"]) == 0
    out = capsys.readouterr()
    names = ["{}_{}_{}".format(c, pos + 1, u) for c, pos, u, _, _ in SITES]
    assert sorted(out.out.split()) == sorted(names)
    with open("sites/discovered.json") as fp:
        sites = json.load(fp)
    assert sites[names[0]]["alts"] == "c3:2000-2150|c3:6000-6100"          # the decoys, not the locus' own tract
    assert sites[names[1]]["alts"] == "c3:10000-10130"
    assert "{}: 2 alt regions".format(names[0]) in out.err.splitlines()
    csv = tmp_path / "samples.csv"
    csv.write_text("".join("s{},{}\n".format(s, b) for s, b in enumerate(bams)))
    calls = _calls(csv, tmp_path / "calls", names + ["HD"])
    noalts = _calls(csv, tmp_path / "calls_noalts", names + ["HD"], "--noalts")
    # the evidence of the indexed samples with the alts: native reader == Python reader
    repo = meta.TREDsRepo()
    for s in (0, EXPANDED):
        for name in names:
            with ingest.BamIngest(bams[s]) as ing:
                ev = ing.extract_locus(repo[name], 150, alts=repo[name].alt, want_names=True)
            py = bam_parser.extract_locus(bams[s], repo, name, 150, True, False, logging.getLogger())
            assert_same_record(py, ev)
            if s == EXPANDED:
                assert ev.nreads > len(ing_noalts(bams[s], repo[name]).names)
    for si, name in enumerate(names):
        cut = sites[name]["cutoff_risk"]
        for s in range(4):
            c, c0 = calls[s], noalts[s]
            if s == EXPANDED:
                assert c[name + ".RDP"] > c0[name + ".RDP"], (name, c, c0)
                assert c[name + ".2"] >= c0[name + ".2"] and c[name + ".2"] >= cut and c[name + ".label"] == "risk"
            else:
                assert {k: v for k, v in c.items() if k.startswith(name)} == \
                       {k: v for k, v in c0.items() if k.startswith(name)}
                assert (c[name + ".1"], c[name + ".2"]) == NORMAL[s][si]
    bare = tmp_path / "bare"
    bare.mkdir()
    monkeypatch.chdir(str(bare))
    c0 = _calls(csv, tmp_path / "calls0", ["HD"])
    for s in range(4):
        assert {k: v for k, v in calls[s].items() if k.startswith("HD")} == {k: v for k, v in c0[s].items() if k.startswith("HD")}


def ing_noalts(bam, t):
    from tredparse_b200 import ingest
    with ingest.BamIngest(bam) as ing:
        return ing.extract_locus(t, 150, alts=(), want_names=True)
