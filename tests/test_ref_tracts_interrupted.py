"""Interrupted reference tracts (DESIGN §4.5.1): pure tracts of one motif joined across short interruptions by the
tract scan (tredsw_ref_tracts_ex, its serial host emulation and oracle/chain_oracle.chained_tracts), the locus rule
of strprofile.locus_for in chain mode against oracle/chain_oracle.locus, and `loci --max-interruption`; on the GPU, the
kernels against the emulation and the oracle, and the workflow on a cohort whose discovered site is an interrupted
tract and whose expanded sample has most of its in-repeat reads mismapped onto interrupted decoys."""
import ctypes
import json
import os

import numpy as np
import pytest

from test_ref_tracts import (ENV, MOTIFS, UNITS, _big_fasta, _calls, _canon, _random_contigs, _rc, _write,
                             ing_noalts)

GRID = [(g, p) for g in (1, 3, 20) for p in ((9, 10), (3, 4), (1, 1))]


def _interrupted(rng, g, unit=None):
    """one planted interrupted tract: a rotation of a unit of UNITS on either strand, 1 to 3 interruptions among
    substitutions (some by an N), insertions of 1 to g + 1 bases (phase shifts), deletions of 1 or 2 bases, copies of
    another unit and homopolymers; lowercase at times"""
    from tredparse_b200 import simulate
    u = unit or UNITS[int(rng.integers(len(UNITS)))]
    r = int(rng.integers(len(u)))
    u = u[r:] + u[:r]
    if rng.random() < 0.5:
        u = _rc(u)
    k = len(u)
    n = int(rng.integers(4, max(5, 100 // k) + 4))
    edits = []
    for c in sorted(set(int(x) for x in rng.integers(1, n, int(rng.integers(1, 4))))):
        x = rng.random()
        if x < 0.3:
            edits.append((c, "sub", "N" if rng.random() < 0.15 else "ACGT"[int(rng.integers(4))]))
        elif x < 0.65:
            ins = "".join(rng.choice(list("ACGT"), int(rng.integers(1, g + 2))))
            if rng.random() < 0.1:
                ins = ins[:-1] + "N"
            edits.append((c, "ins", ins))
        elif x < 0.85:
            edits.append((c, "del", int(rng.integers(1, 3))))
        elif x < 0.93:
            v = UNITS[(UNITS.index(unit) + 1) % len(UNITS)] if unit else "CAG" if k != 3 else "AC"
            edits.append((c, "ins", v * 3))
        else:
            edits.append((c, "ins", "A" * (k + 2)))
    t = simulate.interrupted_tract(u, n, edits)
    return t.lower() if rng.random() < 0.2 else t


def _interrupted_contigs(seed, g, n=4, length=6000):
    """_random_contigs with interrupted tracts planted over them, one at the first base of ctg0 and one at the last
    base of ctg1"""
    rng = np.random.default_rng(seed + 77)
    out = _random_contigs(seed, n, length)
    for ci in range(n):
        s = list(out["ctg{}".format(ci)])
        pos = int(rng.integers(0, 200)) if ci else 0
        while pos < length - 400:
            t = _interrupted(rng, g)
            s[pos:pos + len(t)] = list(t)
            pos += len(t) + int(rng.integers(20, 500))
        if ci == 1:
            t = _interrupted(rng, g)
            s[-len(t):] = list(t)
        out["ctg{}".format(ci)] = "".join(s)
    return out


def _tuples(res):
    t = res["tracts"]
    return [tuple(int(x) for x in r) for r in zip(t["contig"], t["start"], t["length"], t["period"], t["code"],
                                                  res["segments"])]


def _check_grid(fa, contigs, step=0, **kw):
    """every (g, purity) of GRID: the scan == the oracle; -> the chains seen"""
    from oracle import chain_oracle
    chains = 0
    for g, pur in GRID:
        want = chain_oracle.chained_tracts(contigs, MOTIFS, 3, 30, g, *pur)
        got = fa.tracts(MOTIFS, step_bytes=step, max_interrupt=g, purity=pur, **kw)
        assert _tuples(got) == want, (g, pur)
        assert got["stats"]["tracts"] == len(want)
        chains += sum(1 for t in want if t[5] > 1)
        if pur == (1, 1):
            assert all(t[5] == 1 for t in want)
    return chains


# ---------------------------------------------------------------------------------------------------------------
# the rule: emulation of the device code == oracle
# ---------------------------------------------------------------------------------------------------------------
def test_interrupted_tract_planting():
    from tredparse_b200 import simulate
    assert simulate.interrupted_tract("CAG", 4) == "CAG" * 4
    assert simulate.interrupted_tract("CAG", 4, [(1, "sub", "T"), (2, "ins", "AA"), (3, "del", 2)]) == \
        "CAG" + "TAG" + "AACAG" + "G"
    with pytest.raises(ValueError):
        simulate.interrupted_tract("CAG", 4, [(1, "dup", 1)])
    sites = [("c1", 100, "CAG", 10), ("c1", 600, "AAGGG", 8)]
    a = simulate.planted_reference([("c1", 1000)], sites, seed=2)
    assert a == simulate.planted_reference([("c1", 1000)], [s + ((),) for s in sites], seed=2)
    b = simulate.planted_reference([("c1", 1000)], [sites[0] + ([(5, "sub", "A")],), sites[1]], seed=2)
    assert b["c1"][100:130] == "CAG" * 5 + "AAG" + "CAG" * 4 and b["c1"][130:] == a["c1"][130:]


@pytest.mark.parametrize("width,crlf", [(1, False), (60, False), (61, False), (80, False), (60, True)])
def test_emulation_equals_the_oracle(tmp_path, width, crlf):
    contigs = _interrupted_contigs(width + 1000 * crlf, 20)
    from tredparse_b200.fasta import Fasta
    fa = Fasta(_write(str(tmp_path / "r.fa"), contigs, width, crlf))
    assert _check_grid(fa, contigs, emulate=True) > 20


def test_the_rule_by_hand(tmp_path):
    from oracle import chain_oracle
    from tredparse_b200.fasta import Fasta
    pieces = ["CAG" * 8 + "TAG" + "CAG" * 8,                  # a substitution: pure pieces of 24 and 26 bases
              "CAG" * 10 + "TT" + "CAG" * 10,                 # 2 inserted bases: joined at g >= 2 only
              "CAG" * 8 + "AG" + "CAG" * 8,                   # a deletion of one base (phase shift)
              "CAG" * 10 + "ATT" * 3 + "CAG" * 10,            # a segment of another code between: never joined
              "CAG" * 10 + "AN" + "CAG" * 10,                 # an N in the interruption: never joined
              "CAG" * 4 + "TAG" + "CAG" * 2 + "TAG" + "CAG" * 2 + "TAG" + "CAG" * 4]   # 6 disagreements in 42
    seq = "".join(p + "GTCA" * 5 for p in pieces)
    at = [int(x) for x in np.cumsum([0] + [len(p) + 20 for p in pieces])]
    fa = Fasta(_write(str(tmp_path / "r.fa"), {"a": seq}, 60))

    def got(g, pur=(9, 10), **kw):
        return [(s, n, m) for _, s, n, _, _, m in _tuples(fa.tracts(["CAG"], max_interrupt=g, purity=pur,
                                                                   emulate=True, **kw))]
    assert got(0) == [(at[1], 30, 1), (at[1] + 32, 30, 1), (at[3], 30, 1), (at[3] + 39, 30, 1), (at[4], 30, 1),
                      (at[4] + 32, 30, 1)]
    assert got(1) == [(at[0], 51, 2), (at[1], 30, 1), (at[1] + 32, 30, 1), (at[2], 48, 2)] + got(0)[2:]
    assert got(2)[:3] == [(at[0], 51, 2), (at[1], 60, 2), (at[2], 48, 2)]
    loose = got(20, (1, 2))                                # (pieces also join across the 20-base spacers)
    assert any(m > 1 for _, _, m in loose)
    assert not any(s < at[3] + 30 < at[3] + 39 < s + n or s <= at[4] + 31 < s + n for s, n, _ in loose)
    # 9 / 10 fails: the pieces alone (here kept with min_len 0); 3 / 4 passes
    assert [t for t in got(1, min_len=0) if t[0] >= at[5]] == [(at[5], 12, 1), (at[5] + 31, 12, 1)]
    assert [t for t in got(1, (3, 4)) if t[0] >= at[5]] == [(at[5], 45, 4)]
    for g in (0, 1, 2, 20):
        assert _tuples(fa.tracts(["CAG"], max_interrupt=g, emulate=True)) == \
            chain_oracle.chained_tracts({"a": seq}, ["CAG"], 3, 30, g, 9, 10)
    # the invariants: g = 0 and purity 1 / 1 are the pure rule
    pure = fa.tracts(["CAG"], emulate=True)
    assert list(pure["segments"]) == [1] * len(pure["tracts"])
    for g, pur in ((0, (9, 10)), (20, (1, 1))):
        x = fa.tracts(["CAG"], max_interrupt=g, purity=pur, emulate=True)
        assert np.array_equal(x["tracts"], pure["tracts"]) and list(x["segments"]) == [1] * len(pure["tracts"])


@pytest.mark.parametrize("seed", [1, 2])
def test_invariants_on_random_contigs(tmp_path, seed):
    from oracle import chain_oracle, tract_oracle
    from tredparse_b200.fasta import Fasta
    contigs = _interrupted_contigs(seed, 3)
    fa = Fasta(_write(str(tmp_path / "r.fa"), contigs, 60))
    pure = fa.tracts(MOTIFS, emulate=True)
    assert [t[:5] for t in chain_oracle.chained_tracts(contigs, MOTIFS, 3, 30, 0)] == \
        tract_oracle.tracts(contigs, MOTIFS, 3, 30)
    for g, pur in ((0, (9, 10)), (0, (1, 2)), (1, (1, 1)), (20, (1, 1))):
        x = fa.tracts(MOTIFS, max_interrupt=g, purity=pur, emulate=True)
        assert np.array_equal(x["tracts"], pure["tracts"]) and not np.any(x["segments"] != 1)


def test_steps_under_a_small_budget(tmp_path):
    from tredparse_b200.fasta import Fasta
    contigs = _interrupted_contigs(7, 20, n=6, length=3000)
    contigs["big"] = _interrupted_contigs(8, 20, n=1, length=9000)["ctg0"]
    fa = Fasta(_write(str(tmp_path / "r.fa"), contigs, 60))
    assert _check_grid(fa, contigs, step=4000, emulate=True) > 20
    assert fa.tracts(MOTIFS, step_bytes=4000, max_interrupt=3, emulate=True)["stats"]["steps"] >= 6


def test_bgzf_gives_the_text_results(tmp_path):
    from tredparse_b200 import simulate
    from tredparse_b200.fasta import Fasta
    contigs = _interrupted_contigs(11, 20)
    src = _write(str(tmp_path / "r.fa"), contigs, 61)
    text = Fasta(src)
    for bs in (97, 0xFF00):
        fa = Fasta(simulate.bgzip_fasta(src, str(tmp_path / "r{}.fa.gz".format(bs)), block_size=bs))
        for g, pur in GRID[::2]:
            a = fa.tracts(MOTIFS, max_interrupt=g, purity=pur, emulate=True)
            b = text.tracts(MOTIFS, max_interrupt=g, purity=pur, emulate=True)
            assert _tuples(a) == _tuples(b) and a["stats"]["blocks"] > 0
        assert _check_grid(fa, contigs, step=3000, emulate=True) > 20


def test_out_of_range_chain_parameters_are_argument_errors(tmp_path):
    from tredparse_b200 import _lib
    from tredparse_b200.fasta import Fasta
    fa = Fasta(_write(str(tmp_path / "r.fa"), {"a": "CAG" * 40}, 60))
    for g, pur in ((21, (9, 10)), (-1, (9, 10)), (1, (0, 10)), (1, (11, 10)), (1, (5, 1001)), (1, (-1, 10))):
        with pytest.raises(_lib.TredswError, match=r"code -2\).*chain parameters out of range"):
            fa.tracts(["CAG"], max_interrupt=g, purity=pur, emulate=True)
    assert len(fa.tracts(["CAG"], max_interrupt=20, purity=(1000, 1000), emulate=True)["tracts"]) == 1


# ---------------------------------------------------------------------------------------------------------------
# the locus and its alt regions in chain mode
# ---------------------------------------------------------------------------------------------------------------
def test_locus_and_alt_regions_in_chain_mode_equal_the_oracles(tmp_path):
    from oracle import chain_oracle, locus_oracle, tract_oracle
    from tredparse_b200 import simulate, strprofile
    from tredparse_b200.fasta import Fasta
    rng = np.random.default_rng(5)
    sites = []
    for i in range(12):
        u = UNITS[i % len(UNITS)]
        t = _interrupted(rng, 3, unit=u)
        sites.append(("c{}".format(i % 3), 1500 + 2500 * (i // 3), t.upper(), 1))
    contigs = simulate.planted_reference([("c0", 12000), ("c1", 12000), ("c2", 12000)], sites, seed=9)
    fa = Fasta(simulate.write_fasta(str(tmp_path / "ref.fa"), contigs, fai=True))
    motifs = []
    seen = 0
    for i, (c, pos, t, _) in enumerate(sites):
        motif = tract_oracle.canonical(UNITS[i % len(UNITS)])
        motifs.append(motif)
        row = {"contig": c, "start": pos - 100, "end": pos + 150, "motif": motif, "z": 5.0}
        for g, pur in ((1, (9, 10)), (3, (9, 10)), (20, (3, 4)), (3, (1, 1))):
            want = chain_oracle.locus(row, contigs, 150, max_interrupt=g, purity=pur)
            try:
                name, got = strprofile.locus_for(row, fa, 150, max_interrupt=g, purity=pur)
            except strprofile.Skip as e:
                assert want == str(e), (i, g, pur)
                continue
            seen += 1
            assert want[0] == name and {k: got[k] for k in want[1]} == want[1], (i, g, pur)
    assert seen > 30
    # g = 0 keeps the pure rule
    def pure(row, **kw):
        try:
            return strprofile.locus_for(row, fa, 150, **kw)
        except strprofile.Skip as e:
            return str(e)
    for i, (c, pos, t, _) in enumerate(sites):
        row = {"contig": c, "start": pos - 100, "end": pos + 150, "motif": motifs[i], "z": 5.0}
        assert pure(row) == pure(row, max_interrupt=0, purity=(1, 2))
        want = locus_oracle.locus(row, contigs, 150)
        got = pure(row)
        assert want == got if isinstance(got, str) else (want[0] == got[0] and
                                                        {k: got[1][k] for k in want[1]} == want[1])
    # the alt regions of each locus from the chain tracts
    tr = fa.tracts(set(motifs), max_interrupt=3, emulate=True)
    otr = [t[:5] for t in chain_oracle.chained_tracts(contigs, motifs, 3, 30, 3, 9, 10)]
    assert _tuples(tr) == chain_oracle.chained_tracts(contigs, motifs, 3, 30, 3, 9, 10)
    for i, (c, pos, t, _) in enumerate(sites):
        row = {"contig": c, "start": pos - 100, "end": pos + 150, "motif": motifs[i], "z": 5.0}
        try:
            _, loc = strprofile.locus_for(row, fa, 150, max_interrupt=3)
        except strprofile.Skip:
            continue
        first, last = [int(x) for x in loc["repeat_location"].split(":")[1].split("-")]
        assert strprofile.alt_regions_for(loc, tr, 150) == \
            tract_oracle.alt_regions(otr, tr["contigs"], (c, first, last), motifs[i], 150)


# ---------------------------------------------------------------------------------------------------------------
# loci --max-interruption
# ---------------------------------------------------------------------------------------------------------------
def _chain_loci_inputs(tmp_path, purities):
    from tredparse_b200 import simulate, strprofile
    site = ("c1", 1000, "GGGAA", 12, [(6, "sub", "C")])           # pieces of 30 and 29 bases
    contigs = simulate.planted_reference([("c1", 4000), ("c2", 3000)], [site, ("c2", 500, "TTCCC", 20)], seed=4)
    simulate.write_fasta(str(tmp_path / "ref.fa"), contigs)
    row = {"contig": "c1", "start": 990, "end": 1070, "motif": "AAGGG", "top_sample": "a", "z": 9.0,
           "counts": {"a": 1.0, "b": 0.0}}
    with open(str(tmp_path / "out.tsv"), "w") as fp:
        strprofile.write_tsv([row], ["a", "b"], fp)
    for s, (num, den) in zip("ab", purities):
        prof = {"sample": s, "read_length": 150, "params": {"purity_num": num, "purity_den": den}}
        (tmp_path / "{}.str_profile.json".format(s)).write_text(json.dumps(prof))


def _loci2(tmp_path, *extra, env=ENV):
    import subprocess
    import sys
    return subprocess.run([sys.executable, "-m", "tredparse_b200.strprofile", "loci", str(tmp_path / "out.tsv"),
                           "--fasta", str(tmp_path / "ref.fa"), "--profiles", str(tmp_path / "a.str_profile.json"),
                           str(tmp_path / "b.str_profile.json"), *extra], cwd=str(tmp_path), env=env,
                          capture_output=True, text=True)


def _sites(tmp_path):
    with open(str(tmp_path / "sites" / "discovered.json")) as fp:
        return json.load(fp)


def test_loci_max_interruption_reads_the_purity_from_the_profiles(tmp_path):
    _chain_loci_inputs(tmp_path, [(9, 10), (9, 10)])
    r = _loci2(tmp_path)
    assert r.returncode == 0, r.stderr
    assert list(_sites(tmp_path)) == ["c1_1001_GGGAA"]                   # the longer pure piece
    assert _sites(tmp_path)["c1_1001_GGGAA"]["repeat_location"] == "c1:1001-1030"
    r = _loci2(tmp_path, "--max-interruption", "1")
    assert r.returncode == 0, r.stderr
    row = _sites(tmp_path)["c1_1001_GGGAA"]
    assert row["repeat_location"] == "c1:1001-1060" and "alts" not in row    # the whole interrupted tract
    # purity 1 / 1 in the profiles: nothing joins
    _chain_loci_inputs(tmp_path, [(1, 1), (1, 1)])
    r = _loci2(tmp_path, "--max-interruption", "1")
    assert r.returncode == 0, r.stderr
    assert _sites(tmp_path)["c1_1001_GGGAA"]["repeat_location"] == "c1:1001-1030"


def test_loci_max_interruption_refuses_profiles_that_disagree_and_fails_cleanly_without_a_device(tmp_path):
    _chain_loci_inputs(tmp_path, [(9, 10), (4, 5)])
    r = _loci2(tmp_path, "--max-interruption", "1")
    assert r.returncode == 2 and "needs one purity" in r.stderr and not os.path.exists(str(tmp_path / "sites"))
    assert _loci2(tmp_path).returncode == 0                               # without it the purity is not read
    r = _loci2(tmp_path, "--max-interruption", "21")
    assert r.returncode == 2 and "0 to 20" in r.stderr
    _chain_loci_inputs(tmp_path, [(9, 10), (9, 10)])
    r = _loci2(tmp_path, "--alts", "--max-interruption", "1", "--out", str(tmp_path / "o.json"),
               env=dict(ENV, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 1 and "no CUDA device" in r.stderr and r.stdout == ""
    assert not os.path.exists(str(tmp_path / "o.json"))


# ---------------------------------------------------------------------------------------------------------------
# on the GPU: the kernels
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("width,crlf", [(1, False), (61, False), (80, False), (60, True)])
def test_gpu_kernels_equal_the_emulation_and_the_oracle(tmp_path, width, crlf):
    from tredparse_b200 import simulate
    from tredparse_b200.fasta import Fasta
    contigs = _interrupted_contigs(width + 1000 * crlf, 20)
    src = _write(str(tmp_path / "r.fa"), contigs, width, crlf)
    for path in (src, simulate.bgzip_fasta(src, str(tmp_path / "r.fa.gz"), block_size=997)):
        fa = Fasta(path)
        for step in (0, 2000):
            assert _check_grid(fa, contigs, step=step) > 20
            for g, pur in GRID:
                dev = fa.tracts(MOTIFS, step_bytes=step, max_interrupt=g, purity=pur)
                emu = fa.tracts(MOTIFS, step_bytes=step, max_interrupt=g, purity=pur, emulate=True)
                assert np.array_equal(dev["tracts"], emu["tracts"]) and np.array_equal(dev["segments"], emu["segments"])
                assert {k: dev["stats"][k] for k in ("steps", "bytes", "bases", "invalid_bases", "tracts")} == \
                       {k: emu["stats"][k] for k in ("steps", "bytes", "bases", "invalid_bases", "tracts")}


def _raw(path, fa, motifs, chain):
    """tredsw_ref_tracts (chain None) or tredsw_ref_tracts_ex with a chain struct or NULL (chain "null") -> the raw
    bytes of the tract array and the segment counts"""
    from tredparse_b200 import _lib
    from tredparse_b200.fasta import canonical_code
    lib = _lib.load()
    names = list(fa.index)
    cs = np.zeros(len(names), dtype=_lib.FAI_ENTRY_DTYPE)
    for i, n in enumerate(names):
        cs[i] = tuple(fa.index[n])
    ms = np.zeros(len(motifs), dtype=_lib.MOTIF_DTYPE)
    for i, m in enumerate(motifs):
        ms[i]["period"], ms[i]["code"] = len(m), canonical_code(m)
    prm = _lib.TractParams(3, 30, 0)
    res = ctypes.c_void_p()
    h = _lib.default_context().handle
    if chain is None:
        rc = lib.tredsw_ref_tracts(h, path.encode(), _lib.ptr(cs), len(cs), _lib.ptr(ms), len(ms), ctypes.byref(prm),
                                   ctypes.byref(res))
    else:
        ch = None if chain == "null" else ctypes.byref(_lib.TractChain(*chain, 0))
        rc = lib.tredsw_ref_tracts_ex(h, path.encode(), _lib.ptr(cs), len(cs), _lib.ptr(ms), len(ms),
                                      ctypes.byref(prm), ch, ctypes.byref(res))
    _lib.check(rc, "tredsw_ref_tracts")
    try:
        v = _lib.TractsView()
        _lib.check(lib.tredsw_ref_tracts_view(res, ctypes.byref(v)), "view")
        n = int(v.n_tracts)
        return ctypes.string_at(v.tracts, n * _lib.TRACT_DTYPE.itemsize), [v.segments[i] for i in range(n)]
    finally:
        lib.tredsw_ref_tracts_free(res)


@pytest.mark.gpu
def test_gpu_ex_without_chaining_is_the_pure_scan_bit_for_bit(tmp_path):
    from tredparse_b200.fasta import Fasta
    contigs = _interrupted_contigs(3, 20)
    path = _write(str(tmp_path / "r.fa"), contigs, 60)
    fa = Fasta(path)
    base, segs = _raw(path, fa, MOTIFS, None)
    assert len(base) > 0 and set(segs) == {1}
    for chain in ("null", (0, 9, 10), (0, 1, 1), (5, 1, 1)):
        assert _raw(path, fa, MOTIFS, chain) == (base, segs), chain
    other, osegs = _raw(path, fa, MOTIFS, (3, 9, 10))
    assert other != base and max(osegs) > 1


@pytest.mark.gpu
def test_gpu_kernels_equal_the_emulation_on_100_mbp(tmp_path):
    from tredparse_b200.fasta import Fasta
    path = _big_fasta(str(tmp_path / "big.fa"), 11, [41000000, 30000000, 20000000, 9000000, 777])
    # interrupted tracts over the random sequence: one every 20 kb
    rng = np.random.default_rng(12)
    fa = Fasta(path)
    with open(path, "r+b") as fp:
        for name, (L, off, lb, lw) in fa.index.items():
            for _ in range(L // 20000):
                t = _interrupted(rng, 3).encode()
                a = int(rng.integers(0, L - len(t)))
                for i, b in enumerate(t):          # base by base: the tract may cross a line break
                    p = a + i
                    fp.seek(off + (p // lb) * lw + p % lb)
                    fp.write(bytes([b]))
    fa = Fasta(path)
    for g, pur in ((3, (9, 10)), (20, (3, 4))):
        dev = fa.tracts(MOTIFS, step_bytes=16 << 20, max_interrupt=g, purity=pur)
        emu = fa.tracts(MOTIFS, step_bytes=16 << 20, max_interrupt=g, purity=pur, emulate=True)
        assert np.array_equal(dev["tracts"], emu["tracts"]) and np.array_equal(dev["segments"], emu["segments"])
        assert dev["stats"]["tracts"] > 4000 and int((dev["segments"] > 1).sum()) > 1000
        assert dev["stats"]["steps"] == 4 and dev["stats"]["bases"] == 100000777


# ---------------------------------------------------------------------------------------------------------------
# on the GPU: an interrupted discovered site, in-repeat reads mismapped onto interrupted decoys
# ---------------------------------------------------------------------------------------------------------------
# the site: 12 copies of GGGAA with one substitution (pure pieces of 30 and 29 bases); the decoys: interrupted tracts
# whose pure pieces are all shorter than 30 bases, so the pure rule lists none of them
SITE = ("c1", 12000, "GGGAA", 12, [(6, "sub", "C")])
DECOYS = [("c3", 2000, "GGGAA", 30, [(c, "sub", "C") for c in (5, 10, 15, 20, 25)]),
          ("c3", 6000, "TTCCC", 20, [(c, "sub", "A") for c in (5, 10, 15)])]
REFS = [("c1", 24000), ("c2", 18000), ("c3", 14000)]
NORMAL = {0: (8, 12), 1: (10, 10), 2: (6, 11)}
EXPANDED, EXP_UNITS, MISMAP = 3, 200, 0.7


def _cohort(d):
    from tredparse_b200 import bamio, simulate
    from tredparse_b200.meta import TREDsRepo
    contigs = simulate.planted_reference(REFS, [SITE] + DECOYS, seed=23)
    simulate.write_fasta(str(d / "ref.fa"), contigs, width=70)
    hd = TREDsRepo()["HD"]
    refs = REFS + [("chr4", hd.repeat_end + 20000)]
    c, pos, u, n, _ = SITE
    end = pos + len(simulate.interrupted_tract(u, n, SITE[4]))
    decoys = [(2, p, p + len(simulate.interrupted_tract(du, dn, de))) for _, p, du, dn, de in DECOYS]
    bams = []
    for s in range(4):
        al = (NORMAL[0][0], EXP_UNITS) if s == EXPANDED else NORMAL[s]
        recs = simulate.reference_records(contigs[c], 0, pos, end, u, al, cov_per_hap=15, flank=1500, seed=100 * s,
                                          tag="s{}x0".format(s), mismap_fraction=MISMAP if s == EXPANDED else 0.0,
                                          mismap_to=decoys)
        recs += simulate.locus_records(hd, 2, (17, 20), 150, 10.0, seed=40 + s, tag="s{}hd".format(s), flank=1000)
        path = str(d / "s{}.bam".format(s))
        bamio.write_bam(path, refs, simulate.coordinate_sort(recs), index=s in (0, 3), aux=True)
        bams.append(path)
    return bams


@pytest.mark.gpu
def test_gpu_interrupted_alt_regions_rescue_mismapped_in_repeat_reads(tmp_path, monkeypatch, capsys):
    from tredparse_b200 import strprofile
    assert _canon("TTCCC") == _canon("GGGAA")
    bams = _cohort(tmp_path)
    work = tmp_path / "w"
    assert strprofile.main(["profile", *bams, "--workdir", str(work)]) == 0
    profs = [str(work / "s{}.str_profile.json".format(s)) for s in range(4)]
    assert strprofile.main(["outliers", *profs, "--tsv", str(tmp_path / "out.tsv")]) == 0
    run = tmp_path / "run"
    run.mkdir()
    monkeypatch.chdir(str(run))
    loci = ["loci", str(tmp_path / "out.tsv"), "--fasta", str(tmp_path / "ref.fa"), "--profiles", *profs, "--alts"]
    # the pure rule: the locus is the longer pure piece, and no decoy is an alt region
    capsys.readouterr()
    assert strprofile.main(loci + ["--out", "pure.json"]) == 0
    with open("pure.json") as fp:
        pure = json.load(fp)
    assert list(pure) == ["c1_12001_GGGAA"] and pure["c1_12001_GGGAA"]["repeat_location"] == "c1:12001-12030"
    assert pure["c1_12001_GGGAA"]["alts"] == ""
    assert strprofile.main(loci + ["--max-interruption", "1"]) == 0
    out = capsys.readouterr()
    name = "c1_12001_GGGAA"
    assert out.out.split()[-1] == name
    with open("sites/discovered.json") as fp:
        sites = json.load(fp)
    assert list(sites) == [name]
    row = sites[name]
    assert row["repeat_location"] == "c1:12001-12060"                     # the whole planted tract
    assert row["prefix"][-1] != "A" and row["suffix"][0] != "G"
    assert row["alts"] == "c3:2000-2150|c3:6000-6100"                    # the decoys, not the locus' own tract
    assert "{}: 2 alt regions".format(name) in out.err.splitlines()
    csv = tmp_path / "samples.csv"
    csv.write_text("".join("s{},{}\n".format(s, b) for s, b in enumerate(bams)))
    calls = _calls(csv, tmp_path / "calls", [name, "HD"])
    noalts = _calls(csv, tmp_path / "calls_noalts", [name, "HD"], "--noalts")
    from tredparse_b200 import meta
    repo = meta.TREDsRepo()
    from tredparse_b200 import ingest
    with ingest.BamIngest(bams[EXPANDED]) as ing:
        ev = ing.extract_locus(repo[name], 150, alts=repo[name].alt, want_names=True)
    assert ev.nreads > len(ing_noalts(bams[EXPANDED], repo[name]).names)
    cut = row["cutoff_risk"]
    for s in range(4):
        c, c0 = calls[s], noalts[s]
        if s == EXPANDED:
            assert c[name + ".RDP"] > c0[name + ".RDP"], (c, c0)
            assert c[name + ".2"] >= c0[name + ".2"] and c[name + ".2"] >= cut and c[name + ".label"] == "risk"
        else:
            assert {k: v for k, v in c.items() if k.startswith(name)} == \
                   {k: v for k, v in c0.items() if k.startswith(name)}
            assert (c[name + ".1"], c[name + ".2"]) == NORMAL[s]
    bare = tmp_path / "bare"
    bare.mkdir()
    monkeypatch.chdir(str(bare))
    c0 = _calls(csv, tmp_path / "calls0", ["HD"])
    for s in range(4):
        assert {k: v for k, v in calls[s].items() if k.startswith("HD")} == \
               {k: v for k, v in c0[s].items() if k.startswith("HD")}
