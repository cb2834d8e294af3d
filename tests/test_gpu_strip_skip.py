"""The fixed-point exit of the packed family kernel's main strips, against the CPU oracle.

Every main strip of phase 1 runs the same score table and suffix potentials, so a strip whose leaving boundary column
equals its entering one is repeated by every later strip; phase 1 stops there and fills the remaining units' scores,
and phase 2 reads the last written boundary slot for any later strip.  These tests hold every record field to the
oracle with the exit on, check that TREDSW_NO_STRIP_SKIP=1 gives the same records and the same executed-cell statistic
(stats[1] counts the full plan), that the skip counter of the context moves only with the exit on, and that the fused
genotyping call is unchanged byte for byte.  Needs a GPU: run with -m gpu."""
import numpy as np
import pytest

from test_gpu_read_lengths import LENS, _Fam, _Set, _catalogue_set, _pool
from test_gpu_strand_pairing import _batch, _families, _oracle, _phase1_cells, _recs, _strand_class

pytestmark = pytest.mark.gpu


def _skip_stats():
    from tredparse_b200 import _lib
    return _lib.default_context().strip_skip_stats()


def _delta(a, b):
    """Counters of the calls between two reads of the context's strip-skip statistics."""
    per = {p: {k: v - a["by_period"].get(p, {}).get(k, 0) for k, v in d.items()} for p, d in b["by_period"].items()}
    return {"cells_skipped": b["cells_skipped"] - a["cells_skipped"],
            "by_period": {p: d for p, d in per.items() if d["items"]}}


def _classify(reads, rfam, recs, monkeypatch, skip):
    """Records, stats and the strip-skip counters of one classify_reads call with the exit on or off."""
    from tredparse_b200 import ssw
    if skip:
        monkeypatch.delenv("TREDSW_NO_STRIP_SKIP", raising=False)
    else:
        monkeypatch.setenv("TREDSW_NO_STRIP_SKIP", "1")
    s0 = _skip_stats()
    out, stats = ssw.classify_reads(reads, rfam, recs, want_stats=True)
    d = _delta(s0, _skip_stats())
    monkeypatch.delenv("TREDSW_NO_STRIP_SKIP", raising=False)
    return out, stats, d


def _both_modes(reads, rfam, recs, expected, monkeypatch, deterministic=False):
    """Records of both modes == the oracle's and each other's.  The grouping kernels keep the order of the reads inside
    a (family, class) group only when the group's reads arrive in one 32-read window of the batch; otherwise the
    single-strand pairs, and with them stats[1] (per lane max(len a, len b)) and stats[2], vary from call to call.
    `deterministic`: the batch is laid out that way, so all four statistics must be equal."""
    got = {}
    for skip in (True, False):
        out, stats, d = _classify(reads, rfam, recs, monkeypatch, skip)
        for r, e in enumerate(expected):
            assert tuple(int(x) for x in out[r]) == tuple(e), (skip, r, len(reads[r]), e, out[r])
        got[skip] = (out, stats, d)
    assert got[True][0].tobytes() == got[False][0].tobytes()
    a, b = got[True][1], got[False][1]
    assert a[0] == b[0] and a[3] == b[3], (a, b)
    if deterministic:
        assert np.array_equal(a, b), (a, b)                     # stats[1]: the planned phase-1 cells in both modes
    off = got[False][2]
    assert off["cells_skipped"] == 0 and all(v["skipped"] == 0 for v in off["by_period"].values()), off
    return got[True][1], got[True][2]


def test_catalogue_clip_and_outside_families_with_ghost_partners(monkeypatch):
    """Catalogue loci (periods 3, 5, 6 as sub-units of 3, 12; GCN / NGC motifs), a clip family and families outside
    the catalogue (periods 7 and 1), in a large ragged batch whose single-strand groups leave ghost partners."""
    fams, clips = _families(151)
    reads = _batch(fams, 101, 11)
    with _pool() as ex:
        exp = list(ex.map(_oracle, fams, reads, clips))
    flat = [r for rs in reads for r in rs]
    rfam = np.concatenate([np.full(len(rs), i, np.int32) for i, rs in enumerate(reads)])
    _, d = _both_modes(flat, rfam, _recs(fams, clips), [e for es in exp for e in es], monkeypatch)
    assert d["cells_skipped"] > 0, d
    assert sum(v["skipped"] for v in d["by_period"].values()) > 0, d


def test_planned_phase1_cells_with_the_exit(monkeypatch):
    """32 reads per family in one grouping window each (deterministic pairs): stats[1] with the exit on equals the
    phase-1 cells of the full nested-strip plan predicted from the strand classes, and all statistics are equal in
    both modes, while strips were skipped."""
    fams, clips = _families(151)
    reads = _batch(fams, 32, 5)
    with _pool() as ex:
        exp = list(ex.map(_oracle, fams, reads, clips))
        cls = list(ex.map(lambda f, rs: [_strand_class(f, r) for r in rs], fams, reads))
    flat = [r for rs in reads for r in rs]
    rfam = np.concatenate([np.full(len(rs), i, np.int32) for i, rs in enumerate(reads)])
    stats, d = _both_modes(flat, rfam, _recs(fams, clips), [e for es in exp for e in es], monkeypatch,
                           deterministic=True)
    pred = sum(_phase1_cells(f, [len(r) for r in rs], cs) for f, rs, cs in zip(fams, reads, cls))
    assert stats[1] == pred, (stats, pred)
    assert 0 < d["cells_skipped"] < pred, d


def test_every_read_length_of_the_packed_kernel(monkeypatch):
    """75-255 bp reads of the catalogue loci (strip tails, odd last rows, families sized for long reads whose strips
    converge long before the plan ends)."""
    lens, cap = LENS["packed"]
    s = _catalogue_set(lens, cap, 3)
    _, d = _both_modes(s.reads, s.rfam, np.concatenate([f.rec for f in s.fams]), s.expected, monkeypatch)
    assert d["cells_skipped"] > 0, d


def test_reads_that_never_converge(monkeypatch):
    """Reads made of the repeat alone (a long expanded allele): the boundary column keeps growing until the last
    strip, so no item skips anything — and the records still equal the oracle's."""
    from tredparse_b200.meta import TREDsRepo
    t = TREDsRepo()["HD"]
    fam = _Fam(t.prefix, t.repeat, t.suffix, 150)
    rng = np.random.default_rng(4)
    reads = []
    for k in range(96):
        rep = (t.repeat * 60)[k % 3:][:150]
        reads.append(rep if k % 2 else "".join({"A": "T", "C": "G", "G": "C", "T": "A"}[c] for c in reversed(rep)))
    reads = [reads[i] for i in rng.permutation(len(reads))]
    s = _Set([fam], [reads])
    _, d = _both_modes(s.reads, s.rfam, fam.rec, s.expected, monkeypatch)
    assert d["by_period"] and all(v["skipped"] == 0 and v["items_no_skip"] == v["items"] for v in d["by_period"].values()), d


def test_candidates_in_skipped_strips_read_the_last_slot(monkeypatch):
    """Phase 2 of candidates whose unit lies in a skipped strip.  A read of k repeat units followed by the first 5
    suffix bases scores its full length against every template with >= k units, ending in the suffix block; at a
    family sized for 255 bp reads (85 units, 22 strips) the strips of a 64-read item of such reads (k <= 41) converge
    after about 12 strips.  Without clipping none of those full-score candidates is tagged (u * 3 > m rules out REPT),
    so phase 2 locates every one of them, those past the fixed point from the aliased slot, and the read ends HANG at
    u = k - 3 (k >= 12); with clipping it is REPT at u = k + 1 after its k-unit candidate is rejected.  (A candidate
    in a skipped strip never wins outright: the same unit of the last computed strip has the same score and fewer
    units, and is tried first.)"""
    from tredparse_b200 import ssw
    from tredparse_b200.meta import TREDsRepo
    t = TREDsRepo()["HD"]
    fam = _Fam(t.prefix, t.repeat, t.suffix, 255)
    assert fam.U == 85
    ks = list(range(10, 42)) * 2
    reads = [t.repeat * k + t.suffix[:5] for k in ks]
    clip = ssw.make_family(t.prefix, t.repeat, t.suffix, fam.U, clip=True)
    for rec, clipped in ((fam.rec, False), (clip, True)):
        exp = _oracle(fam, reads, clipped)
        if clipped:
            assert all(e[0] == 4 and e[1] == k + 1 for e, k in zip(exp, ks)), exp
        else:
            assert all(e[0] == 5 and e[1] == k - 3 for e, k in zip(exp, ks) if k >= 12), exp
        _, d = _both_modes(reads, np.zeros(len(reads), np.int32), rec, exp, monkeypatch)
        assert d["by_period"][3]["skipped"] > 0 and d["cells_skipped"] > 0, d


def test_fused_call_identical_with_and_without_the_exit(monkeypatch):
    """tredsw_genotype_batch on every catalogue locus of a seeded cohort batch: per-read records, calls (PP included),
    tallies and posteriors are identical byte for byte with TREDSW_NO_STRIP_SKIP=1, and strips were skipped."""
    from tredparse_b200 import cohort, simulate
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    names = list(dict.fromkeys(repo.names))
    specs = simulate.cohort_specs(repo, names, 4, readlen=150, seed=20240000)
    problems = [simulate.simulate_from_spec(repo, s) for s in specs]
    res, skipped = {}, {}
    for skip in (True, False):
        if skip:
            monkeypatch.delenv("TREDSW_NO_STRIP_SKIP", raising=False)
        else:
            monkeypatch.setenv("TREDSW_NO_STRIP_SKIP", "1")
        s0 = _skip_stats()
        res[skip] = cohort.CohortBatch(problems).run_host(want_reads=True, want_hist=True, want_stats=True, want_post=True)
        skipped[skip] = _delta(s0, _skip_stats())["cells_skipped"]
    monkeypatch.delenv("TREDSW_NO_STRIP_SKIP", raising=False)
    a, b = res[True], res[False]
    for k in ("reads", "calls", "hist"):
        assert a[k].tobytes() == b[k].tobytes(), k
    # (the posterior entries come in no particular order; stats[1] and [2] depend on the single-strand pairs, which
    #  vary from call to call in a batch of this size — the algorithmic cells, alignments and grid points do not)
    order = ("problem", "kind", "a", "b", "p")
    assert np.sort(a["post"], order=order).tobytes() == np.sort(b["post"], order=order).tobytes()
    assert [a["stats"][i] for i in (0, 3, 4, 5)] == [b["stats"][i] for i in (0, 3, 4, 5)], (a["stats"], b["stats"])
    assert skipped[True] > 0 and skipped[False] == 0, skipped
