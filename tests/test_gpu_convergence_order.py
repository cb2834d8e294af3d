"""The convergence order of the packed family kernel's reads, against the CPU oracle.

The pre-filter predicts from a read's q-grams in the pure repeat how many main strips it needs before its boundary
column reaches its fixed point; the grouping kernels then order every (family, strand class) group by that prediction,
so that the reads of an item stop at about the same strip.  The order only decides which reads share an item: every
record must equal the oracle's in every combination of the order, the strip exit and strand pairing, and the fused
call must not change.  The per-lane counters of the context (lane_planned, lane_skippable) bound what any order can
skip.  Needs a GPU: run with -m gpu."""
import numpy as np
import pytest

from test_gpu_read_lengths import LENS, _Fam, _catalogue_set, _pool
from test_gpu_strand_pairing import _batch, _families, _oracle, _recs
from test_gpu_strip_skip import _delta, _skip_stats

pytestmark = pytest.mark.gpu

SWITCHES = ("TREDSW_NO_CONVERGENCE_ORDER", "TREDSW_NO_STRIP_SKIP", "TREDSW_NO_STRAND_PAIRING")


def _set_modes(monkeypatch, order=True, skip=True, pairing=True):
    for var, on in zip(SWITCHES, (order, skip, pairing)):
        if on:
            monkeypatch.delenv(var, raising=False)
        else:
            monkeypatch.setenv(var, "1")


def _classify(reads, rfam, recs, monkeypatch, **modes):
    from tredparse_b200 import ssw
    _set_modes(monkeypatch, **modes)
    s0 = _skip_stats()
    out = ssw.classify_reads(reads, rfam, recs)
    d = _delta(s0, _skip_stats())
    _set_modes(monkeypatch)
    return out, d


def _all_modes(reads, rfam, recs, expected, monkeypatch):
    """Records of the order on / off x strip exit on / off x pairing on / off: each equal to the oracle's and, byte for
    byte, to each other's.  Returns the strip counters per mode."""
    outs, stats = {}, {}
    for order in (True, False):
        for skip in (True, False):
            for pairing in (True, False):
                mode = (order, skip, pairing)
                out, d = _classify(reads, rfam, recs, monkeypatch, order=order, skip=skip, pairing=pairing)
                for r, e in enumerate(expected):
                    assert tuple(int(x) for x in out[r]) == tuple(e), (mode, r, len(reads[r]), e, out[r])
                outs[mode], stats[mode] = out.tobytes(), d
    assert len(set(outs.values())) == 1
    for d in stats.values():
        for v in d["by_period"].values():
            assert v["lane_skipped"] <= v["lane_skippable"] <= v["lane_planned"], d
    return stats


def test_catalogue_clip_and_outside_families_in_every_mode(monkeypatch):
    """Catalogue loci (periods 3, 5, 6 as sub-units of 3, 12; GCN / NGC motifs), a clip family and families outside
    the catalogue (periods 7 and 1), in a large ragged batch with groups of several items."""
    fams, clips = _families(151)
    reads = _batch(fams, 101, 11)
    with _pool() as ex:
        exp = list(ex.map(_oracle, fams, reads, clips))
    flat = [r for rs in reads for r in rs]
    rfam = np.concatenate([np.full(len(rs), i, np.int32) for i, rs in enumerate(reads)])
    stats = _all_modes(flat, rfam, _recs(fams, clips), [e for es in exp for e in es], monkeypatch)
    assert sum(v["skipped"] for v in stats[(True, True, True)]["by_period"].values()) > 0


def test_every_read_length_in_every_mode(monkeypatch):
    """75-255 bp reads of the catalogue loci."""
    lens, cap = LENS["packed"]
    s = _catalogue_set(lens, cap, 3)
    _all_modes(s.reads, s.rfam, np.concatenate([f.rec for f in s.fams]), s.expected, monkeypatch)


def _mixed_group():
    """128 reads of the pure repeat (their strips never converge) interleaved with 128 reads holding 5 repeat units
    between the flanks inside random sequence (they converge after a few strips), all on the forward strand of HD:
    in arrival order every 64-read item of the group holds both kinds."""
    from tredparse_b200.meta import TREDsRepo
    t = TREDsRepo()["HD"]
    fam = _Fam(t.prefix, t.repeat, t.suffix, 150)
    rng = np.random.default_rng(7)
    reads = []
    for k in range(128):
        reads.append((t.repeat * 60)[k % 3:][:150])
        core = t.prefix + t.repeat * 5 + t.suffix
        left = int(rng.integers(10, 150 - len(core) - 10))
        flank = "".join(rng.choice(list("ACGT"), 150 - len(core)))
        reads.append(flank[:left] + core + flank[left:])
    return fam, reads


def test_ordering_skips_more_in_a_mixed_group(monkeypatch):
    """The mixed group: with the order on, its converging reads share items and skip strips; in arrival order no item
    skips anything.  In both modes the skipped share stays within the per-lane bound.  (The bound itself depends on the
    order: a lane holds two single-strand reads and converges with the later of them.)"""
    fam, reads = _mixed_group()
    exp = _oracle(fam, reads, False)
    rfam = np.zeros(len(reads), np.int32)
    got = {}
    for order in (True, False):
        out, d = _classify(reads, rfam, fam.rec, monkeypatch, order=order)
        for r, e in enumerate(exp):
            assert tuple(int(x) for x in out[r]) == tuple(e), (order, r, e, out[r])
        got[order] = d["by_period"][3]
    on, off = got[True], got[False]
    assert on["skipped"] > off["skipped"], got
    for v in (on, off):
        # four full 64-read items (32 busy lanes each): every lane could skip at least what its warp skipped, so the
        # skipped share is at most the per-lane bound
        assert v["items"] == 4 and v["lane_planned"] == 32 * v["planned"], got
        assert v["lane_skipped"] == 32 * v["skipped"] and v["lane_skippable"] >= v["lane_skipped"], got


def test_lane_counter_of_a_one_read_item(monkeypatch):
    """One read alone in its item: the lane's own skippable strips are the strips its warp skipped."""
    fam, reads = _mixed_group()
    read = [reads[1]]
    exp = _oracle(fam, read, False)
    out, d = _classify(read, np.zeros(1, np.int32), fam.rec, monkeypatch)
    assert tuple(int(x) for x in out[0]) == tuple(exp[0])
    v = d["by_period"][3]
    assert v["items"] == 1 and v["skipped"] > 0, d
    assert v["lane_planned"] == v["planned"] and v["lane_skipped"] == v["lane_skippable"] == v["skipped"], d


def test_fused_call_identical_with_and_without_the_order(monkeypatch):
    """tredsw_genotype_batch on every catalogue locus of a seeded cohort batch: per-read records, calls (PP included),
    tallies and posteriors are identical byte for byte with TREDSW_NO_CONVERGENCE_ORDER=1."""
    from tredparse_b200 import cohort, simulate
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    names = list(dict.fromkeys(repo.names))
    specs = simulate.cohort_specs(repo, names, 4, readlen=150, seed=20240000)
    problems = [simulate.simulate_from_spec(repo, s) for s in specs]
    res = {}
    for order in (True, False):
        _set_modes(monkeypatch, order=order)
        res[order] = cohort.CohortBatch(problems).run_host(want_reads=True, want_hist=True, want_stats=True,
                                                           want_post=True)
    _set_modes(monkeypatch)
    a, b = res[True], res[False]
    for k in ("reads", "calls", "hist"):
        assert a[k].tobytes() == b[k].tobytes(), k
    # (posterior entries come in no particular order; stats[1] and [2] depend on the single-strand pairs)
    order = ("problem", "kind", "a", "b", "p")
    assert np.sort(a["post"], order=order).tobytes() == np.sort(b["post"], order=order).tobytes()
    assert [a["stats"][i] for i in (0, 3, 4, 5)] == [b["stats"][i] for i in (0, 3, 4, 5)], (a["stats"], b["stats"])
