"""Strand pairing in the packed family kernel, against the CPU oracle.

The q-gram pre-filter sorts every read that reaches the Smith-Waterman kernel into a strand class: templates of both
strands may reach the score threshold, or only forward or only reverse-complement ones.  The packed kernel runs two
single-strand reads per lane (read a in the low s16x2 half, read b in the high one).  These tests hold every record
field to the oracle across the classes, ghost partners, pairs of unequal length, N bases, N-motif families, the
sub-unit path, clip families and families outside the catalogue; predict the executed phase-1 cells (stats[1]) from a
restatement of the class split, so that they fail if pairing silently does not happen; and check that
TREDSW_NO_STRAND_PAIRING=1 gives the same records byte for byte.  Needs a GPU: run with -m gpu."""
import math

import numpy as np
import pytest

from test_gpu_read_lengths import B, TAGC, NO_TAG, _Fam, _pool, _random_family, _reads

pytestmark = pytest.mark.gpu

FLANK = 18
BOTH, FWD, RC = 0, 1, 2


def _strand_class(fam, read, q=6):
    """The pre-filter's class of a read (sw_family.cu, prefilter_kernel): None when no strand reaches
    30 - (q-1)(#N+1) shared q-grams, else BOTH / FWD / RC by which strands reach it."""
    fam.kept_by_prefilter(read, q)              # builds fam.grams
    fwd, rev = fam.grams
    hf = hr = run = 0
    for i, c in enumerate(read):
        if c not in B:
            run = 0
            continue
        run += 1
        if run >= q:
            g = read[i - q + 1:i + 1]
            hf += g in fwd
            hr += g in rev
    thr = 30 - (q - 1) * (sum(c not in B for c in read) + 1)
    if hf < thr and hr < thr:
        return None
    if hf >= thr and hr >= thr:
        return BOTH
    return FWD if hf >= thr else RC


def _oracle(fam, reads, clip):
    """Records of the oracle's arg-max (as test_gpu_read_lengths._oracle_records), with clip's max_units_eff."""
    from oracle import evidence_oracle as evo
    from oracle import sw as osw
    k = len(fam.tseqs)
    al = osw.oracle_align_pairs(reads, fam.tseqs, np.repeat(np.arange(len(reads), dtype=np.int32), k),
                                np.tile(np.arange(k, dtype=np.int32), len(reads))).reshape(len(reads), k, -1)
    out = []
    for r, read in enumerate(reads):
        best = None
        ueff = math.ceil(len(read) / fam.P) if clip else fam.U
        for rank in range(k):
            row = [int(x) for x in al[r, rank, :5]]
            u = rank // 2 + 1
            tag = evo.classify_alignment(*row, len(read), len(fam.tseqs[rank]), u, fam.P, ueff)
            if tag and (best is None or (row[0], -u) > (best[2], -best[1])):
                best = (TAGC[tag], u, *row, rank)
        out.append(NO_TAG if best is None else best)
    return out


def _phase1_cells(fam, lens, classes):
    """stats[1] of one family's reads, given in read order within one 32-read window (the grouping kernels then keep
    that order inside each class): per lane max(len a, len b) x 2 halves x the columns of the nested strips."""
    pi = 3 if fam.P == 6 else fam.P                   # instance_period
    g, k = fam.P // pi, (1 if pi >= 12 else 12 // pi)  # sub-units per unit, units per strip (strip_units)
    cols = 2 * FLANK + (-(-fam.U * g // k)) * pi * k
    total = 0
    for c in (BOTH, FWD, RC):
        ls = [n for n, x in zip(lens, classes) if x == c]
        if c == BOTH:
            total += sum(ls) * 2 * cols
        else:
            total += sum(max(ls[i:i + 2]) for i in range(0, len(ls), 2)) * 2 * cols
    return total


def _with_n(read, rng):
    """1-3 bases replaced by N (lowers the pre-filter threshold by q-1 per N)."""
    s = list(read)
    for i in rng.choice(len(s), size=min(len(s), int(rng.integers(1, 4))), replace=False):
        s[i] = "N"
    return "".join(s)


def _families(L):
    """Catalogue loci (periods 3, 5, 6 = 2 sub-units of 3, 12; GCN and NGC motifs), a clip family, and families
    outside the catalogue (periods 7 and 1)."""
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    rng = np.random.default_rng(2024)
    fams, clips = [], []
    for name in ("HD", "SCA10", "SCA36", "ULD", "OPMD", "BPES"):
        t = repo[name]
        fams.append(_Fam(t.prefix, t.repeat, t.suffix, L))
        clips.append(False)
    t = repo["DM1"]
    fams.append(_Fam(t.prefix, t.repeat, t.suffix, L))
    clips.append(True)
    for p in (7, 1):
        fams.append(_random_family(rng, p, FLANK, FLANK, L))
        clips.append(False)
    return fams, clips


def _recs(fams, clips):
    from tredparse_b200 import ssw
    return np.concatenate([ssw.make_family(f.prefix, f.repeat, f.suffix, f.U, clip=c) for f, c in zip(fams, clips)])


def _batch(fams, n_per_fam, seed):
    """n_per_fam reads per family (ragged lengths incl. < 30 bp, a few up to 10 bp longer than the family's read
    length, both strands, some with N bases), in family order."""
    rng = np.random.default_rng(seed)
    reads = []
    for f in fams:
        rs = _reads(f, rng, n_per_fam, f.readlen + 10)
        reads.append([_with_n(r, rng) if i % 7 == 3 and len(r) > 10 else r for i, r in enumerate(rs)])
    return reads


@pytest.fixture(scope="module")
def window_batch():
    """32 reads per family, family f in reads [32 f, 32 f + 32): one warp of the grouping kernels per family, so the
    order of the reads inside each (family, class) group and the pairs it forms are deterministic."""
    L = 151
    fams, clips = _families(L)
    reads = _batch(fams, 32, 5)
    with _pool() as ex:
        exp = list(ex.map(_oracle, fams, reads, clips))
        cls = list(ex.map(lambda f, rs: [_strand_class(f, r) for r in rs], fams, reads))
    return fams, clips, reads, exp, cls


def _classify(fams, clips, reads, monkeypatch, pairing):
    from tredparse_b200 import ssw
    if pairing:
        monkeypatch.delenv("TREDSW_NO_STRAND_PAIRING", raising=False)
    else:
        monkeypatch.setenv("TREDSW_NO_STRAND_PAIRING", "1")
    flat = [r for rs in reads for r in rs]
    rfam = np.concatenate([np.full(len(rs), i, np.int32) for i, rs in enumerate(reads)])
    out, stats = ssw.classify_reads(flat, rfam, _recs(fams, clips), want_stats=True)
    monkeypatch.delenv("TREDSW_NO_STRAND_PAIRING", raising=False)
    return out, stats


def test_records_and_phase1_cells_with_and_without_pairing(window_batch, monkeypatch):
    """Every record equals the oracle's in both modes; stats[1] equals the phase-1 cells predicted from the class
    split (64-read items of single-strand reads, 32-read items of the others), and pairing executes fewer of them."""
    fams, clips, reads, exp, cls = window_batch
    flat_cls = [c for cs in cls for c in cs]
    kept = [c for c in flat_cls if c is not None]
    # the batch covers every class, with odd counts (ghost partners) in some single-strand groups
    assert {BOTH, FWD, RC} <= set(kept), set(kept)
    assert any(sum(1 for c in cs if c == k) % 2 for cs in cls for k in (FWD, RC))
    # pairs of unequal length, and short reads among the single-strand ones
    ss_lens = [len(r) for rs, cs in zip(reads, cls) for r, c in zip(rs, cs) if c in (FWD, RC)]
    assert min(ss_lens) < 60 and max(ss_lens) >= 151
    pred_pair = pred_both = 0
    for f, rs, cs in zip(fams, reads, cls):
        lens = [len(r) for r in rs]
        pred_pair += _phase1_cells(f, lens, cs)
        pred_both += _phase1_cells(f, lens, [BOTH if c is not None else None for c in cs])
    assert pred_pair < pred_both
    expected = [e for es in exp for e in es]
    got = {}
    for pairing in (True, False):
        out, stats = _classify(fams, clips, reads, monkeypatch, pairing)
        for r, e in enumerate(expected):
            assert tuple(int(x) for x in out[r]) == tuple(e), (pairing, r, flat_cls[r], e, out[r])
        assert stats[1] == (pred_pair if pairing else pred_both), (pairing, stats, pred_pair, pred_both)
        got[pairing] = (out, stats)
    assert np.array_equal(got[True][0], got[False][0])
    assert got[True][1][0] == got[False][1][0] and got[True][1][3] == got[False][1][3]


def test_n_motif_families_and_reads_with_n(window_batch):
    """N-motif loci get both-strand reads from the wildcard; reads with N bases occur in every class the batch has."""
    fams, clips, reads, exp, cls = window_batch
    n_motif = [i for i, f in enumerate(fams) if "N" in f.repeat]
    assert n_motif and any(c == BOTH for i in n_motif for c in cls[i])
    with_n = {c for rs, cs in zip(reads, cls) for r, c in zip(rs, cs) if "N" in r and c is not None}
    assert with_n & {FWD, RC}, with_n


def test_pairing_in_a_large_ragged_batch_vs_oracle(monkeypatch):
    """Many warps per group (the order inside a group, and so the pairs, then vary from run to run), unequal class
    counts, ragged reads; families sized for 100 bp reads in the same batch."""
    fams, clips = _families(151)
    f100, c100 = _families(100)
    fams, clips = fams + f100[:3], clips + c100[:3]
    reads = _batch(fams, 101, 9)
    with _pool() as ex:
        exp = list(ex.map(_oracle, fams, reads, clips))
    out, stats = _classify(fams, clips, reads, monkeypatch, True)
    expected = [e for es in exp for e in es]
    for r, e in enumerate(expected):
        assert tuple(int(x) for x in out[r]) == tuple(e), (r, e, out[r])
    out2, stats2 = _classify(fams, clips, reads, monkeypatch, False)
    assert np.array_equal(out, out2)
    assert stats[1] < stats2[1] and stats[0] == stats2[0]


def test_whole_cohort_batch_identical_without_pairing(monkeypatch):
    """The fused genotyping call on every catalogue locus of three samples: per-read records, calls and tallies are
    identical byte for byte with TREDSW_NO_STRAND_PAIRING=1, and the executed phase-1 cells drop with pairing."""
    from tredparse_b200 import cohort, simulate
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    names = list(dict.fromkeys(repo.names))
    specs = simulate.cohort_specs(repo, names, 3, readlen=150, seed=77)
    problems = [simulate.simulate_from_spec(repo, s) for s in specs]
    res = {}
    for pairing in (True, False):
        if pairing:
            monkeypatch.delenv("TREDSW_NO_STRAND_PAIRING", raising=False)
        else:
            monkeypatch.setenv("TREDSW_NO_STRAND_PAIRING", "1")
        res[pairing] = cohort.CohortBatch(problems).run_host(want_reads=True, want_hist=True, want_stats=True)
    monkeypatch.delenv("TREDSW_NO_STRAND_PAIRING", raising=False)
    a, b = res[True], res[False]
    assert a["reads"].tobytes() == b["reads"].tobytes()
    assert a["calls"].tobytes() == b["calls"].tobytes()
    assert a["hist"].tobytes() == b["hist"].tobytes()
    assert a["stats"][0] == b["stats"][0] and a["stats"][1] < b["stats"][1]
