"""The genotyping kernels at read lengths other than 150 / 250 bp, against the CPU oracle.

The read length decides which code runs: the number of nested strips of the packed family kernel and where its last
partial strip ends (max_units = ceil(READLEN / period)), odd query rows, the batch-wide choice between the packed and
the generic kernel (max_read_len * match < 256), the > 48 KB shared-memory attribute path (static + dynamic bytes:
reads of about 300 bp or more),
and the L-dependent boundaries of the likelihood grid.  Real cohorts have 100/101, 125/126, 151, 250/251 and 300 bp
reads plus adapter-trimmed reads of any shorter length.  Needs a GPU: run with -m gpu."""
import itertools
import json
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from oracle import sw as osw

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
TAGC = {"FULL": 1, "PREF": 2, "POST": 3, "REPT": 4, "HANG": 5}
NO_TAG = (0, 0, -1, -1, -1, -1, -1, -1)        # the record of a read without a tag
B = "ACGT"


def _pool():
    return ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1))      # (ctypes releases the GIL)


# ---------------------------------------------------------------------------------------------------------
# 1. the family kernel (ssw.classify_reads), read by read
# ---------------------------------------------------------------------------------------------------------
class _Fam:
    """A template family and what the oracle and the q-gram pre-filter know about it."""

    def __init__(self, prefix, repeat, suffix, readlen):
        from tredparse_b200 import ssw
        from oracle import evidence_oracle as evo
        self.prefix, self.repeat, self.suffix, self.readlen = prefix, repeat, suffix, readlen
        self.P = len(repeat)
        self.U = -(-readlen // self.P)
        self.rec = ssw.make_family(prefix, repeat, suffix, self.U)
        self.tseqs = [x for _, x in evo.template_family(prefix, repeat, suffix, self.U)]
        self.sum_n = sum(len(x) for x in self.tseqs)
        self.grams = None

    def kept_by_prefilter(self, read, q=6):
        """The exact q-gram pre-filter of sw_family.cu (scoring 1/5/7/2: q = 6, 30 - (q-1)(#N+1) shared q-grams of
        either strand needed): a read it drops never reaches the Smith-Waterman kernel."""
        from oracle import evidence_oracle as evo
        if self.grams is None:
            fwd = set()
            u0 = (q - 1 + self.P - 1) // self.P + 1
            for u in range(1, min(self.U, u0 + 1) + 1):
                t = self.prefix + self.repeat * u + self.suffix
                for i in range(len(t) - q + 1):
                    g = t[i:i + q]
                    assert g.count("N") <= 4
                    for fill in itertools.product(B, repeat=g.count("N")):
                        it = iter(fill)
                        fwd.add("".join(next(it) if c == "N" else c for c in g))
            self.grams = (fwd, {evo.rc(g) for g in fwd})
        fwd, rev = self.grams
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
        return hf >= thr or hr >= thr


def _oracle_records(fam, reads):
    """Expected record of every read: (tag, units, score, rb, re, qb, qe, rank) of the arg-max over the family's
    templates in the reference's order — highest score, then fewest units, then the forward strand."""
    from oracle import evidence_oracle as evo
    k = len(fam.tseqs)
    al = osw.oracle_align_pairs(reads, fam.tseqs, np.repeat(np.arange(len(reads), dtype=np.int32), k),
                                np.tile(np.arange(k, dtype=np.int32), len(reads))).reshape(len(reads), k, -1)
    out = []
    for r, read in enumerate(reads):
        best = None
        for rank in range(k):
            row = [int(x) for x in al[r, rank, :5]]
            u = rank // 2 + 1
            tag = evo.classify_alignment(*row, len(read), len(fam.tseqs[rank]), u, fam.P, fam.U)
            if tag and (best is None or (row[0], -u) > (best[2], -best[1])):
                best = (TAGC[tag], u, *row, rank)
        out.append(NO_TAG if best is None else best)
    return out


def _reads(fam, rng, n, cap):
    """n reads of READLEN around the family's repeat on two haplotypes — one whose repeat fits well inside a read,
    one longer than a read — so that FULL, PREF, POST, REPT, HANG and untagged reads all occur; 1 % substitutions,
    either strand.  About half are trimmed from the 3' end to any length in [1, READLEN] (some below 30 bp), a few
    are 1-10 bases longer than READLEN (at most `cap`), and the order is shuffled so that trimmed and full-length
    reads share warps."""
    from oracle import evidence_oracle as evo
    L, P = fam.readlen, fam.P
    h_short, h_long = max(1, (L - 50) // (2 * P)), fam.U + 8
    reads = []
    for k in range(n):
        mode = k % 4
        h = h_short if mode < 2 else h_long
        motif = fam.repeat.replace("N", B[rng.integers(0, 4)])
        pad = L + 40
        hap = "".join(rng.choice(list(B), pad)) + fam.prefix + motif * h + fam.suffix + "".join(rng.choice(list(B), pad))
        rs = pad + len(fam.prefix)
        re_ = rs + P * h
        if mode == 0:                       # anywhere: mostly flanking sequence
            st = rng.integers(0, len(hap) - L - 10)
        elif mode == 2:                     # inside the long repeat
            st = rng.integers(rs, re_ - L + 1)
        else:                               # overlapping one end of the repeat
            st = rng.integers(rs - L + 10, re_ - 10)
        ext = int(rng.integers(1, 11)) if k % 16 == 5 else 0
        ln = min(L + ext, cap) if k % 2 == 0 or ext else int(rng.integers(1, L + 1))
        read = list(hap[st:st + ln])
        for i in range(len(read)):
            if rng.random() < 0.01:
                read[i] = B[rng.integers(0, 4)]
        read = "".join(read)
        reads.append(evo.rc(read) if rng.random() < 0.5 else read)
    return [reads[i] for i in rng.permutation(n)]


LOCI = ("HD", "DM2", "SCA10", "SCA36", "ULD", "OPMD", "BPES")      # periods 3, 4, 5, 6 (as sub-units of 3), 12; GCN, NGC
LENS = {"packed": ((75, 100, 101, 125, 126, 149, 151, 199, 251, 255), 255),
        "generic": ((256, 300), 304),       # up to 304 bp the dynamic shared memory stays below 48 KB, static + dynamic not
        "smem48k": ((320,), 330)}
NREADS = 64


class _Set:
    """Reads of several families in one classify_reads call, with their oracle records."""

    def __init__(self, fams, reads_per_fam):
        self.fams = fams
        self.reads = [r for rs in reads_per_fam for r in rs]
        self.rfam = np.concatenate([np.full(len(rs), i, np.int32) for i, rs in enumerate(reads_per_fam)])
        with _pool() as ex:
            exp = list(ex.map(_oracle_records, fams, reads_per_fam))
            kept = list(ex.map(lambda f, rs: [f.kept_by_prefilter(r) for r in rs], fams, reads_per_fam))
        self.expected = [e for es in exp for e in es]
        self.kept = np.array([k for ks in kept for k in ks])
        self.alg = np.array([len(r) * fams[f].sum_n for r, f in zip(self.reads, self.rfam)], dtype=np.int64)

    def merged(self, other):
        m = _Set.__new__(_Set)
        m.fams, m.reads = self.fams + other.fams, self.reads + other.reads
        m.rfam = np.concatenate([self.rfam, other.rfam + len(self.fams)]).astype(np.int32)
        m.expected, m.kept = self.expected + other.expected, np.concatenate([self.kept, other.kept])
        m.alg = np.concatenate([self.alg, other.alg])
        return m

    def classify(self, kernel):
        """The kernel's records; `kernel` ("packed" / "generic") is checked through the cell counters."""
        from tredparse_b200 import ssw
        out, stats = ssw.classify_reads(self.reads, self.rfam, np.concatenate([f.rec for f in self.fams]),
                                        want_stats=True)
        assert stats[0] == self.alg.sum() and stats[3] == sum(2 * self.fams[f].U for f in self.rfam)
        kept_cells = int(self.alg[self.kept].sum())
        # the generic phase 1 sweeps all m x n cells of every template of every read the pre-filter keeps; the
        # nested packed pass (plus its end-point search) executes far fewer
        if kernel == "generic":
            assert stats[1] == kept_cells, (stats, kept_cells)
        else:
            assert 0 < stats[1] < kept_cells, (stats, kept_cells)
        return out

    def check(self, out):
        for r in range(len(self.reads)):
            assert tuple(int(x) for x in out[r]) == tuple(self.expected[r]), (r, len(self.reads[r]), self.expected[r], out[r])


def _catalogue_set(lengths, cap, seed):
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    rng = np.random.default_rng(seed)
    fams, reads = [], []
    for L in lengths:
        for name in LOCI:
            t = repo[name]
            fams.append(_Fam(t.prefix, t.repeat, t.suffix, L))
            reads.append(_reads(fams[-1], rng, NREADS, cap))
    return _Set(fams, reads)


@pytest.fixture(scope="module")
def catalogue_sets():
    return {k: _catalogue_set(lens, cap, seed) for seed, (k, (lens, cap)) in enumerate(LENS.items())}


@pytest.mark.parametrize("kernel", list(LENS))
def test_family_kernel_vs_oracle_at_every_read_length(catalogue_sets, kernel):
    """tag, units, score, coordinates and template rank of every read == the oracle's arg-max, at lengths whose strip
    tails, odd last rows and kernel choice differ; ragged (trimmed / over-long) reads share warps with full ones."""
    s = catalogue_sets[kernel]
    s.check(s.classify("generic" if kernel != "packed" else "packed"))
    lens = LENS[kernel][0]
    per_len = len(LOCI) * NREADS
    for i, L in enumerate(lens):
        tags = {s.expected[r][0] for r in range(i * per_len, (i + 1) * per_len)}
        assert tags >= {0, 1, 2, 3, 4}, (L, tags)      # untagged, FULL, PREF, POST, REPT
        ln = [len(s.reads[r]) for r in range(i * per_len, (i + 1) * per_len)]
        assert min(ln) < 30 and len({x % 2 for x in ln}) == 2 and (max(ln) > L or L == LENS[kernel][1])


def test_one_long_read_switches_the_whole_batch_to_the_generic_kernel(catalogue_sets):
    """A batch whose longest read is 255 bp runs the packed kernel; the same batch plus one 256 bp read runs every
    family through the generic one (max_read_len * match >= 256) — with identical records for the shared reads."""
    s = catalogue_sets["packed"]
    assert max(len(r) for r in s.reads) == 255
    a = s.classify("packed")
    f = len(s.fams) - len(LOCI)                             # HD at 255 bp
    hd = next(r for r, g in zip(s.reads, s.rfam) if g == f and len(r) == 255)
    extra = _Set([s.fams[f]], [[hd + hd[-1]]])
    assert len(extra.reads[0]) == 256
    both = s.merged(extra)
    b = both.classify("generic")
    assert np.array_equal(a, b[:len(s.reads)])
    both.check(b)


def _random_family(rng, period, flank_p, flank_s, readlen):
    rnd = lambda n: "".join(rng.choice(list(B), n))
    motif = rnd(period)
    while period > 1 and len(set(motif)) == 1:
        motif = rnd(period)
    return _Fam(rnd(flank_p), motif, rnd(flank_s), readlen)


def test_families_outside_the_catalogue_in_one_batch_with_both_kernels(catalogue_sets):
    """Families made through the C ABI: periods 1, 2, 7-11 with 18 bp flanks (packed instantiations no catalogue
    locus uses; period 1 is a homopolymer, where many templates tie on score), periods 13 and 16 and flanks of 17 and
    20 bp (generic).  In one batch with catalogue families both kernels run in one call; every family's records equal
    those it gets alone, and the oracle's."""
    from tredparse_b200 import ssw
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    rng = np.random.default_rng(77)
    L = 151
    shapes = [(p, 18, 18, "packed") for p in (1, 2, 7, 8, 9, 10, 11)] + \
             [(13, 18, 18, "generic"), (16, 18, 18, "generic"), (4, 17, 18, "generic"), (3, 20, 20, "generic"),
              (5, 18, 17, "generic")]
    fams = [_random_family(rng, p, a, b, L) for p, a, b, _ in shapes]
    for name in ("HD", "ULD"):
        t = repo[name]
        fams.append(_Fam(t.prefix, t.repeat, t.suffix, L))
    kinds = [k for *_, k in shapes] + ["packed", "packed"]
    reads = [_reads(f, rng, 40, 255) for f in fams]
    whole = _Set(fams, reads)
    out = ssw.classify_reads(whole.reads, whole.rfam, np.concatenate([f.rec for f in fams]))
    whole.check(out)
    tags = {e[0] for e in whole.expected}
    assert tags >= {0, 1, 2, 3, 4}, tags
    for i, (f, rs, kind) in enumerate(zip(fams, reads, kinds)):
        alone = _Set([f], [rs])
        got = alone.classify(kind)
        assert np.array_equal(got, out[whole.rfam == i]), (i, kind)


# ---------------------------------------------------------------------------------------------------------
# 2. the fused genotyping call (CohortBatch.run_host), problem by problem
# ---------------------------------------------------------------------------------------------------------
CALL_LENS = (100, 101, 125, 151, 251, 300)


def _problems(L):
    """Per read length: both alleles shorter than the read; two expansions well beyond it (REPT reads, the paired-end
    model on, a surface of several hundred points); a haploid problem; an expansion without a paired-end model."""
    import copy
    from tredparse_b200 import simulate
    from tredparse_b200.meta import TREDsRepo
    repo = TREDsRepo()
    specs = [("HD", (L // 9, L // 5)), ("DM1", (13, (L + 90) // 3)), ("HD", (17, (L + 150) // 3)), ("FXS", (30,))]
    ps = [simulate.simulate_problem(repo[n], al, readlen=L, cov_per_hap=15 if i in (1, 2) else 10, seed=1000 * L + i)
          for i, (n, al) in enumerate(specs)]
    nope = copy.copy(ps[2])
    nope.target_lens = np.zeros(0, np.int32)
    return ps + [nope]


def _oracle_problem(pr, maxinsert):
    from test_gpu_cohort import _expected_reads, _models, _oracle_call
    step, w = _models()
    exp = _expected_reads(pr)
    lk, counts, rept = _oracle_call(pr, [(a, b) for a, b in exp if a not in (0, 5)], step, w, maxinsert=maxinsert)
    return exp, lk, counts, rept


def _check_calls(problems, out, expected):
    from tredparse_b200 import cohort
    post = cohort.posteriors(out["post"], len(problems))
    r0 = 0
    for i, (pr, (exp, lk, counts, rept)) in enumerate(zip(problems, expected)):
        what = (pr.tred.name, pr.readlen, pr.alleles, len(pr.target_lens))
        rows = out["reads"][r0:r0 + pr.nreads]
        r0 += pr.nreads
        assert [(int(a), int(b)) if a else (0, 0) for a, b in rows[:, :2]] == exp, what
        c = cohort.decode_call(out["calls"][i])
        for which, name in ((0, "FULL"), (1, "PREF")):
            assert {k: int(v) for k, v in enumerate(out["hist"][i, which]) if v} == counts[name], what
        assert (c["RDP"], c["FDP"], c["PDP"]) == (rept, sum(counts["FULL"].values()), sum(counts["PREF"].values())), what
        assert c["alleles"] == lk.alleles and c["CI"] == lk.CI and c["label"] == lk.label, (what, c, lk.alleles, lk.CI)
        assert abs(c["PP"] - lk.PP) <= 1e-9, what
        if lk.alleles[0] >= 0:
            assert abs(c["lik"] - lk.lik) <= 1e-9 * abs(lk.lik), what
            assert c["n_points"] == len(lk.surface) and c["run_pe"] == bool(lk.run_pe), what
            for name in ("P_h1", "P_h2", "P_h1h2"):
                want, got = getattr(lk, name), post[i][name]
                assert set(got) == set(want), (what, name, sorted(set(got) ^ set(want))[:6])
                for k, v in want.items():
                    assert abs(got[k] - v) <= 1e-9 * abs(v), (what, name, k, got[k], v)
    return post


@pytest.fixture(scope="module")
def call_sets():
    """{L: problems}, and the oracle of every problem at the default search range (maxinsert = 300) and a wider one
    (maxinsert = 400: at 251 / 300 bp the default range of an expansion with one spanned allele stays below 512
    points, the row kernels' threshold)."""
    problems = {L: _problems(L) for L in CALL_LENS}
    flat = [(L, mi, pr) for L in CALL_LENS for mi in (300, 400) for pr in problems[L]]
    with _pool() as ex:
        res = list(ex.map(lambda a: _oracle_problem(a[2], a[1]), flat))
    oracle = {}
    for (L, mi, _), r in zip(flat, res):
        oracle.setdefault((L, mi), []).append(r)
    return problems, oracle


@pytest.mark.parametrize("L", CALL_LENS)
def test_fused_call_vs_oracle_at_every_read_length(call_sets, L):
    """Per-read (tag, h), tallies, alleles, CI, label, PP, lik, surface size and the posteriors P_h1 / P_h2 / P_h1h2
    of every problem == the oracle's (the likelihood thresholds and the near / mid / far grid columns depend on L)."""
    from tredparse_b200 import cohort
    problems, oracle = call_sets
    points = []
    for mi in (300, 400):
        out = cohort.CohortBatch(problems[L], maxinsert=mi).run_host(want_reads=True, want_hist=True, want_stats=True,
                                                                    want_post=True)
        assert out["stats"][5] == 0
        _check_calls(problems[L], out, oracle[(L, mi)])
        points += [(lk.run_pe, rept, len(lk.surface)) for _, lk, _, rept in oracle[(L, mi)]]
    assert any(pe and rept and n > 512 for pe, rept, n in points), (L, points)


def test_one_batch_of_every_read_length_equals_the_batches_per_length(call_sets):
    """All lengths in one CohortBatch: families (locus, L), hist_units of the longest, max_read_len 300 — so every
    family runs through the generic Smith-Waterman kernel instead of the packed one.  Calls are byte-identical,
    per-read records and posteriors equal."""
    from tredparse_b200 import cohort
    problems, oracle = call_sets
    allp = [pr for L in CALL_LENS for pr in problems[L]]
    batch = cohort.CohortBatch(allp)
    assert batch.max_read_len == 300 and batch.hist_units == 100
    assert len(batch.families) == len({(pr.tred.name, pr.readlen) for pr in allp})
    both = batch.run_host(want_reads=True, want_hist=True, want_post=True)
    post = _check_calls(allp, both, [e for L in CALL_LENS for e in oracle[(L, 300)]])
    i0, r0 = 0, 0
    for L in CALL_LENS:
        ps = problems[L]
        one = cohort.CohortBatch(ps).run_host(want_reads=True, want_post=True)
        nr = sum(p.nreads for p in ps)
        assert both["calls"][i0:i0 + len(ps)].tobytes() == one["calls"].tobytes(), L
        assert np.array_equal(both["reads"][r0:r0 + nr], one["reads"]), L
        assert post[i0:i0 + len(ps)] == cohort.posteriors(one["post"], len(ps)), L
        i0, r0 = i0 + len(ps), r0 + nr


# ---------------------------------------------------------------------------------------------------------
# 3. from a BAM: GPU ingest, read-length pre-step and fused call at 101 and 251 bp
# ---------------------------------------------------------------------------------------------------------
def _close(a, b, path=""):
    if isinstance(b, dict):
        assert isinstance(a, dict) and set(a) == set(b), (path, sorted(set(a) ^ set(b))[:6])
        for k in b:
            _close(a[k], b[k], path + "/" + str(k))
    elif isinstance(b, list):
        assert len(a) == len(b), path
        for i, (x, y) in enumerate(zip(a, b)):
            _close(x, y, "{}[{}]".format(path, i))
    elif isinstance(b, float) or isinstance(a, float):
        assert abs(a - b) <= 1e-9 * max(abs(a), abs(b)) + 1e-15, (path, a, b)
    else:
        assert a == b, (path, a, b)


@pytest.mark.parametrize("L", (101, 251))
def test_tred_run_on_a_sample_bam_of_other_read_lengths_equals_the_oracle(tmp_path, L):
    """A simulated whole-sample BAM of L bp reads at 8 loci: tred.run infers readLen = L and its calls equal the CPU
    oracle's (evidence, PE summaries, call, CI, PP, label, posteriors), key by key."""
    from conftest import golden_module
    from tredparse_b200 import bamio, simulate, tred as T
    from tredparse_b200.meta import TREDsRepo
    g = golden_module("make_oracle_bam_fixture")
    repo = TREDsRepo()
    sam = bamio.AlignmentFile(os.path.join(GOLDEN, "t001.mini.bam"))
    refs = list(zip(sam.references, sam.lengths))
    sam.close()
    path = str(tmp_path / "s{}.bam".format(L))
    simulate.write_sample_bam(path, repo, g.NAMES, refs, g.SAMPLE, readlen=L, flank=g.FLANK)
    pre, calls = g.oracle_calls(path, repo)
    assert pre["readLen"] == L
    mine = json.loads(json.dumps(T.run(("s", path, repo, g.NAMES, 300, False, False, True, True, "INFO"))["tredCalls"]))
    for k, v in json.loads(json.dumps(pre)).items():
        _close(mine[k], v, k)
    for n in g.NAMES:
        for k, v in json.loads(json.dumps(calls[n])).items():
            _close(mine[n + "." + k], v, n + "." + k)
    assert any(mine[n + ".1"] > 0 for n in g.NAMES)
