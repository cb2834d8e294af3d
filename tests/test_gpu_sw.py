"""Parity of the CUDA Smith-Waterman paths (through the C ABI) against the reference's golden outputs
and the CPU oracle.  Needs a GPU: run with -m gpu."""
import os

import numpy as np
import pytest

from oracle import sw as osw

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
CASES = [("t001", "HD"), ("t002", "DM1")]
TAGC = {"FULL": 1, "PREF": 2, "POST": 3, "REPT": 4, "HANG": 5}


def _load(name):
    d = np.load(os.path.join(GOLDEN, name))
    reads, T = list(d["reads"]), list(d["templates"])
    nq, nt = len(reads), len(T)
    qidx = np.repeat(np.arange(nq, dtype=np.int32), nt)
    tidx = np.tile(np.arange(nt, dtype=np.int32), nq)
    return d, reads, T, qidx, tidx


@pytest.mark.parametrize("sample,tred", CASES)
def test_pairs_kernel_bit_exact_on_reference_pairs(sample, tred):
    from tredparse_b200 import ssw
    d, reads, T, qidx, tidx = _load("sw_pairs_{}_{}.npz".format(sample, tred))
    out = ssw.align_pairs(reads, T, qidx, tidx, score2=True)
    gold = d["pairs"].reshape(-1, 7).astype(np.int32)
    assert np.array_equal(out[:, :7], gold)


def test_pairs_kernel_synthetic_and_cigar():
    from tredparse_b200 import ssw
    d = np.load(os.path.join(GOLDEN, "sw_pairs_synthetic.npz"))
    q, T = list(d["queries"]), list(d["templates"])
    idx = np.arange(len(q), dtype=np.int32)
    out, cig = ssw.align_pairs(q, T, idx, idx, score2=True, cigar_cap=128)
    assert np.array_equal(out[:, :7], d["pairs"])
    assert np.array_equal(out[:, 7], d["cigar_len"])
    L = d["cigar"].shape[1]
    for i in range(len(q)):
        n = int(d["cigar_len"][i])
        assert np.array_equal(cig[i, :n], d["cigar"][i, :n])


@pytest.mark.parametrize("sample,tred", CASES)
def test_pairs_kernel_cigar_on_reference_pairs(sample, tred):
    from tredparse_b200 import ssw
    d, reads, T, qidx, tidx = _load("sw_pairs_{}_{}.npz".format(sample, tred))
    sel = np.arange(0, len(qidx), 7)            # every 7th pair keeps the traceback scratch small
    out, cig = ssw.align_pairs(reads, T, qidx[sel], tidx[sel], score2=True, cigar_cap=64)
    glen = d["cigar_len"].reshape(-1)[sel]
    gcig = d["cigar"].reshape(len(qidx), -1)[sel]
    assert np.array_equal(out[:, 7], glen)
    for i in range(len(sel)):
        assert np.array_equal(cig[i, :glen[i]], gcig[i, :glen[i]])


def test_pairs_kernel_random_vs_oracle_edge_cases():
    from tredparse_b200 import ssw
    rng = np.random.default_rng(11)
    q, t = [], []
    for _ in range(600):
        q.append("".join(rng.choice(list("ACGTN"), p=[.24, .24, .24, .24, .04], size=int(rng.integers(1, 300)))))
        t.append("".join(rng.choice(list("ACGTN"), p=[.24, .24, .24, .24, .04], size=int(rng.integers(1, 330)))))
    for i in range(0, 600, 2):
        L = max(1, min(len(q[i]), len(t[i])) // 2)
        t[i] = t[i][:3] + q[i][:L] + t[i][3:]
    q += ["NNNNNNNNNN", "A", "ACGT" * 100]
    t += ["ACGTACGTAC", "A", "ACGT" * 120]
    idx = np.arange(len(q), dtype=np.int32)
    a = ssw.align_pairs(q, t, idx, idx, score2=True)
    b = osw.oracle_align_pairs(q, t, idx, idx)
    assert np.array_equal(a[:, :7], b)
    # other scoring parameters (ssw_wrap defaults 2/2/3/1)
    a = ssw.align_pairs(q, t, idx, idx, match=2, mismatch=2, gap_open=3, gap_extend=1, score2=True)
    b = osw.oracle_align_pairs(q, t, idx, idx, match=2, mismatch=2, go=3, ge=1)
    assert np.array_equal(a[:, :7], b)


def _family_for(d, tred_row):
    from tredparse_b200 import ssw
    READLEN = int(d["READLEN"])
    period = int(d["period"])
    return ssw.make_family(tred_row.prefix, tred_row.repeat, tred_row.suffix, -(-READLEN // period))


@pytest.mark.parametrize("sample,tred", CASES)
def test_family_kernel_matches_reference_classification(sample, tred):
    """tag / h / score of every read == arg-max over the reference's own 100 alignments per read, and
    the coordinates reported for the winner == the reference's for that (read, template) pair."""
    from tredparse_b200 import ssw
    from tredparse_b200.meta import TREDsRepo
    d, reads, T, _, _ = _load("sw_pairs_{}_{}.npz".format(sample, tred))
    fam = _family_for(d, TREDsRepo()[tred])
    out, stats = ssw.classify_reads(reads, np.zeros(len(reads), dtype=np.int32), fam, want_stats=True)
    gold = d["best"]
    pairs = d["pairs"].astype(np.int32)
    for r in range(len(reads)):
        if gold[r, 0] == -1:
            assert out[r, 0] == 0, r
            continue
        assert (out[r, 2], out[r, 1], out[r, 0]) == tuple(int(x) for x in gold[r]), r
        rank = out[r, 7]
        assert tuple(out[r, 2:7]) == tuple(pairs[r, rank, :5]), r
    cells = sum(len(x) for x in reads) * sum(len(t) for t in T)
    assert stats[0] == cells and stats[3] == len(reads) * len(T)


def _expected_best(read, db, P, mu, **score_kw):
    from oracle import evidence_oracle as evo
    tseqs = [x for _, x in db]
    al = osw.oracle_align_pairs([read], tseqs, np.zeros(len(tseqs), np.int32),
                                np.arange(len(tseqs), dtype=np.int32), **score_kw)
    res = []
    for (u, tpl), row in zip(db, al):
        tag = evo.classify_alignment(*[int(x) for x in row[:5]], len(read), len(tpl), u, P, mu)
        if tag:
            res.append((int(row[0]), u, tag))
    return max(res, key=lambda x: (x[0], -x[1])) if res else None


def test_family_kernel_fast_and_generic_paths_vs_oracle_across_loci():
    """Simulated reads at loci of every catalogue period (3,4,5,6,12), with N in the motif, 101, 150,
    250 and 300 bp.  Default scoring goes through the packed fast path while every read of the call is
    shorter than 256 bp; a 300 bp read, or match=2 (scores exceed the 8-bit boundary column: 2*150 >= 256),
    forces the generic scalar phase 1 for the whole call.  Every variant must equal the oracle."""
    from tredparse_b200 import ssw
    from tredparse_b200.meta import TREDsRepo
    from oracle import evidence_oracle as evo
    repo = TREDsRepo()
    rng = np.random.default_rng(5)
    B = "ACGT"
    fams, reads, rfam, dbs = [], [], [], []
    for name in ("HD", "DM2", "SCA10", "SCA36", "ULD", "OPMD", "FXS", "FRDA"):
        t = repo[name]
        for readlen in (101, 150, 250, 300):
            P = len(t.repeat)
            mu = -(-readlen // P)
            fams.append(ssw.make_family(t.prefix, t.repeat, t.suffix, mu))
            fi = len(fams) - 1
            db = evo.template_family(t.prefix, t.repeat, t.suffix, mu)
            for _ in range(6):
                h = int(rng.integers(1, mu + 20))
                motif = t.repeat.replace("N", B[rng.integers(0, 4)])
                hap = "".join(rng.choice(list(B), 200)) + t.prefix + motif * h + t.suffix + "".join(rng.choice(list(B), 200))
                st = int(rng.integers(0, len(hap) - readlen))
                read = list(hap[st:st + readlen])
                for k in range(readlen):
                    if rng.random() < 0.01:
                        read[k] = B[rng.integers(0, 4)]
                read = "".join(read)
                if rng.random() < 0.5:
                    read = evo.rc(read)
                reads.append(read)
                rfam.append(fi)
                dbs.append((db, P, mu))
    fams = np.concatenate(fams)
    rfam = np.array(rfam, dtype=np.int32)
    short = [r for r in range(len(reads)) if len(reads[r]) < 256]        # a call of these runs the packed kernel
    for kw_gpu, kw_or in ((dict(), dict()),
                          (dict(match=2, mismatch=10, gap_open=14, gap_extend=4), dict(match=2, mismatch=10, go=14, ge=4))):
        exp = [_expected_best(reads[r], db, P, mu, **kw_or) for r, (db, P, mu) in enumerate(dbs)]
        for sel in (list(range(len(reads))), short):
            out = ssw.classify_reads([reads[r] for r in sel], rfam[sel], fams, **kw_gpu)
            ntag = 0
            for k, r in enumerate(sel):
                e = exp[r]
                if e is None:
                    assert out[k, 0] == 0, r
                else:
                    ntag += 1
                    assert (out[k, 2], out[k, 1], out[k, 0]) == (e[0], e[1], TAGC[e[2]]), (r, e, out[k])
            assert ntag > len(sel) // 3


def test_prefilter_is_exact_on_borderline_reads():
    """The q-gram pre-filter may only drop reads that cannot reach min_score = 30 against any template.
    Adversarial reads sit right at the bound: a 28..40 bp piece of a template (either strand) with 0..3
    substitutions, a 1..3 bp insertion or deletion, or N bases, embedded in random sequence — scores of
    24..40, i.e. just below and just above the filter's reach.  Every read must get exactly the oracle's
    record (tag, units, score), including the N-motif loci where template N is a wildcard."""
    from tredparse_b200 import ssw
    from tredparse_b200.meta import TREDsRepo
    from oracle import evidence_oracle as evo
    repo = TREDsRepo()
    rng = np.random.default_rng(99)
    B = "ACGT"
    rnd = lambda n: "".join(rng.choice(list(B), n))
    fams, reads, rfam, dbs = [], [], [], []
    for name in ("HD", "DM1", "DM2", "SCA10", "SCA36", "ULD", "OPMD", "BPES"):
        t = repo[name]
        P = len(t.repeat)
        mu = -(-150 // P)
        fams.append(ssw.make_family(t.prefix, t.repeat, t.suffix, mu))
        fi = len(fams) - 1
        db = evo.template_family(t.prefix, t.repeat, t.suffix, mu)
        for _ in range(40):
            u = int(rng.integers(1, mu + 1))
            tpl = db[2 * (u - 1) + int(rng.integers(0, 2))][1].replace("N", B[rng.integers(0, 4)])
            L = int(rng.integers(28, 41))
            st = int(rng.integers(0, max(1, len(tpl) - L + 1)))
            piece = list(tpl[st:st + L])
            kind = int(rng.integers(0, 4))
            if kind == 0:
                for _k in range(int(rng.integers(0, 4))):
                    piece[int(rng.integers(0, len(piece)))] = B[rng.integers(0, 4)]
            elif kind == 1:
                pos = int(rng.integers(5, len(piece) - 5))
                piece[pos:pos] = list(rnd(int(rng.integers(1, 4))))
            elif kind == 2:
                pos = int(rng.integers(5, len(piece) - 8))
                del piece[pos:pos + int(rng.integers(1, 4))]
            else:
                for _k in range(int(rng.integers(1, 3))):
                    piece[int(rng.integers(0, len(piece)))] = "N"
            left = int(rng.integers(0, 150 - len(piece) + 1))
            read = rnd(left) + "".join(piece) + rnd(150 - len(piece) - left)
            reads.append(read)
            rfam.append(fi)
            dbs.append((db, P, mu))
    out = ssw.classify_reads(reads, np.array(rfam, dtype=np.int32), np.concatenate(fams))
    tagged = 0
    for r, (db, P, mu) in enumerate(dbs):
        e = _expected_best(reads[r], db, P, mu)
        if e is None:
            assert out[r, 0] == 0, (r, out[r])
        else:
            tagged += 1
            assert (out[r, 2], out[r, 1], out[r, 0]) == (e[0], e[1], TAGC[e[2]]), (r, e, out[r])
    assert 20 < tagged < len(reads) - 20        # the set really straddles the threshold


def test_aligner_api_matches_reference_semantics():
    """ssw.Aligner / PyAlignRes keep the reference's call signature and filter rule."""
    from tredparse_b200.ssw import Aligner
    d = np.load(os.path.join(GOLDEN, "sw_pairs_t001_HD.npz"))
    read, tpl = str(d["reads"][0]), str(d["templates"][30])
    g = d["pairs"][0, 30].astype(int)
    al = Aligner(ref_seq=tpl, match=1, mismatch=5, gap_open=7, gap_extend=2, report_secondary=False)
    min_len = min(len(read), len(tpl)) // 2
    res = al.align(read, min_score=0, min_len=0)
    assert (res.score, res.ref_begin, res.ref_end, res.query_begin, res.query_end) == tuple(g[:5])
    n = int(d["cigar_len"][0, 30])
    assert res._cigar_string == [int(x) for x in d["cigar"][0, 30, :n]]
    assert al.align(read, min_score=10 ** 6, min_len=min_len) is None
    assert sum(l for l, op in res.iter_cigar if op in "MI") == res.query_end - res.query_begin + 1


def test_legacy_libssw_symbols_drop_in():
    """The reference's own ctypes calling sequence (ssw_wrap.py:186-224) against libtredsw.so."""
    import ctypes
    from tredparse_b200 import _lib, ssw

    class CAlignRes(ctypes.Structure):
        _fields_ = [('score', ctypes.c_uint16), ('score2', ctypes.c_uint16), ('ref_begin', ctypes.c_int32),
                    ('ref_end', ctypes.c_int32), ('query_begin', ctypes.c_int32), ('query_end', ctypes.c_int32),
                    ('ref_end2', ctypes.c_int32), ('cigar', ctypes.POINTER(ctypes.c_uint32)),
                    ('cigarLen', ctypes.c_int32)]
    lib = ctypes.CDLL(_lib.LIB_PATH)
    lib.ssw_init.restype = ctypes.c_void_p
    lib.ssw_init.argtypes = [ctypes.POINTER(ctypes.c_int8), ctypes.c_int32, ctypes.POINTER(ctypes.c_int8), ctypes.c_int32, ctypes.c_int8]
    lib.init_destroy.argtypes = [ctypes.c_void_p]
    lib.ssw_align.restype = ctypes.POINTER(CAlignRes)
    lib.ssw_align.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int8), ctypes.c_int32, ctypes.c_uint8,
                              ctypes.c_uint8, ctypes.c_uint8, ctypes.c_uint16, ctypes.c_int32, ctypes.c_int32]
    lib.align_destroy.argtypes = [ctypes.POINTER(CAlignRes)]
    lib.cigar_int_to_len.restype = ctypes.c_int32
    lib.cigar_int_to_op.restype = ctypes.c_char
    d = np.load(os.path.join(GOLDEN, "sw_pairs_t002_DM1.npz"))
    mat = ssw.score_matrix(1, 5)
    for (r, k) in ((0, 0), (3, 57), (10, 99), (50, 20)):
        read, tpl = ssw.encode(str(d["reads"][r])), ssw.encode(str(d["templates"][k]))
        read, tpl = np.ascontiguousarray(read), np.ascontiguousarray(tpl)
        P8 = ctypes.POINTER(ctypes.c_int8)
        prof = lib.ssw_init(read.ctypes.data_as(P8), len(read), mat.ctypes.data_as(P8), 5, 2)
        res = lib.ssw_align(prof, tpl.ctypes.data_as(P8), len(tpl), 7, 2, 1, 0, 0, len(read) // 2)
        c = res.contents
        g = d["pairs"][r, k].astype(int)
        assert (c.score, c.ref_begin, c.ref_end, c.query_begin, c.query_end, c.score2, c.ref_end2) == tuple(g)
        n = int(d["cigar_len"][r, k])
        assert c.cigarLen == n and [c.cigar[i] for i in range(n)] == [int(x) for x in d["cigar"][r, k, :n]]
        lib.init_destroy(prof)
        lib.align_destroy(res)
    assert lib.cigar_int_to_len(0x123) == 0x12 and lib.cigar_int_to_op(0x121) == b"I"
