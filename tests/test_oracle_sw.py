"""Oracle (CPU) Smith-Waterman restatement vs. the reference's own outputs.  No GPU needed."""
import os

import numpy as np
import pytest

from oracle import sw, evidence_oracle as evo

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
CASES = [("t001", "HD"), ("t002", "DM1")]


def _pairs(name):
    d = np.load(os.path.join(GOLDEN, name))
    reads, T = list(d["reads"]), list(d["templates"])
    nq, nt = len(reads), len(T)
    qidx = np.repeat(np.arange(nq, dtype=np.int32), nt)
    tidx = np.tile(np.arange(nt, dtype=np.int32), nq)
    return d, reads, T, qidx, tidx


@pytest.mark.parametrize("sample,tred", CASES)
def test_oracle_matches_reference_golden_pairs(sample, tred):
    """All 7 fields of every (read, template) pair of the reference fixtures — golden values were
    produced by the reference's unmodified ssw.c."""
    d, reads, T, qidx, tidx = _pairs("sw_pairs_{}_{}.npz".format(sample, tred))
    out = sw.oracle_align_pairs(reads, T, qidx, tidx)
    gold = d["pairs"].reshape(-1, 7).astype(np.int32)
    assert out.shape == gold.shape
    assert np.array_equal(out, gold)


def test_pair_count_is_24500():
    n = sum(np.load(os.path.join(GOLDEN, "sw_pairs_{}_{}.npz".format(s, t)))["pairs"].shape[0] * 100
            for s, t in CASES)
    assert n == 24500


def test_oracle_matches_reference_synthetic_pairs_and_cigars():
    d = np.load(os.path.join(GOLDEN, "sw_pairs_synthetic.npz"))
    q, T = list(d["queries"]), list(d["templates"])
    idx = np.arange(len(q), dtype=np.int32)
    out = sw.oracle_align_pairs(q, T, idx, idx)
    assert np.array_equal(out, d["pairs"])
    assert (d["pairs"][:, 0] >= 250).sum() > 10        # 16-bit path of the reference is exercised
    for i in range(len(q)):
        s, rb, re, qb, qe = (int(x) for x in d["pairs"][i, :5])
        c = sw.oracle_cigar(sw.encode(T[i])[rb:re + 1], sw.encode(q[i])[qb:qe + 1], s)
        g = d["cigar"][i, :d["cigar_len"][i]]
        assert c is not None and np.array_equal(c, g)


@pytest.mark.parametrize("sample,tred", CASES)
def test_classification_c_vs_python_and_golden_best(sample, tred):
    d, reads, T, qidx, tidx = _pairs("sw_pairs_{}_{}.npz".format(sample, tred))
    pairs = d["pairs"].astype(np.int32)
    units = d["units"]
    period = int(d["period"])
    READLEN = int(d["READLEN"])
    max_units = -(-READLEN // period)
    for r, read in enumerate(reads):
        res = []
        for k in range(len(T)):
            s, rb, re, qb, qe = (int(x) for x in pairs[r, k, :5])
            tag = evo.classify_alignment(s, rb, re, qb, qe, len(read), len(T[k]), int(units[k]), period, max_units)
            ctag = sw.TAGS[sw.oracle_classify(s, rb, re, qb, qe, len(read), len(T[k]), int(units[k]), period, max_units)]
            assert tag == ctag
            if tag:
                res.append((s, int(units[k]), tag))
        best = max(res, key=lambda x: (x[0], -x[1])) if res else None
        g = d["best"][r]
        if best is None:
            assert g[0] == -1
        else:
            assert (best[0], best[1], best[2]) == (g[0], g[1], sw.TAGS[int(g[2])])
