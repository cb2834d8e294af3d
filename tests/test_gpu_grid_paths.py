"""Every evaluation path, table tier and reduction of the likelihood grid (grid.cu) against the dense oracle.

The grid never materialises the surface unless asked, and which code computes a point is chosen by the data: small
or large surface, near / mid / far column region (thresholds H1 / H2 of big_setup), sorted / duplicated /
arithmetic candidate lists, the pass-A far loop, the four pass-B weight branches, and the table tier (full, without
the paired-end operands, none).  The cases below are tallies, not reads, placed on those edges; `_shape` restates
the kernel's decisions for each so that `test_every_path_is_reached` fails if a case stops reaching its path.

Per case: the materialised surface, n_points, arg-max (Q10), lik, CI, PP and the sparse posteriors == the oracle's;
the non-materialised run (the mode the fused call uses) == the materialised one, byte for byte; alone == inside a
batch of about 40 large surfaces (fewer CTAs per surface); and the three table tiers (TREDSW_GRID_TABLES) give the
same bits.  Needs a GPU: run with -m gpu."""
import multiprocessing
import os
import types
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RTOL = 1e-9
EPS = np.exp(-10)
INT_MAX = 0x7fffffff
SMALL_LIMIT, ITEM_POINTS, ITEM_MAX, NC_MAX, CHUNK = 512, 256, 12, 32, 256


def _tred(expansion=1, recessive=0, risk=36, prerisk=27):
    return types.SimpleNamespace(is_expansion=expansion, is_recessive=recessive, cutoff_risk=risk,
                                 cutoff_prerisk=prerisk, name="synthetic")


def _glens(n, seed=5):
    rng = np.random.default_rng(seed)
    return [int(x) for x in np.clip(np.rint(rng.normal(350, 75, n)), 200, 999)]


def case(name, full=None, pref=None, rept=0, depth=30.0, ploidy=2, nglobal=300, tlens=(), L=150, period=3,
         maxinsert=300, fullsearch=False, pe_ref=57, minpe=76, tred=None, lists=None):
    """One likelihood problem as tallies: FULL / PREF {units: reads}, the REPT count, and the pair lengths.  `lists`
    (h1 list, h2 list in bp) replaces the candidate lists of candidate_ranges for the GPU and the oracle alike."""
    return dict(name=name, full=dict(full or {}), pref=dict(pref or {}), rept=rept, depth=depth, ploidy=ploidy,
                glens=_glens(nglobal) if nglobal else [], tlens=[int(x) for x in tlens], L=L, period=period,
                maxinsert=maxinsert, fullsearch=fullsearch, pe_ref=pe_ref, minpe=minpe, tred=tred or _tred(),
                lists=lists)


def _pe_case(name, tmin, n_target=20, maxinsert=300, **kw):
    """Paired-end model on (PREF reads past the spanning ones): the far region starts at H2 = pe_ref + 1000 - tmin."""
    tl = [tmin + 7 * (i % 13) for i in range(n_target)]
    kw.setdefault("full", {12: 6})
    kw.setdefault("pref", {42: 3, 45: 4})
    kw.setdefault("rept", 3)
    return case(name, tlens=tl, maxinsert=maxinsert, **kw)


def _fa2_case(name, fa2_want):
    """Default search, extension list h2 = [36, 135, 138, 141, ...] (FULL 12 units, PREF 45): column c >= 2 holds
    135 + 3 (c - 1).  tmin puts H2 = 57 + 1000 - tmin on the value of column fa2_want."""
    h = 135 + 3 * (fa2_want - 1)
    return _pe_case(name, tmin=57 + 1000 - h, full={12: 6}, pref={45: 4, 43: 2}, maxinsert=600)


def _cases():
    C = []
    # size edges
    C.append(case("n512_small", full={10: 4, 15: 5}, rept=2, maxinsert=254))          # 2 x 256
    C.append(case("n513_large", full={10: 4, 15: 5}, rept=2, maxinsert=255))          # 2 x 257
    C.append(case("n3x256", full={10: 4, 15: 5, 17: 2}, rept=2, maxinsert=253))       # 3 x 256
    C.append(case("haploid_strided", pref={44: 5}, ploidy=1, maxinsert=3150, depth=15.0))
    C.append(case("haploid_full", full={20: 7, 21: 1}, ploidy=1, depth=15.0))
    C.append(case("n1_1", full={14: 9}, rept=4, maxinsert=600))
    C.append(case("n1_8", full={k: 2 for k in range(8, 16)}, rept=2))
    C.append(case("n1_9", full={k: 2 for k in range(8, 16)}, pref={41: 3}, rept=2))
    C.append(case("fullsearch_256", full={15: 6, 20: 5}, pref={44: 2}, rept=3, fullsearch=True, maxinsert=256))
    C.append(case("fullsearch_257", full={15: 6}, pref={44: 4}, rept=9, fullsearch=True, maxinsert=257,
                  tlens=range(300, 340)))
    C.append(_pe_case("n2_2102", tmin=700, maxinsert=2100))
    # regions: H1 bound by each term, a candidate on H1 / H2, far from the first column, no mid, no far
    C.append(case("H1_span_p1", full={141: 3, 60: 4}, rept=2, period=1, maxinsert=320))       # H1 = 141 + 19 = 160
    C.append(case("H1_partial_far_first", pref={60: 6, 55: 2}, rept=5))                      # H1 = mp = 180 > L + 1
    C.append(case("H1_L1_on_candidate", full={11: 5, 20: 3}, rept=3, L=149))                 # H1 = L + 1 = 150
    C.append(_pe_case("H2_on_candidate", tmin=57 + 1000 - 450))
    C.append(_pe_case("no_far", tmin=80))                                                    # H2 = 977 > 900
    for fa2 in (32, 31, 33, 64, 65):
        C.append(_fa2_case("fa2_%d" % fa2, fa2))
    # paired-end shapes
    C.append(case("pe_below_minpe", full={12: 6}, pref={42: 3, 45: 4}, rept=3, tlens=[5, 20, 40, 60, 75, 30]))
    C.append(case("pe_negative", full={12: 6}, pref={42: 3, 45: 4}, rept=3,
                  tlens=[-5, -300, -999, 400, 420, 450, 600, -1]))
    for n in (63, 64, 65, 129):
        C.append(_pe_case("pe_n%d" % n, tmin=330, n_target=n))
    C.append(_pe_case("pe_global99", tmin=330, nglobal=99))
    C.append(_pe_case("pe_global100", tmin=330, nglobal=100))
    C.append(_pe_case("pe_target4", tmin=330, n_target=4))
    C.append(_pe_case("pe_target5", tmin=330, n_target=5))
    # lists: Q9 duplicates in an unsorted extension; PREF only; a wide --fullsearch grid
    C.append(case("dup_unsorted", full={10: 5, 60: 3}, pref={42: 4}, rept=4))
    C.append(case("pref_only", pref={44: 6, 41: 3}, rept=6))
    C.append(case("fullsearch_400", full={15: 6, 60: 3}, pref={44: 4, 46: 2}, rept=12, fullsearch=True,
                  maxinsert=400, tlens=range(250, 330, 3)))
    # ties of the maximum along an anti-diagonal (PREF + REPT only: the partial term saturates)
    C.append(case("tie_antidiag", pref={44: 5, 46: 3}, rept=60, maxinsert=300))
    C.append(case("tie_antidiag_pe", pref={44: 5, 46: 3}, rept=40, maxinsert=300, tlens=[100, 120, 140] * 3))
    # PP: each (expansion, recessive) mode with its cutoff on the called alleles (20 | 21), small and large surfaces
    for e in (0, 1):
        for r in (0, 1):
            for risk in (19, 20, 21):
                t = _tred(e, r, risk, risk - 5)
                C.append(case("pp_e%d_r%d_c%d_small" % (e, r, risk), full={20: 6, 21: 5}, tred=t))
                C.append(case("pp_e%d_r%d_c%d_large" % (e, r, risk), full={20: 6, 21: 5}, rept=1, fullsearch=True,
                              maxinsert=60, tred=t))
    # the repeat-only term: absent, and floored at -100
    C.append(case("rept0_large", full={15: 6, 30: 5}, fullsearch=True, maxinsert=70))
    C.append(case("rept_floor", full={15: 6}, pref={44: 3}, rept=400, depth=4.0, maxinsert=200))
    # lists in the layout the kernel accepts (a sorted base part, then an ascending extension; tredsw_likelihood_grid
    # takes any such list) that candidate_ranges never builds: a Q9 duplicate in a far chunk of a sorted list (the
    # base ends where the extension starts), and an unsorted list whose far columns are not arithmetic
    base = [30, 45] + [153 + 3 * i for i in range(254)]
    C.append(case("lists_far_dup_sorted", full={10: 3, 15: 4}, rept=76,
                  lists=([30, 45], base + [base[-1] + 3 * i for i in range(300)])))
    C.append(case("lists_far_dup_unsorted", full={10: 3, 15: 4}, rept=40,
                  lists=([30, 45, 900], [30, 45, 900] + [153 + 3 * i for i in range(300)])))
    return C


CASES = _cases()


# ------------------------------------------------------------------------------------------------------------
# the oracle, one process per case (numpy-bound: threads would not run in parallel)
# ------------------------------------------------------------------------------------------------------------
def _oracle(c):
    from oracle import likelihood_oracle as lko
    from test_gpu_cohort import _models
    step, w = _models()
    pe = types.SimpleNamespace(global_lens=c["glens"], target_lens=c["tlens"], ref=c["pe_ref"], MINPE=c["minpe"])
    lk = lko.LikelihoodOracle(c["tred"], c["period"], c["L"], {"FULL": c["full"], "PREF": c["pref"]}, c["rept"],
                              c["ploidy"], c["depth"], pe, step, w, maxinsert=c["maxinsert"], fullsearch=c["fullsearch"])
    if c["lists"]:
        rules = lk.candidate_ranges
        lk.candidate_ranges = lambda *a: (list(c["lists"][0]), list(c["lists"][1]), rules(*a)[2])
    p = c["period"]
    alleles, lik, PP, CIs = lk.evaluate({k * p: v for k, v in c["full"].items()},
                                        {k * p: v for k, v in c["pref"].items()}, c["rept"])
    return dict(surface=[(s[0] + s[1] + s[3], s[4], s[5], s[6]) for s in lk.surface], alleles=alleles, lik=lik,
                PP=PP, CIs=CIs, P_h1=lk.P_h1, P_h2=lk.P_h2, P_h1h2=lk.P_h1h2, h1range=list(lk.h1range),
                h2range=list(lk.h2range), run_pe=bool(lk.run_pe), max_partial=lk.max_partial,
                pdf=None if lk.pemodel is None else lk.pemodel.pdf)


@pytest.fixture(scope="module")
def oracle():
    ctx = multiprocessing.get_context("spawn")
    order = sorted(range(len(CASES)), key=lambda i: -_cost(CASES[i]))         # longest first
    with ProcessPoolExecutor(max_workers=min(16, os.cpu_count() or 1), mp_context=ctx) as ex:
        res = dict(zip(order, ex.map(_oracle, [CASES[i] for i in order])))
    return [res[i] for i in range(len(CASES))]


def _cost(c):
    n = c["maxinsert"]
    return n * n if c["fullsearch"] else n * max(1, len(c["full"]) + 1)


# ------------------------------------------------------------------------------------------------------------
# the GPU
# ------------------------------------------------------------------------------------------------------------
def _add(batch, c, o):
    from tredparse_b200 import models
    rules = models.candidate_ranges
    if c["lists"]:
        models.candidate_ranges = lambda *a: (list(c["lists"][0]), list(c["lists"][1])) + tuple(rules(*a)[2:])
    try:
        i = batch.add(c["tred"], c["period"], c["L"], {k * c["period"]: v for k, v in c["full"].items()},
                      {k * c["period"]: v for k, v in c["pref"].items()}, c["rept"], c["ploidy"], c["depth"],
                      o["pdf"], c["tlens"], c["pe_ref"], c["minpe"], maxinsert=c["maxinsert"],
                      fullsearch=c["fullsearch"])
    finally:
        models.candidate_ranges = rules
    assert i >= 0
    return i


def _run(cs, os_, want_surface=True, tables=None):
    from tredparse_b200 import models
    old = os.environ.pop("TREDSW_GRID_TABLES", None)
    try:
        if tables:
            os.environ["TREDSW_GRID_TABLES"] = tables
        b = models.GridBatch()
        for c, o in zip(cs, os_):
            _add(b, c, o)
        return b.run(want_surface=want_surface)
    finally:
        os.environ.pop("TREDSW_GRID_TABLES", None)
        if old is not None:
            os.environ["TREDSW_GRID_TABLES"] = old


@pytest.fixture(scope="module")
def runs(oracle):
    """Every case alone: {(tables, materialised): GridBatch}."""
    out = []
    for c, o in zip(CASES, oracle):
        out.append({(t, m): _run([c], [o], want_surface=m, tables=t)
                    for t in (None, "nope", "none") for m in (True, False)})
    return out


# ------------------------------------------------------------------------------------------------------------
# the kernel's shape decisions, restated (grid_classify_kernel, big_setup, rows_eval, grid_rows_reduce_kernel)
# ------------------------------------------------------------------------------------------------------------
def _second_occurrence(hs):
    nb = next((i for i in range(1, len(hs)) if hs[i] <= hs[i - 1]), len(hs))
    return [i >= nb and nb > 0 and hs[i] <= hs[nb - 1] and hs[i] in hs[:nb] for i in range(len(hs))]


def _shape(c, o, tables=None, want_post=False):
    """-> (set of path names, dict of the decisions) for the case at a table tier (None = full tables)."""
    paths, d = set(), {}
    L, p = c["L"], c["period"]
    h1s, h2s = o["h1range"], (o["h2range"] if c["ploidy"] != 1 else [0])
    n1, n2 = len(h1s), len(h2s)
    total = n1 * n2
    run_pe = o["run_pe"]
    if c["ploidy"] == 1 or total <= SMALL_LIMIT:
        paths.add("small")
        chunks = -(-total // ITEM_POINTS)
        if chunks > ITEM_MAX:
            paths.add("small_item_strides")
        if c["ploidy"] == 1:
            paths.add("haploid")
        d["small"] = True
        return paths, d
    paths.add("large")
    ok = tables != "none"
    wrapped = [x + 1000 if x < 0 else x for x in c["tlens"]] if run_pe else []
    npe = len(wrapped) if (run_pe and tables is None) else 0
    ks = max([k * p for k in c["full"]], default=-1000000)
    mp = o["max_partial"]
    tmin = min([x for x in wrapped if x >= c["minpe"]], default=INT_MAX)
    H1 = max(ks + 19, mp, L - 9, L + 1)
    H2 = max(H1, c["pe_ref"] + 1000 - tmin) if (run_pe and tmin != INT_MAX) else H1
    l1 = max([i for i, h in enumerate(h2s) if h < H1], default=-1)
    l2 = max([i for i, h in enumerate(h2s) if h < H2], default=-1)
    fam, fa2 = (l1 + 1, l2 + 1) if ok else (n2, n2)
    srt = all(a <= b for a, b in zip(h1s, h1s[1:])) and all(a <= b for a, b in zip(h2s, h2s[1:]))
    dup1, dup2 = _second_occurrence(h1s), _second_occurrence(h2s)
    has_dup = any(dup1) or any(dup2)
    astep = h2s[1] - h2s[0] if n2 > 1 else 1
    h2_arith = astep > 0 and all(h == h2s[0] + i * astep for i, h in enumerate(h2s))
    fstep = h2s[fa2 + 1] - h2s[fa2] if fa2 + 1 < n2 else 0
    fd0 = h2s[fa2] - L if fa2 < n2 else 1
    far_arith = fd0 >= 1 and all(h2s[i] == h2s[fa2] + (i - fa2) * fstep for i in range(fa2, n2))
    nc = min(NC_MAX, max(1, (n1 + 7) // 8))
    d.update(H1=H1, H2=H2, fam=fam, fa2=fa2, sorted=srt, has_dup=has_dup, h2_arith=h2_arith, far_arith=far_arith,
             nc=nc, tmin=tmin, npe=npe)
    # thresholds and regions
    bind = [n for n, v in (("span", ks + 19), ("partial", mp), ("L+1", L + 1)) if v == H1]
    paths.update("H1_bound_by_" + b for b in bind)
    if H1 in h2s:
        paths.add("candidate_on_H1")
    if H2 > H1:
        paths.add("H2_above_H1")
        if H2 in h2s:
            paths.add("candidate_on_H2")
    if ok:
        paths.add("no_mid" if fam == fa2 else "mid")
        paths.add("no_far" if fa2 == n2 else "far")
        if fa2 == 0:
            paths.add("far_from_first_column")
        if 0 < fa2 < n2:
            paths.add("fa2_mod32_%s" % {0: "0", 1: "1", 31: "31"}.get(fa2 % 32, "other"))
    if run_pe:
        paths.add("pe")
        if tmin == INT_MAX:
            paths.add("pe_every_pair_below_minpe")
        if any(x < 0 for x in c["tlens"]):
            paths.add("pe_negative_lengths")
        nt = len(wrapped)
        paths.add("pe_blocks_%s" % ("1" if nt < 64 else "exact" if nt % 64 == 0 else "tail"))
    paths.add("sorted" if srt else "unsorted")
    if has_dup:
        paths.add("q9_duplicates")
    paths.add("h2_arith" if h2_arith else "h2_not_arith")
    if ok and fa2 < n2:
        paths.add("far_arith" if far_arith else "far_not_arith")
    if n1 % 8:
        paths.add("rows_partial_warp_group")
    paths.add("ctas_%s" % ("1" if nc == 1 else "32" if nc == NC_MAX else "some"))
    if n2 > 2048:
        paths.add("n2_above_2048")
    # pass A: first column of each row, mixed_batch<NJ> sequence, far loop
    ngroups = (n2 + 31) >> 5
    g_mid_end = (min(fa2, n2) + 31) >> 5 if ok else ngroups
    arith = far_arith and ok
    for h1 in h1s:
        if h2_arith:
            num = h1 - h2s[0] + astep - 1
            c0 = min(n2, max(0, int(num / astep)))                   # C division truncates toward zero
        elif srt:
            c0 = int(np.searchsorted(h2s, h1, side="left"))
        else:
            c0 = 0
        gb = c0 >> 5
        while gb < g_mid_end:
            nj = 4 if g_mid_end - gb >= 4 else 2 if g_mid_end - gb >= 2 else 1
            paths.add("mixed_batch_%d" % nj)
            gb += nj
        cf = max(32 * gb, c0)
        if arith and srt:
            if cf < n2:
                paths.add("passA_far_fast")                          # (the run without a materialised surface)
                if cf + 96 < n2:
                    paths.add("passA_far_fast_unrolled")
        elif gb < ngroups:
            paths.add("passA_far_loop_arith" if arith else "passA_far_loop_list")
    # pass B: weight branch of each (row, 256-column chunk, lane)
    far_f = {}
    if want_post and ok:
        M = o["lik"]
        hrep = max(h2s)
        for c12pe, ml, a, b in o["surface"]:
            if b == hrep:
                far_f[a] = np.exp(c12pe - M)
    for cb in range(0, n2, CHUNK):
        cend = min(cb + CHUNK, n2)
        h2_last = h2s[cend - 1] if srt else INT_MAX
        all_far = ok and cb >= fa2
        full_chunk = cend - cb == CHUNK
        lane_dup = [has_dup and any(dup2[col] for col in range(cb + lane, cend, 32)) for lane in range(32)]
        for i1, h1 in enumerate(h1s):
            if h2_last < h1:
                continue
            d1 = has_dup and dup1[i1]
            may_emit = want_post and not d1 and far_f.get(h1, 0.0) >= EPS
            for lane in range(32):
                quiet = not d1 and not lane_dup[lane] and not may_emit
                if all_far and full_chunk and srt and h1 <= h2s[cb] and not d1 and not may_emit and lane_dup[lane]:
                    paths.add("passB_far_full_chunk_dup")       # the first branch's test of dup2 is what keeps it out
                if all_far and full_chunk and srt and h1 <= h2s[cb] and quiet:
                    paths.add("passB_far_full_chunk")
                elif all_far and quiet:
                    paths.add("passB_far")
                elif all_far:
                    paths.add("passB_far_tested")
                    if may_emit:
                        paths.add("passB_far_emit")
                    if lane_dup[lane] or d1:
                        paths.add("passB_far_dup")
                else:
                    paths.add("passB_general")
    return paths, d


def _tie_paths(c, o, nce):
    """Rows of different CTAs (row groups of 8 dealt round-robin over nce CTAs) holding the exact maximum."""
    M = max(s[1] for s in o["surface"])
    rows = {o["h1range"].index(s[2]) for s in o["surface"] if s[1] == M}
    return {"tie_across_ctas"} if len({(r // 8) % nce for r in rows}) > 1 else set()


def _pp_paths(c, o):
    t, p = c["tred"], c["period"]
    hs = {h // p for h in o["h1range"] + o["h2range"]}
    mode = "pp_e%d_r%d" % (t.is_expansion, t.is_recessive)
    r = t.cutoff_risk
    return {mode + "_cutoff_pm1"} if {r - 1, r, r + 1} <= hs else set()


# Far columns that are not arithmetic and a Q9 duplicate in a far chunk come only from the lists_* cases: the lists of
# candidate_ranges are a sorted base part, whose values below H1 are spanning keys or max_partial, and an ascending
# extension from max_partial + period, so their far columns are arithmetic and their duplicates lie in the near region.
REQUIRED = {
    "small", "small_item_strides", "haploid", "large",
    "H1_bound_by_span", "H1_bound_by_partial", "H1_bound_by_L+1", "candidate_on_H1", "H2_above_H1",
    "candidate_on_H2", "no_mid", "mid", "no_far", "far", "far_from_first_column",
    "fa2_mod32_0", "fa2_mod32_1", "fa2_mod32_31",
    "pe", "pe_every_pair_below_minpe", "pe_negative_lengths", "pe_blocks_1", "pe_blocks_exact", "pe_blocks_tail",
    "sorted", "unsorted", "q9_duplicates", "h2_arith", "h2_not_arith", "far_arith", "far_not_arith",
    "rows_partial_warp_group", "ctas_1", "ctas_32", "ctas_some", "n2_above_2048",
    "mixed_batch_4", "mixed_batch_2", "mixed_batch_1",
    "passA_far_fast", "passA_far_fast_unrolled", "passA_far_loop_arith", "passA_far_loop_list",
    "passB_far_full_chunk", "passB_far_full_chunk_dup", "passB_far", "passB_far_tested", "passB_far_dup",
    "passB_general",
    "tie_across_ctas",
    "pp_e0_r0_cutoff_pm1", "pp_e0_r1_cutoff_pm1", "pp_e1_r0_cutoff_pm1", "pp_e1_r1_cutoff_pm1",
    "rept_zero", "rept_floored",
}


def _all_paths(c, o):
    paths, d = _shape(c, o)
    if "large" in paths:
        paths |= _tie_paths(c, o, d["nc"])
    paths |= _pp_paths(c, o)
    if c["rept"] == 0 and "large" in paths:
        paths.add("rept_zero")
    if c["rept"]:
        from scipy.stats import poisson
        L, hd = c["L"], c["depth"] / 2
        if any(poisson.pmf(c["rept"], (max(a - L, 1) + max(b - L, 1)) * hd / L) < np.exp(-100)
               for _, _, a, b in o["surface"]):
            paths.add("rept_floored")
    return paths, d


def test_every_path_is_reached(oracle):
    """Each path of REQUIRED is taken by at least one case (the restatement of the kernel's decisions)."""
    reach = {}
    for c, o in zip(CASES, oracle):
        for p in _all_paths(c, o)[0]:
            reach.setdefault(p, []).append(c["name"])
    missing = sorted(REQUIRED - set(reach))
    assert not missing, (missing, {p: reach[p] for p in sorted(reach)})


# ------------------------------------------------------------------------------------------------------------
# assertions
# ------------------------------------------------------------------------------------------------------------
def _close(a, b, rtol):
    return abs(a - b) <= rtol * max(abs(b), 1e-300)


@pytest.mark.parametrize("k", range(len(CASES)), ids=[c["name"] for c in CASES])
def test_case_matches_oracle(oracle, runs, k):
    """Surface point by point (-inf exactly where h1 > h2), n_points, arg-max, lik, CI, PP and P_h1 / P_h2 / P_h1h2."""
    c, o = CASES[k], oracle[k]
    b = runs[k][(None, True)]
    assert b.meta[0][3] == o["h1range"] and (c["ploidy"] == 1 or b.meta[0][4] == o["h2range"])
    assert bool(b.meta[0][5]) == o["run_pe"]
    S = b.surface_of(0)
    it = iter(o["surface"])
    for i1, h1 in enumerate(o["h1range"]):
        for i2, h2 in enumerate([h1] if c["ploidy"] == 1 else o["h2range"]):
            if h1 > h2:
                assert S[i1, i2] == -np.inf, (i1, i2)
                continue
            _, want, a, bb = next(it)
            assert (a, bb) == (h1, h2)
            assert _close(S[i1, i2], want, RTOL), (h1, h2, S[i1, i2], want)
    s = b.summarize(0)
    assert s["n_points"] == len(o["surface"])
    # the share of the points the joint posterior holds (a Q9 duplicate is held once): sum_uniq / sum_all
    M = o["lik"]
    w_all = sum(np.exp(ml - M) for _, ml, _, _ in o["surface"])
    w_uniq = sum(np.exp(ml - M) for ml in {(a, bb): ml for _, ml, a, bb in o["surface"]}.values())
    R = b.results[0]
    assert _close(float(R["sum_uniq"]) / float(R["sum_all"]), w_uniq / w_all, RTOL), (R["sum_uniq"], R["sum_all"])
    assert tuple(s["alleles"]) == tuple(o["alleles"]), (s["alleles"], o["alleles"])
    assert _close(s["lik"], o["lik"], RTOL)
    assert tuple(s["CIs"]) == tuple(o["CIs"])
    assert abs(s["PP"] - o["PP"]) <= 1e-9, (s["PP"], o["PP"])
    for name in ("P_h1", "P_h2", "P_h1h2"):
        assert set(s[name]) == set(o[name]), (name, sorted(set(s[name]) ^ set(o[name]))[:6])
        for key, v in o[name].items():
            assert abs(s[name][key] - v) <= 1e-9 * abs(v), (name, key, s[name][key], v)


@pytest.mark.parametrize("tables", [None, "nope", "none"])
def test_unmaterialised_run_equals_materialised(runs, tables):
    """want_surface=False (pass A's fast far loop) gives byte-identical results and marginals."""
    for c, r in zip(CASES, runs):
        a, b = r[(tables, True)], r[(tables, False)]
        assert a.results.tobytes() == b.results.tobytes(), c["name"]
        assert a.marg.tobytes() == b.marg.tobytes(), c["name"]


def _sums_close(a, b, rtol=1e-12):
    for f in ("sum_all", "sum_path", "sum_uniq"):
        assert _close(float(a[f]), float(b[f]), rtol), (f, a[f], b[f])


@pytest.mark.parametrize("tables", ["nope", "none"])
def test_table_tiers_give_the_same_bits(runs, tables):
    """Tables without the paired-end operands / no tables: the same surface, maximum, arg-max and point count bit for
    bit (LogProd, halved PE operands); sums and marginals within 1e-12 (with no tables a far weight is exp(ml - max)
    instead of exp(c12 + pe - max) * exp(rept): another rounding)."""
    for c, r in zip(CASES, runs):
        a, b = r[(None, True)], r[(tables, True)]
        assert a.surface.tobytes() == b.surface.tobytes(), c["name"]
        for f in ("max_ml", "arg_i1", "arg_i2", "n_points"):
            assert a.results[0][f] == b.results[0][f], (c["name"], f)
        _sums_close(a.results[0], b.results[0])
        assert np.allclose(a.marg, b.marg, rtol=1e-12, atol=0), c["name"]
        if tables == "nope":                      # the nope tier changes nothing in the PE-free cases
            if not a.meta[0][5]:
                assert a.marg.tobytes() == b.marg.tobytes(), c["name"]


@pytest.mark.parametrize("tables", [None, "nope", "none"])
def test_alone_equals_inside_a_batch_of_forty_large_surfaces(oracle, runs, tables):
    """About 40 large surfaces in one call: fewer CTAs per surface (nce), another grouping of the partial sums, and the
    tables of every surface packed next to each other in the arena (a surface that wrote or read past its own table
    layout would change a neighbour's numbers).  max, arg-max and point count are byte-identical; sums and marginals
    within 1e-12."""
    import torch
    big = [k for k in range(len(CASES)) if "large" in _shape(CASES[k], oracle[k])[0]]
    ks = (big * (1 + 40 // len(big)))[:max(40, len(big))]
    b = _run([CASES[k] for k in ks], [oracle[k] for k in ks], want_surface=False, tables=tables)
    target = torch.cuda.get_device_properties(0).multi_processor_count * 6
    nce = max(1, -(-target // len(ks)))
    assert any(_shape(CASES[k], oracle[k])[1]["nc"] > nce for k in ks)       # some surface really loses CTAs
    for j, k in enumerate(ks):
        a = runs[k][(tables, False)]
        ra, rb = a.results[0], b.results[j]
        for f in ("max_ml", "arg_i1", "arg_i2", "n_points"):
            assert ra[f] == rb[f], (CASES[k]["name"], f)
        _sums_close(ra, rb)
        P = b.probs[j]
        m = b.marg[P["off_ph1"]:P["off_ph2"] + P["n_h2"]]
        assert np.allclose(a.marg, m, rtol=1e-12, atol=0), CASES[k]["name"]


def test_bad_table_switch_is_an_error(oracle):
    from tredparse_b200 import _lib
    with pytest.raises(_lib.TredswError, match="TREDSW_GRID_TABLES"):
        _run([CASES[1]], [oracle[1]], tables="fast")


# ------------------------------------------------------------------------------------------------------------
# the same shapes through the fused call (CohortBatch.run_host): reads built to give the intended tallies
# ------------------------------------------------------------------------------------------------------------
_BASES = "ACGT"


def _reads_problem(name, L, full=None, pref=None, rept=0, tlens=(), depth=30.0, ploidy=2, seed=0):
    """FULL reads of h units between the locus' flanks, PREF reads running off the read end inside the repeat, pure
    repeat REPT reads (unique names: none is dropped as the mate of another), random bases around them."""
    from tredparse_b200 import simulate
    from tredparse_b200.meta import TREDsRepo
    from tredparse_b200.ssw import encode
    t = TREDsRepo()[name]
    rng = np.random.default_rng(seed)
    P = len(t.repeat)
    rnd = lambda n: "".join(rng.choice(list(_BASES), n)) if n > 0 else ""
    motif = lambda h: "".join(t.repeat.replace("N", _BASES[rng.integers(0, 4)]) for _ in range(h))
    reads, want = [], []
    for h, n in (full or {}).items():
        for _ in range(n):
            core = t.prefix + motif(h) + t.suffix
            a = int(rng.integers(0, L - len(core) + 1))
            reads.append(rnd(a) + core + rnd(L - len(core) - a))
            want.append(("FULL", h))
    for h, n in (pref or {}).items():
        for _ in range(n):
            reads.append(rnd(L - len(t.prefix) - P * h) + t.prefix + motif(h))
            want.append(("PREF", h))
    for _ in range(rept):
        s = motif(L // P + 2)
        k = int(rng.integers(0, P))
        reads.append(s[k:k + L])
        want.append(("REPT", None))
    pr = simulate.Problem()
    pr.tred, pr.readlen, pr.ploidy, pr.alleles = t, L, ploidy, (name,)
    pr.reads = np.concatenate([encode(r) for r in reads]).astype(np.int8) if reads else np.zeros(0, np.int8)
    pr.roff = np.arange(len(reads) + 1, dtype=np.int64) * L
    pr.global_lens = np.array(_glens(300, seed), dtype=np.int32)
    pr.target_lens = np.array(list(tlens), dtype=np.int32)
    pr.depth = float(depth)
    pr.names = np.arange(len(reads), dtype=np.int64)
    return pr, want


FUSED = [  # (name, locus, readlen, tallies, batch)
    ("far_emit", "DM1", 150, dict(full={13: 8}, pref={40: 3, 44: 4}, rept=74), "a"),
    ("q9_large", "HD", 150, dict(full={36: 5, 15: 4}, pref={20: 3}, rept=3), "a"),
    ("pe_mid_far", "HD", 150, dict(full={15: 6}, pref={41: 3, 44: 4}, rept=3, tlens=[520 + 9 * i for i in range(30)]), "a"),
    ("tie", "HD", 150, dict(pref={42: 4, 44: 3}, rept=60), "a"),
    ("pp_HD", "HD", 250, dict(full={39: 3, 40: 4, 41: 3, 17: 5}, rept=2), "a"),
    ("pp_DM1", "DM1", 250, dict(full={49: 3, 50: 4, 51: 3, 13: 5}), "a"),
    ("pp_FRDA", "FRDA", 250, dict(full={65: 3, 66: 4, 67: 3}, rept=1), "a"),
    ("pp_AR_small", "AR", 250, dict(full={7: 2, 8: 8, 9: 2}), "a"),
    ("pp_AR_large", "AR", 250, dict(full={7: 2, 8: 8, 9: 2}, rept=2), "a"),
    ("q9_small", "HD", 150, dict(full={36: 5, 15: 4}, pref={20: 3}, rept=3), "b"),     # maxinsert 40
    ("fullsearch_1000", "FXS", 150, dict(full={30: 6}, pref={44: 3}, rept=4, ploidy=1, depth=15.0), "c"),
]
FUSED_RUN = {"a": dict(maxinsert=400), "b": dict(maxinsert=40), "c": dict(maxinsert=1000, fullsearch=True)}


def _fused_oracle(k):
    from test_gpu_cohort import _expected_reads, _models, _oracle_call
    name, locus, L, tallies, batch = FUSED[k]
    pr, want = _reads_problem(locus, L, seed=100 + k, **tallies)
    exp = _expected_reads(pr)
    tags = {1: "FULL", 2: "PREF", 3: "PREF", 4: "REPT"}
    got = [(tags.get(a), b if tags.get(a) != "REPT" else None) for a, b in exp]
    assert got == want, (name, [(g, w) for g, w in zip(got, want) if g != w][:5])
    step, w = _models()
    lk, counts, rept = _oracle_call(pr, [(a, b) for a, b in exp if a not in (0, 5)], step, w, **FUSED_RUN[batch])
    o = dict(surface=[(s[0] + s[1] + s[3], s[4], s[5], s[6]) for s in lk.surface], h1range=list(lk.h1range),
             h2range=list(lk.h2range), run_pe=bool(lk.run_pe), max_partial=lk.max_partial, lik=lk.lik * 1.0)
    lk.surface = [None] * len(lk.surface)          # (only its length is compared)
    lk.pemodel, lk.spanning_db, lk.partial_db = None, {}, {}
    return pr, (exp, lk, counts, rept), o


@pytest.fixture(scope="module")
def fused():
    ctx = multiprocessing.get_context("spawn")
    with ProcessPoolExecutor(max_workers=min(16, os.cpu_count() or 1), mp_context=ctx) as ex:
        return list(ex.map(_fused_oracle, range(len(FUSED))))


def test_fused_call_paths_vs_oracle(fused):
    """Every call field and posterior of the fused call == the oracle's: far-column joint entries emitted in pass B
    (may_emit), Q9 duplicates (counted in the marginals and PP, held once in P_h1h2, merged in P_h1 / P_h2), ties, the
    PP boundaries of four inheritance modes and a haploid --fullsearch problem at maxinsert 1000.  With TREDSW_GRID_TABLES=none
    the calls are the same bits apart from PP (another rounding of the far weights)."""
    import torch
    from test_gpu_read_lengths import _check_calls
    from tredparse_b200 import cohort
    reached = set()
    for batch, kw in FUSED_RUN.items():
        ks = [k for k in range(len(FUSED)) if FUSED[k][4] == batch]
        problems = [fused[k][0] for k in ks]
        out = cohort.CohortBatch(problems, **kw).run_host(want_reads=True, want_hist=True, want_post=True)
        post = _check_calls(problems, out, [fused[k][1] for k in ks])
        shapes = {}
        for k in ks:
            pr, (exp, lk, counts, rept), o = fused[k]
            c = dict(full=dict(counts["FULL"]), pref=dict(counts["PREF"]), rept=rept, ploidy=pr.ploidy,
                     tlens=[int(x) for x in pr.target_lens], L=pr.readlen, period=len(pr.tred.repeat),
                     pe_ref=pr.tred.repeat_end - pr.tred.repeat_start + 1, tred=pr.tred)
            c["minpe"] = c["pe_ref"] - 1 + 20
            shapes[k] = (c, o) + _shape(c, o, want_post=True)
        # CTAs per large surface in this call (big_setup: nce = min(nc, ceil(target_ctas / large surfaces)))
        nbig = sum("large" in sh[2] for sh in shapes.values())
        target = torch.cuda.get_device_properties(0).multi_processor_count * 6
        for k, (c, o, paths, d) in shapes.items():
            if "large" in paths:
                paths = paths | _tie_paths(c, o, max(1, min(d["nc"], -(-target // nbig))))
            reached |= {FUSED[k][0] + ":" + p for p in paths}
        old = os.environ.get("TREDSW_GRID_TABLES")
        os.environ["TREDSW_GRID_TABLES"] = "none"
        try:
            bare = cohort.CohortBatch(problems, **kw).run_host(want_post=True)
        finally:
            if old is None:
                os.environ.pop("TREDSW_GRID_TABLES")
            else:
                os.environ["TREDSW_GRID_TABLES"] = old
        a, b = out["calls"], bare["calls"]
        for f in a.dtype.names:
            if f != "pp":
                assert a[f].tobytes() == b[f].tobytes(), (batch, f)
        assert np.allclose(a["pp"], b["pp"], rtol=1e-12, atol=0), batch
        pb = cohort.posteriors(bare["post"], len(problems))
        for i in range(len(problems)):
            for name in ("P_h1", "P_h2", "P_h1h2"):
                assert set(pb[i][name]) == set(post[i][name]), (batch, i, name)
                for key, v in post[i][name].items():
                    assert _close(pb[i][name][key], v, 1e-12), (batch, i, name, key)
    for want in ("far_emit:passB_far_emit", "far_emit:passB_far_tested", "q9_large:q9_duplicates",
                 "q9_large:large", "q9_small:small", "tie:large", "tie:tie_across_ctas", "pp_AR_small:small", "pp_AR_large:large",
                 "fullsearch_1000:small", "pe_mid_far:mid"):
        assert want in reached, (want, sorted(reached))
