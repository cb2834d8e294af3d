"""
Statistical model of the caller — host side.

Keeps the reference's ``tredparse/models.py`` interface: ``StepModel`` (:42-61), ``NoiseModel``
(:64-84), ``mean_std`` (:87-91), ``histogram`` (:94-98), ``IntegratedCaller(bamParser, score, gc,
maxinsert, fullsearch).call()`` (:101-147, 394-415) with result attributes ``alleles, label, CI, PP,
PEDP, PEG, PET, P_h1, P_h2, P_h1h2, P_PEG, P_PET``.

What runs where:
  host   candidate-allele lists (models.py:224-257, duplicates kept — quirk Q9), run_pe decision,
         CI / sparsify / label bookkeeping on the reduced vectors (:304-392);
  GPU    the KDE of the global pair lengths (:428-435, ``tredsw_pe_kde``), the log-likelihood of every
         (h1, h2) candidate pair (:260-273) and the max / arg-max / marginal / PP reductions
         (:277-302, 342-368) — ``tredsw_likelihood_grid``.
``GridBatch`` evaluates many (sample, locus) problems in one launch; ``IntegratedCaller`` is the
single-problem, reference-shaped front end over it.
"""
import json
import logging
import math
from collections import defaultdict

import numpy as np

from . import _lib
from .utils import datafile, listify

SPAN = 1000
FLANKMATCH = 9
MAX_PERIOD = 6
MAX_LOCUS_PERIOD = 20        # the longest motif the STR profile reports (IrrParams.max_period): discovered loci
SMALL_VALUE = math.exp(-10)
REALLY_SMALL_VALUE = math.exp(-100)
MODEL_PREFIX = "illumina_v3.pcrfree"
MIN_SPANNING_PAIRS = 5

_MODELS = None


def _models():
    global _MODELS
    if _MODELS is None:
        with open(datafile("models.json")) as fp:
            _MODELS = json.load(fp)
    return _MODELS


class StepModel:
    """Step-size distributions per motif period (37 bins centred on 18)."""

    def __init__(self, filename=None):
        md = _models()
        self.non_unit_step_by_period = {i + 1: v for i, v in enumerate(md["non_unit_step_by_period"])}
        self.prob_increase = md["prob_increase"]
        self.step_size_by_period = {int(k): np.array(v) for k, v in md["step_size_by_period"].items()}
        # longer periods share the period-6 distribution (models.py:59-60 stops at 17; discovered loci reach 20)
        for i in range(MAX_PERIOD, MAX_LOCUS_PERIOD + 1):
            self.step_size_by_period[i] = self.step_size_by_period[MAX_PERIOD]


class NoiseModel:
    """Logistic model of the stutter probability."""

    def __init__(self, filename=None):
        self.weights = list(_models()["stutter_weights"])

    def predict(self, x):
        z = self.weights[0]
        assert len(self.weights) == len(x) + 1
        for b, xx in zip(self.weights[1:], x):
            z += b * xx
        return 1.0 / (1 + math.exp(-1 * z))


def mean_std(a):
    """"mean+/-stdbp" of the pair distances (tredparse/models.py mean_std: a.mean(), a.std()) — the same reductions
    numpy's mean / std perform (float64 pairwise sums, population variance), called without their wrappers."""
    n = len(a)
    if not n:
        return ""
    a = np.asarray(a)
    if a.dtype.kind not in "iuf" or a.ndim != 1:
        return "{:.0f}+/-{:.0f}bp".format(a.mean(), a.std())
    m = np.add.reduce(a, dtype=np.float64) / n
    x = a - m
    np.multiply(x, x, out=x)
    return "{:.0f}+/-{:.0f}bp".format(m, math.sqrt(np.add.reduce(x) / n))


_HIST_FORMATS = {}


def histogram(a, bins=40):
    """``np.histogram(a, bins=bins, range=(0, SPAN))`` as "edge:count" pairs (tredparse/models.py histogram).  Integer
    inputs (pair distances) take an exact integer path — same counts, without numpy's generic machinery."""
    if not len(a):
        return ""
    a = np.asarray(a)
    if a.dtype.kind in "iu" and SPAN % bins == 0:
        w = SPAN // bins
        if a.min() < 0 or a.max() > SPAN:
            a = a[(a >= 0) & (a <= SPAN)]
        ar = np.bincount(np.minimum(a // w, bins - 1), minlength=bins)
        fmt = _HIST_FORMATS.get(bins)
        if fmt is None:
            fmt = _HIST_FORMATS[bins] = ",".join("{}:%d".format(w * k) for k in range(bins))
        return fmt % tuple(ar.tolist())
    ar, br = np.histogram(a, bins=bins, range=(0, SPAN))
    return ",".join("{}:{}".format(int(b), n) for (n, b) in zip(ar, br))


def pe_kde(global_lens_list, ctx=None):
    """Normalised KDE pdfs on 0..999 for a list of length arrays -> float64 [n, 1000] (GPU)."""
    ctx = ctx or _lib.default_context()
    n = len(global_lens_list)
    off = np.zeros(n + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(x) for x in global_lens_list])
    lens = np.ascontiguousarray(np.concatenate([np.asarray(x, dtype=np.int32) for x in global_lens_list])
                                if n else np.zeros(0, np.int32), dtype=np.int32)
    out = np.zeros((n, SPAN), dtype=np.float64)
    _lib.check(ctx.lib.tredsw_pe_kde(ctx.handle, _lib.ptr(lens), _lib.ptr(off), n, _lib.ptr(out), 0),
               "tredsw_pe_kde")
    return out


def candidate_ranges(obs_spanning, obs_partial, n_obs_rept, period, t2, t3, has_pemodel, maxinsert,
                     fullsearch):
    """Candidate alleles of the grid (models.py:224-257).  Returns None when there is no evidence,
    else (h1range, h2range, run_pe, max_partial_model) — lists in the reference's order, duplicates
    kept; max_partial_model is the partial-pdf clamp after models.py:241-242."""
    max_full = max(obs_spanning.keys()) if obs_spanning else 0
    max_partial = max(obs_partial.keys()) if obs_partial else 0
    reads_above_full = sum(c for k, c in obs_partial.items() if k > max_full + period)
    run_pe = bool(max_partial >= t3 and reads_above_full > 1 and has_pemodel)
    possible = set(obs_spanning.keys())
    mp_model = t2
    if obs_partial:
        if max_partial > mp_model:
            mp_model = max_partial
        possible.add(max_partial)
    if not possible:
        return None
    base = sorted(possible)
    extended = base + list(range(max_partial + period, period * maxinsert + 1, period))
    if fullsearch:
        h1range = h2range = list(range(period, period * maxinsert + 1, period))
    else:
        h1range = base if max_full else extended
        h2range = extended if (n_obs_rept or run_pe) else base
    return h1range, h2range, run_pe, mp_model


class GridBatch:
    """Accumulates likelihood problems and evaluates them with one ``tredsw_likelihood_grid`` call."""

    def __init__(self, ctx=None, score=1.0, gc=.68):
        self.ctx = ctx
        self.score, self.gc = score, gc
        self.step = StepModel()
        self.noise = NoiseModel()
        self.problems = []
        self.ipool = []
        self.dpool = []
        self.n_ipool = 0
        self.n_dpool = 0
        self.n_surface = 0
        self.n_marg = 0
        self._step_off = {}
        self.meta = []

    def _push_i(self, arr):
        arr = np.asarray(arr, dtype=np.int32).ravel()
        off = self.n_ipool
        self.ipool.append(arr)
        self.n_ipool += len(arr)
        return off

    def _push_d(self, arr):
        arr = np.asarray(arr, dtype=np.float64).ravel()
        off = self.n_dpool
        self.dpool.append(arr)
        self.n_dpool += len(arr)
        return off

    def add(self, tred, period, readlen, obs_spanning, obs_partial, n_rept, ploidy, depth, pe_pdf,
            target_lens, pe_ref, minpe, maxinsert=300, fullsearch=False):
        """Queue one problem; returns its index, or -1 when there is no evidence at all
        (models.py:244-245).  pe_pdf: the normalised KDE (1000 doubles) or None (no PE model)."""
        t2, t3 = readlen - 2 * FLANKMATCH, readlen - 3 * FLANKMATCH
        rng = candidate_ranges(obs_spanning, obs_partial, n_rept, period, t2, t3, pe_pdf is not None,
                               maxinsert, fullsearch)
        if rng is None:
            return -1
        h1range, h2range, run_pe, mp_model = rng
        w = self.noise.weights
        P = np.zeros(1, dtype=_lib.GRID_PROBLEM_DTYPE)[0]
        P["period"], P["readlen"], P["ploidy"], P["n_rept"] = period, readlen, ploidy, n_rept
        P["max_partial"], P["run_pe"] = mp_model, int(run_pe)
        P["pe_ref"], P["pe_minpe"] = pe_ref, minpe
        sk = list(obs_spanning.items())
        pk = list(obs_partial.items())
        P["n_span"], P["n_part"] = len(sk), len(pk)
        P["off_span"] = self._push_i([k for k, _ in sk] + [c for _, c in sk])
        P["off_part"] = self._push_i([k for k, _ in pk] + [c for _, c in pk])
        tl = [int(x) for x in target_lens] if run_pe else []
        for x in tl:
            if not (-SPAN <= x < SPAN):
                raise IndexError("paired-end length {} out of range".format(x))
        tl = [x + SPAN if x < 0 else x for x in tl]          # numpy negative-index wrap (models.py:473)
        P["n_target"] = len(tl)
        P["off_target"] = self._push_i(tl)
        n_h2 = 1 if ploidy == 1 else len(h2range)
        P["n_h1"], P["n_h2"] = len(h1range), n_h2
        P["off_h1"] = self._push_i(h1range)
        P["off_h2"] = self._push_i(h2range if ploidy != 1 else [0])
        P["expansion"], P["recessive"] = int(tred.is_expansion), int(tred.is_recessive)
        P["cutoff_risk"] = int(tred.cutoff_risk)
        P["half_depth"] = depth / 2
        P["stutter_a"] = w[0] + w[1] * period
        P["stutter_w2"] = w[2]
        P["stutter_c3"] = w[3] * self.gc
        P["stutter_c4"] = w[4] * self.score
        P["off_pdf"] = self._push_d(pe_pdf) if (run_pe and pe_pdf is not None) else -1
        if period not in self._step_off:
            self._step_off[period] = self._push_d(self.step.step_size_by_period[period])
        P["off_step"] = self._step_off[period]
        P["off_surface"] = self.n_surface
        self.n_surface += len(h1range) * n_h2
        P["off_ph1"] = self.n_marg
        P["off_ph2"] = self.n_marg + len(h1range)
        self.n_marg += len(h1range) + n_h2
        self.problems.append(P)
        self.meta.append((tred, period, ploidy, h1range, h2range, run_pe))
        return len(self.problems) - 1

    def run(self, want_surface=True):
        ctx = self.ctx or _lib.default_context()
        n = len(self.problems)
        self.results = np.zeros(n, dtype=_lib.GRID_RESULT_DTYPE)
        self.surface = np.zeros(self.n_surface if want_surface else 0, dtype=np.float64)
        self.marg = np.zeros(self.n_marg, dtype=np.float64)
        if n == 0:
            return self
        probs = np.array(self.problems, dtype=_lib.GRID_PROBLEM_DTYPE)
        ipool = np.ascontiguousarray(np.concatenate(self.ipool) if self.ipool else np.zeros(1, np.int32), dtype=np.int32)
        dpool = np.ascontiguousarray(np.concatenate(self.dpool) if self.dpool else np.zeros(1, np.float64))
        rc = ctx.lib.tredsw_likelihood_grid(
            ctx.handle, _lib.ptr(probs), n, _lib.ptr(ipool), len(ipool), _lib.ptr(dpool), len(dpool),
            _lib.ptr(self.surface) if want_surface else None, self.n_surface, _lib.ptr(self.marg),
            self.n_marg, _lib.ptr(self.results), 0)
        _lib.check(rc, "tredsw_likelihood_grid")
        self.probs = probs
        return self

    # ---- per-problem post-processing (host) --------------------------------------------------------
    def surface_of(self, i):
        P = self.probs[i]
        return self.surface[P["off_surface"]:P["off_surface"] + P["n_h1"] * P["n_h2"]].reshape(P["n_h1"], P["n_h2"])

    def summarize(self, i, want_joint=True):
        """-> dict(alleles (bp), lik, PP, CIs (units), P_h1, P_h2, P_h1h2) like evaluate() + sparsify()."""
        tred, period, ploidy, h1range, h2range, run_pe = self.meta[i]
        P, R = self.probs[i], self.results[i]
        h1 = h1range[R["arg_i1"]]
        h2 = h1 if ploidy == 1 else h2range[R["arg_i2"]]
        ph1 = self.marg[P["off_ph1"]:P["off_ph1"] + P["n_h1"]]
        ph2 = self.marg[P["off_ph2"]:P["off_ph2"] + P["n_h2"]]
        # a candidate that no evaluated point uses (an h1 above every h2, an h2 below every h1) never
        # becomes a key of the reference's defaultdicts (models.py:277-285)
        P_h1 = defaultdict(float)
        P_h2 = defaultdict(float)
        if ploidy == 1:
            for h, v in zip(h1range, ph1):      # h2 == h1 for every evaluated point
                P_h1[h] += float(v)
                P_h2[h] += float(v)
        else:
            lo1, hi2 = min(h1range), max(h2range)
            for h, v in zip(h1range, ph1):
                if h <= hi2:
                    P_h1[h] += float(v)
            for h, v in zip(h2range, ph2):
                if h >= lo1:
                    P_h2[h] += float(v)
        h1_lo, h1_hi = calc_CI(P_h1)
        h2_lo, h2_hi = calc_CI(P_h2)
        CIs = (h1_lo // period, h1_hi // period, h2_lo // period, h2_hi // period)
        out = {"alleles": (h1, h2), "lik": float(R["max_ml"]),
               "PP": min(1, float(R["sum_path"]) / float(R["sum_all"])), "CIs": CIs,
               "P_h1": sparsify(P_h1, period), "P_h2": sparsify(P_h2, period), "P_h1h2": {},
               "run_pe": run_pe, "n_points": int(R["n_points"])}
        if want_joint and len(self.surface):
            S = self.surface_of(i)
            W = np.exp(S - R["max_ml"])
            joint = {}
            for i1, i2 in zip(*np.nonzero(np.isfinite(S))):
                a = h1range[i1]
                b = a if ploidy == 1 else h2range[i2]
                joint[(a, b)] = float(W[i1, i2])
            out["P_h1h2"] = sparsify(joint, period)
        return out


def sparsify(P, period, epsilon=SMALL_VALUE):
    """Drop entries below epsilon, normalise by the *full* total (models.py:304-317)."""
    Z = {}
    total = sum(v for v in P.values())
    for k, v in P.items():
        if v < epsilon:
            continue
        key = ",".join(str(x // period) for x in listify(k))
        Z[key] = v / total
    return Z


def calc_CI(P):
    """95% interval over sorted keys of a marginal (models.py:319-340, quirk Q11)."""
    cum_sum, lo, hi, in_range = 0, 0, 0, False
    total_prob = sum(P.values())
    k = 0
    for k, v in sorted(P.items()):
        cum_sum += v
        if (not in_range) and cum_sum > .025 * total_prob:
            in_range, lo = True, k
        if cum_sum > .975 * total_prob:
            break
    hi = k
    return lo, hi


def calc_label(tred, alleles):
    """Disease status from the called alleles (models.py:370-392)."""
    a, b = sorted(alleles)
    label = "ok" if a != -1 else "missing"
    pre, risk = tred.cutoff_prerisk, tred.cutoff_risk
    if tred.is_expansion:
        crit = a if tred.is_recessive else b
        if pre <= crit < risk:
            label = "prerisk"
        elif crit >= risk:
            label = "risk"
    else:
        crit = b if tred.is_recessive else a
        if pre <= crit < risk:
            label = "prerisk"
        elif 0 < crit <= risk:
            label = "risk"
    return label


class IntegratedCaller:
    """Maximum-likelihood diploid caller over spanning, partial, repeat-only reads and spanning pairs."""

    def __init__(self, bamParser, score=1.0, gc=.68, maxinsert=300, fullsearch=False, pe=None):
        from .bam_parser import PEextractor
        self.tred = bamParser.tred
        self.stepmodel = StepModel()
        self.noisemodel = NoiseModel()
        self.readlen = bamParser.READLEN
        self.period = bamParser.repeatSize
        self.t1 = self.readlen - FLANKMATCH
        self.t2 = self.readlen - 2 * FLANKMATCH
        self.t3 = self.readlen - 3 * FLANKMATCH
        self.max_partial = self.t2
        self.score, self.gc = score, gc
        self.counts = bamParser.counts
        self.rept = bamParser.rept
        self.ploidy = bamParser.ploidy
        self.half_depth = bamParser.depth / 2
        self.depth = bamParser.depth
        self.maxinsert = maxinsert
        self.fullsearch = fullsearch
        self.logger = logging.getLogger("IntegratedCaller")
        self.logger.setLevel(bamParser.inputParams.getLogLevel())
        self.pe = pe if pe is not None else PEextractor(bamParser)
        pe = self.pe
        self.has_pemodel = len(pe.global_lens) >= 100 and len(pe.target_lens) >= MIN_SPANNING_PAIRS
        self.pe_pdf = pe_kde([pe.global_lens])[0] if self.has_pemodel else None
        self.PEDP = len(pe.target_lens)
        self.PEG = mean_std(pe.global_lens)
        self.PET = mean_std(pe.target_lens)
        self.P_PEG = histogram(pe.global_lens)
        self.P_PET = histogram(pe.target_lens)
        self.logger.debug("Global pairs: {} ({}), Target pairs: {} ({}), Ref: {}bp".format(
            len(pe.global_lens), self.PEG, len(pe.target_lens), self.PET, pe.ref))
        self.P_h1 = self.P_h2 = self.P_h1h2 = ""
        self.surface = None

    def evaluate(self, obs_spanning, obs_partial, n_obs_rept):
        batch = GridBatch(score=self.score, gc=self.gc)
        pe = self.pe
        idx = batch.add(self.tred, self.period, self.readlen, obs_spanning, obs_partial, n_obs_rept,
                        self.ploidy, self.depth, self.pe_pdf, pe.target_lens, pe.ref, pe.MINPE,
                        maxinsert=self.maxinsert, fullsearch=self.fullsearch)
        if idx < 0:
            return None, None, None, None
        batch.run()
        s = batch.summarize(idx)
        self.max_partial = int(batch.probs[idx]["max_partial"])
        self.surface = batch.surface_of(idx)
        self.h1range, self.h2range, self.run_pe = batch.meta[idx][3], batch.meta[idx][4], batch.meta[idx][5]
        self.P_h1, self.P_h2, self.P_h1h2 = s["P_h1"], s["P_h2"], s["P_h1h2"]
        self.logger.debug("CI(h1) = {} - {}".format(*s["CIs"][:2]))
        self.logger.debug("CI(h2) = {} - {}".format(*s["CIs"][2:]))
        return s["alleles"], s["lik"], s["PP"], s["CIs"]

    def calc_label(self, alleles):
        return calc_label(self.tred, alleles)

    def call(self, **kwargs):
        counts = self.counts
        obs_spanning = dict((k * self.period, v) for k, v in counts["FULL"].items())
        obs_partial = dict((k * self.period, v) for k, v in counts["PREF"].items())
        alleles, lik, PP, CIs = self.evaluate(obs_spanning, obs_partial, self.rept)
        if not alleles:
            alleles = (-1, -1)
            lik = PP = -1
        self.alleles = sorted(x // self.period for x in alleles)
        self.lik = lik
        self.label = label = self.calc_label(self.alleles)
        self.CI = "{}-{}|{}-{}".format(*CIs) if CIs else ""
        self.PP = PP
        self.logger.debug("ML estimate: alleles={} loglikelihood={} PP={} label={}".format(
            self.alleles, lik, PP, label))
